"""The default step path in its steady state: the persistent pf step kernel and the post kernel's dynamic work loop with
every CTA iterating over many tiles / work items, de-phased episodes, and the reference's golden trajectories replayed
through it with auto-reset.

At test sizes the occupancy-sized grids give every CTA one tile, so the buffer rotation of the pf kernel (three output
buffers, four env-scratch buffers, two input stages, their mbarrier phase bits, the env scratch staged three to five tiles
ahead) never wraps.  FLEETSTEP_PF_GRID / FLEETSTEP_POST_GRID cap the grids; every capped case reads the geometry back from
the handle (a cap that is ignored fails the test) and asserts >= 24 tiles per CTA: two full cycles of the 3 x 4 rotation.
"""
import numpy as np
import pytest
import torch

from golden_util import Golden, golden_names
from oracle.oracle import OracleFleet
from parity_util import Outputs, knobs, make_case, run_vs_oracle  # noqa: F401  (knobs: fixture)

pytestmark = pytest.mark.gpu

MIN_TILES_PER_CTA = 24


def _handle(consts, tables, E, env_id_offset=0):
    from fleetrl_b200._lib import FleetStepHandle
    return FleetStepHandle(consts, tables, E, device=0, env_id_offset=env_id_offset)


def _envs_per_tile(consts, tables):
    """Tile size of the step kernel under the current variables (read from a one-env handle)."""
    h = _handle(consts, tables, 1)
    B = h.launch_geometry["envs_per_tile"]
    h.close()
    return B


def _assert_capped(gpu, pf_grid, post_grid=None):
    g = gpu.launch_geometry
    assert gpu.step_kernel_name.startswith("fleet_step_pf_kernel"), gpu.step_kernel_name
    assert g["step_grid"] == pf_grid, g
    assert g["step_tiles"] // g["step_grid"] >= MIN_TILES_PER_CTA, g       # every CTA runs >= 24 tiles
    assert g["step_tiles"] * g["envs_per_tile"] >= gpu.E > (g["step_tiles"] - 1) * g["envs_per_tile"], g
    if post_grid is not None:
        assert g["post_grid"] == post_grid, g
    return g


# --------------------------------------------------------------------------------- b. capped-grid parity vs the oracle
# E = 24 * G * B + tail (a short tail tile wherever B > 1); 24 h episodes de-phased over L = 96 steps; 2 L + 10 steps.
# phase: B * D is not a multiple of 4, so the 16-byte phase of the shared obs tile changes from tile to tile.
PIPE = {
    "n8_widest_tile_g2": dict(n_evs=8, G=2),
    "n13_aux_norm_g3": dict(n_evs=13, G=3, over=dict(normalize=1), phase=True),
    "n11_noaux_linear_g5": dict(n_evs=11, G=5, over=dict(aux=0, deg_mode=1), phase=True),
    "n20_ct_two_trips_ring4_stack2_g1_post1": dict(
        n_evs=20, use_case="ct", two_trips=True, G=1, post=1,
        env=dict(FLEETSTEP_RF_RING=4, FLEETSTEP_RF_STACK=2, FLEETSTEP_RF_EXT_SLOTS=40000)),
    "n50_cfg2_shape_g5": dict(n_evs=50, days=8, G=5),
    "n50_cfg2_shape_g1": dict(n_evs=50, days=8, G=1),
    "n50_cfg2_shape_g1_charge_log": dict(n_evs=50, days=8, G=1, charge_log=True),
    "n12_norm_noaux_g2_charge_log": dict(n_evs=12, G=2, over=dict(normalize=1, aux=0), charge_log=True),
    "n9_norm_nocarry_g3_post1": dict(n_evs=9, G=3, post=1, over=dict(normalize=1, carry_degradation_state=0)),
    "n129_g2_post1": dict(n_evs=129, days=6, G=2, post=1),
    "n129_g2_post2": dict(n_evs=129, days=6, G=2, post=2),
}


def _pipe_case(name, knobs):
    cf = dict(PIPE[name])
    G, post, env = cf.pop("G"), cf.pop("post", None), cf.pop("env", {})
    cf.pop("charge_log", None), cf.pop("phase", None)
    knobs(**env)
    consts, tables = make_case(name, **cf)
    B = _envs_per_tile(consts, tables)
    E = MIN_TILES_PER_CTA * G * B + (B // 3 + 1 if B > 1 else 1)
    knobs(FLEETSTEP_PF_GRID=G, FLEETSTEP_POST_GRID=post)
    return consts, tables, E, G, post


@pytest.mark.parametrize("name", sorted(PIPE))
def test_capped_grid_vs_oracle(name, knobs):
    """Every CTA of the pf kernel runs >= 24 tiles (and the post kernel, capped, fetches many work items) while episodes
    end on different steps: the steady state bench.py and a rollout run, checked step by step against the oracle."""
    cf = PIPE[name]
    consts, tables, E, G, post = _pipe_case(name, knobs)
    gpu = _handle(consts, tables, E, env_id_offset=1000)
    g = _assert_capped(gpu, G, post)
    B = g["envs_per_tile"]
    assert E % B or B == 1                                    # a short tail tile (impossible with one env per tile)
    if cf.get("phase"):
        assert (B * gpu.D) % 4 != 0, (B, gpu.D)
    L = consts.episode_steps
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    r = run_vs_oracle(gpu, orc, 2 * L + 10, charge_log=cf.get("charge_log", False), dephase=L)
    if B > 1:
        assert r["mixed_tiles"] > 0, r                        # finishing and running envs in one tile
    gpu.close()


# ----------------------------------------------------------------- c. grid invariance at production geometry (GPU only)
GRIDS = [(None, None), (1, 1), (7, 3), (64, None), (None, 3)]     # (FLEETSTEP_PF_GRID, FLEETSTEP_POST_GRID)


def test_grid_invariance_cfg2(knobs):
    """cfg2-shaped fleet (N = 50, 16,384 envs: ~11 tiles per CTA at the default grid), de-phased: the per-env results
    depend on no scheduling decision, so outputs and state are bit-identical whatever the grids; only the statistics
    (striped atomics, added in a different order) may differ in the last bits."""
    from fleetrl_b200._abi import FIELDS
    from fleetrl_b200.config import default_config
    from fleetrl_b200.schedule import generate_schedule, synthetic_series
    from fleetrl_b200.tables import FleetInputs, build_fleet

    E, N = 16384, 50
    sched = generate_schedule("lmd", N, seed=42)
    price, tariff, load, pv = synthetic_series(seed=7)
    built = build_fleet(default_config("lmd", seed=0), FleetInputs(sched, price, tariff, load, pv), auto_reset=True,
                        carry_degradation_state=True, seed=0, time_picker="random")
    c, tb = built.consts, built.tables
    hs = []
    for pf, post in GRIDS:
        knobs(FLEETSTEP_PF_GRID=pf, FLEETSTEP_POST_GRID=post)
        h = _handle(c, tb, E)
        g = h.launch_geometry
        assert h.step_kernel_name == "fleet_step_pf_kernel<kV=1>"
        if pf is None:
            assert g["step_tiles"] / g["step_grid"] > 10, g
        else:
            assert g["step_grid"] == pf, g
        if post is not None:
            assert g["post_grid"] == post, g
        hs.append(h)
    assert len({(h.launch_geometry["step_grid"], h.launch_geometry["post_grid"]) for h in hs}) == len(GRIDS)
    dev, D = hs[0].device, hs[0].D
    bufs = [dict(obs=torch.zeros((E, D), dtype=torch.float32, device=dev),
                 term=torch.zeros((E, D), dtype=torch.float32, device=dev),
                 rew=torch.zeros(E, dtype=torch.float32, device=dev),
                 done=torch.zeros(E, dtype=torch.uint8, device=dev)) for _ in hs]
    for h, b in zip(hs, bufs):
        h.reset(obs=b["obs"])
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    L = c.episode_steps
    phase = torch.arange(E, device=dev) % L
    fields = [k for k in FIELDS if k != "charge_log"]
    n_done = 0
    for s in range(L + 30):
        a = torch.empty((E, N), dtype=torch.float32, device=dev).uniform_(-1, 1, generator=gen)
        if s % 5 == 0:
            a[:, ::4] = 0.0
        for h, b in zip(hs, bufs):
            h.step(a, b["obs"], b["rew"], b["done"], b["term"])
        d0 = bufs[0]["done"].bool()
        n_done += int(d0.sum())
        ref = {k: hs[0].get(k) for k in fields}
        for i, (h, b) in enumerate(zip(hs[1:], bufs[1:]), 1):
            for k in ("obs", "rew", "done"):
                assert torch.equal(b[k], bufs[0][k]), f"{k} step {s} grids {GRIDS[i]}"
            assert torch.equal(b["term"][d0], bufs[0]["term"][d0]), f"terminal obs step {s} grids {GRIDS[i]}"
            for k in fields:
                assert torch.equal(h.get(k), ref[k]), f"{k} step {s} grids {GRIDS[i]}"
        if s < L:
            m = (phase == s).to(torch.uint8)
            for h, b in zip(hs, bufs):
                h.reset(mask=m, obs=b["obs"])
    assert n_done > E // 4
    st0 = hs[0].stats()
    for i, h in enumerate(hs[1:], 1):
        st = h.stats()
        for k in st0:
            np.testing.assert_allclose(st[k], st0[k], rtol=1e-12, atol=0, err_msg=f"stat {k} grids {GRIDS[i]}")
    for h in hs:
        assert h.check_errors() == 0
        h.close()


# ------------------------------------------------------------------- d. reference goldens through the default kernel
GOLDEN_MIN_EVS = 8
GOLDEN_KEYS = ["soc", "soc_deg", "hours_left", "target_soc", "rf_len", "soh", "fd_cyc", "life"]


def _golden_pf_names():
    return [n for n in golden_names() if Golden(n).consts_dict["num_evs"] >= GOLDEN_MIN_EVS]


def _check_state(r, key, got, row, what):
    """got: [E, N] device values of every replica, r: the golden trajectory; tolerances of test_gpu_golden.py."""
    g = got.cpu().numpy()
    assert (g == g[:1]).all(), f"{key} {what}: replicas differ"
    want = r[key][row]
    if key == "hours_left":
        want = want.astype(np.float32)
    if key == "rf_len":
        want = want.astype(np.int32)
    if key in ("soh", "life"):
        np.testing.assert_allclose(g[0], want, rtol=0, atol=1e-13, err_msg=f"{key} {what}")
    elif key == "fd_cyc":
        np.testing.assert_allclose(g[0], want, rtol=1e-12, atol=1e-18, err_msg=f"{key} {what}")
    else:
        np.testing.assert_array_equal(g[0], want, err_msg=f"{key} {what}")


@pytest.mark.parametrize("replicas", ["one_env", "replicas_grid1"])
@pytest.mark.parametrize("name", _golden_pf_names())
def test_golden_through_pf_autoreset(name, replicas, knobs):
    """The reference's trajectory, episodes chained by the post kernel's auto-reset (set_next_start) instead of explicit
    resets: on a done step terminal_obs is the reference's last row of the episode, obs and state its reset row of the
    next one.  replicas_grid1: 8 B + 1 identical envs on ONE CTA (>= 9 tiles, the last one short), all bit-identical."""
    g = Golden(name)
    r = g.traj
    consts = g.consts(auto_reset=1, start_lo=int(g.start_idx.min()), start_hi=int(g.start_idx.max()))
    if replicas == "one_env":
        E = 1
    else:
        E = 8 * _envs_per_tile(consts, g.tables) + 1
        knobs(FLEETSTEP_PF_GRID=1)
    h = _handle(consts, g.tables, E)
    assert h.step_kernel_name.startswith("fleet_step_pf_kernel"), h.step_kernel_name
    geo = h.launch_geometry
    if replicas != "one_env":
        assert geo["step_grid"] == 1 and geo["step_tiles"] >= 9 and E % geo["envs_per_tile"] == 1, geo
    dev, D = h.device, h.D
    obs = torch.zeros((E, D), dtype=torch.float32, device=dev)
    term = torch.zeros((E, D), dtype=torch.float32, device=dev)
    rew = torch.zeros(E, dtype=torch.float32, device=dev)
    done = torch.zeros(E, dtype=torch.uint8, device=dev)
    nxt = torch.full((E,), int(g.start_idx[0]), dtype=torch.int32, device=dev)
    h.set_next_start(nxt)
    keys = [k for k in GOLDEN_KEYS if k in r]
    L, n_ep = g.n_steps_per_ep, len(g.start_idx)
    assert consts.episode_steps == L

    h.reset(start_idx=torch.full((E,), int(g.start_idx[0]), dtype=torch.int32, device=dev), obs=obs)
    o = obs.cpu().numpy()
    assert (o == o[:1]).all()
    np.testing.assert_array_equal(o[0], r["obs"][0])
    step = 0
    for j in range(n_ep):
        for k in range(L):
            last = k == L - 1
            if last and j + 1 < n_ep:
                nxt.fill_(int(g.start_idx[j + 1]))            # the start the auto-reset after this step draws
            h.step(torch.from_numpy(np.repeat(g.actions[step][None, :], E, 0)).to(dev), obs, rew, done, term)
            what = f"episode {j} step {k}"
            row = j * (L + 1) + k + 1                         # the reference's row after this step
            d = done.cpu().numpy()
            assert (d == int(r["done"][step])).all(), what
            for key, tol in (("reward64", (1e-11, 1e-10)), ("cashflow", (1e-12, 1e-13))):
                v = h.get(key).cpu().numpy()
                assert (v == v[0]).all(), f"{key} {what}: replicas differ"
                np.testing.assert_allclose(v[0], r["reward" if key == "reward64" else key][step], rtol=tol[0], atol=tol[1],
                                           err_msg=f"{key} {what}")
            if last:
                t = term.cpu().numpy()
                assert (t == t[:1]).all(), f"terminal obs {what}: replicas differ"
                np.testing.assert_array_equal(t[0], r["obs"][row], err_msg=f"terminal obs {what}")
                row = (j + 1) * (L + 1)                       # auto-reset has run: the next episode's reset row
            if not last or j + 1 < n_ep:
                o = obs.cpu().numpy()
                assert (o == o[:1]).all(), f"obs {what}: replicas differ"
                np.testing.assert_array_equal(o[0], r["obs"][row], err_msg=f"obs {what}")
                for key in keys:
                    _check_state(r, key, h.get(key), row, what)
            step += 1
    assert int(h.get("ep_count")[0]) == n_ep + 1 and h.stats()["episodes"] == n_ep * E
    assert h.check_errors() == 0
    h.close()


# --------------------------------------------------------------------------------------------- e. output destinations
@pytest.mark.parametrize("mode", ["offset", "no_term", "obs_gap"])
@pytest.mark.parametrize("kernel", ["pf", "generic"])
def test_output_destinations(kernel, mode, knobs):
    """Observation rows that are not 16-byte aligned (element-wise stores), no terminal_obs while envs finish, and no obs
    for a stretch of steps, in a capped, de-phased case whose obs tile changes its 16-byte phase from tile to tile.
    Outputs that exist are compared with the oracle, and the state always is: it must not depend on which outputs were
    passed."""
    name = "n13_aux_norm_g3"
    consts, tables, E, G, _ = _pipe_case(name, knobs)
    knobs(FLEETSTEP_KERNEL=kernel)
    gpu = _handle(consts, tables, E, env_id_offset=1000)
    if kernel == "pf":
        _assert_capped(gpu, G)
    else:
        assert gpu.step_kernel_name == "fleet_step_kernel"
    L = consts.episode_steps
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    r = run_vs_oracle(gpu, orc, 2 * L + 10, charge_log=False, dephase=L, outputs=Outputs(E, gpu.D, gpu.device, mode))
    assert r["mixed_tiles"] > 0, r
    gpu.close()
