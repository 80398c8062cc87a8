"""Env state that fleet_reset never produces, checked against the oracle: target-SOC flips (fleet_environment.py:613-614)
of some vehicles and not others, fleet_set_state, checkpoint resume on the default kernel, and the log ring after it
wraps.

A vehicle whose SOH falls to <= 0.9 gets target 0.9 from the next step on; the device keeps that as a flag per vehicle
(tflip) plus a counter (n_flips) that switches the flag reads on.  Reset runs start with no flip at all, so every case
here writes SOH (or the target) on both sides, starts just above 0.9 so that daily evaluations cross it later, and
asserts that its scenario (mixed tiles, late flips, extension slots in use, ...) actually happened.
"""
import numpy as np
import pytest
import torch

from fleetrl_b200._abi import FIELDS
from oracle import policies as opol
from oracle.oracle import OracleFleet
from parity_util import Outputs, knobs, make_case, run_vs_oracle  # noqa: F401  (knobs: fixture)

pytestmark = pytest.mark.gpu

MIN_TILES_PER_CTA = 24
FLIP = 0.9


def _handle(consts, tables, E, env_id_offset=1000):
    from fleetrl_b200._lib import FleetStepHandle
    return FleetStepHandle(consts, tables, E, device=0, env_id_offset=env_id_offset)


def _capped_envs(consts, tables, G):
    """Env count that gives every CTA of a FLEETSTEP_PF_GRID=G pf kernel >= 24 tiles, plus a short tail tile."""
    h = _handle(consts, tables, 1)
    B = h.launch_geometry["envs_per_tile"]
    h.close()
    return MIN_TILES_PER_CTA * G * B + (B // 3 + 1 if B > 1 else 1)


def _assert_pf_capped(gpu, G):
    g = gpu.launch_geometry
    assert gpu.step_kernel_name == "fleet_step_pf_kernel<kV=1>", gpu.step_kernel_name
    assert g["step_grid"] == G and g["step_tiles"] // G >= MIN_TILES_PER_CTA, g
    return g


def _fields(h):
    return [k for k in FIELDS if k != "charge_log"]


# ------------------------------------------------------------------------------------------------ state blob layout
# fleet_export_state: StateHeader {uint64 magic; int32 E, N, R, S, X, P, L, T}, then the arrays of state_arrays() in
# order; the rainflow arrays only when the incremental rainflow is on.
HEADER = np.dtype([("magic", "<u8"), ("E", "<i4"), ("N", "<i4"), ("R", "<i4"), ("S", "<i4"), ("X", "<i4"), ("P", "<i4"),
                   ("L", "<i4"), ("T", "<i4")])
EF_COUNT, STAT_STRIPES, N_STATS = 6, 64, 10


def parse_blob(blob):
    hd = np.frombuffer(blob[:HEADER.itemsize].tobytes(), HEADER)[0]
    E, N, R, S, X, P = (int(hd[k]) for k in ("E", "N", "R", "S", "X", "P"))
    EN = E * N
    plain = [("env4", "<i4", (E, 4)), ("soc", "<f8", (E, N)), ("hl", "<f4", (E, N)), ("soh", "<f8", (E, N)),
             ("hist", "<f8", (E, R, N)), ("tflip", "u1", (E, N)), ("n_flips", "<i4", ()), ("env_f64", "<f8", (EF_COUNT, E)),
             ("rf_len", "<i4", (E, N)), ("fd_cyc", "<f8", (E, N)), ("life", "<f8", (E, N)), ("n_cycles", "<i4", (E, N)),
             ("last_deg", "<f8", (E, N))]
    rf = [("rf_stack", "<f8", (EN * S,)), ("rf_dc", "<u4", (E, N)), ("rf_acc", "<f8", (E, N, 2)), ("rf_ext", "<i4", (E, N)),
          ("ext_owner", "<i4", (max(P, 1),)), ("ext_val", "<f8", (max(P, 1) * max(X, 1),))]
    tail = [("stats", "<f8", (STAT_STRIPES * N_STATS,))]
    nbytes = lambda lay: sum(np.dtype(d).itemsize * int(np.prod(s)) for _, d, s in lay)
    layout = plain + tail
    if HEADER.itemsize + nbytes(layout) != len(blob):
        layout = plain + rf + tail
    assert HEADER.itemsize + nbytes(layout) == len(blob), "blob size matches no state_arrays() layout"
    out, off = {"header": hd}, HEADER.itemsize
    for name, d, s in layout:
        n = np.dtype(d).itemsize * int(np.prod(s))
        out[name] = np.frombuffer(blob[off:off + n].tobytes(), d).reshape(s)
        off += n
    return out


# ------------------------------------------------------------------------------------ a. partial flips vs the oracle
# delta: init_soh = 0.9 + delta, calibrated on the oracle so that roughly half of the vehicles cross 0.9 at a daily
# evaluation within the first two simulated days (SEI: 6.5e-5 per day at most, linear: 3.4e-6).
FLIP_CASES = {
    "pf_v1_g2": dict(n_evs=8, G=2, delta=3e-5, policies=True),
    "pf_linear_g1": dict(n_evs=10, G=1, delta=2e-6, over=dict(deg_mode=1)),
    "generic_n7": dict(n_evs=7, E=150, delta=3e-5, policies=True),
    "pf_norm_aux_g1": dict(n_evs=13, G=1, delta=3e-5, over=dict(normalize=1)),
    "pf_ct_two_trips_g1": dict(n_evs=12, G=1, delta=3e-5, use_case="ct", two_trips=True, policies=True),
    "pf_nocarry_g1": dict(n_evs=9, G=1, delta=3e-5, over=dict(carry_degradation_state=0)),
}
NIGHT = (18, 0, 8)          # (charging_hour, charging_minute, max_hours) of the night policy


def _soh_writes(E, N, lo=FLIP - 2e-9, hi=FLIP + 2e-9):
    """SOH of envs e % 3 == 0: vehicle n % 3 == 0 just below 0.9, == 1 exactly 0.9 (both flip on the next step),
    == 2 just above (flips later, at a daily evaluation); NaN elsewhere (keep)."""
    w = np.full((E, N), np.nan)
    rows = np.arange(E) % 3 == 0
    for n in range(N):
        w[rows, n] = (lo, FLIP, hi)[n % 3]
    return w


class FlipWatch:
    """Scenario counters of a flip run: tiles with flipped and unflipped vehicles, two vehicles of one lane pair (even N:
    vehicles 2m and 2m+1 of an env, whose contributions the pf kernel pre-adds with a shuffle) that differ, flips of vehicles whose SOH was not written, envs whose flags a reset cleared while others stay set, and
    policy actions that the flip changed (on a sample of envs; the device computes all of them)."""

    def __init__(self, gpu, orc, consts, tables, B, written, policies):
        self.gpu, self.orc, self.c, self.tb, self.B = gpu, orc, consts, tables, B
        self.written, self.policies = written, policies
        self.prev = None
        self.mixed_tiles = self.mixed_pairs = self.late_flips = self.cleared = self.policy_flip_diffs = 0
        self.flips_per_step = []
        self.pol_envs = range(0, gpu.E, max(1, gpu.E // 60))   # rows compared with the restatement
        self.night = {e: opol.NightPolicy(consts, tables, *NIGHT) for e in self.pol_envs}

    def tiles(self, f):
        E, N = f.shape
        pad = np.full((-E % self.B, N), 2, np.int8)
        t = np.concatenate([f.astype(np.int8), pad]).reshape(-1, self.B * N)
        return int((((t == 1).sum(1) > 0) & ((t == 0).sum(1) > 0)).sum())

    def __call__(self, s, a, obs, rew, done, term):
        tgt = self.orc.get("target_soc")
        f = tgt == FLIP
        if s == -1:
            assert not f.any()                                  # a reset run: no flip anywhere
        else:
            self.flips_per_step.append(int(f.sum()))
            self.mixed_tiles += self.tiles(f)
            N = f.shape[1]
            self.mixed_pairs += int((f[:, 0:N - 1:2] != f[:, 1:N:2]).sum())
            new = f & ~self.prev
            self.late_flips += int((new & ~self.written).sum()) if s >= 1 else 0
            if f.any():                                         # a flag only goes away through a reset
                self.cleared += int((self.prev.any(1) & ~f.any(1)).sum())
        if self.policies and f.any():
            self._check_policies(tgt, f)
        self.prev = f

    def _check_policies(self, tgt, f):
        """fleet_policy_actions against oracle/policies.py, fed the ORACLE's target_soc."""
        c, tb, T = self.c, self.tb, self.c.table_len
        t = np.minimum(self.orc.get("time_idx"), T - 1)
        d_dev = self.gpu.policy_actions("distributed").cpu().numpy()
        n_dev = self.gpu.policy_actions("night", None, *NIGHT).cpu().numpy()
        for e in self.pol_envs:
            want_d = opol.distributed(c, tb, int(t[e]), tgt[e]).astype(np.float32)
            np.testing.assert_array_equal(d_dev[e], want_d, err_msg=f"distributed env {e}")
            np.testing.assert_array_equal(n_dev[e], self.night[e].actions(int(t[e]), tgt[e]).astype(np.float32),
                                          err_msg=f"night env {e}")
            if f[e].any():
                unflipped = opol.distributed(c, tb, int(t[e]), np.full(c.num_evs, c.target_soc)).astype(np.float32)
                self.policy_flip_diffs += int((unflipped != want_d).sum())


@pytest.mark.parametrize("name", sorted(FLIP_CASES))
def test_partial_flips_vs_oracle(name, knobs):
    """SOH written just below, at and just above 0.9 for single vehicles after the reset, init_soh just above 0.9:
    flipped and unflipped vehicles share tiles (and lane pairs), the counter goes from 0 to non-zero during the run,
    daily evaluations flip further vehicles later, and (carry_degradation_state=0) resets clear flags while the counter
    stays.  Every output and state field, target_soc included, is compared with the oracle after every step."""
    cf = dict(FLIP_CASES[name])
    G, delta = cf.pop("G", None), cf.pop("delta")
    policies, E = cf.pop("policies", False), cf.pop("E", None)
    knobs(**cf.pop("env", {}))
    cf["over"] = dict(cf.get("over", {}), init_soh=FLIP + delta)
    consts, tables = make_case("flip_" + name, **cf)
    if G is None:
        knobs(FLEETSTEP_KERNEL="generic")
    else:
        E = _capped_envs(consts, tables, G)
        knobs(FLEETSTEP_PF_GRID=G)
    gpu = _handle(consts, tables, E)
    if G is None:
        assert gpu.step_kernel_name == "fleet_step_kernel"
    else:
        _assert_pf_capped(gpu, G)
    N, L = gpu.N, consts.episode_steps
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    w = _soh_writes(E, N)
    written = ~np.isnan(w)
    watch = FlipWatch(gpu, orc, consts, tables, gpu.launch_geometry["envs_per_tile"], written, policies)

    def hook(s, *args):
        if s == -1:
            soh = np.where(written, w, orc.get("soh"))
            orc.set("soh", soh)
            gpu.set("soh", torch.from_numpy(soh))
        watch(s, *args)

    run_vs_oracle(gpu, orc, 2 * L + 10, charge_log=False, dephase=L, hook=hook)
    r = {k: getattr(watch, k) for k in ("mixed_tiles", "mixed_pairs", "late_flips", "cleared", "policy_flip_diffs")}
    assert watch.flips_per_step[0] > 0, r                    # 0 at the reset, > 0 after the first step
    assert r["mixed_tiles"] > 0 and r["late_flips"] > 0, r
    if G is not None and N % 2 == 0:
        assert r["mixed_pairs"] > 0, r
    if not consts.carry_degradation_state:
        assert r["cleared"] > 0, r
    if policies:
        assert r["policy_flip_diffs"] > 0, r
    gpu.close()


# ------------------------------------------------------------------------------------------------ b. fleet_set_state
WRITABLE = ("soc", "hours_left", "soh", "reward64", "cashflow", "rf_len", "fd_cyc", "life", "ep_return", "last_ep_return",
            "n_cycles", "last_deg", "overload", "soc_viol", "charge_log", "target_soc")
READ_ONLY = ("soc_deg", "time_idx", "finish_idx", "ep_count")


def _random_value(name, shape, rng, consts):
    _, dt, _ = FIELDS[name]
    if name == "target_soc":
        return np.where(rng.random(shape) < 0.5, FLIP, consts.target_soc)
    if dt == np.int32:
        return rng.integers(0, 1 << 20, shape).astype(np.int32)
    return rng.uniform(-3, 3, shape).astype(dt)


@pytest.mark.parametrize("kernel", ["pf", "generic"])
def test_set_get_round_trip(kernel, knobs):
    """Every writable field reads back bit for bit after set() and no other field changes; read-only fields, charge_log
    before enable_charge_log and target values other than the configured one and 0.9 are refused without a change."""
    from fleetrl_b200._lib import FleetStepError
    assert set(WRITABLE) | set(READ_ONLY) == set(FIELDS)
    knobs(FLEETSTEP_KERNEL=kernel)
    consts, tables = make_case("set_round_trip", 10)
    E = 20
    gpu = _handle(consts, tables, E)
    assert gpu.step_kernel_name.startswith("fleet_step_pf_kernel" if kernel == "pf" else "fleet_step_kernel")
    dev = gpu.device
    gpu.reset()
    rng = np.random.default_rng(3)
    with pytest.raises(FleetStepError):
        gpu.set("charge_log", np.zeros((E, gpu.N)))
    for s in range(40):
        gpu.step(torch.from_numpy(rng.uniform(-1, 1, (E, gpu.N)).astype(np.float32)).to(dev))
    snap = lambda: {k: gpu.get(k).clone() for k in FIELDS if k != "charge_log" or enabled}
    enabled = False
    blob0 = gpu.export_state()
    for name in READ_ONLY:
        _, dt, per_ev = FIELDS[name]
        with pytest.raises(FleetStepError):
            gpu.set(name, np.zeros((E, gpu.N) if per_ev else E, dt))
    for bad in (0.8, consts.target_soc + 1e-12, np.nan):
        v = np.full((E, gpu.N), consts.target_soc)
        v[3, 2] = bad
        with pytest.raises(FleetStepError, match="target_soc"):
            gpu.set("target_soc", v)
    np.testing.assert_array_equal(gpu.export_state(), blob0)     # nothing above changed the state
    gpu.enable_charge_log(True)
    enabled = True
    for name in WRITABLE:
        _, dt, per_ev = FIELDS[name]
        shape = (E, gpu.N) if per_ev else (E,)
        before = snap()
        v = _random_value(name, shape, rng, consts)
        assert not np.array_equal(v, before[name].cpu().numpy())
        gpu.set(name, v)
        after = snap()
        np.testing.assert_array_equal(after[name].cpu().numpy(), v, err_msg=name)
        for k in before:
            if k != name:
                assert torch.equal(after[k], before[k]), f"set({name}) changed {k}"
    assert gpu.check_errors() == 0
    gpu.close()


@pytest.mark.parametrize("kernel", ["pf", "generic"])
def test_midrun_writes_vs_oracle(kernel, knobs):
    """target_soc written mid-run to a subset, to nobody, then to another subset, and SOC / SOH of single vehicles
    written between them, identically on the device and the oracle: the run stays in parity (observations bit-exact),
    and after each target write the device's flip counter (parsed from the state blob) is the number of 0.9 entries;
    after the empty write it is 0, so the flag reads are off."""
    knobs(FLEETSTEP_KERNEL=kernel)
    consts, tables = make_case("midrun_writes", 9, over=dict(deg_mode=1))
    E = 120
    gpu = _handle(consts, tables, E)
    assert gpu.step_kernel_name.startswith("fleet_step_pf_kernel" if kernel == "pf" else "fleet_step_kernel")
    N, L = gpu.N, consts.episode_steps
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    rng = np.random.default_rng(5)
    subset = lambda m: np.where(m, FLIP, consts.target_soc)
    idx = np.arange(E * N).reshape(E, N)
    targets = {-1: subset(idx % 7 == 0), 30: subset(np.zeros((E, N), bool)), 60: subset(idx % 5 == 1)}
    seen = dict(counts=[], soc_writes=0, soh_writes=0)

    def write(name, v):
        orc.set(name, v)
        gpu.set(name, torch.from_numpy(v))

    def hook(s, *args):
        if s in targets:
            write("target_soc", targets[s])
            n_flips = int(parse_blob(gpu.export_state())["n_flips"])
            assert n_flips == int((targets[s] == FLIP).sum()), (s, n_flips)
            seen["counts"].append(n_flips)
        if s in (15, 45, 90):
            hl = orc.get("hours_left")
            m = (hl > 0) & (rng.random((E, N)) < 0.3)                # present vehicles: their SOC carries on
            write("soc", np.where(m, rng.uniform(0.1, 0.8, (E, N)), orc.get("soc")))
            seen["soc_writes"] += int(m.sum())
            m = rng.random((E, N)) < 0.3
            write("soh", np.where(m, rng.uniform(0.92, 0.99, (E, N)), orc.get("soh")))
            seen["soh_writes"] += int(m.sum())

    run_vs_oracle(gpu, orc, 2 * L + 10, charge_log=False, dephase=L, hook=hook)
    assert seen["counts"][1] == 0 and seen["counts"][0] > 0 and seen["counts"][2] > 0, seen
    assert seen["soc_writes"] > 0 and seen["soh_writes"] > 0, seen
    gpu.close()


# ---------------------------------------------------------------------------------- c. checkpoint resume, pf kernel
RESUME_ENV = dict(FLEETSTEP_RF_RING=4, FLEETSTEP_RF_STACK=2, FLEETSTEP_RF_EXT_SLOTS=40000)


# Per-env sums over the vehicles: the generic kernel adds them in car order, the pf kernel in five interleaved partial
# sums (fleet_step_pf_kernel's epilogue), so between the two kernels these agree to rounding only (the oracle's tolerances).
KERNEL_SUMS = ("reward64", "cashflow", "ep_return", "last_ep_return", "overload", "soc_viol")


def _compare_handles(a, others, s, outs, other_kernel=()):
    """outs: [(obs, rew, done, term)] of a and then of each other handle after step s; handles whose index is in
    other_kernel run the other step kernel (KERNEL_SUMS and the float32 reward to tolerance, all else bit-exact)."""
    oa, ra, da, ta = outs[0]
    d = da.bool()
    fa = {k: a.get(k) for k in _fields(a)}
    for i, (h, (o, r, dn, t)) in enumerate(zip(others, outs[1:])):
        assert torch.equal(o, oa) and torch.equal(dn, da), f"outputs step {s} handle {i}"
        assert torch.equal(t[d], ta[d]), f"terminal obs step {s} handle {i}"
        if i in other_kernel:
            torch.testing.assert_close(r, ra, rtol=1e-6, atol=1e-6, msg=f"reward step {s} handle {i}")
        else:
            assert torch.equal(r, ra), f"reward step {s} handle {i}"
        for k, v in fa.items():
            if i in other_kernel and k in KERNEL_SUMS:
                torch.testing.assert_close(h.get(k), v, rtol=1e-11, atol=1e-9, msg=f"{k} step {s} handle {i}")
            else:
                assert torch.equal(h.get(k), v), f"{k} step {s} handle {i}"


def test_resume_default_kernel(knobs):
    """export_state() of a capped pf handle at a step where a vehicle holds an extension slot, an env's history ring has
    rows the post kernel has not consumed and flips exist; imported into a dirty pf handle and into a generic-kernel
    handle, all three continue bit for bit for two episodes (the exporter still checked against the oracle; the generic
    handle's per-env sums over the vehicles to rounding, see KERNEL_SUMS).  Blobs of
    another ring size or stack depth, truncated, with a corrupted magic or header are refused and change nothing."""
    from fleetrl_b200._lib import FleetStepError
    knobs(**RESUME_ENV)
    consts, tables = make_case("resume_ct", 20, use_case="ct", two_trips=True, over=dict(init_soh=FLIP + 3e-5))
    E = _capped_envs(consts, tables, 1)
    L = consts.episode_steps
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(21)

    def dirty(h, target_mask):
        h.reset()
        for s in range(L + 17):
            h.step(torch.from_numpy(rng.uniform(-1, 1, (E, h.N)).astype(np.float32)).to(dev))
            if s < L // 2:
                h.reset(mask=torch.from_numpy((np.arange(E) % (L // 2) == s).astype(np.uint8)).to(dev))
        h.set("target_soc", np.where(target_mask, FLIP, consts.target_soc))
        return h

    knobs(FLEETSTEP_PF_GRID=1)
    a = _handle(consts, tables, E)
    _assert_pf_capped(a, 1)
    b = dirty(_handle(consts, tables, E), (np.arange(E * 20).reshape(E, 20) % 3) == 0)
    _assert_pf_capped(b, 1)
    knobs(FLEETSTEP_KERNEL="generic")
    c = dirty(_handle(consts, tables, E), np.zeros((E, 20), bool))
    assert c.step_kernel_name == "fleet_step_kernel"
    foreign = {}
    for k, v in (("FLEETSTEP_RF_RING", 8), ("FLEETSTEP_RF_STACK", 4)):
        knobs(FLEETSTEP_KERNEL=None, **{k: v})
        f = _handle(consts, tables, E)
        f.reset()
        foreign[k] = f.export_state()
        f.close()
        knobs(**{k: RESUME_ENV[k]})
    knobs(FLEETSTEP_KERNEL=None)

    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    st = dict(export_step=None, ext=0, behind=0, n_flips=0, steps_after=0, n_done_after=0)
    outs = [(torch.zeros((E, a.D), dtype=torch.float32, device=dev), torch.zeros(E, dtype=torch.float32, device=dev),
             torch.zeros(E, dtype=torch.uint8, device=dev), torch.zeros((E, a.D), dtype=torch.float32, device=dev))
            for _ in range(2)]

    def rejects(blob):
        before = b.export_state()
        with pytest.raises(FleetStepError):
            b.import_state(blob)
        np.testing.assert_array_equal(b.export_state(), before)

    def hook(s, act, obs, rew, done, term):
        if s < L:
            return
        if st["export_step"] is None:
            blob = a.export_state()
            p = parse_blob(blob)
            k_now = p["env4"][:, 0] - p["env4"][:, 1]
            ext, behind, nf = int((p["rf_ext"] >= 0).sum()), int((p["env4"][:, 3] < k_now).sum()), int(p["n_flips"])
            if not (ext and behind and nf):
                return
            st.update(export_step=s, ext=ext, behind=behind, n_flips=nf)
            for k in foreign:
                rejects(foreign[k])
            rejects(blob[:-1])
            bad = blob.copy()
            bad[0] ^= 0xFF
            rejects(bad)
            bad = blob.copy()
            hd = np.frombuffer(bad[:HEADER.itemsize].tobytes(), HEADER).copy()
            hd["R"] = 8
            bad[:HEADER.itemsize] = np.frombuffer(hd.tobytes(), np.uint8)
            rejects(bad)
            for h in (b, c):
                h.import_state(blob)
            _compare_handles(a, (b, c), s, [(obs, rew, done, term)] * 3)
            return
        a_t = torch.from_numpy(act).to(dev)
        for h, (o, r, d, t) in zip((b, c), outs):
            h.step(a_t, o, r, d, t)
        _compare_handles(a, (b, c), s, [(obs, rew, done, term)] + outs, other_kernel=(1,))
        st["steps_after"] += 1
        st["n_done_after"] += int(done.sum())

    io = Outputs(E, a.D, dev)
    run_vs_oracle(a, orc, 4 * L, charge_log=False, dephase=L, outputs=io, hook=hook)
    assert st["export_step"] is not None, st
    assert st["steps_after"] >= 2 * L and st["n_done_after"] >= E, st
    sa = a.stats()
    for h, tol in ((b, 1e-12), (c, 1e-9)):               # striped atomics; c adds its per-env sums in another order
        sh = h.stats()
        for k in sa:
            np.testing.assert_allclose(sh[k], sa[k], rtol=tol, atol=0 if h is b else tol, err_msg=k)
        assert h.check_errors() == 0
    for h in (a, b, c):
        h.close()


def _vec_inputs(n):
    from fleetrl_b200.schedule import generate_schedule, synthetic_series
    from fleetrl_b200.tables import FleetInputs
    sched = generate_schedule("lmd", n, start="2020-01-01 00:00", end="2020-03-31 23:59", seed=11)
    price, tariff, load, pv = synthetic_series(start="2020-01-01 00:00", end="2020-03-31 23:59")
    return FleetInputs(sched, price, tariff, load, pv)


def test_vec_env_state_dict_round_trip_pf(knobs):
    """FleetVecEnv.state_dict() / load_state_dict() with N = 10 (the pf kernel): the restored env continues the
    trajectories of the first one bit for bit, every state field included."""
    from fleetrl_b200 import FleetVecEnv
    from fleetrl_b200.config import default_config
    cfg = default_config("lmd", time_picker="random", end_cutoff=10)
    E, N = 40, 10
    inputs = _vec_inputs(N)
    a_env = FleetVecEnv(cfg, E, inputs=inputs, output="torch", env_id_offset=9, seed=3)
    assert a_env.handle.step_kernel_name.startswith("fleet_step_pf_kernel")
    a_env.reset()
    rng = np.random.default_rng(6)
    acts = [torch.from_numpy(rng.uniform(-1, 1, (E, N)).astype(np.float32)).to(a_env.device) for _ in range(260)]
    for s in range(130):                       # past one episode end and one daily evaluation
        a_env.step(acts[s])
    sd = a_env.state_dict()
    b_env = FleetVecEnv(cfg, E, inputs=inputs, output="torch", env_id_offset=9, seed=3)
    b_env.reset()
    for s in range(50):                        # dirty state before the import
        b_env.step(acts[-1 - s])
    obs_b = b_env.load_state_dict(sd)
    np.testing.assert_array_equal(obs_b.cpu().numpy(), a_env._obs.cpu().numpy())
    n_done = 0
    for s in range(130, 260):
        oa, ra, da, _ = a_env.step(acts[s])
        ob, rb, db, _ = b_env.step(acts[s])
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db), f"step {s}"
        n_done += int(da.sum())
    assert n_done >= E
    for k in _fields(a_env.handle):
        assert torch.equal(a_env.handle.get(k), b_env.handle.get(k)), k
    sa, sb = a_env.stats(), b_env.stats()
    for k in sa:
        np.testing.assert_allclose(sb[k], sa[k], rtol=1e-12, atol=0, err_msg=k)
    a_env.close(); b_env.close()


# --------------------------------------------------------------------------------------------- d. log ring wrap-around
def test_log_ring_wraps(knobs):
    """enable_log(max_rows=r) with r not dividing the episode length, over more than three episodes: get_log is the
    last r rows of the DataLogger frame built from the oracle, Episode column included."""
    import pandas as pd
    from fleetrl_b200 import FleetVecEnv
    from fleetrl_b200.config import default_config
    cfg = default_config("lmd", time_picker="random", end_cutoff=10)
    E, N, r = 8, 6, 61
    env = FleetVecEnv(cfg, E, inputs=_vec_inputs(N), output="torch", env_id_offset=5, seed=3)
    L = int(env.built.consts.episode_steps)
    steps = 3 * L + 17
    total = steps + 1                                   # one row per step plus the first reset row
    assert L % r and total % r and total % r != (total // r) % r
    orc = OracleFleet(env.built.consts, env.built.tables, E, env_id_offset=5)
    env.enable_log(indices=[2, 5], max_rows=r)
    env.reset(); o_obs = orc.reset()
    rng = np.random.default_rng(8)
    want = {i: [dict(kind="reset", obs=o_obs[i].copy(), soh=orc.get("soh")[i].copy())] for i in (2, 5)}
    for s in range(steps):
        a = rng.uniform(-1, 1, (E, N)).astype(np.float32)
        env.step(torch.from_numpy(a).to(env.device))
        o_obs, o_rew, o_cash, o_done, _ = orc.step(a, want_terminal=True)
        for i in (2, 5):
            w = dict(kind="reset" if o_done[i] else "step", obs=o_obs[i].copy(), soh=orc.get("soh")[i].copy())
            if not o_done[i]:
                w.update(action=a[i].copy(), reward=o_rew[i], cash=o_cash[i], time_idx=orc.get("time_idx")[i])
            want[i].append(w)
    for i in (2, 5):
        assert len(want[i]) == total
        log = env.env_method("get_log", indices=[i])[0]
        assert list(log.columns) == list(env.LOG_COLUMNS) and len(log) == r
        n_steps = 0
        for j in range(r):
            g = total - r + j                           # index of the row in the whole frame
            w, row = want[i][g], log.iloc[j]
            assert row["Episode"] == g // L + 1, (j, row["Episode"])
            np.testing.assert_array_equal(row["Observation"], w["obs"], err_msg=f"row {g}")
            np.testing.assert_allclose(row["SOH"], w["soh"], rtol=0, atol=1e-13)
            if w["kind"] == "reset":
                assert row["Reward"] == 0.0 and not np.any(row["Action"])
                continue
            n_steps += 1
            assert row["Time"] == pd.Timestamp(env.built.dates[int(w["time_idx"])])
            np.testing.assert_array_equal(row["Action"], w["action"].astype(np.float64))
            np.testing.assert_allclose(row["Reward"], w["reward"], rtol=1e-11, atol=1e-10)
            np.testing.assert_allclose(row["Cashflow"], w["cash"], rtol=1e-12, atol=1e-13)
        assert n_steps > 0 and log["Episode"].iloc[0] < log["Episode"].iloc[-1]
    env.close()
