"""GPU vs CPU-oracle parity on many envs with auto-reset, random starts and random actions (through the C ABI).

The per-step comparison and its tolerances are those of parity_util.run_vs_oracle.
"""
import numpy as np
import pytest
import torch

from oracle.oracle import OracleFleet
from parity_util import make_case, run_vs_oracle
from synth_tables import make_consts, make_tables

pytestmark = pytest.mark.gpu

CASES = {
    "lmd_7ev": dict(n_evs=7, days=12, use_case="lmd", E=96, steps=230),
    "lmd_50ev": dict(n_evs=50, days=8, use_case="lmd", E=37, steps=120),
    "ct_20ev_two_trips": dict(n_evs=20, days=10, use_case="ct", two_trips=True, E=64, steps=210, episode_hours=48),
    "ut_1h_5ev": dict(n_evs=5, days=30, use_case="ut", sph=1, E=128, steps=110, episode_hours=48,
                      over=dict(include_building=0, include_pv=0)),
    "lmd_1ev": dict(n_evs=1, days=12, use_case="lmd", E=700, steps=110),
    "lmd_300ev": dict(n_evs=300, days=6, use_case="lmd", E=3, steps=100),
    "lmd_9ev_norm_nocarry": dict(n_evs=9, days=12, use_case="lmd", E=40, steps=200,
                                 over=dict(normalize=1, carry_degradation_state=0)),
    "lmd_6ev_linear_noaux": dict(n_evs=6, days=12, use_case="lmd", E=40, steps=200, over=dict(deg_mode=1, aux=0)),
    "lmd_5ev_soh09": dict(n_evs=5, days=12, use_case="lmd", E=16, steps=120, over=dict(init_soh=0.9)),
    "lmd_4ev_no_autoreset": dict(n_evs=4, days=12, use_case="lmd", E=8, steps=110, over=dict(auto_reset=0)),
    "lmd_12ev_nodeg_exact_soc": dict(n_evs=12, days=12, use_case="lmd", E=64, steps=230, over=dict(calc_degradation=0)),
    # ten-day episodes: ten daily evaluations per episode over one persistent rainflow stack per vehicle
    "lmd_9ev_10day_episodes": dict(n_evs=9, days=30, use_case="lmd", E=3, steps=1000, episode_hours=240),
    "lmd_50ev_e36": dict(n_evs=50, days=8, use_case="lmd", E=36, steps=120),
    "ut_10ev_e50": dict(n_evs=10, days=10, use_case="ut", E=50, steps=210, episode_hours=48),
    # no auxiliary block, with and without normalisation: with the "+log" rows below, every pf kernel instance runs here
    "lmd_10ev_noaux": dict(n_evs=10, days=12, use_case="lmd", E=48, steps=200, over=dict(aux=0)),
    "lmd_12ev_norm_noaux": dict(n_evs=12, days=12, use_case="lmd", E=40, steps=200, over=dict(normalize=1, aux=0)),
}


# both step-kernel implementations are exercised: "pf" (persistent software-pipelined kernel, the default where it
# applies: auto-reset, 8 <= N <= 256) and "generic" (any configuration).  "+ringR+stackS[+extX]" shrinks the history ring /
# the inline rainflow stack so that ring flushes between evaluations and stack extension slots are exercised.
KERNELS = ([(n, "pf") for n in sorted(CASES) if CASES[n]["n_evs"] >= 8 and CASES[n]["n_evs"] <= 256
            and CASES[n].get("over", {}).get("auto_reset", 1)]
           + [(n, "generic") for n in sorted(CASES)]
           + [(n, "pf+ring4+stack2") for n in ("lmd_50ev", "ct_20ev_two_trips", "lmd_9ev_norm_nocarry")]
           + [(n, "generic+ring8+stack3") for n in ("lmd_300ev", "lmd_7ev", "lmd_1ev", "lmd_5ev_soh09", "lmd_4ev_no_autoreset")]
           + [("lmd_9ev_10day_episodes", "pf+ring16+stack4"), ("lmd_50ev", "pf+ring128+stack64")]
           # pf rows run the instance without the charge log (the one bench.py and FleetVecEnv use); "+log" rows run the
           # kLog instances (all four normalisation x auxiliary-block combinations, and the ct / ut use cases); generic rows
           # keep the charge log on throughout
           + [("lmd_50ev", "pf+log"), ("lmd_9ev_norm_nocarry", "pf+log"), ("lmd_10ev_noaux", "pf+log"),
              ("lmd_12ev_norm_noaux", "pf+log"), ("ct_20ev_two_trips", "pf+log"), ("ut_10ev_e50", "pf+log")])


@pytest.mark.parametrize("name,kernel", KERNELS)
def test_gpu_vs_oracle(name, kernel, monkeypatch):
    from fleetrl_b200._lib import FleetStepHandle
    monkeypatch.setenv("FLEETSTEP_KERNEL", kernel.split("+")[0])
    if "+stack" in kernel:
        monkeypatch.setenv("FLEETSTEP_RF_EXT_SLOTS", "40000")      # tiny inline stacks: every vehicle may need an extension slot
    else:
        monkeypatch.delenv("FLEETSTEP_RF_EXT_SLOTS", raising=False)
    for var, key in (("FLEETSTEP_RF_RING", "ring"), ("FLEETSTEP_RF_STACK", "stack"), ("FLEETSTEP_RF_EXT", "ext")):
        val = [t[len(key):] for t in kernel.split("+")[1:] if t.startswith(key)]
        if val:
            monkeypatch.setenv(var, val[0])
        else:
            monkeypatch.delenv(var, raising=False)

    cs = dict(CASES[name])
    E, steps = cs.pop("E"), cs.pop("steps")
    consts, tables = make_case(name, **cs)
    orc = OracleFleet(consts, tables, E, env_id_offset=1000)
    gpu = FleetStepHandle(consts, tables, E, device=0, env_id_offset=1000)
    charge_log = kernel.startswith("generic") or "+log" in kernel
    run_vs_oracle(gpu, orc, steps, charge_log=charge_log)
    gpu.close()


def test_rainflow_stack_capacity_is_loud(monkeypatch):
    """A rainflow stack that outgrows its inline entries + extension slot raises error flag bit 3 (never silent)."""
    from fleetrl_b200._lib import FleetStepError, FleetStepHandle
    monkeypatch.setenv("FLEETSTEP_RF_STACK", "2")
    monkeypatch.setenv("FLEETSTEP_RF_EXT", "1")
    tables, T = make_tables(seed=5, n_evs=8, days=6)
    consts = make_consts(tables, T, 8)
    gpu = FleetStepHandle(consts, tables, 32, device=0)
    dev = gpu.device
    obs = torch.zeros((32, gpu.D), dtype=torch.float32, device=dev)
    rew = torch.zeros(32, dtype=torch.float32, device=dev)
    done = torch.zeros(32, dtype=torch.uint8, device=dev)
    gpu.reset(obs=obs)
    rng = np.random.default_rng(0)
    for s in range(100):
        gpu.step(torch.from_numpy(rng.uniform(-1, 1, (32, 8)).astype(np.float32)).to(dev), obs, rew, done)
    with pytest.raises(FleetStepError, match="rainflow stack capacity"):
        gpu.check_errors()
    gpu.close()


def test_sei_stress_accuracy():
    """The post kernel's SEI cycle stress (rainflow_sei_degradation.py:68-79, dod ** kd2 as exp(kd2 * log(dod))) against
    extended precision: relative error below 5e-14 over the whole argument range (fd_cyc is stated at rel 1e-12 vs the reference)."""
    import ctypes as C
    from fleetrl_b200._lib import load_library
    L = load_library()
    rng = np.random.default_rng(0)
    eff = np.concatenate([rng.uniform(0, 1, 1_000_000), 10 ** rng.uniform(-9, 0, 500_000),
                          1 - 10 ** rng.uniform(-12, -1, 250_000), 10 ** rng.uniform(-14, -9, 10_000),
                          [1.0, 0.5, 0.25, 0.7071067811865476, 0.7071067811865475, 1e-9, 9.99e-10, 0.0]])
    mean = rng.uniform(0, 1, len(eff))
    dev = torch.device("cuda", 0)
    e_d, m_d = torch.from_numpy(eff).to(dev), torch.from_numpy(mean).to(dev)
    out = torch.empty_like(e_d)
    assert L.fleet_debug_stress(C.c_void_p(e_d.data_ptr()), C.c_void_p(m_d.data_ptr()), C.c_void_p(out.data_ptr()),
                                len(eff), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)) == 0
    got = out.cpu().numpy()
    ld = np.longdouble
    with np.errstate(divide="ignore"):
        want = (1 / (ld(1.4e5) * eff.astype(ld) ** ld(-0.501) + ld(-1.23e5)) * np.exp(ld(1.04) * (mean.astype(ld) - ld(0.5))))
    want = want.astype(np.float64)
    assert got[-1] == 0.0 and want[-1] == 0.0            # dod == 0: no stress
    rel = np.abs(got[:-1] - want[:-1]) / np.abs(want[:-1])
    assert rel.max() < 5e-14, (rel.max(), eff[rel.argmax()])


@pytest.mark.parametrize("kernel,n_evs", [("pf", 8), ("generic", 3)])
def test_year_long_evaluation_episode(kernel, n_evs, monkeypatch):
    """The reference's evaluation / benchmark callers run ONE episode of n_steps = 8600 hours (agent_eval/
    basic_evaluation.py:64, benchmarking/uncontrolled_charging.py:45-51): 34,400 quarter-hour steps, 358 daily evaluations
    over one ever-growing soc_log per vehicle.  The device keeps a 16-row ring and the persistent three-point stack
    instead of the log; cycle counts must stay bit-exact and SOH within 1e-12 over the whole year."""
    from fleetrl_b200._lib import FleetStepHandle
    monkeypatch.setenv("FLEETSTEP_KERNEL", kernel)
    hours, E = 8600, 2
    tables, T = make_tables(seed=11, n_evs=n_evs, days=362)
    consts = make_consts(tables, T, n_evs, episode_hours=hours, use_case="lmd", auto_reset=1 if kernel == "pf" else 0)
    steps = hours * 4
    assert consts.episode_steps == steps
    orc = OracleFleet(consts, tables, E, env_id_offset=3)
    gpu = FleetStepHandle(consts, tables, E, device=0, env_id_offset=3)
    assert gpu.device_bytes < 64 << 20                  # no per-episode history on the device
    dev = gpu.device
    obs = torch.zeros((E, gpu.D), dtype=torch.float32, device=dev)
    rew = torch.zeros(E, dtype=torch.float32, device=dev)
    done = torch.zeros(E, dtype=torch.uint8, device=dev)
    start = np.zeros(E, np.int32)
    o_obs = orc.reset(start_idx=start)
    gpu.reset(start_idx=torch.from_numpy(start).to(dev), obs=obs)
    np.testing.assert_array_equal(obs.cpu().numpy(), o_obs)
    rng = np.random.default_rng(3)
    block = rng.uniform(-1, 1, (steps, E, n_evs)).astype(np.float32)
    block[:, 0, :] = 1.0                                # env 0: uncontrolled charging (uncontrolled_charging.py:51-54)
    block[rng.random(block.shape) < 0.1] = 0.0
    a_dev = torch.from_numpy(block).to(dev)
    n_eval = 0
    for s in range(steps):
        o_obs, o_rew, _, o_done = orc.step(block[s])
        gpu.step(a_dev[s], obs, rew, done)
        last = s == steps - 1
        if s % 96 == 58 or last or s < 200:             # every step at first, then once per day and at the end
            np.testing.assert_array_equal(done.cpu().numpy(), o_done, err_msg=f"done step {s}")
            for k in ("time_idx", "rf_len", "n_cycles", "hours_left"):
                np.testing.assert_array_equal(gpu.get(k).cpu().numpy(), orc.get(k), err_msg=f"{k} step {s}")
            np.testing.assert_allclose(gpu.get("soh").cpu().numpy(), orc.get("soh"), rtol=0, atol=1e-12, err_msg=f"soh step {s}")
            np.testing.assert_allclose(gpu.get("fd_cyc").cpu().numpy(), orc.get("fd_cyc"), rtol=1e-10, atol=1e-18)
            np.testing.assert_allclose(gpu.get("soc").cpu().numpy(), orc.get("soc"), rtol=0, atol=1e-11, err_msg=f"soc step {s}")
            np.testing.assert_allclose(gpu.get("reward64").cpu().numpy(), o_rew, rtol=1e-11, atol=1e-9)
            if not last or kernel != "pf":              # (the pf case auto-resets after the last step)
                np.testing.assert_allclose(obs.cpu().numpy(), o_obs, rtol=0, atol=2e-6, err_msg=f"obs step {s}")
            n_eval += 1
    assert o_done.all() and n_eval > 358
    assert orc.get("n_cycles").max() > 2000             # thousands of cycles per vehicle went through the stack
    assert gpu.check_errors() == 0 and orc.err_flags() == 0
    gpu.close()
