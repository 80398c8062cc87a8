"""Flush units of the post kernel against the oracle.

An env whose history ring would wrap with the next sample and that has no daily evaluation and no reset in the same step
is a flush-only entry: the step kernel puts it on a list of its own, and the post kernel consumes those entries in units
of 32 consecutive vehicles of the flattened (entry x N) index space, one unit per warp, after the other work items.  A
unit therefore covers the tail of one env and the head of the next whenever N is not a multiple of 32.

Every case caps the post kernel's grid (FLEETSTEP_POST_GRID) so that each warp fetches many units per launch, de-phases
the episodes, and asserts from the state read before each step (env4 = {t, t_start, ep_count, k_done}, the stack depths
and extension slots) that its scenario happened: flush-only entries in the same step as flush + evaluation or
flush + reset entries, units whose lanes cover two envs, and, for the deep-stack case, a flush lane that holds an
extension slot (the rf_vehicle_slow path).
"""
import numpy as np
import pytest

from oracle.oracle import OracleFleet
from parity_util import knobs, make_case, run_vs_oracle  # noqa: F401  (knobs: fixture)
from test_gpu_state import parse_blob

pytestmark = pytest.mark.gpu


# N, CTA size of the post kernel, env count, post grid; "slow": 2-entry inline stacks, so deep stacks live in extension slots
CASES = {
    "n50_straddle_64thr": dict(n_evs=50, E=400, post=2, threads=64, chunks=1),
    "n20_32thr": dict(n_evs=20, E=600, post=3, threads=32, chunks=1),
    "n70_chunked_items": dict(n_evs=70, E=300, post=2, threads=64, chunks=2),
    "n33": dict(n_evs=33, E=400, post=2, threads=64, chunks=1),
    "n20_ct_slow_path_ext": dict(n_evs=20, E=400, post=2, threads=32, chunks=1, use_case="ct", two_trips=True,
                                 env=dict(FLEETSTEP_RF_RING=4, FLEETSTEP_RF_STACK=2, FLEETSTEP_RF_EXT_SLOTS=40000),
                                 slow=True),
}


def _straddling_units(n_flush, N):
    """Units whose 32 lanes cover vehicles of two or more entries: one per entry boundary f * N (0 < f < n_flush) that
    does not fall on a unit boundary.  Independent of the order in which the entries were pushed."""
    return sum(1 for f in range(1, n_flush) if (f * N) % 32)


@pytest.mark.parametrize("name", sorted(CASES))
def test_flush_units_vs_oracle(name, knobs):
    from fleetrl_b200._lib import FleetStepHandle
    cf = dict(CASES[name])
    E, post, threads, chunks = cf.pop("E"), cf.pop("post"), cf.pop("threads"), cf.pop("chunks")
    env, slow = cf.pop("env", {}), cf.pop("slow", False)
    knobs(FLEETSTEP_POST_GRID=post, **env)
    consts, tables = make_case(name, days=8, **cf)
    N, L, T = consts.num_evs, consts.episode_steps, consts.table_len
    gpu = FleetStepHandle(consts, tables, E, device=0, env_id_offset=1000)
    assert gpu.launch_geometry["post_grid"] == post, gpu.launch_geometry
    assert threads == (32 if N <= 32 else 64) and chunks == -(-N // threads)
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    trig_row = (np.asarray(tables["hour"]) == 14) & (np.asarray(tables["minute"]) == 45)

    st = dict(steps_both=0, flush_only=0, flush_eval=0, flush_reset=0, straddle=0, max_units_per_warp=0, slow_ext=0)

    def hook(s, *_):
        p = parse_blob(gpu.export_state())
        R, S = int(p["header"]["R"]), int(p["header"]["S"])
        t, t0, k_done = p["env4"][:, 0], p["env4"][:, 1], p["env4"][:, 3]
        k = t - t0                                             # the coming step is step k of the episode
        flush = k + 1 - k_done >= R - 1
        trig = trig_row[np.minimum(t, T - 2) + 1] & bool(consts.calc_degradation)
        reset = t + 1 == t0 + L
        only = flush & ~trig & ~reset
        n_only = int(only.sum())
        st["flush_only"] += n_only
        st["flush_eval"] += int((flush & trig).sum())
        st["flush_reset"] += int((flush & reset).sum())
        if n_only and (flush & (trig | reset)).any():
            st["steps_both"] += 1
        st["straddle"] += _straddling_units(n_only, N)
        st["max_units_per_warp"] = max(st["max_units_per_warp"], -(-n_only * N // 32) / (post * threads // 32))
        if slow:
            depth = (p["rf_dc"] & 0xFFFF).astype(np.int64)
            deep = (depth > S) & (p["rf_ext"] >= 0)            # starts on rf_vehicle_slow with an extension slot
            st["slow_ext"] += int((deep & only[:, None]).sum())

    run_vs_oracle(gpu, orc, 2 * L + 10, charge_log=False, dephase=L, hook=hook)
    assert st["steps_both"] > 0 and st["flush_eval"] > 0 and st["flush_reset"] > 0, st
    assert st["straddle"] > 0 and st["max_units_per_warp"] >= 4, st
    if slow:
        assert st["slow_ext"] > 0, st
    gpu.close()
