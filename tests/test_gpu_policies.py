"""On-device rule-based baseline policies (fleet_policy_actions) vs the NumPy restatement of the reference's benchmark
scripts (oracle/policies.py), stepping the fleet with the policy's own actions so that times, departures, auto-resets
and the night policy's window state all evolve.  Actions are float32 on both sides: bit-exact."""
import numpy as np
import pytest
import torch

from fleetrl_b200.config import default_config
from fleetrl_b200.policies import night_params
from fleetrl_b200.schedule import generate_schedule, synthetic_series
from fleetrl_b200.tables import FleetInputs
from oracle import policies as opol

pytestmark = pytest.mark.gpu


def _inputs(use_case, n):
    sched = generate_schedule(use_case, n, start="2020-01-01 00:00", end="2020-03-31 23:59", seed=5)
    price, tariff, load, pv = synthetic_series(start="2020-01-01 00:00", end="2020-03-31 23:59")
    return FleetInputs(sched, price, tariff, load, pv)


# id -> (use case, N, env_config overrides).  1h: a 1-hour grid, where the night window opens only at charging minute 0
# (target 1.0 puts it at 23:00 for this schedule); 33: the (env, EV) index i / N crosses a warp inside an env; tuned: the
# distributed rule and night_params read target_soc and charging_eff, the fleet's trajectory obc_max_power (below evse).
CASES = {
    "lmd-6": ("lmd", 6, {}),
    "ct-4": ("ct", 4, {}),
    "ut-5": ("ut", 5, {}),
    "lmd-4-1h": ("lmd", 4, dict(freq="1h", minutes=60, time_steps_per_hour=1, target_soc=1.0)),
    "lmd-33": ("lmd", 33, {}),
    "ct-6-tuned": ("ct", 6, dict(target_soc=0.95, charging_eff=0.82, obc_max_power=3.0)),
}


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("policy", ["uncontrolled", "distributed", "night"])
def test_policy_actions_match_reference_rules(case, policy):
    from fleetrl_b200 import FleetVecEnv
    use_case, n_evs, over = CASES[case]
    cfg = default_config(use_case, time_picker="random", end_cutoff=10, episode_length=48 if use_case == "ct" else 24,
                         **over)
    E = 24
    env = FleetVecEnv(cfg, E, inputs=_inputs(use_case, n_evs), output="torch", seed=9)
    c, tb = env.built.consts, env.built.tables
    env.reset()
    for k, v in over.items():
        if hasattr(c, k):
            assert getattr(c, k) == v, k
    npar = night_params(env.built)
    assert 0 <= npar.charging_hour <= 23 and npar.charging_minute in (0, 15, 30, 45)
    night = [opol.NightPolicy(c, tb, npar.charging_hour, npar.charging_minute, npar.max_hours) for _ in range(E)]
    n_nonzero = 0
    for s in range(260):
        t = env.handle.get("time_idx").cpu().numpy()
        tgt = env.handle.get("target_soc").cpu().numpy()
        a_dev = env.baseline_actions(policy)
        want = np.empty((E, n_evs), dtype=np.float32)
        for e in range(E):
            if policy == "uncontrolled":
                a = opol.uncontrolled(n_evs)
            elif policy == "distributed":
                a = opol.distributed(c, tb, int(t[e]), tgt[e])
            else:
                a = night[e].actions(int(t[e]), tgt[e])
            want[e] = a.astype(np.float32)
        np.testing.assert_array_equal(a_dev.cpu().numpy(), want, err_msg=f"{policy} step {s}")
        n_nonzero += int((want != 0).sum())
        env.step(a_dev)
    assert n_nonzero > 0
    if policy == "night":
        # the window opened and closed at least once somewhere
        assert any(p.charging_start != 0 for p in night)
    env.close()
