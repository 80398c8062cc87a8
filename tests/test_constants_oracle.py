"""The oracle against relations that hold between runs differing in one configuration constant
(tests/constant_relations.py): the temperature factor of the SEI fade, and reward weights that must not feed back into
the state.  The same relations run on the device in tests/test_gpu_constants.py."""
import numpy as np
import pytest

from constant_relations import OracleSide, check_reward_weights, check_temperature
from parity_util import make_case

# use case, N, extra constants: lmd at the default constants, ct (lunch-time targets, 4.6 kW chargers) with another
# target and efficiency; both with a grid connection small enough for overloads of rel >= 1.1
CASES = {
    "lmd_n6": dict(use_case="lmd", n_evs=6, over=dict(grid_connection=70.0)),
    "ct_n5_two_trips": dict(use_case="ct", n_evs=5, two_trips=True, over=dict(target_soc=0.95, charging_eff=0.86,
                                                                             grid_connection=40.0)),
}


def _maker(name, E):
    cf = dict(CASES[name])
    base_over = cf.pop("over", {})

    def make(**over):
        consts, tables = make_case(name, days=8, **cf, over=dict(base_over, **over))
        return OracleSide(consts, tables, E, env_id_offset=5)
    return make, make_case(name, days=8, **cf)[1]


@pytest.mark.parametrize("temperature", [5.0, 15.0, 35.0, 40.0])
@pytest.mark.parametrize("name", sorted(CASES))
def test_temperature_scales_cycle_fade(name, temperature):
    make, tables = _maker(name, 24)
    r = check_temperature(make, tables, temperature, steps=100)
    assert r["n_ratio"] > 24, r
    assert r["worst"] <= 1e-14, r


@pytest.mark.parametrize("name", sorted(CASES))
def test_reward_weights_do_not_feed_back(name):
    make, tables = _maker(name, 24)
    n = check_reward_weights(make, tables, steps=130)
    assert n["invalid"] > 0 and n["overload"] > 0 and n["departures"] > 0 and n["price"] > 0, n


def test_s_temp_reference_values():
    """s_temp(25) = 1; the factor grows with temperature (k_temp > 0) and matches a float64 evaluation."""
    from constant_relations import s_temp
    assert s_temp(25.0) == 1
    v = [float(s_temp(t)) for t in (5.0, 15.0, 25.0, 35.0, 40.0)]
    assert all(a < b for a, b in zip(v, v[1:]))
    for t in (5.0, 40.0):
        f64 = np.exp(6.93e-2 * (t - 25) * ((25 + 273.15) / (t + 273.15)))
        assert abs(f64 - float(s_temp(t))) <= 4 * np.finfo(np.float64).eps * f64
