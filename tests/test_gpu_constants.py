"""The step, post and policy kernels away from the default configuration constants.

Every other parity test runs one set of EvConfig / ScoreConfig / company constants, and at several of those values a
term disappears (temperature 25 C makes the SEI temperature factor exactly 1) or two constants become interchangeable
(charging_eff == discharging_eff, lc_batt_cap == init_battery_cap, obc_max_power above every evse_max_power).

a. A seeded sweep of constant draws against the oracle, each non-degenerate in all of those, on the capped-grid pf kernel
   and on the generic kernel with the charge log; every draw asserts that its scenarios happened.
b. The oracle-independent relations of tests/constant_relations.py on the device, at the cfg2 fleet shape.
c. An env_config of the custom use case with ignore_* flags, resolved by build_fleet and stepped against the oracle.
"""
import functools

import numpy as np
import pytest
import torch

from constant_relations import STATE_FIELDS, check_reward_weights, check_temperature
from oracle import policies as opol
from oracle.oracle import OracleFleet
from parity_util import knobs, make_case, run_vs_oracle  # noqa: F401  (knobs: fixture)
from test_gpu_pipeline import MIN_TILES_PER_CTA, _assert_capped, _envs_per_tile, _handle

pytestmark = pytest.mark.gpu

TEMPS = (5.0, 15.0, 35.0, 40.0)
TARGETS = (0.7, 0.8, 0.95, 1.0)
EVSE = dict(lmd=11.0, ut=22.0, ct=4.6)
CAP0 = dict(lmd=60.0, ut=50.0, ct=16.7)
SOH_09 = (1, 2, 7, 9)          # draws starting at SOH 0.9: every target flips to 0.9 at the first step

# use case, N, steps per hour, normalize, kernel (pf: grid capped at G CTAs; generic: FLEETSTEP_KERNEL=generic, E envs).
# N runs from below the pf range (8 <= N <= 256) to above it; the caretaker fleets have a lunch-time trip.
STRUCT = [
    dict(use_case="lmd", n_evs=8, sph=4, normalize=0, kernel="pf", G=2),
    dict(use_case="lmd", n_evs=13, sph=4, normalize=1, kernel="pf", G=3),
    dict(use_case="ct", n_evs=20, sph=4, normalize=1, kernel="pf", G=1),
    dict(use_case="ut", n_evs=11, sph=4, normalize=0, kernel="pf", G=2),
    dict(use_case="lmd", n_evs=9, sph=1, normalize=1, kernel="pf", G=2),
    dict(use_case="ut", n_evs=50, sph=1, normalize=0, kernel="pf", G=1),
    dict(use_case="ct", n_evs=16, sph=4, normalize=0, kernel="pf", G=2),
    dict(use_case="lmd", n_evs=5, sph=4, normalize=1, kernel="generic", E=96),
    dict(use_case="ct", n_evs=7, sph=4, normalize=0, kernel="generic", E=96),
    dict(use_case="ut", n_evs=6, sph=1, normalize=1, kernel="generic", E=96),
    dict(use_case="ct", n_evs=5, sph=1, normalize=1, kernel="generic", E=96),
    dict(use_case="lmd", n_evs=260, sph=4, normalize=0, kernel="generic", E=12),
]


def _draw(i, st, rng):
    """Constant overrides of draw i (see the module docstring and _check_draws for what each draw must satisfy)."""
    uc, N = st["use_case"], st["n_evs"]
    evse, cap0 = EVSE[uc], CAP0[uc]
    eta_c = rng.uniform(0.8, 0.98)
    eta_d = rng.uniform(0.8, 0.98)
    while abs(eta_d - eta_c) < 0.03:
        eta_d = rng.uniform(0.8, 0.98)
    target = TARGETS[(i + i // 4) % 4]
    over = dict(
        normalize=st["normalize"], temperature=TEMPS[i % 4], target_soc=target,
        init_soh=0.9 if i in SOH_09 else 1.0,
        charging_eff=eta_c, discharging_eff=eta_d,
        obc_max_power=evse * (rng.uniform(0.35, 0.9) if i % 2 == 0 else rng.uniform(1.1, 3.0)),
        lc_batt_cap=cap0 * (rng.uniform(0.6, 0.9) if i % 2 else rng.uniform(1.1, 1.6)),
        target_soc_lunch=rng.uniform(0.5, 0.8), min_laxity=rng.uniform(1.2, 3.5), def_soc=rng.uniform(0.2, 0.8),
        soc_eps=(0.0, 0.001, 0.02, 0.05)[(i // 2) % 4], fully_charged_reward=(0.0, 0.4, 2.5)[i % 3],
        fixed_markup=rng.uniform(0, 30), variable_multiplier=rng.uniform(1.0, 2.5),
        feed_in_deduction=rng.uniform(0.0, 0.5),
        price_multiplier=0.0 if i % 4 == 3 else rng.uniform(0.5, 8.0),
        penalty_invalid_action=0.0 if i % 5 == 2 else -rng.uniform(0.05, 0.6),
        penalty_overcharging=0.0 if i % 5 == 3 else -rng.uniform(0.001, 0.02),
        penalty_overloading=0.0 if i % 5 == 4 else rng.uniform(0.3, 2.0),
        clip_overcharging=-rng.uniform(0.05, 0.5),
        grid_connection=rng.uniform(0.35, 0.6) * (50.0 + N * evse),
    )
    table_target = target if i % 3 == 2 else 0.85      # tables derived from another target: SOC above the target
    return over, table_target


def _draws():
    rng = np.random.default_rng(20261021)
    out = {}
    for i, st in enumerate(STRUCT):
        over, table_target = _draw(i, st, rng)
        name = f"d{i:02d}_{st['use_case']}_n{st['n_evs']}_{'15min' if st['sph'] == 4 else '1h'}_{st['kernel']}"
        out[name] = dict(st, over=over, table_target=table_target)
    return out


DRAWS = _draws()


def _soc_above_target(cf):
    """Vehicles arrive above their target: the tables' target is higher, or the flip lowers the target to 0.9."""
    o = cf["over"]
    return cf["table_target"] > o["target_soc"] or (o["init_soh"] == 0.9 and o["target_soc"] > 0.9)


def _check_draws():
    """What the draws cover together (a draw table that loses one of these fails every case)."""
    d = list(DRAWS.values())
    o = [x["over"] for x in d]
    assert all(x["charging_eff"] != x["discharging_eff"] and x["lc_batt_cap"] != CAP0[y["use_case"]] for x, y in zip(o, d))
    assert all(x["temperature"] in TEMPS for x in o) and {x["temperature"] for x in o} == set(TEMPS)
    below = [x["obc_max_power"] < EVSE[y["use_case"]] for x, y in zip(o, d)]
    assert sum(below) == len(d) // 2
    flips = {x["target_soc"] for x in o if x["init_soh"] == 0.9}
    assert min(flips) < 0.9 < max(flips)                             # the flip raises and lowers the target
    assert any(x["soc_eps"] == 0 for x in o) and any(x["fully_charged_reward"] == 0 for x in o)
    for k in ("price_multiplier", "penalty_invalid_action", "penalty_overcharging", "penalty_overloading"):
        assert any(x[k] == 0 for x in o) and any(x[k] != 0 for x in o), k
    assert {y["use_case"] for y in d} == {"lmd", "ct", "ut"} and {y["sph"] for y in d} == {1, 4}
    assert {y["normalize"] for y in d} == {0, 1} and {y["kernel"] for y in d} == {"pf", "generic"}
    assert min(y["n_evs"] for y in d) < 8 and max(y["n_evs"] for y in d) > 256
    assert sum(_soc_above_target(y) for y in d) >= len(d) // 3
    assert any(x["init_soh"] == 0.9 and y["normalize"] for x, y in zip(o, d))   # flipped aux terms, normalised


@pytest.mark.parametrize("name", sorted(DRAWS))
def test_constant_draw_vs_oracle(name, knobs):
    _check_draws()
    cf = DRAWS[name]
    uc, N, sph = cf["use_case"], cf["n_evs"], cf["sph"]
    two_trips = uc == "ct"
    consts, tables = make_case(name, N, days=8, use_case=uc, sph=sph, two_trips=two_trips, over=cf["over"],
                               table_target=cf["table_target"])
    if cf["kernel"] == "pf":
        G = cf["G"]
        B = _envs_per_tile(consts, tables)
        E = MIN_TILES_PER_CTA * G * B + (B // 3 + 1 if B > 1 else 1)
        knobs(FLEETSTEP_PF_GRID=G)
        gpu = _handle(consts, tables, E, env_id_offset=1000)
        _assert_capped(gpu, G)
        charge_log = False
    else:
        E = cf["E"]
        knobs(FLEETSTEP_KERNEL="generic")
        gpu = _handle(consts, tables, E, env_id_offset=1000)
        assert gpu.step_kernel_name == "fleet_step_kernel"
        charge_log = True
    c = consts
    P = min(c.obc_max_power, c.evse_max_power)
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    there, time_left = np.asarray(tables["there"]), np.asarray(tables["time_left"])
    hour = np.asarray(tables["hour"])
    T = c.table_len
    n_pol = min(E, 8)
    seen = dict(obc=0, flip=0, lunch=0, overload=0, neg_demand=0, policy=0)
    pre = {}

    def hook(s, a, *_):
        if s >= 0:
            t = pre["t"]
            th = there[:, t].T                                              # [E, N] presence during the step
            a64 = a.astype(np.float64)
            if c.obc_max_power < c.evse_max_power:                          # energy = requested at the obc limit
                seen["obc"] += int(((th == 1) & (a64 > 0) & (orc.get("charge_log") == P * a64 * c.dt)).sum())
            seen["neg_demand"] += int(((th == 1) & (a64 >= 0) & (pre["soc"] > pre["target"])).sum())
            ntl = time_left[:, t + 1].T
            lunch = (hour[t + 1] > 11) & (hour[t + 1] < 15)
            seen["lunch"] += int(((pre["hl"] != 0) & (ntl == 0) & lunch[:, None]).sum())
            seen["overload"] += int((orc.get("overload") / c.grid_connection + 1 >= 1.1).sum())
            seen["flip"] += int((orc.get("target_soc") == 0.9).sum())
        pre.update(t=orc.get("time_idx"), soc=orc.get("soc"), target=orc.get("target_soc"), hl=orc.get("hours_left"))
        # the distributed rule at every env's current time (reads lc_batt_cap, evse_max_power and charging_eff)
        got = gpu.policy_actions("distributed").cpu().numpy()[:n_pol]
        for e in range(n_pol):
            want = opol.distributed(c, tables, min(int(pre["t"][e]), T - 1), pre["target"][e]).astype(np.float32)
            np.testing.assert_array_equal(got[e], want, err_msg=f"distributed policy step {s} env {e}")
        seen["policy"] += int((got != 0).sum())

    L = c.episode_steps
    run_vs_oracle(gpu, orc, 2 * L + 10, charge_log=charge_log, dephase=L, hook=hook)
    assert seen["overload"] > 0 and seen["policy"] > 0, seen
    if _soc_above_target(cf):
        assert seen["neg_demand"] > 0, seen
    if c.obc_max_power < c.evse_max_power:
        assert seen["obc"] > 0, seen
    if c.init_soh == 0.9:
        assert seen["flip"] > 0, seen
    if c.is_caretaker:
        assert seen["lunch"] > 0, seen
    gpu.close()


# ------------------------------------------------------------------------------- b. relations at the cfg2 fleet shape
class DeviceSide:
    """A FleetStepHandle seen through the interface of constant_relations (outputs and state stay on the device)."""

    def __init__(self, consts, tables, E):
        self.h = _handle(consts, tables, E)
        self.consts, self.E, self.N = consts, E, int(consts.num_evs)
        dev, D = self.h.device, self.h.D
        self.obs = torch.zeros((E, D), dtype=torch.float32, device=dev)
        self.term = torch.zeros((E, D), dtype=torch.float32, device=dev)
        self.rew = torch.zeros(E, dtype=torch.float32, device=dev)
        self.done = torch.zeros(E, dtype=torch.uint8, device=dev)

    def reset(self):
        self.h.reset(obs=self.obs)

    def step(self, a):
        self.h.step(torch.from_numpy(a).to(self.h.device), self.obs, self.rew, self.done, self.term)
        return dict(obs=self.obs, term=self.term, done=self.done.cpu().numpy().astype(bool),
                    reward=self.h.get("reward64").cpu().numpy(), cashflow=self.h.get("cashflow").cpu().numpy())

    def state(self):
        return {k: self.h.get(k) for k in STATE_FIELDS}

    def get(self, name):
        return self.h.get(name).cpu().numpy()

    def stats(self):
        return self.h.stats()


@functools.lru_cache(maxsize=1)
def _cfg2():
    from fleetrl_b200.config import default_config
    from fleetrl_b200.schedule import generate_schedule, synthetic_series
    from fleetrl_b200.tables import FleetInputs, build_fleet
    sched = generate_schedule("lmd", 50, seed=42)
    price, tariff, load, pv = synthetic_series(seed=7)
    built = build_fleet(default_config("lmd", seed=0), FleetInputs(sched, price, tariff, load, pv), auto_reset=True,
                        carry_degradation_state=True, seed=0, time_picker="random")
    return built.consts, built.tables


def _cfg2_maker(E=16384):
    from fleetrl_b200._abi import FleetConsts
    c, tb = _cfg2()
    sides = []

    def make(**over):
        sd = DeviceSide(FleetConsts.from_dict(dict(c.to_dict(), **over)), tb, E)
        sides.append(sd)
        return sd
    return make, tb, sides


@pytest.mark.parametrize("temperature", [5.0, 40.0])
def test_temperature_relation_cfg2(temperature):
    make, tb, sides = _cfg2_maker()
    r = check_temperature(make, tb, temperature, steps=97)
    assert r["n_ratio"] > 16384, r
    assert r["worst"] <= 1e-14, r
    for sd in sides:
        assert sd.h.check_errors() == 0
        sd.h.close()


def test_reward_weights_relation_cfg2():
    make, tb, sides = _cfg2_maker()
    n = check_reward_weights(make, tb, steps=126)
    assert n["invalid"] > 0 and n["overload"] > 0 and n["departures"] > 0 and n["price"] > 0, n
    for sd in sides:
        assert sd.h.check_errors() == 0
        sd.h.close()


# ------------------------------------------------------------------------------------ c. env_config to the device
def test_custom_env_config_to_device(knobs):
    """The custom use case (evse 120 kW above the on-board charger's 100 kW, 500 kW grid) with ignore_price_reward and
    ignore_invalid_penalty and another target SOC, from env_config through build_fleet to the device, against the oracle
    on the constants build_fleet resolved."""
    from fleetrl_b200 import FleetVecEnv
    from fleetrl_b200.config import default_config
    from fleetrl_b200.schedule import generate_schedule, synthetic_series
    from fleetrl_b200.tables import FleetInputs
    start, end = "2020-01-01 00:00", "2020-02-29 23:59"
    cfg = default_config("custom", gen_schedule=True, gen_n_evs=9, gen_start_date=start, gen_end_date=end, end_cutoff=10,
                         custom_ev_battery_size_in_kwh=300, max_batt_cap_in_all_use_cases=300,
                         custom_weekday_distance_mean=150, ignore_price_reward=True, ignore_invalid_penalty=True,
                         target_soc=0.8, seed=3)
    price, tariff, load, pv = synthetic_series(start=start, end=end, seed=6)
    inputs = FleetInputs(generate_schedule("lmd", 1, start=start, end=end, seed=5), price, tariff, load, pv)
    env = FleetVecEnv(cfg, 300, inputs=inputs, seed=11)
    c, tb = env.built.consts, env.built.tables
    assert c.num_evs == 9 and c.price_multiplier == 0 and c.penalty_invalid_action == 0 and c.target_soc == 0.8
    assert c.penalty_overloading == 1 and c.penalty_overcharging == -0.0055
    assert c.evse_max_power == 120 and c.obc_max_power == 100 and c.grid_connection == 500
    assert c.init_battery_cap == 300 and c.lc_batt_cap == 300
    orc = OracleFleet(c, tb, env.num_envs, threads=8)
    there = np.asarray(tb["there"])
    seen = dict(obc=0, overload=0)
    pre = {}

    def hook(s, a, *_):
        if s >= 0:
            a64 = a.astype(np.float64)
            th = there[:, pre["t"]].T
            seen["obc"] += int(((th == 1) & (a64 > 0) & (orc.get("charge_log") == c.obc_max_power * a64 * c.dt)).sum())
            seen["overload"] += int((orc.get("overload") / c.grid_connection + 1 >= 1.1).sum())
        pre["t"] = orc.get("time_idx")

    L = c.episode_steps
    run_vs_oracle(env.handle, orc, 2 * L + 10, charge_log=True, dephase=L, hook=hook)
    assert seen["obc"] > 0 and seen["overload"] > 0, seen
    st = env.handle.stats()
    assert st["penalty"] == st["reward"]                              # price_multiplier 0
    env.close()
