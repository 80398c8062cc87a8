"""Relations between runs that differ in one configuration constant, checked without a reference implementation.

The oracle (oracle/fleet_oracle.c) and the kernels are written from the same reference lines, so a constant both read
the same wrong way is invisible to a parity test.  These relations follow from the reference's formulas alone and are
run on both sides: on OracleFleet (tests/test_constants_oracle.py) and on the device (tests/test_gpu_constants.py).

A "side" is any object with
    consts, E, N
    reset()                       reset every env through the counter RNG
    step(a)                       a: float32 [E, N] NumPy; -> dict(obs, term, done, reward, cashflow): obs / term as the
                                  side keeps them (NumPy or torch), done bool [E], reward / cashflow float64 [E] (NumPy)
    state()                       dict name -> array of every state field (NumPy or torch)
    get(name)                     one field as NumPy
    stats()                       dict of the FLEET_S_* statistics

temperature   two fleets that differ only in `temperature` are bit-identical up to each env's first 14:45 evaluation;
              there the cycle fade of every vehicle scales by s_temp(T) (rainflow_sei_degradation.py:72-79).
reward_weights  price_multiplier, the penalty weights, clip_overcharging and fully_charged_reward change the reward
              only: obs, terminal obs, done, cashflow and every state field stay bit-identical.  The reward is affine in
              price_multiplier, penalty_invalid_action, penalty_overloading and fully_charged_reward; the invalid-action
              and overload terms have closed forms (ev_charger.py:120-122,180-182, score_config.py:33-41); the penalty
              statistic is reward - cashflow * price_multiplier (fleet_environment.py:659), also at price_multiplier 0.
"""
import numpy as np
import torch

from oracle.oracle import OracleFleet

# every state field except the ones that carry the reward (reward64, ep_return, last_ep_return) and the charge log
STATE_FIELDS = ("soc", "hours_left", "soc_deg", "soh", "target_soc", "time_idx", "finish_idx", "rf_len", "fd_cyc",
                "life", "ep_count", "n_cycles", "last_deg", "overload", "soc_viol")
EPS = float(np.finfo(np.float64).eps)

# weight -> increment: the reward is affine in each of them
AFFINE = dict(price_multiplier=1.7, penalty_invalid_action=-0.35, penalty_overloading=0.6, fully_charged_reward=0.8)
# further single-constant changes that must leave everything but the reward alone (absolute values)
REWARD_ONLY = dict(price_multiplier=0.0, clip_overcharging=-0.45, penalty_overcharging=-0.013)


class OracleSide:
    def __init__(self, consts, tables, E, env_id_offset=0):
        self.o = OracleFleet(consts, tables, E, env_id_offset=env_id_offset)
        self.consts, self.E, self.N = consts, E, int(consts.num_evs)

    def reset(self):
        self.o.reset()

    def step(self, a):
        obs, rew, cash, done, term = self.o.step(a, want_terminal=True)
        return dict(obs=obs, term=term, done=done.astype(bool), reward=rew, cashflow=cash)

    def state(self):
        return {k: self.o.get(k) for k in STATE_FIELDS}

    def get(self, name):
        return self.o.get(name)

    def stats(self):
        return self.o.stats()


def s_temp(temperature):
    """Temperature stress factor of the SEI model (rainflow_sei_degradation.py:72-73) in extended precision."""
    ld = np.longdouble
    k_temp, t_ref, t = ld(6.93e-2), ld(25), ld(temperature)
    return np.exp(k_temp * (t - t_ref) * ((t_ref + ld(273.15)) / (t + ld(273.15))))


def actions(rng, s, E, N):
    """Random actions with exact zeros every fifth step and everybody charging every seventh (overloads)."""
    a = rng.uniform(-1, 1, (E, N)).astype(np.float32)
    if s % 5 == 0:
        a[rng.random((E, N)) < 0.3] = 0.0
    if s % 7 == 0:
        a[:] = 1.0
    return a


def _same(x, y):
    if isinstance(x, np.ndarray):
        return np.array_equal(x, y)
    return bool(torch.equal(x, y))


def _rows(x, mask):
    """x[mask] for a NumPy bool mask over the leading (env) axis of a NumPy or torch array."""
    if isinstance(x, np.ndarray):
        return x[mask]
    return x[torch.from_numpy(mask).to(x.device)]


def _assert_same_rows(x, y, mask, what):
    assert _same(_rows(x, mask), _rows(y, mask)), what


def _assert_identical(out_a, out_b, st_a, st_b, mask, what, outputs=("reward", "cashflow"), skip=()):
    """Outputs and state of the envs in `mask` are bit-identical (state fields in `skip` excepted)."""
    assert np.array_equal(out_a["done"][mask], out_b["done"][mask]), f"done {what}"
    for k in outputs:
        assert np.array_equal(out_a[k][mask], out_b[k][mask]), f"{k} {what}"
    _assert_same_rows(out_a["obs"], out_b["obs"], mask, f"obs {what}")
    _assert_same_rows(out_a["term"], out_b["term"], mask & out_a["done"], f"terminal obs {what}")
    for k in STATE_FIELDS:
        if k not in skip:
            _assert_same_rows(st_a[k], st_b[k], mask, f"{k} {what}")


def check_temperature(make, tables, temperature, steps, seed=3):
    """make(temperature=...) -> side.  Returns dict(n_ratio, worst): vehicles whose cycle fade was compared at their
    env's first evaluation, and the largest relative deviation of fd_cyc(T) / fd_cyc(25) from s_temp(T)."""
    base, warm = make(temperature=25.0), make(temperature=float(temperature))
    want = float(s_temp(temperature))
    assert want != 1.0
    hour, minute = np.asarray(tables["hour"]), np.asarray(tables["minute"])
    E, N = base.E, base.N
    base.reset()
    warm.reset()
    rng = np.random.default_rng(seed)
    evaluated = np.zeros(E, bool)
    n_ratio, worst = 0, 0.0
    for s in range(steps):
        t = base.get("time_idx")
        assert np.array_equal(t, warm.get("time_idx")), f"time_idx before step {s}"
        ev = (hour[t + 1] == 14) & (minute[t + 1] == 45)              # this step ends on a 14:45 row: evaluation
        a = actions(rng, s, E, N)
        out_b, out_w = base.step(a), warm.step(a)
        st_b, st_w = base.state(), warm.state()
        _assert_identical(out_b, out_w, st_b, st_w, ~evaluated & ~ev, f"step {s} before the first evaluation")
        first = ev & ~evaluated
        if first.any():
            # the evaluation changes the fade and the SOH it leaves behind, nothing that this step computed before it
            _assert_identical(out_b, out_w, st_b, st_w, first, f"step {s} at the first evaluation",
                              skip=("soh", "fd_cyc", "life", "last_deg"))
            fa, fw = _rows(st_b["fd_cyc"], first), _rows(st_w["fd_cyc"], first)
            nz = fa != 0
            assert bool((fw[~nz] == 0).all()), f"step {s}: cycle fade at {temperature} C without one at 25 C"
            if bool(nz.any()):
                rel = abs(fw[nz] / fa[nz] - want) / want
                worst = max(worst, float(rel.max()))
                n_ratio += int(nz.sum())
        evaluated |= ev
    assert evaluated.all(), "some envs never reached a 14:45 evaluation"
    return dict(n_ratio=n_ratio, worst=worst)


def overload_term(overload, grid):
    """score_config.py:33-41 for the overload of one step (rel >= 1.1), per unit of penalty_overloading."""
    rel = overload / grid + 1
    pen = -700 / (1 + np.exp(-15.77350877 * (rel - 1.33298382)))
    return np.where((overload > 0) & (rel >= 1.1), pen, 0.0)


def invalid_term(tables, t, a):
    """ev_charger.py:120-122,180-182 per unit of penalty_invalid_action: sum of a^2 over absent vehicles with |a| > 0.05."""
    there = np.asarray(tables["there"])[:, t].T                           # [E, N] presence at each env's time
    a64 = a.astype(np.float64)
    return np.where((there == 0) & (np.abs(a64) > 0.05), a64 * a64, 0.0).sum(1)


def check_reward_weights(make, tables, steps, seed=5):
    """make(**over) -> side.  Returns counts of the events the relations were exercised on."""
    base = make()
    c = base.consts
    variants = {}
    for k, d in AFFINE.items():
        for m in (1, 2):
            variants[(k, m)] = make(**{k: getattr(c, k) + m * d})
    for k, v in REWARD_ONLY.items():
        assert getattr(c, k) != v
        variants[(k, "set")] = make(**{k: v})
    sides = [base] + list(variants.values())
    for sd in sides:
        sd.reset()
    E, N = base.E, base.N
    rng = np.random.default_rng(seed)
    n = dict(invalid=0, overload=0, departures=0, price=0)
    r_sum = np.zeros(E)
    for s in range(steps):
        t = base.get("time_idx")
        a = actions(rng, s, E, N)
        outs = [sd.step(a) for sd in sides]
        st0 = base.state()
        r0 = outs[0]["reward"]
        r = {}
        for (key, sd), out in zip(variants.items(), outs[1:]):
            _assert_identical(outs[0], out, st0, sd.state(), np.ones(E, bool), f"step {s}, {key[0]} changed",
                              outputs=("cashflow",))
            r[key] = out["reward"]
        for k, d in AFFINE.items():
            r1, r2 = r[(k, 1)], r[(k, 2)]
            tol = 1e-13 + 4 * N * EPS * (np.abs(r0) + np.abs(r1) + np.abs(r2))
            dev = np.abs((r2 - r0) - 2 * (r1 - r0))
            assert (dev <= tol).all(), f"step {s}: reward not affine in {k} (worst {dev.max():.3g})"
            if k == "penalty_invalid_action":
                want = d * invalid_term(tables, t, a)
            elif k == "penalty_overloading":
                want = d * overload_term(base.get("overload"), c.grid_connection)
            else:
                want = None
            if want is not None:
                dev = np.abs((r1 - r0) - want)
                assert (dev <= tol).all(), f"step {s}: {k} term (worst {dev.max():.3g})"
                n["invalid" if k == "penalty_invalid_action" else "overload"] += int((want != 0).sum())
            elif k == "fully_charged_reward":
                n["departures"] += int((r1 != r0).sum())
            else:
                n["price"] += int((r1 != r0).sum())
        r_sum += r0
    for (key, sd) in [(("base", None), base)] + list(variants.items()):
        st = sd.stats()
        pm = sd.consts.price_multiplier
        if pm == 0:
            assert st["penalty"] == st["reward"], f"{key}: penalty statistic at price_multiplier 0"
        else:
            want = st["reward"] - st["cashflow"] * pm
            assert abs(st["penalty"] - want) <= 1e-12 * max(1.0, abs(st["reward"]), abs(st["cashflow"] * pm)), \
                f"{key}: penalty statistic {st['penalty']!r} != reward - cashflow * price_multiplier {want!r}"
    np.testing.assert_allclose(base.stats()["reward"], r_sum.sum(), rtol=1e-12)
    return n
