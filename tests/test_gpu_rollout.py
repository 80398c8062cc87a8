"""Device RolloutBuffer (fleet_rollout_*, FleetRolloutBuffer, collect_rollouts) against the NumPy restatement of SB3's
RolloutBuffer and collect_rollouts loop (oracle/rollout_buffer.py).  Every comparison is bit for bit: float arrays are
compared as their uint32 patterns, so even the sign of a zero counts."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from fleetrl_b200._lib import FleetStepError
from fleetrl_b200.rollout import FleetRolloutBuffer, collect_rollouts
from oracle import rollout_buffer as ref

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _bits_equal(got, want, what):
    g = np.ascontiguousarray(got.cpu().numpy() if isinstance(got, torch.Tensor) else got, dtype=np.float32)
    w = np.ascontiguousarray(want, dtype=np.float32)
    assert g.shape == w.shape, f"{what}: shape {g.shape} vs {w.shape}"
    bad = g.view(np.uint32) != w.view(np.uint32)
    assert not bad.any(), f"{what}: {bad.sum()} of {bad.size} differ, first at {np.argwhere(bad)[:3].tolist()}"


def _random_fill(rng, T, E, p_start=0.1):
    """rewards, values, episode_starts [T, E], last_values, dones [E]: float32, with random episode starts and dones."""
    rew = (rng.standard_normal((T, E)) * 2).astype(np.float32)
    val = rng.standard_normal((T, E)).astype(np.float32)
    starts = (rng.random((T, E)) < p_start).astype(np.float32)
    starts[0] = 1.0
    return rew, val, starts, rng.standard_normal(E).astype(np.float32), rng.random(E) < 0.2


# ---------------------------------------------------------------- GAE

@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (0.99, 1.0), (1.0, 1.0), (0.0, 0.5)])
@pytest.mark.parametrize("E", [1, 33, 1000, 65536])
@pytest.mark.parametrize("T", [1, 2, 64])
def test_gae_bit_for_bit(T, E, gamma, lam):
    rng = np.random.default_rng(T * 100003 + E)
    rew, val, starts, lv, dones = _random_fill(rng, T, E)
    buf = FleetRolloutBuffer(T, E, 1, 1, DEV, gamma=gamma, gae_lambda=lam)
    buf.rewards.copy_(_t(rew)); buf.values.copy_(_t(val)); buf.episode_starts.copy_(_t(starts))
    buf.pos, buf.full = T, True
    buf.compute_returns_and_advantage(_t(lv), _t(dones))
    o = ref.RolloutBuffer(T, 1, 1, gae_lambda=lam, gamma=gamma, n_envs=E)
    o.rewards[...], o.values[...], o.episode_starts[...] = rew, val, starts
    o.full = True
    o.compute_returns_and_advantage(lv, dones)
    _bits_equal(buf.advantages, o.advantages, "advantages")
    _bits_equal(buf.returns, o.returns, "returns")


def test_gae_input_forms():
    """last_values [E, 1] and dones as bool, uint8 or float give the same result."""
    rng = np.random.default_rng(3)
    T, E = 5, 77
    rew, val, starts, lv, dones = _random_fill(rng, T, E)
    buf = FleetRolloutBuffer(T, E, 1, 1, DEV, gamma=0.9, gae_lambda=0.8)
    buf.rewards.copy_(_t(rew)); buf.values.copy_(_t(val)); buf.episode_starts.copy_(_t(starts))
    buf.pos, buf.full = T, True
    outs = []
    for lvt, dt in ((_t(lv), _t(dones)), (_t(lv[:, None]), _t(dones.astype(np.uint8))), (_t(lv), _t(dones.astype(np.float32)))):
        buf.compute_returns_and_advantage(lvt, dt)
        outs.append(buf.advantages.clone())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


# ---------------------------------------------------------------- add

def _transition(rng, E, D, N, start_dtype):
    start = rng.random(E) < 0.3
    start_t = {"bool": _t(start), "uint8": _t(start.astype(np.uint8)), "float32": _t(start.astype(np.float32)),
               "float64": _t(start.astype(np.float64))}[start_dtype]
    return dict(obs=rng.standard_normal((E, D)).astype(np.float32), action=(rng.standard_normal((E, N)) * 2).astype(np.float32),
                reward=rng.standard_normal(E).astype(np.float32), start=start, start_t=start_t,
                value=rng.standard_normal((E, 1)).astype(np.float32), log_prob=rng.standard_normal(E).astype(np.float32))


@pytest.mark.parametrize("start_dtype", ["bool", "uint8", "float32", "float64"])
@pytest.mark.parametrize("E,D,N", [(33, 375, 50), (64, 388, 50), (1000, 45, 7), (1, 1, 1)])
def test_add_slots_bit_for_bit(E, D, N, start_dtype):
    """Slot contents equal SB3's add.  D = 375 with E = 33 puts slots and rows off 16-byte boundaries; the obs are also
    passed as a view one float into an allocation."""
    rng = np.random.default_rng(E * 7 + D)
    T = 3
    buf = FleetRolloutBuffer(T, E, D, N, DEV)
    o = ref.RolloutBuffer(T, D, N, n_envs=E)
    for t in range(T):
        x = _transition(rng, E, D, N, start_dtype)
        raw = torch.zeros(E * D + 1, device=DEV)
        raw[1:] = _t(x["obs"].ravel())
        obs = raw[1:].view(E, D) if t == 1 else _t(x["obs"])
        reward = _t(x["reward"].astype(np.float64)) if t == 2 else _t(x["reward"])   # float64 is cast, as SB3 does
        buf.add(obs, _t(x["action"]), reward, x["start_t"], _t(x["value"]), _t(x["log_prob"]))
        o.add(x["obs"], x["action"], x["reward"], x["start"], x["value"], x["log_prob"])
    assert buf.full and buf.pos == T
    for name in ("observations", "actions", "rewards", "episode_starts", "values", "log_probs"):
        _bits_equal(getattr(buf, name), getattr(o, name), name)


def test_add_error_paths():
    E, D, N, T = 8, 5, 3, 2
    buf = FleetRolloutBuffer(T, E, D, N, DEV)
    rng = np.random.default_rng(0)
    x = _transition(rng, E, D, N, "bool")
    args = [_t(x["obs"]), _t(x["action"]), _t(x["reward"]), x["start_t"], _t(x["value"]), _t(x["log_prob"])]

    def bad(i, v):
        a = list(args)
        a[i] = v
        with pytest.raises(FleetStepError):
            buf.add(*a)
        assert buf.pos == 0

    bad(0, torch.from_numpy(x["obs"]))                                  # host tensor
    bad(0, _t(x["obs"])[:, :4].contiguous())                            # shape
    bad(0, _t(x["obs"]).t().contiguous().t())                          # not contiguous
    bad(1, _t(x["action"].T.copy()).t())                                # not contiguous
    bad(2, _t(x["reward"][:-1]))                                        # shape
    bad(3, x["start_t"].to(torch.int32))                                # neither a flag nor a float
    bad(4, x["value"])                                                  # not a tensor
    buf.add(*args)
    buf.add(*args)
    with pytest.raises(FleetStepError):
        buf.add(*args)                                                  # full
    buf.reset()
    assert buf.pos == 0 and not buf.full
    with pytest.raises(FleetStepError):
        buf._write(T, obs=args[0])                                      # slot outside the buffer (C side)
    for kw in (dict(gamma=1.5), dict(gae_lambda=-0.1), dict(gamma=float("nan"))):
        with pytest.raises(FleetStepError):
            FleetRolloutBuffer(T, E, D, N, DEV, **kw)
    with pytest.raises(FleetStepError):
        FleetRolloutBuffer(0, E, D, N, DEV)


def test_not_full_raises():
    buf = FleetRolloutBuffer(2, 4, 3, 2, DEV)
    with pytest.raises(FleetStepError):
        buf.compute_returns_and_advantage(torch.zeros(4, device=DEV), torch.zeros(4, dtype=torch.bool, device=DEV))
    with pytest.raises(FleetStepError):
        next(buf.get(2))


def test_c_entry_points_reject_bad_input():
    buf = FleetRolloutBuffer(2, 4, 3, 2, DEV)
    lib, d = buf.lib, buf._desc
    z = torch.zeros(4, device=DEV)
    u = torch.zeros(4, dtype=torch.uint8, device=DEV)
    assert lib.fleet_rollout_gae(C.byref(d), 1.5, 0.9, z.data_ptr(), u.data_ptr(), None) == -1
    assert b"gamma" in lib.fleet_rollout_last_error()
    assert lib.fleet_rollout_gae(C.byref(d), 0.9, 2.0, z.data_ptr(), u.data_ptr(), None) == -1
    assert lib.fleet_rollout_gae(C.byref(d), 0.9, 0.9, None, u.data_ptr(), None) == -1
    assert lib.fleet_rollout_gather(C.byref(d), None, -1, *([None] * 7)) == -1
    assert lib.fleet_rollout_add(C.byref(d), -1, z.data_ptr(), *([None] * 6)) == -1
    empty = type(d)(2, 4, 3, 2, *([None] * 8))
    assert lib.fleet_rollout_add(C.byref(empty), 0, *([None] * 7)) == -1
    assert b"NULL" in lib.fleet_rollout_last_error()
    zero = type(d)(2, 0, 3, 2, *[getattr(d, f) for f, _ in d._fields_[4:]])
    assert lib.fleet_rollout_gae(C.byref(zero), 0.9, 0.9, z.data_ptr(), u.data_ptr(), None) == -1
    assert lib.fleet_rollout_gather(C.byref(d), None, 0, *([None] * 7)) == 0     # nothing to gather


# ---------------------------------------------------------------- get

def _filled_pair(rng, T, E, D, N, gamma=0.99, lam=0.95):
    buf = FleetRolloutBuffer(T, E, D, N, DEV, gamma=gamma, gae_lambda=lam)
    o = ref.RolloutBuffer(T, D, N, gae_lambda=lam, gamma=gamma, n_envs=E)
    for t in range(T):
        x = _transition(rng, E, D, N, "bool")
        if t == 0:
            x["start"][:] = True
            x["start_t"] = _t(x["start"])
        buf.add(_t(x["obs"]), _t(x["action"]), _t(x["reward"]), x["start_t"], _t(x["value"]), _t(x["log_prob"]))
        o.add(x["obs"], x["action"], x["reward"], x["start"], x["value"], x["log_prob"])
    lv, dones = rng.standard_normal(E).astype(np.float32), rng.random(E) < 0.2
    buf.compute_returns_and_advantage(_t(lv), _t(dones))
    o.compute_returns_and_advantage(lv, dones)
    return buf, o


@pytest.mark.parametrize("T,E,D,N", [(7, 33, 388, 50), (5, 40, 375, 50), (3, 1, 6, 2)])
def test_get_with_indices_bit_for_bit(T, E, D, N):
    rng = np.random.default_rng(T * E + D)
    buf, o = _filled_pair(rng, T, E, D, N)
    perm = rng.permutation(T * E)
    bs = 37 if T * E > 37 else 2
    assert (T * E) % bs
    got = list(buf.get(bs, indices=perm))
    want = list(o.get(bs, indices=perm))
    assert len(got) == len(want) and got[-1].observations.shape[0] == (T * E) % bs
    for g, w in zip(got, want):
        for name, gv, wv in zip(g._fields, g, w):
            _bits_equal(gv, wv, name)
    assert buf.observations.shape == (T, E, D)       # the [T, E, ...] layout stays after get()
    with pytest.raises(FleetStepError):
        next(buf.get(bs, indices=np.arange(T * E) + 1))
    with pytest.raises(FleetStepError):
        next(buf.get(bs, indices=np.arange(T * E - 1)))


def test_randperm_covers_each_index_once():
    T, E, D, N = 16, 300, 4, 2
    buf = FleetRolloutBuffer(T, E, D, N, DEV)
    buf.pos, buf.full = T, True
    tag = torch.arange(T * E, dtype=torch.float32, device=DEV).view(E, T).t().contiguous()   # flat k -> k
    buf.log_probs.copy_(tag)
    buf.observations.copy_(tag[:, :, None].expand(T, E, D))
    g = torch.Generator(device=DEV)
    g.manual_seed(5)
    orders = []
    for epoch in range(2):
        batches = list(buf.get(1000, generator=g))
        assert [b.old_log_prob.shape[0] for b in batches] == [1000] * 4 + [800]
        k = torch.cat([b.old_log_prob for b in batches])
        assert torch.equal(torch.sort(k).values, torch.arange(T * E, dtype=torch.float32, device=DEV))
        for b in batches:
            assert torch.equal(b.observations, b.old_log_prob[:, None].expand(-1, D))
        orders.append(k)
    assert not torch.equal(orders[0], orders[1])
    (whole,) = list(buf.get())
    assert whole.observations.shape == (T * E, D)


# ---------------------------------------------------------------- end to end over FleetVecNormalize

class _Policy:
    """Deterministic elementwise policy; actions exceed +-1 for part of the entries."""

    def __init__(self, N):
        self.N, self.calls = N, []

    def predict_values(self, obs):
        return obs[:, :8].sum(1, keepdim=True) * 0.1

    def forward(self, obs):
        a = torch.tanh(obs[:, :self.N] * 0.7 + 0.1) * 1.8
        out = (a, self.predict_values(obs), -0.5 * (a * a).sum(1))
        self.calls.append(out)
        return out


def _fleet(E=512, N=10):
    from synth_tables import make_consts, make_tables
    from fleetrl_b200 import FleetVecEnv, FleetVecNormalize
    tables, Tt = make_tables(n_evs=N, days=12, seed=7)
    consts = make_consts(tables, Tt, N)
    env = FleetVecEnv(None, E, built=SimpleNamespace(consts=consts, tables=tables, rc=None), output="torch")
    vn = FleetVecNormalize(env)
    obs = vn.reset()
    # de-phase the episodes (env e is e mod L steps into its episode) so that dones fall inside the rollout
    L = int(consts.episode_steps)
    phase = torch.arange(E, device=DEV) % L
    a = torch.full((E, N), 0.3, device=DEV)
    for s in range(L):
        obs, _, _ = vn.step_raw(a)
        env.handle.reset(mask=(phase == s).to(torch.uint8), obs=env._obs)
    obs, _, _ = vn.step_raw(a)
    return env, vn, obs


def test_collect_rollouts_matches_restated_loop():
    E, N, T = 512, 10, 40
    env_a, vn_a, obs_a = _fleet(E, N)
    env_b, vn_b, obs_b = _fleet(E, N)
    assert torch.equal(obs_a, obs_b)
    D = env_a.obs_dim
    pol = _Policy(N)
    buf = FleetRolloutBuffer(T, E, D, N, DEV, gamma=0.98, gae_lambda=0.95)
    ones = torch.ones(E, dtype=torch.bool, device=DEV)
    last_obs, last_starts = collect_rollouts(vn_a, pol, buf, obs_a, ones)
    assert buf.full and len(pol.calls) == T

    # the same env stepped through the restated loop, fed the same policy outputs
    k, rewards, dones_seq = [0], [], []

    def policy_np(obs):
        out = [x.cpu().numpy() for x in pol.calls[k[0]]]
        k[0] += 1
        return out

    def env_step(a):
        o, r, d = vn_b.step_raw(_t(a))
        rewards.append(r.cpu().numpy().copy())
        dones_seq.append(d.cpu().numpy().astype(bool))
        return o.cpu().numpy().copy(), r.cpu().numpy().copy(), dones_seq[-1], [{"TimeLimit.truncated": False}] * E

    o = ref.RolloutBuffer(T, D, N, gae_lambda=0.95, gamma=0.98, n_envs=E)
    o_last, o_starts = ref.collect_rollouts(env_step, policy_np, lambda x: pol.predict_values(_t(x)).cpu().numpy(), o, T,
                                            obs_b.cpu().numpy(), np.ones(E, bool), gamma=0.98)
    for name in ("observations", "actions", "rewards", "episode_starts", "values", "log_probs", "advantages", "returns"):
        _bits_equal(getattr(buf, name), getattr(o, name), name)
    _bits_equal(last_obs, o_last, "last obs")
    np.testing.assert_array_equal(last_starts.cpu().numpy().astype(bool), o_starts)

    starts = buf.episode_starts.cpu().numpy()
    assert (starts[0] == 1).all()
    for t in range(1, T):
        np.testing.assert_array_equal(starts[t], dones_seq[t - 1].astype(np.float32))
    n_done = sum(int(d.sum()) for d in dones_seq[:-1])
    assert n_done >= E // 4, n_done                               # episodes end inside the rollout
    acts = buf.actions.cpu().numpy()
    assert (np.abs(acts) > 1).any()                                # stored unclipped
    for t in range(T):
        d = dones_seq[t]
        _bits_equal(buf.rewards[t].cpu().numpy()[d], rewards[t][d], f"rewards at done envs, step {t}")   # no bootstrap term


def test_collect_rollouts_does_not_synchronise():
    E, N, T = 512, 10, 8
    env, vn, obs = _fleet(E, N)
    buf = FleetRolloutBuffer(T, E, env.obs_dim, N, DEV)
    pol = _Policy(N)
    starts = torch.ones(E, dtype=torch.bool, device=DEV)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        obs, starts = collect_rollouts(vn, pol, buf, obs, starts)
        obs, starts = collect_rollouts(vn, pol, buf, obs, starts)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert buf.full and torch.isfinite(buf.returns).all()


# ---------------------------------------------------------------- 64-bit offsets

def test_offsets_past_2_31_elements():
    """One buffer of 85 x 65 536 x 388 floats (8.6 GB): the last slot's add and a gather of its rows."""
    T, E, D, N = 85, 65536, 388, 2
    assert T * E * D > 2 ** 31
    buf = FleetRolloutBuffer(T, E, D, N, DEV)
    try:
        g = torch.Generator(device=DEV)
        g.manual_seed(1)
        obs = torch.randn((E, D), device=DEV, generator=g)
        act = torch.randn((E, N), device=DEV, generator=g)
        val = torch.randn(E, device=DEV, generator=g)
        buf.pos = T - 1
        buf.add(obs, act, val * 2, torch.zeros(E, dtype=torch.bool, device=DEV), val, -val)
        assert buf.full
        assert torch.equal(buf.observations[T - 1], obs) and torch.equal(buf.actions[T - 1], act)
        assert torch.equal(buf.log_probs[T - 1], -val)
        envs = torch.tensor([0, 1, E - 2, E - 1], device=DEV)
        s = buf._get_samples(envs * T + (T - 1))                     # flat index of (env, step T-1)
        assert torch.equal(s.observations, obs[envs]) and torch.equal(s.actions, act[envs])
        assert torch.equal(s.old_values, val[envs]) and torch.equal(s.old_log_prob, -val[envs])
        s0 = buf._get_samples(torch.tensor([(E - 1) * T], device=DEV))   # a row of slot 0 is still zero
        assert not s0.observations.any()
    finally:
        del buf
        torch.cuda.empty_cache()
