"""Device VecNormalize (fleet_norm_*, FleetVecNormalize) against the NumPy restatement of SB3's VecNormalize
(oracle/vec_normalize.py).

Outputs are checked two ways: bit for bit against SB3's formula evaluated in NumPy with the statistics read back from the
device, and within one float32 ulp of the restatement's own outputs (whose statistics agree to rel 1e-12; an absolute
1e-12 covers results so close to 0 that a 1e-16 difference of the statistics exceeds their ulp)."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from fleetrl_b200._lib import FleetNormHandle, FleetStepError
from oracle.vec_normalize import VecNormalize

pytestmark = pytest.mark.gpu

EPS, CLIP = 1e-8, 10.0
DEV = torch.device("cuda", 0)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


class _ArrayVenv:
    """Feeds prepared batches to the restatement like a VecEnv."""

    def __init__(self, E, D):
        self.num_envs = E
        self.observation_space = SimpleNamespace(shape=(D,))
        self.next = None

    def reset(self):
        return self.next

    def step_async(self, actions):
        pass

    def step_wait(self):
        obs, rew, done, term = self.next
        infos = [{"terminal_observation": term[i]} if done[i] else {} for i in range(len(done))]
        return obs, rew, done, infos


def _formula_obs(x, st):
    return np.clip((x - st["obs_mean"]) / np.sqrt(st["obs_var"] + EPS), -CLIP, CLIP).astype(np.float32)


def _formula_rew(r, st):
    return np.clip(r.astype(np.float64) / np.sqrt(st["ret_var"][()] + EPS), -CLIP, CLIP).astype(np.float32)


def _within_ulp(a, b, what):
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    tol = np.spacing(np.maximum(np.abs(a), np.abs(b))).astype(np.float64) + 1e-12
    bad = np.abs(a.astype(np.float64) - b.astype(np.float64)) > tol
    assert not bad.any(), f"{what}: {bad.sum()} elements beyond 1 ulp, first {np.argwhere(bad)[:3].tolist()}"


def _rel(a, b, rtol, what):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=0, err_msg=what)


def _mean_close(a, b, var, rtol, what):
    """Means to rel rtol of the data's scale sqrt(var + mean^2): a mean near 0 has no relative accuracy of its own."""
    b = np.asarray(b, np.float64)
    tol = rtol * np.sqrt(np.asarray(var) + b * b)
    bad = np.abs(np.asarray(a) - b) > tol
    assert not bad.any(), f"{what}: {np.asarray(a)[bad][:3]} vs {b[bad][:3]}"


def _check_stats(st, ref, rtol=1e-12):
    _mean_close(st["obs_mean"], ref.obs_rms.mean, ref.obs_rms.var, rtol, "obs mean")
    _rel(st["obs_var"], ref.obs_rms.var, rtol, "obs var")
    _rel(st["obs_count"][()], ref.obs_rms.count, 1e-15, "obs count")
    _mean_close(st["ret_mean"][()], ref.ret_rms.mean, ref.ret_rms.var, rtol, "ret mean")
    _rel(st["ret_var"][()], ref.ret_rms.var, rtol, "ret var")
    _rel(st["ret_count"][()], ref.ret_rms.count, 1e-15, "ret count")
    _rel(st["returns"], ref.returns, rtol, "returns")


class _Pair:
    """A FleetNormHandle and the restatement fed the same batches."""

    def __init__(self, E, D, **kw):
        self.E, self.D = E, D
        self.h = FleetNormHandle(E, D, 0, **kw)
        self.venv = _ArrayVenv(E, D)
        self.ref = VecNormalize(self.venv, obs_shape=(D,), **kw)
        self.m = torch.zeros(self.h.moments_len, dtype=torch.float64, device=DEV)
        self.out = torch.zeros((E, D), dtype=torch.float32, device=DEV)
        self.tout = torch.zeros((E, D), dtype=torch.float32, device=DEV)
        self.rout = torch.zeros(E, dtype=torch.float32, device=DEV)

    def reset(self, x):
        self.venv.next = x
        want = self.ref.reset()
        xd = _t(x)
        self.h.reset_returns()
        self.h.moments(xd, None, self.m)
        self.h.apply(self.m, xd, self.out)
        st = self.h.get_state()
        got = self.out.cpu().numpy()
        np.testing.assert_array_equal(got, _formula_obs(x, st))
        _within_ulp(got, want, "reset obs")
        return st

    def step(self, x, r, done, term, check=True, rtol=1e-12):
        self.venv.next = (x, r, done, term)
        w_obs, w_rew, _, infos = self.ref.step(None)
        d = _t(done.astype(np.uint8))
        self.h.moments(_t(x), _t(r), self.m)
        self.h.apply(self.m, _t(x), self.out, _t(r), self.rout, d, _t(term), self.tout)
        st = self.h.get_state()
        if check:
            _check_stats(st, self.ref, rtol)
            got, rew, tg = self.out.cpu().numpy(), self.rout.cpu().numpy(), self.tout.cpu().numpy()
            np.testing.assert_array_equal(got, _formula_obs(x, st))
            np.testing.assert_array_equal(rew, _formula_rew(r, st))
            _within_ulp(got, w_obs, "obs")
            _within_ulp(rew, w_rew, "reward")
            idx = np.nonzero(done)[0]
            if len(idx):
                np.testing.assert_array_equal(tg[idx], _formula_obs(term[idx], st))
                _within_ulp(tg[idx], np.stack([infos[i]["terminal_observation"] for i in idx]), "terminal obs")
            assert (st["returns"][idx] == 0).all()
        return st


def _batch(rng, E, D, loc=None, sc=None):
    loc = rng.uniform(-2, 2, D) if loc is None else loc
    sc = rng.uniform(0.1, 3, D) if sc is None else sc
    return (rng.standard_normal((E, D)) * sc + loc).astype(np.float32)


def _step_data(rng, E, D, p_done=0.05, **kw):
    return (_batch(rng, E, D, **kw), (rng.standard_normal(E) * 2 + 0.3).astype(np.float32), rng.random(E) < p_done,
            _batch(rng, E, D, **kw))


@pytest.mark.parametrize("D", [1, 5, 45, 388, 389])
@pytest.mark.parametrize("E", [1, 37, 4099, 65536])
def test_kernel_matches_restatement(E, D):
    rng = np.random.default_rng(E * 1000 + D)
    p = _Pair(E, D)
    p.reset(_batch(rng, E, D))
    for _ in range(2 if E * D > 1e6 else 4):
        p.step(*_step_data(rng, E, D, p_done=0.2))


def test_chained_steps_with_random_done():
    """200 steps over several chunks, returns carried and zeroed by random done flags."""
    rng = np.random.default_rng(7)
    E, D = 1100, 7
    p = _Pair(E, D, gamma=0.95)
    p.reset(_batch(rng, E, D))
    loc, sc = rng.uniform(-1, 1, D), rng.uniform(0.5, 2, D)
    for s in range(200):
        p.step(*_step_data(rng, E, D, p_done=0.03, loc=loc, sc=sc))


def test_constant_columns_and_clipping():
    rng = np.random.default_rng(8)
    E, D = 3000, 9
    p = _Pair(E, D)
    p.reset(_batch(rng, E, D))
    clipped = [0, 0, 0, 0]
    for s in range(6):
        x, r, done, term = _step_data(rng, E, D, p_done=0.1)
        x[:, 2] = 0.25                       # constant columns
        x[:, 5] = -3.0
        out = rng.random((E, D)) < 0.01      # outliers on both sides
        x[out] = np.where(rng.random(out.sum()) < 0.5, 1e3, -1e3).astype(np.float32)
        r[:2], r[2:4] = 1e5, -1e5                # rare large rewards, beyond 10 sd of the returns
        p.step(x, r, done, term)
        got, rew = p.out.cpu().numpy(), p.rout.cpu().numpy()
        clipped = [clipped[0] + (got == CLIP).sum(), clipped[1] + (got == -CLIP).sum(),
                   clipped[2] + (rew == CLIP).sum(), clipped[3] + (rew == -CLIP).sum()]
    assert min(clipped) > 0, clipped


def test_large_offset_small_spread():
    """Mean 1e4, sd 1e-2.  The moments are sums about K = the running mean, so once the statistics are near the data
    they keep full precision.  From the 1e-4 prior (K = 0) the first update cancels: its variance agrees to rel 1e-6."""
    rng = np.random.default_rng(9)
    E, D = 4099, 6
    loc, sc = 1e4 + rng.uniform(-1, 1, D), np.full(D, 1e-2)
    p = _Pair(E, D)
    p.reset(_batch(rng, E, D, loc=loc, sc=sc))
    _check_stats(p.h.get_state(), p.ref, rtol=1e-6)
    # continue from the restatement's statistics: the steady state of a run
    st = dict(obs_mean=p.ref.obs_rms.mean, obs_var=p.ref.obs_rms.var, obs_count=np.float64(p.ref.obs_rms.count))
    p.h.set_state(**st)
    for s in range(5):
        p.step(*_step_data(rng, E, D, loc=loc, sc=sc))


def test_deterministic():
    rng = np.random.default_rng(10)
    E, D = 65536, 45
    hs = [FleetNormHandle(E, D, 0) for _ in range(2)]
    m = torch.zeros(hs[0].moments_len, dtype=torch.float64, device=DEV)
    out = torch.zeros((E, D), dtype=torch.float32, device=DEV)
    rout = torch.zeros(E, dtype=torch.float32, device=DEV)
    data = [_step_data(rng, E, D) for _ in range(4)]
    for h in hs:
        for x, r, done, term in data:
            h.moments(_t(x), _t(r), m)
            h.apply(m, _t(x), out, _t(r), rout, _t(done.astype(np.uint8)))
    a, b = hs[0].get_state(), hs[1].get_state()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


def test_sharded_moments_add():
    """Two objects over the halves of a batch, their moments vectors added in place of the all-reduce, hold the statistics
    of one object over the whole batch."""
    rng = np.random.default_rng(11)
    E, D = 10000, 33
    E1 = 4321
    whole = FleetNormHandle(E, D, 0)
    halves = [FleetNormHandle(E1, D, 0), FleetNormHandle(E - E1, D, 0)]
    mw = torch.zeros(whole.moments_len, dtype=torch.float64, device=DEV)
    mh = [torch.zeros_like(mw) for _ in range(2)]
    sl = [slice(0, E1), slice(E1, E)]
    for s in range(5):
        x, r, done, term = _step_data(rng, E, D, p_done=0.1)
        ow, rw = torch.zeros((E, D), device=DEV), torch.zeros(E, device=DEV)
        whole.moments(_t(x), _t(r), mw)
        whole.apply(mw, _t(x), ow, _t(r), rw, _t(done.astype(np.uint8)))
        for h, m, q in zip(halves, mh, sl):
            h.moments(_t(x[q]), _t(r[q]), m)
        total = mh[0] + mh[1]
        for h, q in zip(halves, sl):
            o, ro = torch.zeros((q.stop - q.start, D), device=DEV), torch.zeros(q.stop - q.start, device=DEV)
            h.apply(total, _t(x[q]), o, _t(r[q]), ro, _t(done[q].astype(np.uint8)))
            _within_ulp(o.cpu().numpy(), ow[q].cpu().numpy(), "sharded obs")
            _within_ulp(ro.cpu().numpy(), rw[q].cpu().numpy(), "sharded reward")
        sw, s0, s1 = whole.get_state(), halves[0].get_state(), halves[1].get_state()
        for k in ("obs_mean", "obs_var", "obs_count", "ret_mean", "ret_var", "ret_count"):
            np.testing.assert_array_equal(s0[k], s1[k], err_msg=k)
        for k in ("obs_var", "obs_count", "ret_var", "ret_count"):
            _rel(s0[k], sw[k], 1e-12, k)
        _mean_close(s0["obs_mean"], sw["obs_mean"], sw["obs_var"], 1e-12, "obs mean")
        _mean_close(s0["ret_mean"], sw["ret_mean"], sw["ret_var"], 1e-12, "ret mean")
        _rel(np.concatenate([s0["returns"], s1["returns"]]), sw["returns"], 1e-15, "returns")


# ---------------------------------------------------------------- FleetVecNormalize over FleetVecEnv, end to end

def _inputs():
    from fleetrl_b200.schedule import generate_schedule, synthetic_series
    from fleetrl_b200.tables import FleetInputs
    sched = generate_schedule("lmd", 6, start="2020-01-01 00:00", end="2020-03-31 23:59", seed=11)
    price, tariff, load, pv = synthetic_series(start="2020-01-01 00:00", end="2020-03-31 23:59")
    return FleetInputs(sched, price, tariff, load, pv)


class _OracleVenv:
    """OracleFleet as the VecEnv the restatement wraps: float32 rewards, like FleetVecEnv."""

    def __init__(self, orc):
        self.orc, self.num_envs = orc, orc.E
        self.observation_space = SimpleNamespace(shape=(orc.D,))

    def reset(self):
        return self.orc.reset()

    def step_async(self, actions):
        self.a = actions

    def step_wait(self):
        obs, rew, _, done, term = self.orc.step(self.a, want_terminal=True)
        done = done.astype(bool)
        return obs, rew.astype(np.float32), done, [{"terminal_observation": term[i]} if done[i] else {} for i in range(len(done))]


def _make(output, E=48, **kw):
    from fleetrl_b200 import FleetVecEnv, FleetVecNormalize
    from fleetrl_b200.config import default_config
    from oracle.oracle import OracleFleet
    cfg = default_config("lmd", time_picker="random", end_cutoff=10)
    env = FleetVecEnv(cfg, E, inputs=_inputs(), output=output, env_id_offset=77, seed=3)
    orc = OracleFleet(env.built.consts, env.built.tables, E, env_id_offset=77)
    return FleetVecNormalize(env, **kw), VecNormalize(_OracleVenv(orc), obs_shape=(env.obs_dim,), **kw), orc


def _np(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


@pytest.mark.parametrize("output", ["torch", "numpy"])
def test_wrapper_end_to_end(output):
    E, N = 48, 6
    vn, ref, orc = _make(output)
    assert vn.training and vn.norm_obs and vn.norm_reward
    _within_ulp(_np(vn.reset()), ref.reset(), "reset obs")
    np.testing.assert_array_equal(_np(vn.get_original_obs()), ref.get_original_obs())
    rng = np.random.default_rng(0)
    n_done = 0
    for s in range(200):
        a = rng.uniform(-1, 1, (E, N)).astype(np.float32)
        obs, rew, done, infos = vn.step(a if output == "numpy" else torch.from_numpy(a).to(DEV))
        w_obs, w_rew, w_done, w_infos = ref.step(a)
        assert isinstance(obs, np.ndarray) == (output == "numpy")
        np.testing.assert_array_equal(_np(done), w_done)
        np.testing.assert_array_equal(_np(vn.get_original_obs()), ref.get_original_obs())   # raw obs, bit for bit
        _within_ulp(_np(obs), w_obs, f"obs step {s}")
        np.testing.assert_allclose(_np(rew), w_rew, rtol=1e-5, atol=1e-6)   # raw f32 rewards may differ by an ulp
        np.testing.assert_allclose(_np(vn.get_original_reward()), ref.get_original_reward(), rtol=1e-6, atol=1e-6)
        st = vn.handle.get_state()
        _mean_close(st["obs_mean"], ref.obs_rms.mean, ref.obs_rms.var, 1e-12, "obs mean")
        _rel(st["obs_var"], ref.obs_rms.var, 1e-12, "obs var")
        np.testing.assert_allclose(st["returns"], ref.returns, rtol=1e-5, atol=1e-6)
        for i in np.nonzero(w_done)[0]:
            _within_ulp(_np(infos[int(i)]["terminal_observation"]), w_infos[i]["terminal_observation"], "terminal obs")
            np.testing.assert_allclose(infos[int(i)]["episode"]["r"], orc.get("last_ep_return")[i], rtol=1e-11)   # raw
            assert st["returns"][i] == 0.0
            n_done += 1
        assert vn.env_method("is_done", indices=[0, 1]) == [bool(w_done[0]), bool(w_done[1])]
    assert n_done >= 2 * E
    np.testing.assert_allclose(vn.ret_rms.var, ref.ret_rms.var, rtol=1e-5)
    assert vn.get_attr("num_cars", indices=[0]) == [N]
    vn.close()


def test_frozen_statistics_and_raw_rewards():
    E, N = 48, 6
    vn, ref, _ = _make("torch")
    vn.reset(); ref.reset()
    rng = np.random.default_rng(1)
    for s in range(20):
        a = rng.uniform(-1, 1, (E, N)).astype(np.float32)
        vn.step(torch.from_numpy(a).to(DEV)); ref.step(a)
    vn.training = ref.training = False
    vn.norm_reward = ref.norm_reward = False
    before = vn.state_dict()
    for s in range(30):
        a = rng.uniform(-1, 1, (E, N)).astype(np.float32)
        obs, rew, done, _ = vn.step(torch.from_numpy(a).to(DEV))
        w_obs, w_rew, _, _ = ref.step(a)
        assert torch.equal(rew, vn.get_original_reward())                 # norm_reward=False: raw rewards
        _within_ulp(obs.cpu().numpy(), w_obs, "frozen obs")
    after = vn.state_dict()
    for k in ("obs_mean", "obs_var", "obs_count", "ret_mean", "ret_var", "ret_count"):
        np.testing.assert_array_equal(after[k], before[k], err_msg=k)
    # loading saved statistics from any object with mean / var / count
    D = vn.handle.D
    rng2 = np.random.default_rng(2)
    saved = SimpleNamespace(mean=rng2.normal(0, 1, D), var=rng2.uniform(0.1, 2, D), count=1234.5)
    vn.obs_rms = saved
    ref.obs_rms.mean, ref.obs_rms.var, ref.obs_rms.count = saved.mean, saved.var, saved.count
    np.testing.assert_array_equal(vn.obs_rms.mean, saved.mean)
    assert vn.obs_rms.count == 1234.5
    x = rng2.normal(0, 1, (5, D)).astype(np.float32)
    np.testing.assert_array_equal(vn.normalize_obs(x), ref.normalize_obs(x))
    vn.ret_rms = SimpleNamespace(mean=0.5, var=4.0, count=10.0)
    vn.norm_reward = ref.norm_reward = True
    ref.ret_rms.var = np.float64(4.0)
    r = rng2.normal(0, 50, 17).astype(np.float32)
    np.testing.assert_array_equal(vn.normalize_reward(r), ref.normalize_reward(r).astype(np.float32))
    vn.close()


def test_state_dict_resumes_bit_for_bit():
    from fleetrl_b200 import FleetVecEnv, FleetVecNormalize
    from fleetrl_b200.config import default_config
    E, N = 32, 6
    cfg = default_config("lmd", time_picker="random", end_cutoff=10)
    inputs = _inputs()
    mk = lambda: FleetVecNormalize(FleetVecEnv(cfg, E, inputs=inputs, output="torch", env_id_offset=9, seed=3))
    a = mk()
    a.reset()
    rng = np.random.default_rng(6)
    acts = [torch.from_numpy(rng.uniform(-1, 1, (E, N)).astype(np.float32)).to(DEV) for _ in range(240)]
    for s in range(130):
        a.step(acts[s])
    env_sd, norm_sd = a.venv.state_dict(), a.state_dict()
    b = mk()
    b.venv.load_state_dict(env_sd)
    b.load_state_dict(norm_sd)
    for s in range(130, 240):
        oa, ra, da, _ = a.step(acts[s])
        ob, rb, db, _ = b.step(acts[s])
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db), f"step {s}"
        idx = da.nonzero().flatten()                     # rows of running envs keep older terminal rows
        assert torch.equal(a.terminal_observations[idx], b.terminal_observations[idx])
    sa, sb = a.state_dict(), b.state_dict()
    for k in sa:
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)
    a.close(); b.close()


def test_unaligned_views_leave_neighbours_untouched():
    rng = np.random.default_rng(12)
    E, D = 37, 5
    x, r, done, term = _step_data(rng, E, D, p_done=0.3)
    ref = _Pair(E, D)
    ref.reset(x)
    ref.step(x, r, done, term, check=False)
    h = FleetNormHandle(E, D, 0)
    sentinel = np.float32(-777.25)
    bufs = {k: torch.full((E * D + 2,), float(sentinel), device=DEV) for k in ("x", "out", "term", "tout")}
    bufs["x"][1:1 + E * D] = _t(x.ravel()); bufs["term"][1:1 + E * D] = _t(term.ravel())
    v = {k: b[1:1 + E * D].view(E, D) for k, b in bufs.items()}
    assert all(t.data_ptr() % 16 for t in v.values())
    m = torch.zeros(h.moments_len, dtype=torch.float64, device=DEV)
    rout = torch.zeros(E, dtype=torch.float32, device=DEV)
    h.moments(v["x"], None, m)
    h.apply(m, v["x"], v["out"])
    h.moments(v["x"], _t(r), m)
    h.apply(m, v["x"], v["out"], _t(r), rout, _t(done.astype(np.uint8)), v["term"], v["tout"])
    assert torch.equal(v["out"], ref.out) and torch.equal(rout, ref.rout)
    idx = np.nonzero(done)[0]
    tout = v["tout"].cpu().numpy()
    np.testing.assert_array_equal(tout[idx], ref.tout.cpu().numpy()[idx])
    assert (tout[~done] == sentinel).all()                              # rows of running envs untouched
    for k, b in bufs.items():
        assert b[0].item() == sentinel and b[-1].item() == sentinel, k
    np.testing.assert_array_equal(v["x"].cpu().numpy(), x)                # raw obs intact


@pytest.mark.parametrize("kw", [dict(E=0), dict(D=0), dict(clip_obs=0.0), dict(clip_reward=-1.0), dict(gamma=1.5),
                                dict(gamma=-0.1), dict(epsilon=-1e-9), dict(clip_obs=float("nan"))])
def test_bad_arguments_raise(kw):
    args = dict(E=4, D=3)
    args.update(kw)
    E, D = args.pop("E"), args.pop("D")
    with pytest.raises(FleetStepError):
        FleetNormHandle(E, D, 0, **args)


def test_bad_buffers_raise():
    h = FleetNormHandle(8, 3, 0)
    m = torch.zeros(h.moments_len, dtype=torch.float64, device=DEV)
    x = torch.zeros((8, 3), device=DEV)
    with pytest.raises(FleetStepError):
        h.moments(x.double(), None, m)
    with pytest.raises(FleetStepError):
        h.apply(m, x[:4].contiguous(), torch.zeros((4, 3), device=DEV))     # an update needs all E rows
    with pytest.raises(FleetStepError):
        h.apply(None, x, None)                                              # output missing
    out = torch.zeros((4, 3), device=DEV)
    h.apply(None, x[:4].contiguous(), out)                                  # normalise-only works on any row count
