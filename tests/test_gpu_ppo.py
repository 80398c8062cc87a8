"""fleet_ppo_* (the PPO loss kernels), ppo_loss, FleetMlpPolicy and ppo_train against the float64 restatement of SB3's
PPO (oracle/ppo.py), on the same float32 inputs.

Tolerances.  The kernels compute every element-wise term in float32 (u = 2^-24) and every sum in float64, so the error
of a result is the first-order propagation of the float32 roundings of each row; the float64 sums add nothing visible.
_bounds() writes that propagation out per row from the oracle's float64 intermediates:
  * log_prob: each of the N terms -(a-mu)^2/(2 sigma^2) - log sigma - log sqrt(2 pi) takes <= 4 roundings of its largest
    part plus the error of expf / logf (<= 2 ulp each) on sigma, and the float64 sum is rounded once:
    e_lp = u (|lp| + 4 sum_n (|t_n| + 2));
  * log_ratio = lp - old_log_prob rounds once more, ratio = expf(log_ratio) adds <= 2 ulp:
    e_lr = e_lp + u |lp - old|,  e_r = r (e_lr + 2u);
  * the normalised advantage (A - m) / (s + 1e-8) takes three roundings, and m, s are rounded to float32:
    e_adv = 4u |A_hat| + 2u (|m| + |A|) / s;
  * each statistic and gradient then follows from its derivative w.r.t. these; see _bounds.
Where a ratio or a value difference lies near a clip bound, a rounding could flip the branch; the inputs are drawn with
a margin of 1e-3 around every bound (far above e_r), so every branch is the oracle's and clip_fraction is exact.
The bounds are worst cases (all roundings aligned) and doubled for the second-order terms; the target of 1e-5 relative
holds wherever e_lp is below it, which is the case for N <= 50 rows of the drawn magnitudes."""
import ctypes as C
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from fleetrl_b200._lib import FleetPpoBatch, FleetPpoParams, FleetStepError, load_library
from fleetrl_b200.ppo import STATS, FleetMlpPolicy, log_prob, ppo_loss, ppo_train
from fleetrl_b200.rollout import FleetRolloutBuffer, RolloutBufferSamples, collect_rollouts
from oracle import ppo as ref

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
U = 2.0 ** -24
F64 = torch.float64
LSP = math.log(math.sqrt(2 * math.pi))
MARGIN = 1e-3


def draw(rng, B, N, clip_range=0.2, clip_range_vf=0.5):
    """float32 inputs: about a third of the ratios outside [1 - eps, 1 + eps], about a third of the value clips active,
    and no ratio or value difference within MARGIN of a bound (as the oracle computes them from these float32 inputs)."""
    f = np.float32
    log_std = rng.uniform(-1.0, 0.3, N).astype(f)
    mean = rng.standard_normal((B, N)).astype(f)
    actions = (mean + np.exp(log_std) * rng.standard_normal((B, N))).astype(f)
    lp = ref.log_prob(torch.from_numpy(mean).double(), torch.from_numpy(log_std).double(),
                      torch.from_numpy(actions).double()).numpy()
    delta = rng.normal(0, 0.2, B)
    for _ in range(20):
        old = (lp - delta).astype(f)
        r = np.exp(lp - old.astype(np.float64))
        near = (np.abs(r - (1 - clip_range)) < MARGIN) | (np.abs(r - (1 + clip_range)) < MARGIN)
        if not near.any():
            break
        delta[near] += 3 * MARGIN
    values = rng.standard_normal(B).astype(f)
    dv = rng.normal(0, 0.5, B)
    for _ in range(20):
        old_v = (values - dv).astype(f)
        near = np.abs(np.abs(values.astype(np.float64) - old_v) - clip_range_vf) < MARGIN
        if not near.any():
            break
        dv[near] += 3 * MARGIN
    adv = rng.normal(0.3, 1.5, B).astype(f)
    ret = (values + rng.standard_normal(B)).astype(f)
    return dict(mean=mean, log_std=log_std, values=values, actions=actions, old_log_prob=old, old_values=old_v,
                advantages=adv, returns=ret)


def to_dev(x):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(DEV) for k, v in x.items()}


def samples(t):
    return RolloutBufferSamples(None, t["actions"], t["old_values"], t["old_log_prob"], t["advantages"], t["returns"])


def device_loss(t, stats=None, **kw):
    """ppo_loss forward and backward on the device: loss, stats [5], grad_mean, grad_log_std, grad_values."""
    mean = t["mean"].clone().requires_grad_(True)
    log_std = t["log_std"].clone().requires_grad_(True)
    values = t["values"].clone().requires_grad_(True)
    stats = torch.zeros(5, dtype=F64, device=DEV) if stats is None else stats
    loss = ppo_loss(mean, log_std, values, samples(t), stats=stats, **kw)
    loss.backward()
    return loss.detach(), stats, mean.grad, log_std.grad, values.grad


def _bounds(x, kw, o):
    """Per-result error bounds (see the module docstring) from the oracle's float64 intermediates."""
    d64 = lambda k: torch.from_numpy(x[k]).double()   # noqa: E731
    mean, log_std, actions, adv = d64("mean"), d64("log_std"), d64("actions"), d64("advantages")
    B, N = mean.shape
    sig = torch.exp(log_std)
    d = actions - mean
    t1 = d * d / (2 * sig * sig)
    terms = -t1 - torch.log(sig) - LSP
    lp = terms.sum(1)
    old = d64("old_log_prob")
    e_lp = U * (lp.abs() + 4 * (terms.abs() + 2).sum(1))
    e_lr = e_lp + U * (lp - old).abs()
    r = torch.exp(lp - old)
    e_r = r * (e_lr + 2 * U)
    norm = kw["normalize_advantage"] and B > 1
    if norm:
        m, s = adv.mean(), adv.std()
        a = (adv - m) / (s + 1e-8)
        e_adv = 4 * U * a.abs() + 2 * U * (m.abs() + adv.abs()) / s
    else:
        a, e_adv = adv, torch.zeros_like(adv)
    w = o["w"]
    b = {}
    b["policy_gradient_loss"] = ((a.abs() * e_r + r * e_adv + 2 * U * (a * r).abs()).sum() / B).item()
    b["approx_kl"] = (((r - 1).abs() * e_lr + 2 * U * r).sum() / B).item()
    vp = o["vp"]
    ret = d64("returns")
    e = ret - vp
    b["value_loss"] = ((2 * e.abs() * 2 * U * (ret.abs() + vp.abs() + d64("old_values").abs()) + 2 * U * e * e).sum()
                       / B).item()
    b["entropy_loss"] = 4 * U * N * (1 + log_std.abs().max().item())
    b["clip_fraction"] = 0.0
    g = -a * w * r / B
    e_g = w * (a.abs() * e_r + r * e_adv) / B + 4 * U * g.abs()
    q = d * d / (sig * sig)
    gm = (g[:, None] * d / (sig * sig)).abs()
    b["grad_mean"] = e_g[:, None] * (d / (sig * sig)).abs() + 8 * U * gm
    b["grad_log_std"] = (e_g[:, None] * (q - 1).abs() + 8 * U * g.abs()[:, None] * (q + 1)).sum(0) + 2 * U
    # returns - values_pred; with clipping values_pred = old_values + (values - old_values) rounds twice
    e_e = 2 * U * (ret.abs() + vp.abs() + d64("values").abs() + d64("old_values").abs())
    b["grad_values"] = 2 * U * o["gv"].abs() + kw["vf_coef"] * 2 / B * e_e * o["vmask"]
    return b


def _oracle(x, kw):
    c = {k: torch.from_numpy(v) for k, v in x.items()}
    loss, st, gm, gls, gv = ref.loss_and_grads(c["mean"], c["log_std"], c["values"], c["actions"], c["old_log_prob"],
                                               c["old_values"], c["advantages"], c["returns"], **kw)
    # the branch weights and the value prediction, for the bounds
    d64 = {k: v.double() for k, v in c.items()}
    lp = ref.log_prob(d64["mean"], d64["log_std"], d64["actions"])
    r = torch.exp(lp - d64["old_log_prob"])
    B = len(r)
    adv = d64["advantages"]
    a = (adv - adv.mean()) / (adv.std() + 1e-8) if kw["normalize_advantage"] and B > 1 else adv
    lo, hi = 1 - kw["clip_range"], 1 + kw["clip_range"]
    l1, l2 = a * r, a * torch.clamp(r, lo, hi)
    passes = ((r >= lo) & (r <= hi)).double()
    w = torch.where(l1 < l2, torch.ones_like(r), torch.where(l1 > l2, passes, 0.5 + 0.5 * passes))
    if kw["clip_range_vf"] is None:
        vp, vmask = d64["values"], torch.ones_like(r)
    else:
        dv = d64["values"] - d64["old_values"]
        c_ = kw["clip_range_vf"]
        vp, vmask = d64["old_values"] + torch.clamp(dv, -c_, c_), ((dv >= -c_) & (dv <= c_)).double()
    return dict(loss=loss.item(), stats={k: v.item() for k, v in st.items()}, grad_mean=gm, grad_log_std=gls,
                grad_values=gv, w=w, vp=vp, vmask=vmask, gv=gv, r=r)


def _check(name, got, want, bound):
    got = got.detach().double().cpu()
    diff = (got - want).abs()
    assert bool((diff <= 2 * bound).all()), \
        f"{name}: max |diff| {diff.max().item():.3e}, bound {torch.as_tensor(bound).max().item():.3e}"


@pytest.mark.parametrize("norm", [True, False])
@pytest.mark.parametrize("clip_range_vf", [None, 0.5])
@pytest.mark.parametrize("N", [1, 20, 50, 300])
@pytest.mark.parametrize("B", [1, 2, 33, 4096, 65536])
def test_loss_and_gradients_match_oracle(B, N, clip_range_vf, norm):
    rng = np.random.default_rng(B * 1009 + N * 7 + (clip_range_vf is None) * 2 + int(norm))
    x = draw(rng, B, N)
    t = to_dev(x)
    base = dict(clip_range=0.2, clip_range_vf=clip_range_vf, normalize_advantage=norm, vf_coef=0.5)
    o = _oracle(x, dict(base, ent_coef=0.0))

    # log_prob: the rollout-time entry point
    lp = log_prob(t["mean"], t["log_std"], t["actions"]).double().cpu()
    lp_ref = ref.log_prob(*(torch.from_numpy(x[k]).double() for k in ("mean", "log_std", "actions")))
    sig = torch.exp(torch.from_numpy(x["log_std"]).double())
    d = torch.from_numpy(x["actions"]).double() - torch.from_numpy(x["mean"]).double()
    terms = -(d * d) / (2 * sig * sig) - torch.log(sig) - LSP
    _check("log_prob", lp, lp_ref, U * (lp_ref.abs() + 4 * (terms.abs() + 2).sum(1)))

    if B >= 4096:
        cf = o["stats"]["clip_fraction"]
        assert 0.15 < cf < 0.5, cf                                   # about a third of the ratios are clipped
    for ent_coef in (0.0, 0.01):
        kw = dict(base, ent_coef=ent_coef)
        loss, st, gm, gls, gv = device_loss(t, **kw)
        bnd = _bounds(x, kw, o)
        want = dict(o["stats"])
        ent = want["entropy_loss"]
        for i, k in enumerate(STATS):
            _check(k, st[i], torch.tensor(want[k], dtype=F64), bnd[k] + 1e-15)
        assert st[3].item() * B == round(want["clip_fraction"] * B)   # exact: no ratio near a bound
        want_loss = o["loss"] + ent_coef * ent
        loss_b = bnd["policy_gradient_loss"] + 0.5 * bnd["value_loss"] + ent_coef * bnd["entropy_loss"] + U * abs(want_loss)
        _check("loss", loss, torch.tensor(want_loss, dtype=F64), loss_b + 1e-12)
        _check("grad_mean", gm, o["grad_mean"], bnd["grad_mean"])
        _check("grad_log_std", gls, o["grad_log_std"] - ent_coef, bnd["grad_log_std"] + U * (o["grad_log_std"].abs() + ent_coef))
        _check("grad_values", gv, o["grad_values"], bnd["grad_values"] + 1e-30)
        # the stated target, where the float32 log-probabilities allow it
        if N <= 50 and B >= 33:
            scale = o["grad_mean"].abs().max().item()
            assert (gm.double().cpu() - o["grad_mean"]).abs().max().item() <= 1e-5 * scale
            assert abs(st[1].item() - want["value_loss"]) <= 1e-5 * abs(want["value_loss"])


def test_unchanged_policy_ratio_is_exactly_one():
    rng = np.random.default_rng(7)
    B, N = 4096, 50
    x = draw(rng, B, N)
    t = to_dev(x)
    t["old_log_prob"] = log_prob(t["mean"], t["log_std"], t["actions"])
    kw = dict(clip_range=0.2, clip_range_vf=None, normalize_advantage=True, ent_coef=0.0, vf_coef=0.5)
    loss, st, gm, gls, gv = device_loss(t, **kw)
    assert st[3].item() == 0.0 and st[4].item() == 0.0             # clip_fraction, approx_kl: bit for bit
    # the plain policy gradient: g_i = -A_hat_i / B
    adv = t["advantages"].double().cpu()
    m, s = np.float32(adv.mean().item()), np.float32(adv.std().item())
    a = (adv - float(m)) / (float(s) + 1e-8)
    mean, act = t["mean"].double().cpu(), t["actions"].double().cpu()
    var = torch.exp(t["log_std"].double().cpu()) ** 2
    want = (-a / B)[:, None] * (act - mean) / var
    assert (gm.double().cpu() - want).abs().max().item() <= 1e-5 * want.abs().max().item()
    assert abs(st[0].item() - (-a.mean().item())) <= 1e-6            # policy_loss = -mean(A_hat) ~ 0


def test_calls_are_bit_identical():
    rng = np.random.default_rng(9)
    t = to_dev(draw(rng, 65536, 50))
    kw = dict(clip_range=0.2, clip_range_vf=0.5, normalize_advantage=True, ent_coef=0.01, vf_coef=0.5)
    a = device_loss(t, **kw)
    b = device_loss(t, **kw)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_error_paths():
    L = load_library()
    rng = np.random.default_rng(2)
    t = to_dev(draw(rng, 64, 5))
    ptr = {k: v.data_ptr() for k, v in t.items()}
    order = ("mean", "log_std", "actions", "values", "old_log_prob", "old_values", "advantages", "returns")

    def batch(B=64, N=5, **null):
        return FleetPpoBatch(B, N, 0, *[None if null.get(k) else ptr[k] for k in order])

    ok = FleetPpoParams(0.2, -1.0, 0.0, 0.5, 1, 0)
    need = L.fleet_ppo_workspace_bytes(64, 5)
    assert need > 0 and L.fleet_ppo_workspace_bytes(0, 5) == 0 and L.fleet_ppo_workspace_bytes(64, 0) == 0
    ws = torch.zeros(need, dtype=torch.uint8, device=DEV)
    out = torch.zeros(2 * 64, dtype=torch.float32, device=DEV)
    stats = torch.zeros(5, dtype=F64, device=DEV)
    loss = torch.zeros((), dtype=torch.float32, device=DEV)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda x: C.c_void_p(x.data_ptr())   # noqa: E731

    def call(b, prm=ok, nbytes=need):
        return L.fleet_ppo_loss(C.byref(b), C.byref(prm), p(loss), p(stats), p(out), p(ws), nbytes, s)

    assert call(batch()) == 0
    bad = [call(batch(B=0)), call(batch(N=0)), call(batch(mean=True)), call(batch(returns=True)),
           call(batch(), FleetPpoParams(0.0, -1.0, 0.0, 0.5, 1, 0)), call(batch(), FleetPpoParams(-0.1, -1.0, 0.0, 0.5, 1, 0)),
           call(batch(), nbytes=need - 1), call(batch(old_values=True), FleetPpoParams(0.2, 0.5, 0.0, 0.5, 1, 0)),
           L.fleet_ppo_loss(None, C.byref(ok), p(loss), p(stats), p(out), p(ws), need, s),
           L.fleet_ppo_loss(C.byref(batch()), None, p(loss), p(stats), p(out), p(ws), need, s),
           L.fleet_ppo_loss(C.byref(batch()), C.byref(ok), p(loss), None, p(out), p(ws), need, s),
           L.fleet_ppo_loss(C.byref(batch()), C.byref(ok), p(loss), p(stats), p(out), None, need, s),
           L.fleet_ppo_log_prob(C.byref(batch(actions=True)), p(out), s), L.fleet_ppo_log_prob(C.byref(batch()), None, s),
           L.fleet_ppo_loss_backward(C.byref(batch()), C.byref(ok), None, p(out), p(out), p(out), p(out), p(ws), need, s),
           L.fleet_ppo_loss_backward(C.byref(batch()), C.byref(ok), p(loss), p(out), p(out), p(out), p(out), p(ws),
                                     need - 1, s)]
    assert all(rc == -1 for rc in bad), bad
    assert b"workspace" in L.fleet_ppo_last_error()
    # the Python layer checks shapes, dtypes, devices and contiguity
    with pytest.raises(FleetStepError):
        ppo_loss(t["mean"][:, :4], t["log_std"], t["values"], samples(t))
    with pytest.raises(FleetStepError):
        ppo_loss(t["mean"].double(), t["log_std"], t["values"], samples(t))
    with pytest.raises(FleetStepError):
        ppo_loss(t["mean"].cpu(), t["log_std"], t["values"], samples(t))
    with pytest.raises(FleetStepError):
        ppo_loss(t["mean"].t().contiguous().t(), t["log_std"], t["values"], samples(t))
    torch.cuda.synchronize()


def test_offsets_past_2_31_elements():
    """One minibatch of 42,949,673 x 50 actions (2^31 + 2 elements, 8.6 GB per array), ratio 1 by construction: the
    rows past element 2^31 against their closed forms."""
    N = 50
    B = 2 ** 31 // N + 1
    assert B * N > 2 ** 31
    g = torch.Generator(device=DEV)
    g.manual_seed(3)
    t = {}
    try:
        t["mean"] = torch.randn((B, N), device=DEV, generator=g)
        t["actions"] = torch.randn((B, N), device=DEV, generator=g)
        t["log_std"] = torch.linspace(-0.5, 0.2, N, device=DEV)
        for k in ("values", "old_values", "advantages", "returns"):
            t[k] = torch.randn(B, device=DEV, generator=g)
        t["old_log_prob"] = log_prob(t["mean"], t["log_std"], t["actions"])
        tail = slice(B - 64, B)
        lp_tail = log_prob(t["mean"][tail].contiguous(), t["log_std"], t["actions"][tail].contiguous())
        assert torch.equal(lp_tail, t["old_log_prob"][tail])
        kw = dict(clip_range=0.2, clip_range_vf=None, normalize_advantage=False, ent_coef=0.0, vf_coef=0.5)
        loss, st, gm, gls, gv = device_loss(t, **kw)
        assert st[3].item() == 0.0 and st[4].item() == 0.0
        adv = t["advantages"][tail].double()
        var = torch.exp(t["log_std"].double()) ** 2
        want = (-adv / B)[:, None] * (t["actions"][tail].double() - t["mean"][tail].double()) / var
        assert (gm[tail].double() - want).abs().max().item() <= 1e-5 * want.abs().max().item()
        want_v = 0.5 * 2 * (t["values"][tail].double() - t["returns"][tail].double()) / B
        assert (gv[tail].double() - want_v).abs().max().item() <= 1e-5 * want_v.abs().max().item()
        vl = ((t["returns"].double() - t["values"].double()) ** 2).mean().item()
        assert abs(st[1].item() - vl) <= 1e-6 * vl
        assert abs(st[0].item() - (-t["advantages"].double().mean().item())) <= 1e-6
        del gm
    finally:
        t.clear()
        torch.cuda.empty_cache()


# ---------------------------------------------------------------- end to end

def _fleet(E, N):
    from synth_tables import make_consts, make_tables
    from fleetrl_b200 import FleetVecEnv, FleetVecNormalize
    tables, Tt = make_tables(n_evs=N, days=12, seed=7)
    consts = make_consts(tables, Tt, N)
    env = FleetVecEnv(None, E, built=SimpleNamespace(consts=consts, tables=tables, rc=None), output="torch")
    vn = FleetVecNormalize(env)
    return env, vn, vn.reset()


def _adam_bound(lr, steps, b1=0.9, b2=0.999):
    """Largest total difference between two Adam trajectories of `steps` steps from the same point: each step moves a
    parameter by at most lr * |m_hat| / sqrt(v_hat) <= lr * (1 - b1) / (1 - b1^t) * sqrt((1 - b2^t) / (1 - b2))
    * sum_{j<t} (b1 / sqrt(b2))^j, whatever the gradients; two trajectories can differ by twice the sum."""
    tot = 0.0
    for t in range(1, steps + 1):
        s = sum((b1 / math.sqrt(b2)) ** j for j in range(t))
        tot += (1 - b1) / (1 - b1 ** t) * math.sqrt((1 - b2 ** t) / (1 - b2)) * s
    return 2 * lr * tot


def test_collect_and_train_end_to_end():
    E, N, T, bs, epochs = 256, 10, 16, 1024, 2
    env, vn, obs = _fleet(E, N)
    D = env.obs_dim
    torch.manual_seed(0)
    policy = FleetMlpPolicy(D, N, DEV)
    init = {k: v.detach().clone() for k, v in policy.state_dict().items()}
    buf = FleetRolloutBuffer(T, E, D, N, DEV, gamma=0.99, gae_lambda=0.95)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(5)
    first = []
    step = policy.optimizer.step

    def record_step(*a, **k):   # the clipped gradient of the first minibatch
        if not first:
            first.extend(p.grad.detach().clone() for p in policy.parameters())
        return step(*a, **k)

    policy.optimizer.step = record_step
    starts = torch.ones(E, dtype=torch.bool, device=DEV)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        obs, starts = collect_rollouts(vn, policy, buf, obs, starts)
        stats = ppo_train(policy, buf, n_epochs=epochs, batch_size=bs, generator=gen)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    after = {k: v.detach().double().cpu() for k, v in policy.state_dict().items()}

    # the float64 restatement from the same parameters, on the same buffer, with the same permutations
    o = ref.MlpPolicy(D, N)
    o.load_state_dict({k: v.double().cpu() for k, v in init.items()})
    o.make_optimizer()
    n = T * E
    flat = {k: getattr(buf, k).transpose(0, 1).reshape(n, -1).squeeze(-1).double().cpu()
            for k in ("observations", "actions", "values", "log_probs", "advantages", "returns")}
    g2 = torch.Generator(device=DEV)
    g2.manual_seed(5)
    perms = [torch.randperm(n, device=DEV, generator=g2).cpu() for _ in range(epochs)]
    o_first = []
    out, steps = ref.train(o, flat, perms, bs, n_epochs=epochs,
                           on_step=lambda p: o_first or o_first.extend(q.grad.clone() for q in p.parameters()))
    assert steps == epochs * math.ceil(n / bs)

    for name, gd, go in zip(dict(policy.named_parameters()), first, o_first):
        scale = go.abs().max().item()
        assert (gd.double().cpu() - go).abs().max().item() <= 1e-4 * scale + 1e-9, name
    bound = _adam_bound(3e-4, steps)
    moved = 0.0
    for k, v in o.state_dict().items():
        assert (after[k] - v).abs().max().item() <= bound, (k, bound)
        moved = max(moved, (v - init[k].double().cpu()).abs().max().item())
    assert moved > 1e-4

    assert stats["train/n_updates"] == out["train/n_updates"] == epochs and stats["train/clip_range"] == 0.2
    for k in ("train/entropy_loss", "train/policy_gradient_loss", "train/value_loss", "train/approx_kl", "train/loss",
              "train/std"):
        assert stats[k].is_cuda and stats[k].dim() == 0
        assert abs(stats[k].item() - out[k]) <= 1e-3 * abs(out[k]) + 1e-6, (k, stats[k].item(), out[k])
    assert abs(stats["train/clip_fraction"].item() - out["train/clip_fraction"]) <= 2.0 / bs
    assert abs(stats["train/explained_variance"].item() - out["train/explained_variance"]) <= 1e-9
