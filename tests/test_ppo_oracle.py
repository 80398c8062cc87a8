"""The float64 restatement of SB3's PPO loss and train loop (oracle/ppo.py) against closed forms, and FleetMlpPolicy's
layout and initialisation against SB3 2.3.2's MlpPolicy.  CPU only."""
import math

import numpy as np
import pytest
import torch

from oracle import ppo as ref

F64 = torch.float64


def closed_form(mean, log_std, values, actions, old_lp, old_v, adv, ret, clip_range=0.2, clip_range_vf=None,
                normalize_advantage=True, ent_coef=0.0, vf_coef=0.5):
    """The gradients of PPO's loss written out (ppo_loss's backward), with torch's rules at the edges: clamp passes the
    gradient on its closed interval, minimum splits a tie in half, the normalised advantage carries none."""
    B = len(adv)
    sig = torch.exp(log_std)
    var = sig * sig
    d = actions - mean
    lp = (-(d * d) / (2 * var) - torch.log(sig) - math.log(math.sqrt(2 * math.pi))).sum(1)
    a = (adv - adv.mean()) / (adv.std() + 1e-8) if normalize_advantage and B > 1 else adv
    r = torch.exp(lp - old_lp)
    lo, hi = 1 - clip_range, 1 + clip_range
    l1, l2 = a * r, a * torch.clamp(r, lo, hi)
    passes = ((r >= lo) & (r <= hi)).to(F64)
    w = torch.where(l1 < l2, torch.ones_like(r), torch.where(l1 > l2, passes, 0.5 + 0.5 * passes))
    g = -a * w * r / B
    grad_mean = g[:, None] * d / var
    grad_log_std = (g[:, None] * (d * d / var - 1)).sum(0) - ent_coef
    if clip_range_vf is None:
        vp, vmask = values, torch.ones_like(values)
    else:
        dv = values - old_v
        vp = old_v + torch.clamp(dv, -clip_range_vf, clip_range_vf)
        vmask = ((dv >= -clip_range_vf) & (dv <= clip_range_vf)).to(F64)
    grad_values = vf_coef * 2 * (vp - ret) / B * vmask
    return grad_mean, grad_log_std, grad_values, dict(r=r, a=a, w=w, vmask=vmask, lo=lo, hi=hi)


def draw(rng, B, N, clip_range=0.2, clip_range_vf=0.5):
    """Inputs with about a third of the ratios outside the clip range and a third of the value clips active."""
    log_std = rng.uniform(-1.0, 0.3, N)
    mean = rng.standard_normal((B, N))
    actions = mean + np.exp(log_std) * rng.standard_normal((B, N))
    lp = ref.log_prob(torch.tensor(mean), torch.tensor(log_std), torch.tensor(actions)).numpy()
    old_lp = lp - rng.normal(0, 0.2, B)
    values = rng.standard_normal(B)
    old_v = values - rng.normal(0, 0.5, B)
    adv = rng.normal(0.3, 1.5, B)
    ret = values + rng.standard_normal(B)
    return [torch.tensor(x) for x in (mean, log_std, values, actions, old_lp, old_v, adv, ret)]


@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("clip_range_vf", [None, 0.5])
@pytest.mark.parametrize("ent_coef", [0.0, 0.01])
def test_gradients_match_closed_form(normalize, clip_range_vf, ent_coef):
    rng = np.random.default_rng(11 + int(normalize) + (clip_range_vf is None) * 2 + int(ent_coef * 400))
    B, N = 2000, 7
    x = draw(rng, B, N)
    kw = dict(clip_range=0.2, clip_range_vf=clip_range_vf, normalize_advantage=normalize, ent_coef=ent_coef, vf_coef=0.5)
    _, _, gm, gls, gv = ref.loss_and_grads(*x, **kw)
    cm, cls, cv, info = closed_form(*x, **kw)
    np.testing.assert_allclose(gm.numpy(), cm.numpy(), rtol=1e-10, atol=1e-15)
    np.testing.assert_allclose(gls.numpy(), cls.numpy(), rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(gv.numpy(), cv.numpy(), rtol=1e-10, atol=1e-15)
    # the draw covers clipped and unclipped samples with both signs of the advantage, and both value-clip states
    r, a = info["r"], info["a"]
    inside = (r >= info["lo"]) & (r <= info["hi"])
    for sel in (inside & (a > 0), inside & (a < 0), (r > info["hi"]) & (a > 0), (r > info["hi"]) & (a < 0),
                (r < info["lo"]) & (a > 0), (r < info["lo"]) & (a < 0)):
        assert int(sel.sum()) > 20
    assert 0.2 < float((~inside).double().mean()) < 0.45
    if clip_range_vf is not None:
        assert 0.1 < float(info["vmask"].mean()) < 0.9


def _at_ratio_one(B=5, N=3, seed=0):
    """Inputs whose old_log_prob is the policy's own: every ratio is exactly 1."""
    rng = np.random.default_rng(seed)
    mean, log_std, values, actions, _, old_v, adv, ret = draw(rng, B, N)
    old_lp = ref.log_prob(mean, log_std, actions).detach()
    return [mean, log_std, values, actions, old_lp, old_v, adv, ret]


def test_clamp_bound_is_inclusive():
    """clip_range = 0: every ratio (exactly 1) lies on both bounds.  With an inclusive clamp the tied minimum still
    passes the whole gradient: g = -A / B.  Value clip: values - old_values exactly c passes its gradient too."""
    x = _at_ratio_one()
    x[5] = x[2] - 0.5                      # values - old_values = 0.5 exactly
    _, st, gm, _, gv = ref.loss_and_grads(*x, clip_range=0.0, clip_range_vf=0.5, normalize_advantage=False)
    mean, log_std, _, actions, _, _, adv, ret = x
    B = len(adv)
    var = torch.exp(log_std) ** 2
    np.testing.assert_allclose(gm.numpy(), (-adv / B)[:, None].numpy() * ((actions - mean) / var).numpy(), rtol=1e-12)
    np.testing.assert_allclose(gv.numpy(), (0.5 * 2 * (x[2] - ret) / B).numpy(), rtol=1e-12)
    assert float(st["clip_fraction"]) == 0.0 and float(st["approx_kl"]) == 0.0


def test_minimum_splits_a_tie():
    """torch.min of two equal tensors sends half of the gradient to each side: the rule the kernels restate."""
    a = torch.tensor([1.5, -2.0], dtype=F64, requires_grad=True)
    b = torch.tensor([1.5, -3.0], dtype=F64, requires_grad=True)
    torch.min(a, b).sum().backward()
    assert a.grad.tolist() == [0.5, 0.0] and b.grad.tolist() == [0.5, 1.0]
    # in the loss: a ratio of exactly 1 inside the range ties both surrogates; the halves add up to the whole gradient
    x = _at_ratio_one(seed=3)
    _, _, gm, _, _ = ref.loss_and_grads(*x, clip_range=0.2, normalize_advantage=False)
    cm, _, _, info = closed_form(*x, clip_range=0.2, normalize_advantage=False)
    assert bool((info["w"] == 1.0).all())
    np.testing.assert_allclose(gm.numpy(), cm.numpy(), rtol=1e-12)


def test_single_sample_is_not_normalised():
    rng = np.random.default_rng(5)
    x = draw(rng, 1, 4)
    l_on, _, *g_on = ref.loss_and_grads(*x, normalize_advantage=True)
    l_off, _, *g_off = ref.loss_and_grads(*x, normalize_advantage=False)
    assert float(l_on) == float(l_off)
    for a, b in zip(g_on, g_off):
        assert torch.equal(a, b)
    cm, _, _, info = closed_form(*x, normalize_advantage=True)
    assert torch.equal(info["a"], x[6])


def _loop_setup(seed=0, n=96, D=6, N=2):
    torch.manual_seed(seed)
    pol = ref.MlpPolicy(D, N)
    pol.make_optimizer()
    g = torch.Generator().manual_seed(seed)
    flat = dict(observations=torch.randn(n, D, dtype=F64, generator=g), actions=torch.randn(n, N, dtype=F64, generator=g),
                values=torch.randn(n, dtype=F64, generator=g), log_probs=-2 + 0.3 * torch.randn(n, dtype=F64, generator=g),
                advantages=torch.randn(n, dtype=F64, generator=g), returns=torch.randn(n, dtype=F64, generator=g))
    return pol, flat, g


def test_loop_bookkeeping():
    pol, flat, g = _loop_setup()
    n, bs, epochs = 96, 40, 3
    perms = [torch.randperm(n, generator=g) for _ in range(epochs)]
    steps, log = [], []
    out, n_steps = ref.train(pol, flat, perms, bs, n_epochs=epochs, on_step=lambda p: steps.append(1), log=log)
    assert n_steps == len(steps) == epochs * math.ceil(n / bs)
    assert out["train/n_updates"] == epochs
    last = [s["approx_kl"] for e, s in log if e == epochs - 1]
    assert len(last) == math.ceil(n / bs)
    assert out["train/approx_kl"] == pytest.approx(sum(last) / len(last), rel=1e-15)
    every = [s["approx_kl"] for _, s in log]
    assert out["train/approx_kl"] != pytest.approx(sum(every) / len(every), rel=1e-6)
    assert out["train/policy_gradient_loss"] == pytest.approx(sum(s["policy_gradient_loss"] for _, s in log) / len(log))


def test_target_kl_stops_before_the_step():
    pol, flat, g = _loop_setup(seed=1)
    before = {k: v.clone() for k, v in pol.state_dict().items()}
    perms = [torch.randperm(96, generator=g) for _ in range(4)]
    log = []
    out, n_steps = ref.train(pol, flat, perms, 32, n_epochs=4, target_kl=1e-9, log=log)
    assert n_steps == 0 and len(log) == 1 and out["train/n_updates"] == 1
    assert log[0][1]["approx_kl"] > 1.5e-9
    for k, v in pol.state_dict().items():
        assert torch.equal(v, before[k]), k


# SB3 2.3.2, PPO("MlpPolicy", env with Box(obs_dim) observations and Box(action_dim) actions).policy.state_dict()
SB3_MLP_POLICY_KEYS = [
    ("log_std", ("N",)),
    ("mlp_extractor.policy_net.0.weight", (64, "D")),
    ("mlp_extractor.policy_net.0.bias", (64,)),
    ("mlp_extractor.policy_net.2.weight", (64, 64)),
    ("mlp_extractor.policy_net.2.bias", (64,)),
    ("mlp_extractor.value_net.0.weight", (64, "D")),
    ("mlp_extractor.value_net.0.bias", (64,)),
    ("mlp_extractor.value_net.2.weight", (64, 64)),
    ("mlp_extractor.value_net.2.bias", (64,)),
    ("action_net.weight", ("N", 64)),
    ("action_net.bias", ("N",)),
    ("value_net.weight", (1, 64)),
    ("value_net.bias", (1,)),
]


def test_policy_state_dict_has_sb3_keys():
    from fleetrl_b200.ppo import FleetMlpPolicy
    D, N = 388, 50
    sd = FleetMlpPolicy(D, N, "cpu").state_dict()
    want = [(k, tuple({"D": D, "N": N}.get(s, s) for s in shape)) for k, shape in SB3_MLP_POLICY_KEYS]
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == want
    # and it loads into the float64 restatement, whose names are the same
    o = ref.MlpPolicy(D, N)
    o.load_state_dict(sd)


def test_policy_orthogonal_initialisation():
    from fleetrl_b200.ppo import FleetMlpPolicy
    torch.manual_seed(0)
    p = FleetMlpPolicy(388, 50, "cpu", log_std_init=-0.5)
    gains = {"mlp_extractor.policy_net.0": 2.0, "mlp_extractor.policy_net.2": 2.0, "mlp_extractor.value_net.0": 2.0,
             "mlp_extractor.value_net.2": 2.0, "action_net": 0.01 ** 2, "value_net": 1.0}
    sd = p.state_dict()
    for name, g2 in gains.items():
        w = sd[name + ".weight"].double()
        short = w @ w.T if w.shape[0] <= w.shape[1] else w.T @ w
        np.testing.assert_allclose(short.numpy(), g2 * np.eye(short.shape[0]), atol=1e-5 * g2)
        assert not sd[name + ".bias"].any()
    assert torch.equal(sd["log_std"], torch.full((50,), -0.5))
    opt = p.optimizer
    assert isinstance(opt, torch.optim.Adam) and opt.defaults["eps"] == 1e-5 and opt.defaults["lr"] == 3e-4
