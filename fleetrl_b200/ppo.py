"""PPO's update on the device: stable-baselines3 2.3.2's MlpPolicy (common/policies.py, ActorCriticPolicy) and the body of
PPO.train (ppo/ppo.py) over a full FleetRolloutBuffer.

The policy and value networks are torch modules (cuBLAS).  The per-minibatch work around them, the diagonal-Gaussian
log-probability, the clipped surrogate and value loss with advantage normalisation, and the gradients of that loss, are
kernels of libfleetstep (fleet_ppo_*): three launches per minibatch, forward and backward, and no host synchronisation.
ppo_loss is the torch.autograd.Function over them; ppo_train is the epoch / minibatch loop.

Differences from SB3, all deliberate:
  * reductions (the advantages' mean and std, the minibatch means, the log-probability's sum over the action dimensions)
    run in float64, so the loss and the statistics are more accurate than SB3's float32 ones and differ from them at
    float32 rounding level; approx_kl is averaged from float64 terms ((ratio - 1) - log_ratio);
  * the statistics ppo_train returns are 0-dim device tensors, not Python floats: reading them is the caller's one sync;
  * only what PPO's MlpPolicy needs for a Box observation and a Box action: no gSDE, no shared layers
    (share_features_extractor), no Discrete / MultiDiscrete actions.
"""
import ctypes as C
import math
from functools import partial

import torch
from torch import nn

from ._lib import FleetPpoBatch, FleetPpoParams, FleetStepError, _dptr, _stream_ptr, load_library
from .rollout import FleetRolloutBuffer, RolloutBufferSamples

STATS = ("policy_gradient_loss", "value_loss", "entropy_loss", "clip_fraction", "approx_kl")   # fleet_ppo_loss order

_WORKSPACE = {}   # device -> zero-filled uint8 tensor; the kernels leave it reusable, so one per device is shared


def _lib_check(lib, rc, what):
    if rc != 0:
        raise FleetStepError(f"{what}: {lib.fleet_ppo_last_error().decode()} (code {rc})")


def _tensor(t, shape, name, device):
    """t as it must reach the kernels: a contiguous float32 tensor of `shape` on `device` (a trailing 1 is accepted)."""
    if not isinstance(t, torch.Tensor):
        raise FleetStepError(f"{name}: expected a torch tensor on {device}, got {type(t).__name__}")
    if t.device != device:
        raise FleetStepError(f"{name}: expected a tensor on {device}, got one on {t.device}")
    if tuple(t.shape) != tuple(shape) and not (t.dim() == len(shape) + 1 and tuple(t.shape) == tuple(shape) + (1,)):
        raise FleetStepError(f"{name}: expected shape {tuple(shape)}, got {tuple(t.shape)}")
    if t.dtype != torch.float32:
        raise FleetStepError(f"{name}: expected float32, got {t.dtype}")
    if not t.is_contiguous():
        raise FleetStepError(f"{name}: expected a contiguous tensor")
    return t.reshape(shape)


def _device(t):
    d = t.device
    if d.type != "cuda":
        raise FleetStepError("the PPO kernels run on a CUDA device; there is no CPU fallback")
    return d


def _workspace(lib, device, B, N):
    need = int(lib.fleet_ppo_workspace_bytes(int(B), int(N)))
    ws = _WORKSPACE.get(device)
    if ws is None or ws.numel() < need:
        ws = torch.zeros(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _WORKSPACE[device] = ws
    return ws


def _batch(mean, log_std, actions, values=None, old_log_prob=None, old_values=None, advantages=None, returns=None):
    B, N = mean.shape
    return FleetPpoBatch(B, N, 0, *[None if t is None else t.data_ptr() for t in
                                    (mean, log_std, actions, values, old_log_prob, old_values, advantages, returns)])


def log_prob(mean_actions, log_std, actions):
    """DiagGaussianDistribution(N).proba_distribution(mean_actions, log_std).log_prob(actions) with fleet_ppo_log_prob:
    float32 [B].  No autograd (rollout time)."""
    dev = _device(mean_actions)
    if mean_actions.dim() != 2:
        raise FleetStepError(f"mean_actions: expected [B, N], got shape {tuple(mean_actions.shape)}")
    B, N = mean_actions.shape
    mean_actions = _tensor(mean_actions.detach(), (B, N), "mean_actions", dev)
    log_std = _tensor(log_std.detach(), (N,), "log_std", dev)
    actions = _tensor(actions.detach(), (B, N), "actions", dev)
    lib = load_library()
    out = torch.empty(B, dtype=torch.float32, device=dev)
    b = _batch(mean_actions, log_std, actions)
    with torch.cuda.device(dev):
        _lib_check(lib, lib.fleet_ppo_log_prob(C.byref(b), _dptr(out), _stream_ptr(dev)), "fleet_ppo_log_prob")
    return out


def _params(clip_range, clip_range_vf, normalize_advantage, ent_coef, vf_coef):
    return FleetPpoParams(float(clip_range), -1.0 if clip_range_vf is None else float(clip_range_vf), float(ent_coef),
                          float(vf_coef), int(bool(normalize_advantage)), 0)


class _PpoLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mean_actions, log_std, values, samples, params, stats):
        dev = _device(mean_actions)
        if mean_actions.dim() != 2:
            raise FleetStepError(f"mean_actions: expected [B, N], got shape {tuple(mean_actions.shape)}")
        B, N = mean_actions.shape
        ts = [_tensor(mean_actions, (B, N), "mean_actions", dev), _tensor(log_std, (N,), "log_std", dev),
              _tensor(samples.actions, (B, N), "actions", dev), _tensor(values, (B,), "values", dev),
              _tensor(samples.old_log_prob, (B,), "old_log_prob", dev),
              _tensor(samples.old_values, (B,), "old_values", dev),
              _tensor(samples.advantages, (B,), "advantages", dev), _tensor(samples.returns, (B,), "returns", dev)]
        if stats is None:
            stats = torch.zeros(len(STATS), dtype=torch.float64, device=dev)
        elif stats.device != dev or stats.dtype != torch.float64 or stats.shape != (len(STATS),) or not stats.is_contiguous():
            raise FleetStepError(f"stats: expected a contiguous float64 tensor of shape ({len(STATS)},) on {dev}")
        lib = load_library()
        ws = _workspace(lib, dev, B, N)
        coef = torch.empty((2, B), dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        b = _batch(*ts)
        with torch.cuda.device(dev):
            _lib_check(lib, lib.fleet_ppo_loss(C.byref(b), C.byref(params), _dptr(loss), _dptr(stats), _dptr(coef),
                                               _dptr(ws), ws.numel(), _stream_ptr(dev)), "fleet_ppo_loss")
        ctx.save_for_backward(*ts, coef)
        ctx.params = params
        ctx.values_shape = values.shape
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        ts = ctx.saved_tensors
        coef = ts[-1]
        mean_actions, log_std = ts[0], ts[1]
        dev = mean_actions.device
        B, N = mean_actions.shape
        lib = load_library()
        ws = _workspace(lib, dev, B, N)
        g = grad_loss.detach().to(dtype=torch.float32).contiguous()
        grad_mean = torch.empty_like(mean_actions)
        grad_log_std = torch.empty_like(log_std)
        grad_values = torch.empty(B, dtype=torch.float32, device=dev)
        b = _batch(*ts[:-1])
        with torch.cuda.device(dev):
            _lib_check(lib, lib.fleet_ppo_loss_backward(C.byref(b), C.byref(ctx.params), _dptr(g), _dptr(coef),
                                                        _dptr(grad_mean), _dptr(grad_log_std), _dptr(grad_values),
                                                        _dptr(ws), ws.numel(), _stream_ptr(dev)),
                       "fleet_ppo_loss_backward")
        return grad_mean, grad_log_std, grad_values.reshape(ctx.values_shape), None, None, None


def ppo_loss(mean_actions, log_std, values, samples: RolloutBufferSamples, clip_range=0.2, clip_range_vf=None,
             normalize_advantage=True, ent_coef=0.0, vf_coef=0.5, stats=None):
    """PPO.train's loss of one minibatch (ppo.py), as a 0-dim float32 device tensor with a backward on the device.

    mean_actions float32 [B, N], log_std [N] and values [B] or [B, 1] are the policy's outputs (they carry the
    gradient); samples the RolloutBufferSamples of the minibatch.  stats: an optional float64 [5] device tensor to which
    this minibatch's policy_gradient_loss, value_loss, entropy_loss, clip_fraction and approx_kl are added (STATS)."""
    return _PpoLoss.apply(mean_actions, log_std, values, samples,
                          _params(clip_range, clip_range_vf, normalize_advantage, ent_coef, vf_coef), stats)


class _MlpExtractor(nn.Module):
    """SB3's MlpExtractor with net_arch dict(pi=[64, 64], vf=[64, 64]) and Tanh."""

    def __init__(self, feature_dim):
        super().__init__()
        self.policy_net = nn.Sequential(nn.Linear(feature_dim, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        self.value_net = nn.Sequential(nn.Linear(feature_dim, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        self.latent_dim_pi = self.latent_dim_vf = 64

    def forward_actor(self, features):
        return self.policy_net(features)

    def forward_critic(self, features):
        return self.value_net(features)


class FleetMlpPolicy(nn.Module):
    """SB3 2.3.2's ActorCriticPolicy with PPO's MlpPolicy defaults for a Box(obs_dim) observation and a Box(action_dim)
    action: separate pi / vf networks of two 64-wide Tanh layers, action_net, value_net, a state-independent log_std,
    orthogonal initialisation (gains sqrt(2), 0.01, 1; zero biases) and Adam(lr, eps=1e-5).  The attribute names are
    SB3's, so state_dict() has exactly the keys and shapes of an SB3 PPO("MlpPolicy").policy and loads into one.

    Learning-rate schedules belong to the caller: set optimizer.param_groups[i]["lr"] before each ppo_train call, as
    SB3's _update_learning_rate does."""

    def __init__(self, obs_dim, action_dim, device, lr=3e-4, log_std_init=0.0):
        super().__init__()
        self.obs_dim, self.action_dim = int(obs_dim), int(action_dim)
        self.log_std = nn.Parameter(torch.ones(self.action_dim) * log_std_init, requires_grad=True)
        self.mlp_extractor = _MlpExtractor(self.obs_dim)
        self.action_net = nn.Linear(64, self.action_dim)
        self.value_net = nn.Linear(64, 1)
        for module, gain in ((self.mlp_extractor, math.sqrt(2)), (self.action_net, 0.01), (self.value_net, 1.0)):
            module.apply(partial(self._init_weights, gain=gain))
        self.to(device)
        self.device = self.log_std.device
        self.optimizer = torch.optim.Adam(self.parameters(), lr=lr, eps=1e-5)

    @staticmethod
    def _init_weights(module, gain=1.0):
        """BasePolicy.init_weights: orthogonal weights, zero biases."""
        if isinstance(module, nn.Linear):
            nn.init.orthogonal_(module.weight, gain=gain)
            if module.bias is not None:
                module.bias.data.fill_(0.0)

    def loss_inputs(self, obs):
        """(mean_actions [B, N], log_std [N], values [B]): what ppo_loss takes (evaluate_actions without the distribution)."""
        features = obs.float()
        mean_actions = self.action_net(self.mlp_extractor.forward_actor(features))
        values = self.value_net(self.mlp_extractor.forward_critic(features)).flatten()
        return mean_actions, self.log_std, values

    def forward(self, obs, deterministic=False):
        """ActorCriticPolicy.forward: (actions [E, N], values [E, 1], log_prob [E]).  Sampling is Normal.rsample,
        mean + randn * exp(log_std); the log-probability is fleet_ppo_log_prob."""
        features = obs.float()
        values = self.value_net(self.mlp_extractor.forward_critic(features))
        mean_actions = self.action_net(self.mlp_extractor.forward_actor(features))
        std = torch.ones_like(mean_actions) * self.log_std.exp()
        actions = mean_actions if deterministic else mean_actions + torch.randn_like(mean_actions) * std
        return actions, values, log_prob(mean_actions, self.log_std, actions)

    def predict_values(self, obs):
        return self.value_net(self.mlp_extractor.forward_critic(obs.float()))


def ppo_train(policy: FleetMlpPolicy, buffer: FleetRolloutBuffer, n_epochs=10, batch_size=64, clip_range=0.2,
              clip_range_vf=None, normalize_advantage=True, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, target_kl=None,
              generator=None):
    """The body of SB3's PPO.train (ppo.py) over a full buffer: n_epochs passes of buffer.get(batch_size, generator), each
    minibatch running the policy, ppo_loss, zero_grad, backward, clip_grad_norm_(max_grad_norm) and optimizer.step.

    Returns SB3's logged values under its train/* names as 0-dim float64 device tensors: entropy_loss,
    policy_gradient_loss, value_loss and clip_fraction (means over every minibatch), approx_kl (the mean over the last
    epoch), loss (the last minibatch's, float32), explained_variance (over the whole buffer; NaN when var(returns) is 0)
    and std (mean of exp(log_std)); and the Python numbers n_updates (epochs run by this call; SB3 adds them to its
    running _n_updates) and clip_range.

    With target_kl=None (SB3's default) the call never synchronises the host.  With target_kl set, each minibatch reads
    its approx_kl (one sync per minibatch) and, like SB3, stops before the optimizer step once it exceeds
    1.5 * target_kl; that epoch still counts in n_updates."""
    if not buffer.full:
        raise FleetStepError("ppo_train: the buffer is not full")
    dev = buffer.device
    policy.train(True)
    n = buffer.buffer_size * buffer.n_envs
    n_batches = -(-n // int(batch_size))
    acc = torch.zeros((n_epochs, n_batches, len(STATS)), dtype=torch.float64, device=dev)
    params = _params(clip_range, clip_range_vf, normalize_advantage, ent_coef, vf_coef)
    loss, n_updates, ran, last_epoch_batches = None, 0, 0, 0
    for epoch in range(n_epochs):
        continue_training = True
        last_epoch_batches = 0
        for j, data in enumerate(buffer.get(batch_size, generator=generator)):
            mean_actions, log_std, values = policy.loss_inputs(data.observations)
            loss = _PpoLoss.apply(mean_actions, log_std, values, data, params, acc[epoch, j])
            ran += 1
            last_epoch_batches += 1
            if target_kl is not None and float(acc[epoch, j, 4]) > 1.5 * target_kl:
                continue_training = False
                break
            policy.optimizer.zero_grad()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(policy.parameters(), max_grad_norm)
            policy.optimizer.step()
        n_updates += 1
        if not continue_training:
            break

    rows = acc.view(-1, len(STATS))[:ran]
    means = rows.sum(0) / ran
    last = acc[n_updates - 1, :last_epoch_batches, 4].sum() / last_epoch_batches
    values, returns = buffer.values.double().flatten(), buffer.returns.double().flatten()
    var_y = returns.var(unbiased=False)
    explained_var = torch.where(var_y == 0, torch.full_like(var_y, float("nan")),
                                1 - (returns - values).var(unbiased=False) / var_y)
    return {
        "train/entropy_loss": means[2],
        "train/policy_gradient_loss": means[0],
        "train/value_loss": means[1],
        "train/approx_kl": last,
        "train/clip_fraction": means[3],
        "train/loss": loss.detach(),
        "train/explained_variance": explained_var,
        "train/std": policy.log_std.detach().double().exp().mean(),
        "train/n_updates": n_updates,
        "train/clip_range": clip_range,
    }
