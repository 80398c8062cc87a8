"""stable-baselines3 2.3.2's DiagGaussianDistribution (common/distributions.py) and the loss and loop of PPO.train
(ppo/ppo.py), restated line by line in torch float64 on the CPU with autograd.  The reference for fleet_ppo_* and for
fleetrl_b200.ppo.ppo_train.

Inputs are cast to float64 here; every reduction SB3 makes is a float64 torch reduction.
"""
import torch
from torch import nn
from torch.distributions import Normal


F64 = torch.float64


def distribution(mean_actions, log_std):
    """DiagGaussianDistribution.proba_distribution: Normal(mean, ones_like(mean) * log_std.exp())."""
    action_std = torch.ones_like(mean_actions) * log_std.exp()
    return Normal(mean_actions, action_std)


def log_prob(mean_actions, log_std, actions):
    """DiagGaussianDistribution.log_prob: sum_independent_dims(Normal.log_prob(actions))."""
    return distribution(mean_actions, log_std).log_prob(actions).sum(dim=1)


def entropy(mean_actions, log_std):
    return distribution(mean_actions, log_std).entropy().sum(dim=1)


def loss(mean_actions, log_std, values, actions, old_log_prob, old_values, advantages, returns, clip_range=0.2,
         clip_range_vf=None, normalize_advantage=True, ent_coef=0.0, vf_coef=0.5):
    """The loss of one minibatch of PPO.train and the five values it logs (0-dim tensors):
    (loss, dict(policy_gradient_loss, value_loss, entropy_loss, clip_fraction, approx_kl))."""
    log_prob_ = log_prob(mean_actions, log_std, actions)
    entropy_ = entropy(mean_actions, log_std)
    values = values.flatten()
    if normalize_advantage and len(advantages) > 1:
        advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
    ratio = torch.exp(log_prob_ - old_log_prob)
    policy_loss_1 = advantages * ratio
    policy_loss_2 = advantages * torch.clamp(ratio, 1 - clip_range, 1 + clip_range)
    policy_loss = -torch.min(policy_loss_1, policy_loss_2).mean()
    clip_fraction = torch.mean((torch.abs(ratio - 1) > clip_range).to(F64))
    if clip_range_vf is None:
        values_pred = values
    else:
        values_pred = old_values + torch.clamp(values - old_values, -clip_range_vf, clip_range_vf)
    value_loss = nn.functional.mse_loss(returns, values_pred)
    entropy_loss = -torch.mean(entropy_)
    total = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
    with torch.no_grad():
        log_ratio = log_prob_ - old_log_prob
        approx_kl = torch.mean((torch.exp(log_ratio) - 1) - log_ratio)
    stats = dict(policy_gradient_loss=policy_loss.detach(), value_loss=value_loss.detach(),
                 entropy_loss=entropy_loss.detach(), clip_fraction=clip_fraction, approx_kl=approx_kl)
    return total, stats


def loss_and_grads(mean_actions, log_std, values, actions, old_log_prob, old_values, advantages, returns, **kw):
    """loss() on float64 copies of the inputs, with the gradients of the loss w.r.t. mean_actions, log_std, values."""
    d = lambda a: torch.as_tensor(a).to(F64).clone()   # noqa: E731
    mean_actions, log_std, values = (d(t).requires_grad_(True) for t in (mean_actions, log_std, values))
    total, stats = loss(mean_actions, log_std, values, d(actions), d(old_log_prob), d(old_values), d(advantages),
                        d(returns), **kw)
    total.backward()
    return total.detach(), stats, mean_actions.grad, log_std.grad, values.grad


class MlpPolicy(nn.Module):
    """ActorCriticPolicy with MlpPolicy's networks in float64 (the attribute names and order of fleetrl_b200's
    FleetMlpPolicy, so load_state_dict copies one into the other)."""

    def __init__(self, obs_dim, action_dim, lr=3e-4):
        super().__init__()
        self.log_std = nn.Parameter(torch.zeros(action_dim, dtype=F64))
        self.mlp_extractor = nn.Module()
        mk = lambda: nn.Sequential(nn.Linear(obs_dim, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())   # noqa: E731
        self.mlp_extractor.policy_net = mk()
        self.mlp_extractor.value_net = mk()
        self.action_net = nn.Linear(64, action_dim)
        self.value_net = nn.Linear(64, 1)
        self.to(F64)
        self.lr = lr

    def make_optimizer(self):
        self.optimizer = torch.optim.Adam(self.parameters(), lr=self.lr, eps=1e-5)

    def loss_inputs(self, obs):
        mean = self.action_net(self.mlp_extractor.policy_net(obs))
        return mean, self.log_std, self.value_net(self.mlp_extractor.value_net(obs)).flatten()


def explained_variance(y_pred, y_true):
    """common/utils.py explained_variance."""
    var_y = torch.var(y_true, unbiased=False)
    return float("nan") if var_y == 0 else float(1 - torch.var(y_true - y_pred, unbiased=False) / var_y)


def train(policy, flat, perms, batch_size, n_epochs=10, clip_range=0.2, clip_range_vf=None, normalize_advantage=True,
          ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, target_kl=None, on_step=None, log=None):
    """PPO.train over flattened rollout data (SB3's swap_and_flatten order): flat = dict of float64 tensors
    observations [n, D], actions [n, N], values, log_probs, advantages, returns [n]; perms = one index permutation per
    epoch.  on_step(policy) is called before each optimizer step (after clipping); log, a list, receives
    (epoch, stats) of every minibatch.  Returns SB3's logged values and the
    number of optimizer steps."""
    entropy_losses, pg_losses, value_losses, clip_fractions = [], [], [], []
    n_updates, steps, continue_training, total = 0, 0, True, None
    n = flat["observations"].shape[0]
    for epoch in range(n_epochs):
        approx_kl_divs = []
        perm = perms[epoch]
        for start in range(0, n, batch_size):
            idx = perm[start:start + batch_size]
            mean, log_std, values = policy.loss_inputs(flat["observations"][idx])
            total, st = loss(mean, log_std, values, flat["actions"][idx], flat["log_probs"][idx], flat["values"][idx],
                             flat["advantages"][idx], flat["returns"][idx], clip_range=clip_range,
                             clip_range_vf=clip_range_vf, normalize_advantage=normalize_advantage, ent_coef=ent_coef,
                             vf_coef=vf_coef)
            pg_losses.append(st["policy_gradient_loss"].item())
            clip_fractions.append(st["clip_fraction"].item())
            value_losses.append(st["value_loss"].item())
            entropy_losses.append(st["entropy_loss"].item())
            approx_kl_divs.append(st["approx_kl"].item())
            if log is not None:
                log.append((epoch, {k: v.item() for k, v in st.items()}))
            if target_kl is not None and approx_kl_divs[-1] > 1.5 * target_kl:
                continue_training = False
                break
            policy.optimizer.zero_grad()
            total.backward()
            nn.utils.clip_grad_norm_(policy.parameters(), max_grad_norm)
            if on_step is not None:
                on_step(policy)
            policy.optimizer.step()
            steps += 1
        n_updates += 1
        if not continue_training:
            break
    mean = lambda xs: sum(xs) / len(xs)   # noqa: E731
    return {
        "train/entropy_loss": mean(entropy_losses),
        "train/policy_gradient_loss": mean(pg_losses),
        "train/value_loss": mean(value_losses),
        "train/approx_kl": mean(approx_kl_divs),
        "train/clip_fraction": mean(clip_fractions),
        "train/loss": total.item(),
        "train/explained_variance": explained_variance(flat["values"], flat["returns"]),
        "train/std": torch.exp(policy.log_std).mean().item(),
        "train/n_updates": n_updates,
        "train/clip_range": clip_range,
    }, steps
