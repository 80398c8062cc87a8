"""FleetRolloutBuffer — stable-baselines3 2.3.2's RolloutBuffer (common/buffers.py) on the device, and collect_rollouts, the
loop of OnPolicyAlgorithm.collect_rollouts (common/on_policy_algorithm.py) over FleetVecEnv / FleetVecNormalize.

SB3's buffer is a set of host NumPy arrays: it cannot take CUDA observations, and at FleetVecEnv's sizes it would pull
every observation batch over PCIe.  This one keeps the transitions in torch-owned HBM and runs add, the GAE scan and the
minibatch gather as kernels of libfleetstep (fleet_rollout_*), with SB3's attribute names, defaults and float32
arithmetic: advantages and returns equal SB3's bit for bit.

Differences from SB3, all deliberate:
  * the attributes keep their [T, E, ...] layout after get(): there is no swap_and_flatten copy, the gather kernel maps
    SB3's env-major flat sample index k to step k % T, env k // T; the samples are the same;
  * get() draws its permutation with torch.randperm on the device (optionally from `generator`), so the order differs
    from SB3's np.random.permutation; `indices=` injects a permutation;
  * reset() rewinds pos / full without clearing memory;
  * compute_returns_and_advantage and get raise until the buffer is full; add on a full buffer raises;
  * collect_rollouts does no timeout bootstrapping: SB3 adds gamma * V(terminal_obs) to the reward only where
    infos[i]["TimeLimit.truncated"] is true, and FleetVecEnv reports it false, as the reference's step returns
    truncated=False.
"""
from typing import NamedTuple

import torch

from ._lib import FleetRolloutBuf, FleetStepError, _dptr, _stream_ptr, load_library


class RolloutBufferSamples(NamedTuple):
    """SB3's type_aliases.RolloutBufferSamples."""
    observations: torch.Tensor
    actions: torch.Tensor
    old_values: torch.Tensor
    old_log_prob: torch.Tensor
    advantages: torch.Tensor
    returns: torch.Tensor


_ARRAYS = ("observations", "actions", "rewards", "episode_starts", "values", "log_probs", "advantages", "returns")


class FleetRolloutBuffer:
    """RolloutBuffer(buffer_size, observation_space, action_space, device, gae_lambda, gamma, n_envs) for a Box observation
    of obs_dim and a Box action of action_dim, on a CUDA device.  observations [T, E, obs_dim], actions [T, E, action_dim]
    and rewards, episode_starts, values, log_probs, advantages, returns [T, E] are float32 tensors."""

    def __init__(self, buffer_size, num_envs, obs_dim, action_dim, device, gamma=0.99, gae_lambda=1.0):
        self.lib = load_library()
        self.buffer_size, self.n_envs = int(buffer_size), int(num_envs)
        self.obs_dim, self.action_dim = int(obs_dim), int(action_dim)
        if min(self.buffer_size, self.n_envs, self.obs_dim, self.action_dim) < 1:
            raise FleetStepError("buffer_size, num_envs, obs_dim and action_dim must be >= 1")
        if not (0.0 <= float(gamma) <= 1.0 and 0.0 <= float(gae_lambda) <= 1.0):
            raise FleetStepError("gamma and gae_lambda must be in [0, 1]")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise FleetStepError("FleetRolloutBuffer lives on a CUDA device; there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.gamma, self.gae_lambda = gamma, gae_lambda
        T, E = self.buffer_size, self.n_envs
        f = dict(dtype=torch.float32, device=self.device)
        self.observations = torch.zeros((T, E, self.obs_dim), **f)
        self.actions = torch.zeros((T, E, self.action_dim), **f)
        for name in _ARRAYS[2:]:
            setattr(self, name, torch.zeros((T, E), **f))
        self._desc = FleetRolloutBuf(T, E, self.obs_dim, self.action_dim, *[getattr(self, n).data_ptr() for n in _ARRAYS])
        self.reset()

    @property
    def num_envs(self):
        return self.n_envs

    def reset(self):
        """Rewind to slot 0 (SB3 also zeroes the arrays; every slot is written again before it is read)."""
        self.pos = 0
        self.full = False

    def size(self):
        return self.buffer_size if self.full else self.pos

    # ---- inputs
    def _check(self, rc, what):
        if rc != 0:
            raise FleetStepError(f"{what}: {self.lib.fleet_rollout_last_error().decode()} (code {rc})")

    def _tensor(self, t, shape, name, flags=False):
        """t on this device, of `shape` (a trailing 1 of values / log-probs is accepted), contiguous; float dtypes are cast
        to float32 as SB3's assignment casts.  flags=True: bool and uint8 pass through as uint8 (episode starts, dones)."""
        if not isinstance(t, torch.Tensor):
            raise FleetStepError(f"{name}: expected a torch tensor on {self.device}, got {type(t).__name__}")
        if t.device != self.device:
            raise FleetStepError(f"{name}: expected a tensor on {self.device}, got one on {t.device}")
        if tuple(t.shape) != tuple(shape) and not (t.dim() == len(shape) + 1 and tuple(t.shape) == tuple(shape) + (1,)):
            raise FleetStepError(f"{name}: expected shape {tuple(shape)}, got {tuple(t.shape)}")
        if not t.is_contiguous():
            raise FleetStepError(f"{name}: expected a contiguous tensor")
        if flags and t.dtype in (torch.bool, torch.uint8):
            return t.view(torch.uint8)
        if not t.dtype.is_floating_point:
            raise FleetStepError(f"{name}: expected a floating-point tensor, got {t.dtype}")
        return t.reshape(shape) if t.dtype == torch.float32 else t.reshape(shape).float()

    def _write(self, slot, obs=None, action=None, reward=None, episode_start=None, value=None, log_prob=None):
        """fleet_rollout_add into `slot` for the fields given; the others keep their contents."""
        E = self.n_envs
        obs = None if obs is None else self._tensor(obs, (E, self.obs_dim), "obs")
        action = None if action is None else self._tensor(action, (E, self.action_dim), "action")
        reward = None if reward is None else self._tensor(reward, (E,), "reward")
        value = None if value is None else self._tensor(value, (E,), "value")
        log_prob = None if log_prob is None else self._tensor(log_prob, (E,), "log_prob")
        start = None
        if episode_start is not None:
            start = self._tensor(episode_start, (E,), "episode_start", flags=True)
            if start.dtype == torch.float32:    # a float flag is stored as it is, like SB3's float32 assignment
                self.episode_starts[slot].copy_(start)
                start = None
        with torch.cuda.device(self.device):
            self._check(self.lib.fleet_rollout_add(self._desc, int(slot), _dptr(obs), _dptr(action), _dptr(reward),
                                                   _dptr(start), _dptr(value), _dptr(log_prob), _stream_ptr(self.device)),
                        "fleet_rollout_add")

    # ---- RolloutBuffer
    def add(self, obs, action, reward, episode_start, value, log_prob):
        """Store one transition of every env in slot pos (SB3's signature; values [E, 1] are flattened)."""
        if self.full:
            raise FleetStepError("add: the buffer is full; call reset() first")
        self._write(self.pos, obs, action, reward, episode_start, value, log_prob)
        self._advance()

    def _advance(self):
        self.pos += 1
        if self.pos == self.buffer_size:
            self.full = True

    def compute_returns_and_advantage(self, last_values, dones):
        """GAE(lambda) advantages and returns = advantages + values, SB3's float32 arithmetic bit for bit.
        last_values [E] or [E, 1]: the value of the observation after the last step; dones [E] (bool / uint8 / float)."""
        if not self.full:
            raise FleetStepError("compute_returns_and_advantage: the buffer is not full")
        E = self.n_envs
        lv = self._tensor(last_values, (E,), "last_values")
        d = self._tensor(dones, (E,), "dones", flags=True)
        if d.dtype != torch.uint8:
            d = d.to(torch.uint8)
        with torch.cuda.device(self.device):
            self._check(self.lib.fleet_rollout_gae(self._desc, float(self.gamma), float(self.gae_lambda), _dptr(lv), _dptr(d),
                                                   _stream_ptr(self.device)), "fleet_rollout_gae")

    def get(self, batch_size=None, generator=None, indices=None):
        """Yield RolloutBufferSamples over a permutation of the T*E samples, batch_size at a time (the last batch may be
        smaller).  SB3's flat sample k is env k // T, step k % T.  indices: an injected permutation (int, length T*E)."""
        if not self.full:
            raise FleetStepError("get: the buffer is not full")
        n = self.buffer_size * self.n_envs
        if indices is None:
            perm = torch.randperm(n, device=self.device, generator=generator)
        else:
            perm = torch.as_tensor(indices).to(device=self.device, dtype=torch.int64).contiguous()
            if perm.shape != (n,):
                raise FleetStepError(f"indices: expected {n} indices, got shape {tuple(perm.shape)}")
            if n and bool(((perm < 0) | (perm >= n)).any()):
                raise FleetStepError(f"indices: every index must lie in [0, {n})")
        if batch_size is None:
            batch_size = n
        start = 0
        while start < n:
            yield self._get_samples(perm[start:start + batch_size])
            start += batch_size

    def _get_samples(self, batch_inds):
        b = batch_inds.shape[0]
        f = dict(dtype=torch.float32, device=self.device)
        out = RolloutBufferSamples(torch.empty((b, self.obs_dim), **f), torch.empty((b, self.action_dim), **f),
                                   *[torch.empty(b, **f) for _ in range(4)])
        with torch.cuda.device(self.device):
            self._check(self.lib.fleet_rollout_gather(self._desc, _dptr(batch_inds), int(b), *[_dptr(t) for t in out],
                                                      _stream_ptr(self.device)), "fleet_rollout_gather")
        return out


def collect_rollouts(venv, policy, buffer: FleetRolloutBuffer, last_obs, last_episode_starts):
    """OnPolicyAlgorithm.collect_rollouts on the device: fill `buffer` with buffer_size steps of `venv` (FleetVecEnv or
    FleetVecNormalize, through step_raw) and compute its advantages and returns, with no host synchronisation.

    policy: anything with forward(obs) -> (actions, values, log_probs) and predict_values(obs), e.g. an SB3
    ActorCriticPolicy on the env's GPU.  Like SB3, the buffer stores the unclipped actions, the env is stepped with
    clamp(actions, -1, 1), and episode_starts are the previous step's dones.  No timeout bootstrapping (module docstring).
    First call: last_obs = venv.reset(), last_episode_starts = ones(E) (SB3's _setup_learn).  Returns the
    (last_obs, last_episode_starts) the next call takes: views of venv's output buffers, valid until venv steps again.
    """
    buffer.reset()
    with torch.no_grad():
        for t in range(buffer.buffer_size):
            actions, values, log_probs = policy.forward(last_obs)
            # step_raw overwrites the buffers last_obs and last_episode_starts view: store them first, the reward after
            buffer._write(t, obs=last_obs, action=actions, episode_start=last_episode_starts, value=values,
                          log_prob=log_probs)
            new_obs, rewards, dones = venv.step_raw(torch.clamp(actions, -1.0, 1.0))
            buffer._write(t, reward=rewards)
            buffer._advance()
            last_obs, last_episode_starts = new_obs, dones
        buffer.compute_returns_and_advantage(policy.predict_values(last_obs), last_episode_starts)
    return last_obs, last_episode_starts
