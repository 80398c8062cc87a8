"""NumPy restatement of stable-baselines3 2.3.2's RolloutBuffer (common/buffers.py: reset, add,
compute_returns_and_advantage, swap_and_flatten, get, _get_samples) and of the loop body of
OnPolicyAlgorithm.collect_rollouts (common/on_policy_algorithm.py), line by line, for Box observations and actions.

TEST INFRASTRUCTURE ONLY: the reference that tests/test_gpu_rollout.py checks fleetrl_b200's device RolloutBuffer against.
The product package never imports this module.  Tensors are NumPy arrays here (SB3's .cpu().numpy() calls are dropped).

The float32 order of compute_returns_and_advantage, as NumPy 2 evaluates SB3's lines when gamma and gae_lambda are Python
floats (as PPO passes them) and the arrays are float32: a Python float meeting a float32 array is rounded to float32, the
product gamma * gae_lambda is formed in double first, and every array intermediate is float32:
    g  = float32(gamma)            gl = float32(gamma * gae_lambda)
    t = T-1:  nnt = 1 - float32(dones);        nv = last_values
    t < T-1:  nnt = 1 - episode_starts[t+1];   nv = values[t+1]
    delta = (rewards[t] + (g * nv) * nnt) - values[t]
    lgl   = delta + (gl * nnt) * lgl          # lgl = 0 before t = T-1
    advantages[t] = lgl;   returns = advantages + values
"""
import numpy as np


class RolloutBuffer:
    def __init__(self, buffer_size, obs_dim, action_dim, gae_lambda=1, gamma=0.99, n_envs=1):
        self.buffer_size = buffer_size
        self.obs_shape = (obs_dim,)
        self.action_dim = action_dim
        self.n_envs = n_envs
        self.gae_lambda = gae_lambda
        self.gamma = gamma
        self.pos = 0
        self.full = False
        self.generator_ready = False
        self.reset()

    @staticmethod
    def swap_and_flatten(arr: np.ndarray) -> np.ndarray:
        shape = arr.shape
        if len(shape) < 3:
            shape = (*shape, 1)
        return arr.swapaxes(0, 1).reshape(shape[0] * shape[1], *shape[2:])

    def size(self) -> int:
        if self.full:
            return self.buffer_size
        return self.pos

    def reset(self) -> None:
        self.observations = np.zeros((self.buffer_size, self.n_envs, *self.obs_shape), dtype=np.float32)
        self.actions = np.zeros((self.buffer_size, self.n_envs, self.action_dim), dtype=np.float32)
        self.rewards = np.zeros((self.buffer_size, self.n_envs), dtype=np.float32)
        self.returns = np.zeros((self.buffer_size, self.n_envs), dtype=np.float32)
        self.episode_starts = np.zeros((self.buffer_size, self.n_envs), dtype=np.float32)
        self.values = np.zeros((self.buffer_size, self.n_envs), dtype=np.float32)
        self.log_probs = np.zeros((self.buffer_size, self.n_envs), dtype=np.float32)
        self.advantages = np.zeros((self.buffer_size, self.n_envs), dtype=np.float32)
        self.generator_ready = False
        self.pos = 0
        self.full = False

    def compute_returns_and_advantage(self, last_values: np.ndarray, dones: np.ndarray) -> None:
        # Convert to numpy
        last_values = np.array(last_values, dtype=np.float32).flatten()

        last_gae_lam = 0
        for step in reversed(range(self.buffer_size)):
            if step == self.buffer_size - 1:
                next_non_terminal = 1.0 - dones.astype(np.float32)
                next_values = last_values
            else:
                next_non_terminal = 1.0 - self.episode_starts[step + 1]
                next_values = self.values[step + 1]
            delta = self.rewards[step] + self.gamma * next_values * next_non_terminal - self.values[step]
            last_gae_lam = delta + self.gamma * self.gae_lambda * next_non_terminal * last_gae_lam
            self.advantages[step] = last_gae_lam
        # TD(lambda) estimator, see Github PR #375 or "Telescoping in TD(lambda)"
        # in David Silver Lecture 4: https://www.youtube.com/watch?v=PnHCvfgC_ZA
        self.returns = self.advantages + self.values

    def add(self, obs, action, reward, episode_start, value, log_prob) -> None:
        log_prob = np.asarray(log_prob)
        if len(log_prob.shape) == 0:
            # Reshape 0-d tensor to avoid error
            log_prob = log_prob.reshape(-1, 1)

        # Reshape to handle multi-dim and discrete action spaces, see GH #970 #1392
        action = np.asarray(action).reshape((self.n_envs, self.action_dim))

        self.observations[self.pos] = np.array(obs)
        self.actions[self.pos] = np.array(action)
        self.rewards[self.pos] = np.array(reward)
        self.episode_starts[self.pos] = np.array(episode_start)
        self.values[self.pos] = np.array(value).flatten()
        self.log_probs[self.pos] = np.array(log_prob)
        self.pos += 1
        if self.pos == self.buffer_size:
            self.full = True

    def get(self, batch_size=None, indices=None):
        assert self.full, ""
        if indices is None:      # injected for parity runs; SB3 always draws it here
            indices = np.random.permutation(self.buffer_size * self.n_envs)
        # Prepare the data
        if not self.generator_ready:
            _tensor_names = ["observations", "actions", "values", "log_probs", "advantages", "returns"]

            for tensor in _tensor_names:
                self.__dict__[tensor] = self.swap_and_flatten(self.__dict__[tensor])
            self.generator_ready = True

        # Return everything, don't create minibatches
        if batch_size is None:
            batch_size = self.buffer_size * self.n_envs

        start_idx = 0
        while start_idx < self.buffer_size * self.n_envs:
            yield self._get_samples(indices[start_idx : start_idx + batch_size])
            start_idx += batch_size

    def _get_samples(self, batch_inds: np.ndarray):
        data = (
            self.observations[batch_inds],
            self.actions[batch_inds],
            self.values[batch_inds].flatten(),
            self.log_probs[batch_inds].flatten(),
            self.advantages[batch_inds].flatten(),
            self.returns[batch_inds].flatten(),
        )
        return data   # SB3: RolloutBufferSamples(*tuple(map(self.to_torch, data)))


def collect_rollouts(env_step, policy, predict_values, rollout_buffer, n_rollout_steps, last_obs, last_episode_starts,
                     gamma=0.99, low=-1.0, high=1.0):
    """The loop of OnPolicyAlgorithm.collect_rollouts for a Box action space without squashing.  env_step(actions) ->
    (new_obs, rewards, dones, infos); policy(obs) -> (actions, values, log_probs); predict_values(obs) -> values.
    Returns (last_obs, last_episode_starts) as SB3 leaves self._last_obs / self._last_episode_starts."""
    n_steps = 0
    rollout_buffer.reset()
    while n_steps < n_rollout_steps:
        actions, values, log_probs = policy(last_obs)
        clipped_actions = np.clip(actions, low, high)
        new_obs, rewards, dones, infos = env_step(clipped_actions)
        n_steps += 1
        # Handle timeout by bootstrapping with value function
        for idx, done in enumerate(dones):
            if (
                done
                and infos[idx].get("terminal_observation") is not None
                and infos[idx].get("TimeLimit.truncated", False)
            ):
                terminal_value = predict_values(infos[idx]["terminal_observation"][None])[0]
                rewards[idx] += gamma * terminal_value
        rollout_buffer.add(last_obs, actions, rewards, last_episode_starts, values, log_probs)
        last_obs = new_obs
        last_episode_starts = dones
    values = predict_values(new_obs)
    rollout_buffer.compute_returns_and_advantage(last_values=values, dones=dones)
    return last_obs, last_episode_starts
