"""NumPy restatement of stable-baselines3 2.3.2's VecNormalize (common/vec_env/vec_normalize.py) and RunningMeanStd
(common/running_mean_std.py), line by line, for Box observations.

TEST INFRASTRUCTURE ONLY: the reference that tests/test_gpu_normalize.py checks fleetrl_b200's device VecNormalize
against.  The product package never imports this module.

One deliberate deviation from SB3, shared with the device implementation: RunningMeanStd.update reduces the batch mean
and variance in float64.  SB3 calls np.mean / np.var on the array as it comes, i.e. in float32 for FleetEnv's
observations, so its statistics carry float32 rounding; these are more accurate and differ from SB3's at that level.
Everything after the batch moments (update_from_moments, the normalisation formulas, the returns) is SB3's float64
arithmetic in SB3's order.
"""
import numpy as np


class RunningMeanStd:
    def __init__(self, epsilon: float = 1e-4, shape=()):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = epsilon

    def update(self, arr: np.ndarray) -> None:
        arr = np.asarray(arr, dtype=np.float64)          # the deviation: SB3 reduces in arr's own dtype
        batch_mean = np.mean(arr, axis=0)
        batch_var = np.var(arr, axis=0)
        batch_count = arr.shape[0]
        self.update_from_moments(batch_mean, batch_var, batch_count)

    def update_from_moments(self, batch_mean, batch_var, batch_count) -> None:
        delta = batch_mean - self.mean
        tot_count = self.count + batch_count

        new_mean = self.mean + delta * batch_count / tot_count
        m_a = self.var * self.count
        m_b = batch_var * batch_count
        m_2 = m_a + m_b + np.square(delta) * self.count * batch_count / (self.count + batch_count)
        new_var = m_2 / (self.count + batch_count)

        new_count = batch_count + self.count

        self.mean = new_mean
        self.var = new_var
        self.count = new_count


class VecNormalize:
    """SB3's VecNormalize over any object with num_envs, reset() and step_async / step_wait returning
    (obs, rewards, dones, infos) with infos[i]["terminal_observation"] for finished envs."""

    def __init__(self, venv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                 epsilon=1e-8, obs_shape=None):
        self.venv = venv
        self.num_envs = venv.num_envs
        self.obs_rms = RunningMeanStd(shape=obs_shape if obs_shape is not None else venv.observation_space.shape)
        self.ret_rms = RunningMeanStd(shape=())
        self.clip_obs = clip_obs
        self.clip_reward = clip_reward
        self.returns = np.zeros(self.num_envs)
        self.gamma = gamma
        self.epsilon = epsilon
        self.training = training
        self.norm_obs = norm_obs
        self.norm_reward = norm_reward
        self.old_obs = np.array([])
        self.old_reward = np.array([])

    def step_async(self, actions):
        self.venv.step_async(actions)

    def step_wait(self):
        obs, rewards, dones, infos = self.venv.step_wait()
        self.old_obs = obs
        self.old_reward = rewards

        if self.training and self.norm_obs:
            self.obs_rms.update(obs)

        obs = self.normalize_obs(obs)

        if self.training:
            self._update_reward(rewards)
        rewards = self.normalize_reward(rewards)

        # Normalize the terminal observations
        for idx, done in enumerate(dones):
            if not done:
                continue
            if "terminal_observation" in infos[idx]:
                infos[idx]["terminal_observation"] = self.normalize_obs(infos[idx]["terminal_observation"])

        self.returns[dones] = 0
        return obs, rewards, dones, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def _update_reward(self, reward: np.ndarray) -> None:
        self.returns = self.returns * self.gamma + reward
        self.ret_rms.update(self.returns)

    def _normalize_obs(self, obs, obs_rms):
        return np.clip((obs - obs_rms.mean) / np.sqrt(obs_rms.var + self.epsilon), -self.clip_obs, self.clip_obs)

    def normalize_obs(self, obs):
        obs_ = np.array(obs, copy=True)
        if self.norm_obs:
            obs_ = self._normalize_obs(obs, self.obs_rms).astype(np.float32)
        return obs_

    def normalize_reward(self, reward):
        if self.norm_reward:
            reward = np.clip(reward / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward, self.clip_reward)
        return reward

    def get_original_obs(self):
        return self.old_obs.copy()

    def get_original_reward(self):
        return self.old_reward.copy()

    def reset(self):
        obs = self.venv.reset()
        self.old_obs = obs
        self.returns = np.zeros(self.num_envs)
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)
