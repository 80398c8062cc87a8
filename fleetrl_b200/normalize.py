"""FleetVecNormalize — stable-baselines3 2.3.2's VecNormalize (common/vec_env/vec_normalize.py) on the device.

The reference trains with make_vec_env(FleetEnv) -> VecNormalize -> PPO and evaluates with saved VecNormalize statistics.
SB3's wrapper is NumPy-only: it would pull every observation batch to the host.  This one keeps the running statistics,
the discounted returns and the normalised outputs in HBM (libfleetstep's fleet_norm_*: two kernel launches per training
step, no host synchronisation) with SB3's arithmetic, order of operations and defaults.

Differences from SB3, all deliberate:
  * the batch mean / variance are reduced in float64 (SB3 reduces in the observation dtype, float32), so the statistics
    are more accurate than SB3's and differ from them at float32 rounding level;
  * normalised rewards are float32 (SB3 returns float64 under NumPy 2);
  * obs_rms / ret_rms return snapshots; assign an object with mean / var / count to load statistics (that is how saved
    SB3 statistics come in).  SB3's pickles (VecNormalize.load) and sync_envs_normalization need SB3's own class.
With sync=True and an initialised multi-rank torch.distributed, every training step all-reduces the batch moments
(2*D+4 float64) between the two kernels, so that all ranks of FleetVecEnv.sharded keep identical statistics.
"""
import numpy as np
import torch

from . import dist as _dist
from ._lib import FleetNormHandle

try:  # pragma: no cover - stable-baselines3 is third party and not part of the build image
    from stable_baselines3.common.vec_env import VecEnvWrapper as _WrapperBase
except Exception:
    _WrapperBase = object


class RunningMeanStd:
    """Snapshot of a running mean / variance (the attributes of SB3's common/running_mean_std.RunningMeanStd)."""

    def __init__(self, mean, var, count):
        self.mean, self.var, self.count = mean, var, count

    def __repr__(self):
        return f"RunningMeanStd(mean={self.mean!r}, var={self.var!r}, count={self.count!r})"


class FleetVecNormalize(_WrapperBase):
    """VecNormalize over a FleetVecEnv (torch or numpy output), same constructor arguments and defaults as SB3's.

    When stable-baselines3 is importable this class IS a stable_baselines3 VecEnvWrapper; without it the same protocol is
    duck-typed.  torch mode returns device tensors that the next step overwrites; numpy mode returns fresh arrays.
    """

    def __init__(self, venv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                 epsilon=1e-8, sync=True):
        if _WrapperBase is not object:
            _WrapperBase.__init__(self, venv)
        self.venv = venv
        self.num_envs = venv.num_envs
        self.observation_space, self.action_space = venv.observation_space, venv.action_space
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = float(clip_obs), float(clip_reward), float(gamma), float(epsilon)
        self.sync = bool(sync)
        E, D = venv.num_envs, venv.obs_dim
        self.handle = FleetNormHandle(E, D, venv.device, clip_obs, clip_reward, gamma, epsilon)
        self._flags = [bool(training), bool(norm_obs), bool(norm_reward)]
        self.handle.set_flags(*self._flags)
        dev = venv.device
        self._obs_n = torch.zeros((E, D), dtype=torch.float32, device=dev)
        self._term_n = torch.zeros((E, D), dtype=torch.float32, device=dev)
        self._rew_n = torch.zeros(E, dtype=torch.float32, device=dev)
        self._moments = torch.zeros(self.handle.moments_len, dtype=torch.float64, device=dev)
        self._actions = None

    # ---- the attributes SB3 callers toggle (evaluation: training = False, norm_reward = False)
    def _flag(i):
        def get(self):
            return self._flags[i]

        def put(self, value):
            self._flags[i] = bool(value)
            self.handle.set_flags(*self._flags)
        return property(get, put)

    training, norm_obs, norm_reward = _flag(0), _flag(1), _flag(2)
    del _flag

    # ---- running statistics (each read synchronises; assigning loads them)
    @property
    def obs_rms(self):
        s = self.handle.get_state()
        return RunningMeanStd(s["obs_mean"], s["obs_var"], float(s["obs_count"]))

    @obs_rms.setter
    def obs_rms(self, rms):
        self.handle.set_state(obs_mean=np.broadcast_to(np.asarray(rms.mean, np.float64), (self.handle.D,)),
                              obs_var=np.broadcast_to(np.asarray(rms.var, np.float64), (self.handle.D,)),
                              obs_count=np.float64(rms.count))

    @property
    def ret_rms(self):
        s = self.handle.get_state()
        return RunningMeanStd(s["ret_mean"][()], s["ret_var"][()], float(s["ret_count"]))

    @ret_rms.setter
    def ret_rms(self, rms):
        self.handle.set_state(ret_mean=np.float64(np.reshape(rms.mean, ())), ret_var=np.float64(np.reshape(rms.var, ())),
                              ret_count=np.float64(rms.count))

    @property
    def returns(self):
        return self.handle.get_state()["returns"]

    def state_dict(self):
        """Statistics and discounted returns (float64): load_state_dict resumes bit for bit."""
        return self.handle.get_state()

    def load_state_dict(self, d):
        self.handle.set_state(**{k: d[k] for k in self.handle.STATE})

    # ---- VecEnv protocol
    def _is_numpy(self):
        return self.venv.output == "numpy"

    def _out(self, t):
        return t.cpu().numpy() if self._is_numpy() else t

    def _update_and_normalize(self, obs, rew=None, done=None, term=None):
        m = None
        if self._flags[0]:
            m = self._moments
            self.handle.moments(obs, rew, m)
            if self.sync:
                _dist.all_reduce_moments(m)
        self.handle.apply(m, obs, self._obs_n, rew, None if rew is None else self._rew_n, done, term,
                          None if term is None else self._term_n)

    def reset(self, **kwargs):
        self.venv.reset(**kwargs)
        self.handle.reset_returns()
        self._update_and_normalize(self.venv._obs)
        return self._out(self._obs_n)

    def step_async(self, actions):
        self._actions = actions

    def step_raw(self, actions: torch.Tensor):
        """Hot-loop variant for on-device rollouts: views of the normalised obs, normalised rewards and done flags, no
        infos, no host synchronisation.  Normalised terminal rows of finished envs are in `terminal_observations`."""
        v = self.venv
        v.handle.step(actions, v._obs, v._rew, v._done, v._term)
        self._update_and_normalize(v._obs, v._rew, v._done, v._term)
        return self._obs_n, self._rew_n, v._done

    @property
    def terminal_observations(self):
        return self._term_n

    def step_wait(self):
        v = self.venv
        E, N = v.num_envs, v.num_cars
        a = torch.as_tensor(np.asarray(self._actions, dtype=np.float32) if self._is_numpy() else self._actions,
                            dtype=torch.float32).to(v.device).reshape(E, N).contiguous()
        obs, rew, done = self.step_raw(a)
        if self._is_numpy():
            done_np = done.cpu().numpy().astype(bool)
            v._last_done = done_np
            infos = v._infos(np.nonzero(done_np)[0], terminal_obs=self._term_n)
            return obs.cpu().numpy(), rew.cpu().numpy(), done_np, infos
        return obs, rew, done.bool(), v._infos(None, terminal_obs=self._term_n)

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    # ---- normalisation of arbitrary batches with the current statistics (no update)
    def _as_rows(self, x, width):
        t = torch.as_tensor(x, dtype=torch.float32).to(self.venv.device)
        return t.reshape((-1, width) if width else (-1,)).contiguous()

    def normalize_obs(self, obs):
        """(obs - mean) / sqrt(var + eps) clipped to +-clip_obs, as float32 (a copy when norm_obs is off)."""
        is_np = not isinstance(obs, torch.Tensor)
        x = self._as_rows(obs, self.handle.D)
        out = torch.empty_like(x)
        self.handle.apply(None, x, out)
        out = out.reshape(np.shape(obs))
        return out.cpu().numpy() if is_np else out

    def normalize_reward(self, reward):
        """reward / sqrt(ret_var + eps) clipped to +-clip_reward, as float32 (unchanged when norm_reward is off)."""
        if not self._flags[2]:
            return reward
        is_np = not isinstance(reward, torch.Tensor)
        r = self._as_rows(reward, 0)
        out = torch.empty_like(r)
        self.handle.apply(None, reward=r, reward_out=out)
        out = out.reshape(np.shape(reward))
        return out.cpu().numpy() if is_np else out

    def get_original_obs(self):
        """The raw observations of the last reset / step (a copy)."""
        return self._out(self.venv._obs.clone())

    def get_original_reward(self):
        """The raw rewards of the last step (a copy, float32)."""
        return self._out(self.venv._rew.clone())

    # ---- pass-through to the wrapped env
    def get_attr(self, attr_name, indices=None):
        return self.venv.get_attr(attr_name, indices)

    def set_attr(self, attr_name, value, indices=None):
        return self.venv.set_attr(attr_name, value, indices)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        return self.venv.env_method(method_name, *args, indices=indices, **kwargs)

    def env_is_wrapped(self, wrapper_class, indices=None):
        return self.venv.env_is_wrapped(wrapper_class, indices)

    def seed(self, seed=None):
        return self.venv.seed(seed)

    def close(self):
        self.handle.close()
        self.venv.close()
