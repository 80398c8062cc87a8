"""FleetVecEnv — the SB3-shaped VecEnv over the CUDA step (one handle per GPU), and FleetEnv — the gym-shaped
single environment, both mirroring the reference's interface for this path:

  FleetEnv(env_config)                  fleetrl/fleet_env/fleet_environment.py:76
  reset() -> (obs float32[D], {})       :330-434
  step(a) -> (obs, reward, done, False, {})   :436-702
  observation_space / action_space      :316-325
  env_method helpers                    :741-799  (is_done, get_time, get_start_time, set_start_time, get_dist_factor, get_log)
  VecEnv protocol (stable-baselines3==2.3.2, third party): num_envs, reset, step_async/step_wait/step, close,
  get_attr/set_attr/env_method/env_is_wrapped/seed, auto-reset with infos[i]["terminal_observation"],
  "TimeLimit.truncated" and Monitor's infos[i]["episode"] — call sites benchmarking/*.py, agent_eval/basic_evaluation.py:68-90.

All computation happens in libfleetstep.so; this module only owns buffers and bookkeeping.  Tensors returned in
"torch" mode are views of the buffers the kernel wrote (no host round-trip); "numpy" mode goes through
fleet_step_host (pinned buffers, H2D/D2H inside the library).
"""
import numpy as np
import pandas as pd
import torch

from . import dist as _dist
from ._abi import STATS
from ._lib import FleetStepHandle
from .spaces import action_box, observation_box
from .tables import BuiltFleet, FleetInputs, build_fleet


class LazyInfos:
    """List-like `infos` of a VecEnv step that materialises a dict only when indexed (65k dicts per step would
    dominate the step time).  Entries of finished envs carry "terminal_observation", "TimeLimit.truncated" and the
    Monitor-style "episode" record; all others are {} like the reference's `info` (fleet_environment.py:235,702)."""

    def __init__(self, n, done_idx, terminal_obs, ep_returns, ep_len):
        self._n = n
        self._done = {int(i): k for k, i in enumerate(done_idx)}
        self._term, self._ret, self._len = terminal_obs, ep_returns, ep_len

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(self._n))]
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        k = self._done.get(int(i))
        if k is None:
            return {}
        return {"terminal_observation": self._term[k], "TimeLimit.truncated": False,
                "episode": {"r": float(self._ret[k]), "l": int(self._len), "t": 0.0}}

    def __iter__(self):
        return (self[i] for i in range(self._n))


try:  # pragma: no cover - stable-baselines3 is third party and not part of the build image
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase
except Exception:
    _VecEnvBase = object


class FleetVecEnv(_VecEnvBase):
    """num_envs identical FleetEnvs stepped by one kernel launch pair per step on one GPU.

    When stable-baselines3 is importable this class IS a stable_baselines3 VecEnv (BaseAlgorithm._wrap_env accepts it as
    is); without it the same protocol is duck-typed.

    env_config: dict or JSON path with the reference's keys; `inputs` optionally supplies the schedule / price /
    load / PV frames in memory (synthetic fleets) instead of CSV files under env_config["data_path"].
    output: "torch" (CUDA tensors, zero-copy) or "numpy".
    env_id_offset: global id of local env 0 (use `FleetVecEnv.sharded` under torchrun).
    """

    def __init__(self, env_config, num_envs, device=0, inputs: FleetInputs = None, output="torch", env_id_offset=0,
                 carry_degradation_state=True, seed=None, built: BuiltFleet = None):
        self.built = built or build_fleet(env_config, inputs, auto_reset=True,
                                          carry_degradation_state=carry_degradation_state, seed=seed)
        c = self.built.consts
        self.num_envs, self.num_cars = int(num_envs), int(c.num_evs)
        self.handle = FleetStepHandle(c, self.built.tables, self.num_envs, device=device, env_id_offset=env_id_offset)
        self.device = self.handle.device
        self.obs_dim = self.handle.D
        self.observation_space = observation_box(self.obs_dim, bool(c.normalize))
        self.action_space = action_box(self.num_cars)
        if _VecEnvBase is not object:
            _VecEnvBase.__init__(self, self.num_envs, self.observation_space, self.action_space)
        self.output = output
        if output not in ("torch", "numpy"):
            raise ValueError("output must be 'torch' or 'numpy'")
        E, D = self.num_envs, self.obs_dim
        dev = self.device
        self._obs = torch.zeros((E, D), dtype=torch.float32, device=dev)
        self._term = torch.zeros((E, D), dtype=torch.float32, device=dev)
        self._log_idx = []
        self._last_done = np.zeros(E, dtype=bool)
        self._night = None          # night-charging window parameters (fleetrl_b200/policies.py), derived on first use
        self._rew = torch.zeros(E, dtype=torch.float32, device=dev)
        self._done = torch.zeros(E, dtype=torch.uint8, device=dev)
        self._actions = None
        self.render_mode = None
        self._start_override = None
        # env_config["log_data"]=True (the reference's evaluation runs use one env): log the first envs (at most 8)
        if self.built.rc is not None and self.built.rc.cfg.get("log_data", False):
            self.enable_log(indices=list(range(min(E, 8))))
        if output == "numpy":
            self._h_act = torch.zeros((E, self.num_cars), dtype=torch.float32).pin_memory()
            self._h_obs = torch.zeros((E, D), dtype=torch.float32).pin_memory()
            self._h_rew = torch.zeros(E, dtype=torch.float32).pin_memory()
            self._h_done = torch.zeros(E, dtype=torch.uint8).pin_memory()

    # ---- construction helpers
    @classmethod
    def sharded(cls, env_config, total_envs, **kw):
        """One shard per rank under torchrun: contiguous env ranges, GPU = LOCAL_RANK."""
        rank, world_size, local_rank = _dist.world()
        lo, hi = _dist.shard_range(total_envs, rank, world_size)
        return cls(env_config, hi - lo, device=local_rank, env_id_offset=lo, **kw)

    # ---- VecEnv protocol
    def reset(self, start_idx=None):
        """All envs.  start_idx (int array [E]) injects the episode starts (parity runs); default: device RNG over
        the configured time picker's range."""
        s = None
        if start_idx is not None:
            s = torch.as_tensor(np.asarray(start_idx), dtype=torch.int32, device=self.device).contiguous()
        self.handle.reset(start_idx=s, obs=self._obs)
        return self._out(self._obs)

    def step_async(self, actions):
        self._actions = actions

    def step_wait(self):
        a = self._actions
        E, N = self.num_envs, self.num_cars
        if self.output == "numpy":
            self._h_act.numpy()[...] = np.asarray(a, dtype=np.float32).reshape(E, N)
            self.handle.step_host(self._h_act.numpy(), self._h_obs.numpy(), self._h_rew.numpy(), self._h_done.numpy(), self._term)
            # fresh arrays like DummyVecEnv / SubprocVecEnv return them: the pinned buffers are overwritten by the next step
            obs, rew, done = self._h_obs.numpy().copy(), self._h_rew.numpy().copy(), self._h_done.numpy().astype(bool)
            done_idx = np.nonzero(done)[0]
            self._last_done = done
        else:
            a = torch.as_tensor(a, dtype=torch.float32, device=self.device).reshape(E, N).contiguous()
            self.handle.step(a, self._obs, self._rew, self._done, self._term)
            obs, rew, done = self._obs, self._rew, self._done.bool()
            done_idx = None
        return obs, rew, done, self._infos(done_idx)

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def _infos(self, done_idx, terminal_obs=None):
        """infos of the step just taken; terminal_obs: the [E, D] buffer holding the terminal rows (default: this env's
        own, a wrapper passes its normalised copy)."""
        if done_idx is None:   # torch mode: one small D2H of the done flags (use step_raw() to avoid it)
            done_idx = torch.nonzero(self._done).flatten().cpu().numpy()
            self._last_done = np.zeros(self.num_envs, dtype=bool)
            self._last_done[done_idx] = True
        if len(done_idx) == 0:
            return LazyInfos(self.num_envs, [], None, None, 0)
        idx_t = torch.as_tensor(done_idx, device=self.device, dtype=torch.long)
        term = (self._term if terminal_obs is None else terminal_obs).index_select(0, idx_t)   # finished envs' rows only
        if self.output == "numpy":
            term = term.cpu().numpy()
        rets = self.handle.get("last_ep_return").index_select(0, idx_t).cpu().numpy()
        return LazyInfos(self.num_envs, done_idx, term, rets, int(self.built.consts.episode_steps))

    def step_raw(self, actions: torch.Tensor):
        """Hot-loop variant for on-device rollouts: CUDA tensors in, views of the output buffers back, no infos,
        no host synchronisation.  Finished envs are flagged in `done`; their last observation is in
        `self.terminal_observations`."""
        self.handle.step(actions, self._obs, self._rew, self._done, self._term)
        return self._obs, self._rew, self._done

    @property
    def terminal_observations(self):
        return self._term

    # ---- evaluation log (DataLogger.log_data, utils/data_logger/data_logger.py:21-68) for selected envs
    LOG_COLUMNS = ("Episode", "Time", "Observation", "Action", "Reward", "Cashflow", "Penalties", "Grid overloading",
                   "SOC violation", "Degradation", "Charging energy", "SOH")

    def enable_log(self, indices=(0,), max_rows=None):
        """Record the reference's per-step log rows for the given envs (evaluation runs).  The rows are written on the
        device by the library (fleet_enable_log: a ring of max_rows rows per env, default four episodes) and only read
        back by get_log; rows follow fleet_environment.py:420-432 (reset row) and :679-690 (one row per step that does
        not end the episode).  Call it before reset()."""
        self._log_idx = [int(i) for i in self._indices(indices)]
        L = int(self.built.consts.episode_steps)
        self.handle.enable_log(self._log_idx, int(max_rows) if max_rows else 4 * L)

    def _log_frames(self):
        """DataLogger.log as one DataFrame per logged env (columns LOG_COLUMNS)."""
        return {rec["env"]: _log_frame(rec, self.built) for rec in self.handle.read_log()}

    def baseline_actions(self, policy, out=None):
        """Actions [E, N] (float32, on the device) of one of the reference's rule-based benchmark policies at every env's
        current time: "uncontrolled" (benchmarking/uncontrolled_charging.py), "distributed" (distributed_charging.py) or
        "night" (night_charging.py; its window parameters are derived from the schedule once)."""
        if policy == "night":
            if self._night is None:
                from .policies import night_params
                self._night = night_params(self.built)
            n = self._night
            return self.handle.policy_actions("night", out, n.charging_hour, n.charging_minute, n.max_hours)
        return self.handle.policy_actions(policy, out)

    def close(self):
        self.handle.close()

    def seed(self, seed=None):
        return [None] * self.num_envs

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * len(self._indices(indices))

    def get_attr(self, attr_name, indices=None):
        idx = self._indices(indices)
        if attr_name == "num_cars":
            return [self.num_cars] * len(idx)
        if attr_name in ("observation_space", "action_space", "render_mode"):
            return [getattr(self, attr_name)] * len(idx)
        if attr_name == "episode_soh":
            soh = self.handle.get("soh").cpu().numpy()
            return [soh[i] for i in idx]
        raise AttributeError(attr_name)

    def set_attr(self, attr_name, value, indices=None):
        raise AttributeError(f"{attr_name} is not settable on the batched environment")

    def env_method(self, method_name, *args, indices=None, **kwargs):
        idx = self._indices(indices)
        return getattr(self, "_m_" + method_name)(idx, *args, **kwargs)

    # ---- env_method surface of the reference (fleet_environment.py:741-799)
    def _m_is_done(self, idx):
        """episode.done of the step just taken (fleet_environment.py:750); an env that has been auto-reset since is in a
        new episode, whose own flag is False, but SB3 callers ask right after the step that returned done=True."""
        return [bool(self._last_done[i]) for i in idx]

    def _m_get_time(self, idx):
        t = self.handle.get("time_idx").cpu().numpy()
        return [pd.Timestamp(self.built.dates[min(int(t[i]), len(self.built.dates) - 1)]) for i in idx]

    def _m_get_start_time(self, idx):
        f = self.handle.get("finish_idx").cpu().numpy() - int(self.built.consts.episode_steps)
        return [pd.Timestamp(self.built.dates[int(f[i])]) for i in idx]

    def _m_set_start_time(self, idx, start_time):
        # like the reference (fleet_environment.py:765-773) this has no lasting effect: reset() picks the start
        return [None for _ in idx]

    def _m_get_dist_factor(self, idx):
        """hours_needed / (hours_left + 0.001) from the SCHEDULE columns at the current time (:782-799)."""
        c, tb = self.built.consts, self.built.tables
        t = self.handle.get("time_idx").cpu().numpy()
        tgt = self.handle.get("target_soc").cpu().numpy()
        out = []
        for i in idx:
            ti = min(int(t[i]), c.table_len - 1)
            there = tb["there"][:, ti].astype(np.float64)
            cl = tgt[i] * there - tb["soc_on_return"][:, ti]
            hn = cl * c.lc_batt_cap / (c.evse_max_power * c.charging_eff)
            out.append(np.divide(hn, np.add(tb["time_left"][:, ti], 0.001)))
        return out

    def _m_get_log(self, idx):
        """Per-step log of the envs selected with enable_log() in the reference's DataLogger columns; for other envs the
        reduced episode statistics kept on the device (the same quantities summed over envs and steps)."""
        frames = self._log_frames() if self._log_idx else {}
        return [frames[i] if i in frames else pd.DataFrame([self.stats()]) for i in idx]

    # ---- statistics
    def stats(self, all_reduce=False):
        s = self.handle.stats_tensor()
        if all_reduce:
            _dist.all_reduce_stats(s)
        return dict(zip(STATS, s.cpu().tolist()))

    # ---- checkpointing (the env state is a handful of device tensors)
    _STATE_FIELDS = ("soc", "hours_left", "soh", "rf_len", "fd_cyc", "life", "ep_return", "target_soc")

    def state_dict(self):
        """Readable copies of the main state fields plus "blob": the complete device state (history ring, rainflow
        stacks, counters, statistics) as one opaque array — what load_state_dict restores."""
        d = {k: self.handle.get(k).cpu() for k in self._STATE_FIELDS}
        d["time_idx"] = self.handle.get("time_idx").cpu()
        d["finish_idx"] = self.handle.get("finish_idx").cpu()
        d["blob"] = torch.from_numpy(self.handle.export_state())
        d["last_obs"] = self._obs.cpu()
        return d

    def load_state_dict(self, d):
        """Resume exactly where state_dict() was taken (same env_config and num_envs): the next step() continues the
        trajectories bit for bit.  Returns the observation the envs were in."""
        self.handle.import_state(d["blob"].numpy())
        self._obs.copy_(d["last_obs"].to(self.device))
        return self._out(self._obs)

    def _indices(self, indices):
        if indices is None:
            return list(range(self.num_envs))
        if isinstance(indices, int):
            return [indices]
        return list(indices)

    def _out(self, t):
        return t.cpu().numpy() if self.output == "numpy" else t


LOG_COLUMNS = FleetVecEnv.LOG_COLUMNS


def _log_frame(rec, built):
    """One env's rows of the device-side log ring (FleetStepHandle.read_log) as the reference's DataLogger frame."""
    L = int(built.consts.episode_steps)
    first = rec["rows_total"] - len(rec["kind"])          # rows that fell out of the ring
    rows = []
    for r in range(len(rec["kind"])):
        kind = int(rec["kind"][r])
        rows.append({"Episode": (first + r) // L + 1,                                  # data_logger.py:51
                     "Time": pd.Timestamp(built.dates[int(rec["time_idx"][r])]),
                     "Observation": rec["obs"][r], "Action": rec["action"][r],
                     "Reward": float(rec["reward"][r]), "Cashflow": float(rec["cashflow"][r]),
                     "Penalties": float(rec["penalties"][r]), "Grid overloading": float(rec["overload"][r]),
                     "SOC violation": float(rec["soc_viol"][r]),
                     "Degradation": rec["degradation"][r] if kind == 2 else 0.0,
                     "Charging energy": rec["charging_energy"][r], "SOH": rec["soh"][r]})
    return pd.DataFrame(rows, columns=list(LOG_COLUMNS))


class FleetEnv:
    """Drop-in for the reference's gym.Env: ONE environment, NumPy in / NumPy out, no auto-reset.

    It is the E=1 case of the batched kernels (useful for evaluation scripts and parity checks; for training use
    FleetVecEnv)."""

    metadata = {"render_modes": []}

    def __init__(self, env_config, inputs: FleetInputs = None, device=0, log_rows=None):
        self.built = build_fleet(env_config, inputs, auto_reset=False, carry_degradation_state=True)
        c = self.built.consts
        self.num_cars = int(c.num_evs)
        self.handle = FleetStepHandle(c, self.built.tables, 1, device=device)
        # env_config["log_data"] (fleet_environment.py:129,420,679): keep the DataLogger rows on the device (ring of
        # log_rows rows, default four episodes) and hand them out as the reference's frame in get_log()
        self.log_data = bool(self.built.rc.cfg.get("log_data", False)) if self.built.rc is not None else False
        if self.log_data:
            self.handle.enable_log([0], int(log_rows) if log_rows else 4 * int(c.episode_steps))
        dev = self.handle.device
        self.observation_space = observation_box(self.handle.D, bool(c.normalize))
        self.action_space = action_box(self.num_cars)
        self._obs = torch.zeros((1, self.handle.D), dtype=torch.float32, device=dev)
        self._rew = torch.zeros(1, dtype=torch.float32, device=dev)
        self._done = torch.zeros(1, dtype=torch.uint8, device=dev)
        self.info = {}
        self._start_idx = None
        self.render_mode = "human"

    def reset(self, start_time=None, **kwargs):
        """start_time (str / Timestamp) replaces the time picker for this reset (the reference does that by swapping
        env.time_picker); default: the configured picker (static index, or device RNG over its range)."""
        if start_time is not None:
            t0 = int(np.searchsorted(self.built.dates, np.datetime64(pd.Timestamp(start_time))))
            s = torch.tensor([t0], dtype=torch.int32, device=self.handle.device)
        else:
            s = None
        self.handle.reset(start_idx=s, obs=self._obs)
        return self._obs[0].cpu().numpy(), self.info

    def step(self, actions):
        a = np.asarray(actions, dtype=np.float32).reshape(1, self.num_cars)
        if np.isnan(a).any():
            raise TypeError("The parsed action value was not recognised")     # ev_charger.py:209
        self.handle.step(torch.from_numpy(a).to(self.handle.device), self._obs, self._rew, self._done)
        reward = float(self.handle.get("reward64")[0].item())
        return self._obs[0].cpu().numpy(), reward, bool(self._done[0].item()), False, self.info

    def close(self):
        self.handle.close()
        return None

    def render(self):
        return None

    # env_method helpers (fleet_environment.py:741-799)
    def is_done(self):
        return bool(self._done[0].item())

    def get_time(self):
        t = int(self.handle.get("time_idx")[0].item())
        return pd.Timestamp(self.built.dates[min(t, len(self.built.dates) - 1)])

    def get_start_time(self):
        f = int(self.handle.get("finish_idx")[0].item()) - int(self.built.consts.episode_steps)
        return pd.Timestamp(self.built.dates[f])

    def set_start_time(self, start_time):
        return None

    def get_log(self):
        """DataLogger.log (data_logger.py:55-68) when the env was built with log_data=True, else the reduced statistics."""
        if not self.log_data:
            return pd.DataFrame([self.handle.stats()])
        return _log_frame(self.handle.read_log()[0], self.built)
