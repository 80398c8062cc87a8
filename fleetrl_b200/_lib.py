"""ctypes binding of libfleetstep.so (include/fleetstep.h) over torch CUDA tensors.

torch is plumbing here: it owns device buffers and streams; every computation happens inside the CUDA library.
There is deliberately NO fallback: if the shared library or a CUDA device is missing the calls raise.
"""
import ctypes as C
import os

import numpy as np
import torch

from ._abi import ABI_VERSION, FIELDS, STATS, FleetConsts, FleetTables

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FLEETSTEP_LIB") or os.path.join(_HERE, "libfleetstep.so")   # FLEETSTEP_LIB: diagnostic builds
_LIB = None

_TORCH_DTYPES = {np.float64: torch.float64, np.float32: torch.float32, np.int32: torch.int32, np.uint8: torch.uint8}

EXPORTS = [
    "fleet_abi_version", "fleet_create", "fleet_destroy", "fleet_obs_dim", "fleet_num_evs", "fleet_num_envs",
    "fleet_reset", "fleet_step", "fleet_step_host", "fleet_set_next_start", "fleet_get_state", "fleet_set_state",
    "fleet_field_info", "fleet_get_stats", "fleet_reset_stats", "fleet_check_errors", "fleet_launch_count",
    "fleet_device_bytes", "fleet_last_error", "fleet_set_timing", "fleet_get_timing", "fleet_step_kernel_name", "fleet_policy_actions", "fleet_policy_reset", "fleet_enable_charge_log",
    "fleet_debug_stress", "fleet_enable_log", "fleet_log_layout", "fleet_read_log", "fleet_state_bytes", "fleet_export_state", "fleet_import_state",
    "fleet_launch_geometry",
    "fleet_norm_create", "fleet_norm_destroy", "fleet_norm_set_flags", "fleet_norm_moments_len", "fleet_norm_moments",
    "fleet_norm_apply", "fleet_norm_reset_returns", "fleet_norm_get_state", "fleet_norm_set_state", "fleet_norm_last_error",
    "fleet_rollout_add", "fleet_rollout_gae", "fleet_rollout_gather", "fleet_rollout_last_error",
]


class FleetStepError(RuntimeError):
    pass


class FleetRolloutBuf(C.Structure):
    """struct FleetRolloutBuf of fleetstep.h: sizes and the device pointers of a rollout buffer's eight arrays."""
    _fields_ = [(n, C.c_int32) for n in ("buffer_size", "num_envs", "obs_dim", "action_dim")] + \
               [(n, C.c_void_p) for n in ("observations", "actions", "rewards", "episode_starts", "values", "log_probs",
                                          "advantages", "returns")]


def load_library(path: str = LIB_PATH):
    """Load libfleetstep.so and declare the prototypes.  Raises if the library has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(path):
        raise FleetStepError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` or `make`. "
            "fleetrl_b200 has no CPU fallback.")
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.fleet_abi_version.restype = C.c_int
    L.fleet_create.argtypes = [C.POINTER(FleetConsts), C.POINTER(FleetTables), i32, i32, i64, C.POINTER(vp)]
    L.fleet_destroy.argtypes = [vp]
    for f in ("fleet_obs_dim", "fleet_num_evs", "fleet_num_envs"):
        getattr(L, f).argtypes = [vp]
    L.fleet_reset.argtypes = [vp, vp, vp, vp, vp]
    L.fleet_step.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.fleet_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.fleet_set_next_start.argtypes = [vp, vp]
    L.fleet_get_state.argtypes = [vp, i32, vp, vp]
    L.fleet_set_state.argtypes = [vp, i32, vp, vp]
    L.fleet_field_info.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i64)]
    L.fleet_get_stats.argtypes = [vp, vp, vp]
    L.fleet_reset_stats.argtypes = [vp, vp]
    L.fleet_check_errors.argtypes = [vp, C.POINTER(C.c_uint32), vp]
    L.fleet_launch_count.argtypes = [vp]
    L.fleet_launch_count.restype = i64
    L.fleet_device_bytes.argtypes = [vp]
    L.fleet_device_bytes.restype = i64
    L.fleet_policy_actions.argtypes = [vp, i32, i32, i32, i32, vp, vp]
    L.fleet_policy_reset.argtypes = [vp, vp]
    L.fleet_enable_charge_log.argtypes = [vp, i32]
    L.fleet_debug_stress.argtypes = [vp, vp, vp, i32, vp]
    L.fleet_enable_log.argtypes = [vp, vp, i32, i32]
    L.fleet_log_layout.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.fleet_read_log.argtypes = [vp, vp, vp, vp]
    L.fleet_state_bytes.argtypes = [vp]
    L.fleet_state_bytes.restype = i64
    L.fleet_export_state.argtypes = [vp, vp, vp]
    L.fleet_import_state.argtypes = [vp, vp, vp]
    L.fleet_step_kernel_name.argtypes = [vp]
    L.fleet_step_kernel_name.restype = C.c_char_p
    L.fleet_launch_geometry.argtypes = [vp] + [C.POINTER(i32)] * 4
    L.fleet_set_timing.argtypes = [vp, i32]
    L.fleet_get_timing.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i64)]
    L.fleet_last_error.argtypes = [vp]
    L.fleet_last_error.restype = C.c_char_p
    f64 = C.c_double
    L.fleet_norm_create.argtypes = [i32, i32, i32, f64, f64, f64, f64, C.POINTER(vp)]
    L.fleet_norm_destroy.argtypes = [vp]
    L.fleet_norm_set_flags.argtypes = [vp, i32, i32, i32]
    L.fleet_norm_moments_len.argtypes = [vp]
    L.fleet_norm_moments.argtypes = [vp, vp, vp, vp, vp]
    L.fleet_norm_apply.argtypes = [vp, vp, i64] + [vp] * 8
    L.fleet_norm_reset_returns.argtypes = [vp, vp]
    L.fleet_norm_get_state.argtypes = [vp] * 9
    L.fleet_norm_set_state.argtypes = [vp] * 9
    L.fleet_norm_last_error.argtypes = [vp]
    L.fleet_norm_last_error.restype = C.c_char_p
    rb = C.POINTER(FleetRolloutBuf)
    L.fleet_rollout_add.argtypes = [rb, i32] + [vp] * 7
    L.fleet_rollout_gae.argtypes = [rb, f64, f64, vp, vp, vp]
    L.fleet_rollout_gather.argtypes = [rb, vp, i64] + [vp] * 7
    L.fleet_rollout_last_error.argtypes = []
    L.fleet_rollout_last_error.restype = C.c_char_p
    if L.fleet_abi_version() != ABI_VERSION:
        raise FleetStepError("libfleetstep.so ABI version does not match fleetrl_b200/_abi.py")
    _LIB = L
    return L


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _dptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class FleetStepHandle:
    """One GPU's worth of environments: thin, checked wrapper over the C ABI."""

    def __init__(self, consts: FleetConsts, tables: dict, num_envs: int, device=0, env_id_offset: int = 0):
        if not torch.cuda.is_available():
            raise FleetStepError("no CUDA device available; fleetrl_b200 has no CPU fallback")
        self.lib = load_library()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.consts = consts
        tb, keep = FleetTables.from_arrays(tables)
        h = C.c_void_p()
        rc = self.lib.fleet_create(C.byref(consts), C.byref(tb), int(num_envs), self.device.index, int(env_id_offset),
                                   C.byref(h))
        self._h = h
        if rc != 0:
            msg = self.lib.fleet_last_error(h).decode() if h else "fleet_create failed"
            if h:
                self.lib.fleet_destroy(h)
            self._h = None
            raise FleetStepError(f"fleet_create: {msg} (code {rc})")
        del keep
        self.E = self.lib.fleet_num_envs(h)
        self.N = self.lib.fleet_num_evs(h)
        self.D = self.lib.fleet_obs_dim(h)
        self._next_start = None

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None):
            self.lib.fleet_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise FleetStepError(f"{what}: {self.lib.fleet_last_error(self._h).decode()} (code {rc})")

    def _chk_tensor(self, t, shape, dtype, name):
        if t is None:
            return
        if t.device != self.device or t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
            raise FleetStepError(f"{name}: expected contiguous {dtype} tensor of shape {tuple(shape)} on {self.device}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}")

    # -- the path
    def reset(self, start_idx=None, mask=None, obs=None):
        self._chk_tensor(start_idx, (self.E,), torch.int32, "start_idx")
        self._chk_tensor(mask, (self.E,), torch.uint8, "mask")
        self._chk_tensor(obs, (self.E, self.D), torch.float32, "obs")
        self._check(self.lib.fleet_reset(self._h, _dptr(start_idx), _dptr(mask), _dptr(obs), _stream_ptr(self.device)),
                    "fleet_reset")

    def step(self, actions, obs=None, reward=None, done=None, terminal_obs=None):
        self._chk_tensor(actions, (self.E, self.N), torch.float32, "actions")
        self._chk_tensor(obs, (self.E, self.D), torch.float32, "obs")
        self._chk_tensor(reward, (self.E,), torch.float32, "reward")
        self._chk_tensor(done, (self.E,), torch.uint8, "done")
        self._chk_tensor(terminal_obs, (self.E, self.D), torch.float32, "terminal_obs")
        self._check(self.lib.fleet_step(self._h, _dptr(actions), _dptr(obs), _dptr(reward), _dptr(done),
                                        _dptr(terminal_obs), _stream_ptr(self.device)), "fleet_step")

    def step_unchecked(self, actions_ptr, obs_ptr, reward_ptr, done_ptr, term_ptr, stream_ptr):
        """Hot-loop variant: raw integer pointers, no tensor validation (bench / rollout loops)."""
        rc = self.lib.fleet_step(self._h, actions_ptr, obs_ptr, reward_ptr, done_ptr, term_ptr, stream_ptr)
        if rc != 0:
            self._check(rc, "fleet_step")

    def step_host(self, actions, obs, reward, done, terminal_obs=None):
        """NumPy / pinned-host call: H2D copy, step, D2H copies, stream sync — all inside the library."""
        self._chk_tensor(terminal_obs, (self.E, self.D), torch.float32, "terminal_obs")
        for a, shape, dt, nm in ((actions, (self.E, self.N), np.float32, "actions"), (obs, (self.E, self.D), np.float32, "obs"),
                                 (reward, (self.E,), np.float32, "reward"), (done, (self.E,), np.uint8, "done")):
            if a is not None and (a.dtype != dt or tuple(a.shape) != shape or not a.flags.c_contiguous):
                raise FleetStepError(f"{nm}: expected C-contiguous {dt} array of shape {shape}")
        self._check(self.lib.fleet_step_host(self._h, actions.ctypes.data, None if obs is None else obs.ctypes.data,
                                             None if reward is None else reward.ctypes.data,
                                             None if done is None else done.ctypes.data, _dptr(terminal_obs),
                                             _stream_ptr(self.device)),
                    "fleet_step_host")

    def set_next_start(self, next_start):
        self._chk_tensor(next_start, (self.E,), torch.int32, "next_start")
        self._next_start = next_start  # keep alive
        self._check(self.lib.fleet_set_next_start(self._h, _dptr(next_start)), "fleet_set_next_start")

    # -- state access
    def get(self, name):
        fid, dt, per_ev = FIELDS[name]
        out = torch.empty((self.E, self.N) if per_ev else (self.E,), dtype=_TORCH_DTYPES[dt], device=self.device)
        self._check(self.lib.fleet_get_state(self._h, fid, _dptr(out), _stream_ptr(self.device)), f"fleet_get_state({name})")
        return out

    def set(self, name, value):
        fid, dt, per_ev = FIELDS[name]
        v = torch.as_tensor(value, dtype=_TORCH_DTYPES[dt], device=self.device).contiguous()
        self._chk_tensor(v, (self.E, self.N) if per_ev else (self.E,), _TORCH_DTYPES[dt], name)
        if name == "target_soc":
            # the device keeps a vehicle's target as one flag: raised to 0.9 (fleet_environment.py:613-614) or not
            target = float(self.consts.target_soc)
            bad = (v != 0.9) & (v != target)
            if bool(bad.any()):
                raise FleetStepError(f"set(target_soc): {v[bad][0].item()!r} is neither the configured target {target!r} "
                                     "nor 0.9, the only values a vehicle's target can take")
        self._check(self.lib.fleet_set_state(self._h, fid, _dptr(v), _stream_ptr(self.device)), f"fleet_set_state({name})")
        torch.cuda.current_stream(self.device).synchronize()

    def stats_tensor(self):
        out = torch.empty(len(STATS), dtype=torch.float64, device=self.device)
        self._check(self.lib.fleet_get_stats(self._h, _dptr(out), _stream_ptr(self.device)), "fleet_get_stats")
        return out

    def stats(self):
        return dict(zip(STATS, self.stats_tensor().cpu().tolist()))

    def reset_stats(self):
        self._check(self.lib.fleet_reset_stats(self._h, _stream_ptr(self.device)), "fleet_reset_stats")

    def check_errors(self):
        flags = C.c_uint32(0)
        self._check(self.lib.fleet_check_errors(self._h, C.byref(flags), _stream_ptr(self.device)), "fleet_check_errors")
        return int(flags.value)

    POLICIES = {"uncontrolled": 0, "distributed": 1, "night": 2}

    def policy_actions(self, policy, out=None, charging_hour=0, charging_minute=0, max_hours=0):
        """Actions [E, N] float32 of a rule-based baseline policy at every env's current time (benchmarking/*.py)."""
        if out is None:
            out = torch.empty((self.E, self.N), dtype=torch.float32, device=self.device)
        self._chk_tensor(out, (self.E, self.N), torch.float32, "actions")
        self._check(self.lib.fleet_policy_actions(self._h, self.POLICIES[policy], int(charging_hour), int(charging_minute),
                                                  int(max_hours), _dptr(out), _stream_ptr(self.device)), "fleet_policy_actions")
        return out

    def policy_reset(self):
        self._check(self.lib.fleet_policy_reset(self._h, _stream_ptr(self.device)), "fleet_policy_reset")

    def enable_charge_log(self, enable=True):
        """Keep EvCharger's per-vehicle charge_log of every step (field "charge_log"); off by default."""
        self._check(self.lib.fleet_enable_charge_log(self._h, 1 if enable else 0), "fleet_enable_charge_log")

    # -- device-side DataLogger (data_logger.py:21-68) for selected envs
    def enable_log(self, env_ids, rows_per_env):
        ids = np.ascontiguousarray(env_ids, dtype=np.int32)
        self._check(self.lib.fleet_enable_log(self._h, ids.ctypes.data, len(ids), int(rows_per_env)), "fleet_enable_log")
        self._log_ids = ids

    def read_log(self):
        """-> list (one entry per logged env) of dicts of arrays, oldest row first: ep_count, time_idx, reward, cashflow,
        penalties, overload, soc_viol, kind (1 reset row / 2 step with daily degradation / 0 other step), action [rows, N],
        degradation [rows, N], charging_energy [rows, N], soh [rows, N], obs [rows, D]."""
        n, cap, rd = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        self._check(self.lib.fleet_log_layout(self._h, C.byref(n), C.byref(cap), C.byref(rd)), "fleet_log_layout")
        n, cap, rd = n.value, cap.value, rd.value
        rows = np.zeros((max(n, 1), max(cap, 1), max(rd, 1)))
        counts = np.zeros(max(n, 1), np.int64)
        self._check(self.lib.fleet_read_log(self._h, rows.ctypes.data, counts.ctypes.data, _stream_ptr(self.device)), "fleet_read_log")
        N, out = self.N, []
        for l in range(n):
            cnt = int(counts[l])
            r = rows[l, :cnt] if cnt <= cap else np.roll(rows[l], -(cnt % cap), axis=0)
            out.append({"env": int(self._log_ids[l]), "rows_total": cnt, "ep_count": r[:, 0].astype(np.int64),
                        "time_idx": r[:, 1].astype(np.int64), "reward": r[:, 2], "cashflow": r[:, 3], "penalties": r[:, 4],
                        "overload": r[:, 5], "soc_viol": r[:, 6], "kind": r[:, 7].astype(np.int64),
                        "action": r[:, 8:8 + N], "degradation": r[:, 8 + N:8 + 2 * N],
                        "charging_energy": r[:, 8 + 2 * N:8 + 3 * N], "soh": r[:, 8 + 3 * N:8 + 4 * N],
                        "obs": r[:, 8 + 4 * N:].astype(np.float32)})
        return out

    # -- checkpoint / resume
    def export_state(self):
        """The complete env state of the handle as one opaque uint8 array (fleet_export_state)."""
        buf = np.empty(int(self.lib.fleet_state_bytes(self._h)), np.uint8)
        self._check(self.lib.fleet_export_state(self._h, buf.ctypes.data, _stream_ptr(self.device)), "fleet_export_state")
        return buf

    def import_state(self, blob):
        b = np.ascontiguousarray(blob, dtype=np.uint8)
        if b.size != int(self.lib.fleet_state_bytes(self._h)):
            raise FleetStepError("import_state: blob size does not match this handle")
        self._check(self.lib.fleet_import_state(self._h, b.ctypes.data, _stream_ptr(self.device)), "fleet_import_state")

    def set_timing(self, enable=True):
        self._check(self.lib.fleet_set_timing(self._h, 1 if enable else 0), "fleet_set_timing")

    def get_timing(self):
        """(step-kernel ms, post-kernel ms, steps) summed over the steps since set_timing (at most the last 1024)."""
        a, b, n = C.c_double(0), C.c_double(0), C.c_int64(0)
        self._check(self.lib.fleet_get_timing(self._h, C.byref(a), C.byref(b), C.byref(n)), "fleet_get_timing")
        return a.value, b.value, int(n.value)

    @property
    def step_kernel_name(self):
        """Name of the step kernel fleet_create selected for this handle."""
        return self.lib.fleet_step_kernel_name(self._h).decode()

    @property
    def launch_geometry(self):
        """dict(step_grid, step_tiles, envs_per_tile, post_grid): the launch geometry fleet_create chose (after the
        FLEETSTEP_PF_GRID / FLEETSTEP_POST_GRID caps)."""
        v = [C.c_int32(0) for _ in range(4)]
        self._check(self.lib.fleet_launch_geometry(self._h, *[C.byref(x) for x in v]), "fleet_launch_geometry")
        return dict(zip(("step_grid", "step_tiles", "envs_per_tile", "post_grid"), (x.value for x in v)))

    @property
    def launch_count(self):
        return int(self.lib.fleet_launch_count(self._h))

    @property
    def device_bytes(self):
        return int(self.lib.fleet_device_bytes(self._h))

    @property
    def raw(self):
        return self._h


class FleetNormHandle:
    """Device VecNormalize statistics for [E][D] float32 batches (fleet_norm_*): thin, checked wrapper over the C ABI."""

    def __init__(self, num_envs: int, obs_dim: int, device=0, clip_obs=10.0, clip_reward=10.0, gamma=0.99, epsilon=1e-8):
        if not torch.cuda.is_available():
            raise FleetStepError("no CUDA device available; fleetrl_b200 has no CPU fallback")
        self.lib = load_library()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        h = C.c_void_p()
        rc = self.lib.fleet_norm_create(int(num_envs), int(obs_dim), self.device.index, float(clip_obs), float(clip_reward),
                                        float(gamma), float(epsilon), C.byref(h))
        self._h = h
        if rc != 0:
            msg = self.lib.fleet_norm_last_error(h).decode() if h else "fleet_norm_create failed"
            if h:
                self.lib.fleet_norm_destroy(h)
            self._h = None
            raise FleetStepError(f"fleet_norm_create: {msg} (code {rc})")
        self.E, self.D = int(num_envs), int(obs_dim)
        self.moments_len = int(self.lib.fleet_norm_moments_len(h))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.fleet_norm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise FleetStepError(f"{what}: {self.lib.fleet_norm_last_error(self._h).decode()} (code {rc})")

    _chk_tensor = FleetStepHandle._chk_tensor

    def set_flags(self, training, norm_obs, norm_reward):
        self._check(self.lib.fleet_norm_set_flags(self._h, int(bool(training)), int(bool(norm_obs)), int(bool(norm_reward))),
                    "fleet_norm_set_flags")

    def moments(self, obs, reward, out):
        """Batch moments of obs [E, D] (and of the new returns when reward [E] is given) into out (float64 [2D+4])."""
        self._chk_tensor(obs, (self.E, self.D), torch.float32, "obs")
        self._chk_tensor(reward, (self.E,), torch.float32, "reward")
        self._chk_tensor(out, (self.moments_len,), torch.float64, "moments")
        if out is None:
            raise FleetStepError("moments: an output tensor is required")
        self._check(self.lib.fleet_norm_moments(self._h, _dptr(obs), _dptr(reward), _dptr(out), _stream_ptr(self.device)),
                    "fleet_norm_moments")

    def apply(self, moments=None, obs=None, obs_out=None, reward=None, reward_out=None, done=None, terminal_obs=None,
              terminal_obs_out=None):
        """Merge `moments` (None: no update) and normalise; see fleet_norm_apply."""
        rows = next((t.shape[0] for t in (obs, reward, done) if t is not None), self.E)
        self._chk_tensor(moments, (self.moments_len,), torch.float64, "moments")
        for t, nm in ((obs, "obs"), (obs_out, "obs_out"), (terminal_obs, "terminal_obs"), (terminal_obs_out, "terminal_obs_out")):
            self._chk_tensor(t, (rows, self.D), torch.float32, nm)
        self._chk_tensor(reward, (rows,), torch.float32, "reward")
        self._chk_tensor(reward_out, (rows,), torch.float32, "reward_out")
        self._chk_tensor(done, (rows,), torch.uint8, "done")
        self._check(self.lib.fleet_norm_apply(self._h, _dptr(moments), int(rows), _dptr(obs), _dptr(obs_out), _dptr(reward),
                                              _dptr(reward_out), _dptr(done), _dptr(terminal_obs), _dptr(terminal_obs_out),
                                              _stream_ptr(self.device)), "fleet_norm_apply")

    def reset_returns(self):
        self._check(self.lib.fleet_norm_reset_returns(self._h, _stream_ptr(self.device)), "fleet_norm_reset_returns")

    STATE = ("obs_mean", "obs_var", "obs_count", "ret_mean", "ret_var", "ret_count", "returns")

    def _shapes(self):
        return ((self.D,), (self.D,), (), (), (), (), (self.E,))

    def get_state(self):
        """dict of float64 NumPy arrays: obs_mean [D], obs_var [D], obs_count, ret_mean, ret_var, ret_count, returns [E]."""
        out = {k: np.zeros(s, np.float64) for k, s in zip(self.STATE, self._shapes())}
        self._check(self.lib.fleet_norm_get_state(self._h, *[out[k].ctypes.data for k in self.STATE], _stream_ptr(self.device)),
                    "fleet_norm_get_state")
        return out

    def set_state(self, **parts):
        """Set any of the get_state() entries; the others stay."""
        bad = set(parts) - set(self.STATE)
        if bad:
            raise KeyError(f"unknown state entries {sorted(bad)}")
        keep = {}
        for k, s in zip(self.STATE, self._shapes()):
            if parts.get(k) is not None:
                a = np.array(parts[k], dtype=np.float64, order="C")
                if a.shape != s and a.size == 1 and s == ():
                    a = a.reshape(())
                if a.shape != s:
                    raise FleetStepError(f"{k}: expected shape {s}, got {a.shape}")
                keep[k] = a
        self._check(self.lib.fleet_norm_set_state(self._h, *[keep[k].ctypes.data if k in keep else None for k in self.STATE],
                                                  _stream_ptr(self.device)), "fleet_norm_set_state")
