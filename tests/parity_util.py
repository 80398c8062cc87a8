"""Per-step comparison of a FleetStepHandle with the CPU oracle (oracle/fleet_oracle.c), shared by test_gpu_parity.py
and test_gpu_pipeline.py, and the `knobs` fixture of the tests that set the library's diagnostic variables.

Bit-exact (asserted with array_equal): done, time index, hours_left, target flags, SOC / soc_deg (see below), rainflow cycle
counts / rainflow_length, observations (float32), terminal observations, start indices drawn by the device RNG.
Tolerance: reward rel 1e-11 / abs 1e-10 (deterministic re-association of the per-env sum, exp), cashflow rel 1e-12 (regrouped
revenue factor), SOH abs 1e-13, fd_cyc rel 1e-11.
"""
import zlib

import numpy as np
import pytest
import torch

from synth_tables import make_consts, make_tables

EXACT = ["time_idx", "finish_idx", "hours_left", "target_soc", "rf_len", "n_cycles", "ep_count"]
KNOBS = ("FLEETSTEP_KERNEL", "FLEETSTEP_PF_GRID", "FLEETSTEP_POST_GRID", "FLEETSTEP_RF_RING", "FLEETSTEP_RF_STACK",
         "FLEETSTEP_RF_EXT", "FLEETSTEP_RF_EXT_SLOTS")


@pytest.fixture
def knobs(monkeypatch):
    """Start from the default kernel selection and geometry; returns a setter for the diagnostic variables (None: unset)."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)

    def set_knobs(**kv):
        for k, v in kv.items():
            if v is None:
                monkeypatch.delenv(k, raising=False)
            else:
                monkeypatch.setenv(k, str(v))
    return set_knobs


def make_case(name, n_evs, days=12, use_case="lmd", sph=4, episode_hours=24, two_trips=False, over=None,
              table_target=0.85):
    """(consts, tables) of a synthetic fleet; the tables' seed is derived from `name`, so a case is stable across runs.
    table_target: the target SOC the tables' SOC_on_return is derived from (independent of the constants' target_soc)."""
    over = dict(over or {})
    cap0 = dict(lmd=60.0, ut=50.0, ct=16.7)[use_case]
    tables, T = make_tables(n_evs=n_evs, days=days, sph=sph, seed=zlib.crc32(name.encode()) % 1000, two_trips=two_trips,
                            cap=cap0, target_soc=table_target)
    if not over.get("include_building", 1):
        tables = dict(tables, load=None)
    if not over.get("include_pv", 1):
        tables = dict(tables, pv=None)
    return make_consts(tables, T, n_evs, sph=sph, episode_hours=episode_hours, use_case=use_case, **over), tables


class Outputs:
    """Where each step writes its observations.

    plain    obs / terminal_obs are tensors of their own;
    offset   obs starts 4 bytes, terminal_obs 8 bytes into a larger buffer (16-byte bulk stores do not apply: the kernels
             take their element-wise paths); the bytes of the buffers outside the views must stay untouched;
    no_term  terminal_obs=None (finishing envs write no terminal observation);
    obs_gap  obs=None (and terminal_obs=None) for steps [gap[0], gap[1]), then obs again.
    """
    SENTINEL = -12345.5

    def __init__(self, E, D, dev, mode="plain", gap=(60, 130)):
        self.mode, self.gap = mode, gap
        if mode == "offset":
            self._obs_buf = torch.full((E * D + 8,), self.SENTINEL, dtype=torch.float32, device=dev)
            self._term_buf = torch.full((E * D + 8,), self.SENTINEL, dtype=torch.float32, device=dev)
            self.obs = self._obs_buf[1:1 + E * D].view(E, D)
            self.term = self._term_buf[2:2 + E * D].view(E, D)
            assert self.obs.data_ptr() % 16 == 4 and self.term.data_ptr() % 16 == 8
        else:
            self.obs = torch.zeros((E, D), dtype=torch.float32, device=dev)
            self.term = torch.full((E, D), -7.0, dtype=torch.float32, device=dev)

    def at(self, s):
        """(obs, terminal_obs) to pass at step s (None: not passed)."""
        if self.mode == "no_term":
            return self.obs, None
        if self.mode == "obs_gap" and self.gap[0] <= s < self.gap[1]:
            return None, None
        return self.obs, self.term

    def check_untouched(self, s):
        if self.mode != "offset":
            return
        E, D = self.obs.shape
        for buf, lo in ((self._obs_buf, 1), (self._term_buf, 2)):
            outside = torch.cat([buf[:lo], buf[lo + E * D:]])
            assert bool((outside == self.SENTINEL).all()), f"step {s}: bytes outside the output view were written"


def mixed_tiles(done, B):
    """Number of tiles of B envs (tail tile included) in which some envs finish and others keep running."""
    E = len(done)
    pad = np.full(-E % B, 2, np.int64)                   # padding counts as neither finishing nor running
    d = np.concatenate([done.astype(np.int64), pad]).reshape(-1, B)
    fin, run = (d == 1).sum(1), (d == 0).sum(1)
    return int(((fin > 0) & (run > 0)).sum())


def run_vs_oracle(gpu, orc, steps, *, charge_log, dephase=0, outputs=None, action_seed=7, hook=None):
    """Reset both sides through the counter RNG, then step them with the same random actions and compare every output
    and state field after every step.

    dephase=L: after each of the first L steps, env e with e % L == s is reset again (masked reset on both sides), so
    that episodes end on different steps (the de-phased steady state of a long rollout).
    hook(s, actions, obs, reward, done, terminal_obs), if given, runs after the reset (s = -1, actions and step outputs
    None) and at the end of every step s, once that step has been compared: it may write state on both sides or step
    further handles with the same actions.
    Returns dict(n_done, mixed_tiles): finished episodes, and tiles (of the handle's launch geometry) that had finishing
    and running envs in the same step."""
    E, N, D = gpu.E, gpu.N, gpu.D
    dev = gpu.device
    consts = orc.consts
    assert D == orc.D
    B = gpu.launch_geometry["envs_per_tile"]
    io = outputs or Outputs(E, D, dev)
    rng = np.random.default_rng(action_seed)
    rew = torch.zeros(E, dtype=torch.float32, device=dev)
    done = torch.zeros(E, dtype=torch.uint8, device=dev)

    if charge_log:
        gpu.enable_charge_log(True)          # EvCharger's charge_log of every step (FLEET_F_CHARGE_LOG)
    o_obs = orc.reset()                      # start indices from the counter RNG on both sides
    obs0, _ = io.at(-1)
    gpu.reset(obs=obs0)
    np.testing.assert_array_equal(gpu.get("time_idx").cpu().numpy(), orc.get("time_idx"))
    np.testing.assert_array_equal(obs0.cpu().numpy(), o_obs)
    if hook:
        hook(-1, None, obs0, None, None, None)

    # SOC / soc_deg are bit-exact for a given SOH.  Once a vehicle has been through a daily SEI evaluation its SOH agrees
    # with the oracle to 1e-13 only (device pow/exp vs libm, and the incremental rainflow adds a vehicle's cycle
    # stress terms in commit order, not list order), so its capacity and hence its SOC may differ in the last
    # bit: exact equality is asserted where degradation cannot interfere, the stated 1e-12 otherwise.
    soc_exact = (not consts.calc_degradation) or consts.deg_mode == 1
    n_done = n_mixed = 0
    for s in range(steps):
        a = rng.uniform(-1, 1, (E, N)).astype(np.float32)
        if s % 5 == 0:
            a[rng.random((E, N)) < 0.3] = 0.0          # exact zeros: plateaus in the SOC history
        if s % 7 == 0:
            a[:] = 1.0                                  # everybody charges: overload penalties
        obs, term = io.at(s)
        o_obs, o_rew, o_cash, o_done, o_term = orc.step(a, want_terminal=True)
        gpu.step(torch.from_numpy(a).to(dev), obs, rew, done, term)
        g_done = done.cpu().numpy()
        np.testing.assert_array_equal(g_done, o_done, err_msg=f"done step {s}")
        for k in EXACT:
            np.testing.assert_array_equal(gpu.get(k).cpu().numpy(), orc.get(k), err_msg=f"{k} step {s}")
        for k in ("soc", "soc_deg"):
            g_v, o_v = gpu.get(k).cpu().numpy(), orc.get(k)
            if soc_exact:
                np.testing.assert_array_equal(g_v, o_v, err_msg=f"{k} step {s}")
            else:
                np.testing.assert_allclose(g_v, o_v, rtol=0, atol=1e-12, err_msg=f"{k} step {s}")
                assert (g_v != o_v).mean() < 1e-2, f"{k} step {s}: too many non-identical elements"
        if charge_log:
            g_cl, o_cl = gpu.get("charge_log").cpu().numpy(), orc.get("charge_log")
            if soc_exact:
                np.testing.assert_array_equal(g_cl, o_cl, err_msg=f"charge_log step {s}")
            else:
                np.testing.assert_allclose(g_cl, o_cl, rtol=0, atol=1e-10, err_msg=f"charge_log step {s}")
        np.testing.assert_allclose(gpu.get("reward64").cpu().numpy(), o_rew, rtol=1e-11, atol=1e-10, err_msg=f"reward step {s}")
        np.testing.assert_allclose(gpu.get("cashflow").cpu().numpy(), o_cash, rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(rew.cpu().numpy(), o_rew.astype(np.float32), rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(gpu.get("soh").cpu().numpy(), orc.get("soh"), rtol=0, atol=1e-13, err_msg=f"soh step {s}")
        np.testing.assert_allclose(gpu.get("fd_cyc").cpu().numpy(), orc.get("fd_cyc"), rtol=1e-11, atol=1e-18)
        np.testing.assert_allclose(gpu.get("life").cpu().numpy(), orc.get("life"), rtol=0, atol=1e-13)
        np.testing.assert_allclose(gpu.get("overload").cpu().numpy(), orc.get("overload"), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(gpu.get("soc_viol").cpu().numpy(), orc.get("soc_viol"), rtol=1e-12, atol=1e-15)
        if obs is not None:
            np.testing.assert_array_equal(obs.cpu().numpy(), o_obs, err_msg=f"obs step {s}")
        if consts.auto_reset and o_done.any():
            idx = np.nonzero(o_done)[0]
            if term is not None:
                np.testing.assert_array_equal(term.cpu().numpy()[idx], o_term[idx], err_msg=f"terminal obs step {s}")
            n_done += len(idx)
        n_mixed += mixed_tiles(g_done, B)
        if s < dephase:
            m = (np.arange(E) % dephase == s).astype(np.uint8)
            o_r = orc.reset(mask=m)
            gpu.reset(mask=torch.from_numpy(m).to(dev), obs=obs)
            idx = np.nonzero(m)[0]
            np.testing.assert_array_equal(gpu.get("time_idx").cpu().numpy(), orc.get("time_idx"), err_msg=f"reset {s}")
            if obs is not None:
                np.testing.assert_array_equal(obs.cpu().numpy()[idx], o_r[idx], err_msg=f"reset obs step {s}")
        io.check_untouched(s)
        if hook:
            hook(s, a, obs, rew, done, term)
    if consts.auto_reset:
        assert n_done > 0
    g_stats, o_stats = gpu.stats(), orc.stats()
    for k in o_stats:
        np.testing.assert_allclose(g_stats[k], o_stats[k], rtol=1e-9, atol=1e-9, err_msg=f"stat {k}")
    assert gpu.check_errors() == 0 and orc.err_flags() == 0
    return dict(n_done=n_done, mixed_tiles=n_mixed)
