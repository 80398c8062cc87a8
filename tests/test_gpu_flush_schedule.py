"""Which envs the step kernel puts on the post kernel's work list, against an integer model of the rule.

The rainflow state of a vehicle is read only by the daily 14:45 evaluations, and every reset restarts it.  So the step
kernel consumes history samples only while an evaluation remains in the episode:
  * WL_TRIGGER  the step reaches a 14:45 row: consume the pending samples, then evaluate;
  * WL_FLUSH    an evaluation remains in the episode after this step's, and the ring would wrap with the next sample
                (k + 1 - k_done >= R - 1);
  * WL_RESET    the episode is over.
After the last evaluation of an episode the ring wraps over samples nobody consumed and k_done falls behind.

work_flags() below restates that rule over env4 = {t, t_start, ep_count, k_done} and the time table.  The GPU cases
predict from the state exported before each step which envs push which flags, and check the k_done the post kernel
leaves behind, while run_vs_oracle compares every output and state field with the oracle.  Each case asserts that its
scenarios happened.  The year-long evaluation episode runs under the same rule in
test_gpu_parity.py::test_year_long_evaluation_episode.
"""
import numpy as np
import pytest

from parity_util import knobs, make_case, run_vs_oracle  # noqa: F401  (knobs: fixture)


def trigger_rows(hour, minute):
    """(trig, nxt): trig[t] = row t is 14:45; nxt[t] = the first 14:45 row at or after t (len(trig): none), t <= T."""
    trig = (np.asarray(hour) == 14) & (np.asarray(minute) == 45)
    T = len(trig)
    nxt = np.full(T + 1, T, np.int64)
    for t in range(T - 1, -1, -1):
        nxt[t] = t if trig[t] else nxt[t + 1]
    return trig, nxt


def work_flags(env4, trig, nxt, L, R, calc_deg=True, auto_reset=True):
    """(trigger, reset, flush): the work-list flags each env pushes in its coming step (all False for a frozen env)."""
    T = len(trig)
    t, t0, k_done = (env4[:, j].astype(np.int64) for j in (0, 1, 3))
    k, t_fin = t - t0, t0 + L
    live = np.full(len(t), True) if auto_reset else t < t_fin
    tr = np.minimum(t, T - 2)                                # the step_row the kernel reads
    trigger = live & bool(calc_deg) & trig[tr + 1]
    reset = live & bool(auto_reset) & (t + 1 == t_fin)
    n2 = nxt[np.minimum(tr + 2, T)]                          # the next 14:45 row at or after t + 2
    ahead = live & bool(calc_deg) & (n2 < T) & (n2 <= t_fin)
    flush = ahead & (k + 1 - k_done >= R - 1)
    return trigger, reset, flush


def k_done_after(env4, trigger, reset, flush):
    """k_done after the step of envs that do not reset (a reset starts the next episode at k_done = 0)."""
    k = env4[:, 0].astype(np.int64) - env4[:, 1]
    return np.where(reset, 0, np.where(trigger | flush, k + 1, env4[:, 3]))


def episode_counts(L, R=16, sph=4, new=True):
    """Per-episode work of the rule over every start slot of a day (24-hour days with one 14:45 row each), per episode:
    flush-only entries, history samples consumed, and rows scanned inside an evaluation entry per evaluation."""
    spd = 24 * sph
    T = L + 3 * spd
    step = np.arange(T)
    trig, nxt = trigger_rows((step // sph) % 24, (step % sph) * (60 // sph))
    env4 = np.zeros((spd, 4), np.int64)
    env4[:, 0] = env4[:, 1] = np.arange(spd)
    flush_only = consumed = eval_rows = evals = 0
    for _ in range(L):
        k = env4[:, 0] - env4[:, 1]
        trigger, reset, flush = work_flags(env4, trig, nxt, L, R)
        if not new:                                          # the previous rule: ring-wrap flush in every step
            flush = k + 1 - env4[:, 3] >= R - 1
        pend = k + 1 - env4[:, 3]
        flush_only += int((flush & ~trigger & ~reset).sum())
        consumed += int(pend[trigger | flush].sum())
        eval_rows += int(pend[trigger].sum())
        evals += int(trigger.sum())
        env4[:, 3] = np.where(trigger | flush, k + 1, env4[:, 3])
        env4[:, 0] += 1
    return dict(flush_only=flush_only / spd, consumed=consumed / spd, eval_rows=eval_rows / max(evals, 1))


def test_model_counts():
    """The model at the cfg2 (24-hour episodes) and cfg3 (48-hour) shapes with R = 16: the previous rule consumes
    every sample and flushes every 14 steps; the gated rule roughly halves what cfg2 consumes and flushes, and leaves
    what an evaluation entry scans as it was."""
    old, new = episode_counts(96, new=False), episode_counts(96)
    assert old == pytest.approx(dict(flush_only=5.375, consumed=89.28125, eval_rows=7.71875))
    assert new == pytest.approx(dict(flush_only=2.71875, consumed=48.5, eval_rows=7.71875))
    old, new = episode_counts(192, new=False), episode_counts(192)
    assert old == pytest.approx(dict(flush_only=11.375, consumed=185.28125, eval_rows=6.859375))
    assert new == pytest.approx(dict(flush_only=8.71875, consumed=144.5, eval_rows=6.859375))


def test_model_cases():
    """The rule on a six-row table with 14:45 at rows 1 and 5, L = 4, R = 3 (a wrap flush at two pending samples)."""
    trig, nxt = trigger_rows([14] * 6, [0, 45, 0, 0, 0, 45])
    env4 = np.array([[3, 2, 0, 0],     # row 5 <= t_fin = 6 and two samples pending: wrap flush
                     [4, 2, 0, 0],     # evaluates at row 5; no row >= 6: nothing ahead
                     [5, 3, 0, 0],     # past T - 2: the kernel reads row 4, which evaluates; nothing ahead
                     [2, 0, 0, 0],     # the ring would wrap, but row 5 is after t_fin = 4: no flush
                     [0, 0, 0, 0],     # evaluates at row 1, the first step of the episode
                     [2, 1, 0, 0],     # row 5 <= t_fin = 5 and two samples pending: wrap flush
                     [2, 1, 0, 1],     # one sample pending: nothing
                     [4, 1, 0, 0],     # the last step: evaluates at row 5, then resets
                     [3, 2, 0, 1]])    # the next step evaluates, one sample pending: the evaluation consumes it
    trigger, reset, flush = work_flags(env4, trig, nxt, L=4, R=3)
    assert list(trigger) == [False, True, True, False, True, False, False, True, False]
    assert list(flush) == [True, False, False, False, False, True, False, False, False]
    assert list(reset) == [False, False, False, False, False, False, False, True, False]
    assert list(k_done_after(env4, trigger, reset, flush)) == [2, 3, 3, 0, 1, 2, 1, 0, 1]
    assert not work_flags(env4, trig, nxt, L=4, R=3, calc_deg=False)[2].any()


# name -> make_case arguments plus: E, post grid, steps in episodes, kernel, knobs, and which scenarios must occur
CASES = {
    "lmd_n50_24h": dict(n_evs=50, E=400, post=2, episodes=3),
    "ct_n20_48h_ring4_stack2": dict(n_evs=20, E=400, post=3, episodes=2, use_case="ct", two_trips=True, episode_hours=48,
                                    env=dict(FLEETSTEP_RF_RING=4, FLEETSTEP_RF_STACK=2, FLEETSTEP_RF_EXT_SLOTS=40000),
                                    need=("between_evals", "slow_ext")),
    "lmd_n9_nocarry": dict(n_evs=9, E=300, post=2, episodes=3, over=dict(carry_degradation_state=0)),
    "lmd_n7_generic_frozen": dict(n_evs=7, E=600, post=2, episodes=3, kernel="generic", over=dict(auto_reset=0),
                                  need=("frozen",)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_schedule_vs_model(name, knobs):
    from fleetrl_b200._lib import FleetStepHandle
    from oracle.oracle import OracleFleet
    from test_gpu_state import parse_blob
    cf = dict(CASES[name])
    E, post, episodes, kernel = cf.pop("E"), cf.pop("post"), cf.pop("episodes"), cf.pop("kernel", None)
    env, need = cf.pop("env", {}), cf.pop("need", ())
    knobs(FLEETSTEP_POST_GRID=post, FLEETSTEP_KERNEL=kernel, **env)
    consts, tables = make_case(name, days=8, **cf)
    L, auto = consts.episode_steps, bool(consts.auto_reset)
    gpu = FleetStepHandle(consts, tables, E, device=0, env_id_offset=1000)
    assert gpu.launch_geometry["post_grid"] == post, gpu.launch_geometry
    if kernel:
        assert gpu.step_kernel_name == "fleet_step_kernel", gpu.step_kernel_name
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    trig, nxt = trigger_rows(tables["hour"], tables["minute"])
    n_trig = np.concatenate([[0], np.cumsum(trig)])        # n_trig[t + 1]: 14:45 rows <= t
    st = dict(checked=0, wrapped=0, wrapped_then_eval=0, one_pending=0, trig_first=0, trig_last=0, between_evals=0,
              slow_ext=0, frozen=0, flush_only=0)
    prev = {}
    wrapped_ep = np.full(E, -1)                              # ep_count of an env when its ring was seen wrapped

    def hook(s, *_):
        p = parse_blob(gpu.export_state())
        R, S = int(p["header"]["R"]), int(p["header"]["S"])
        env4 = p["env4"].astype(np.int64)
        t, t0, ep, k_done = env4[:, 0], env4[:, 1], env4[:, 2], env4[:, 3]
        k = t - t0
        if prev:                                             # the k_done the post kernel left behind
            keep = np.full(E, True)
            if s < L:                                        # envs re-reset by the de-phasing after this step
                keep = np.arange(E) % L != s
            np.testing.assert_array_equal(k_done[keep], prev["k_done"][keep], err_msg=f"k_done after step {s}")
            st["checked"] += int(keep.sum())
        live = np.full(E, True) if auto else t < t0 + L
        wrapped = live & (k - k_done > R - 1)
        st["wrapped"] += int(wrapped.sum())
        wrapped_ep[wrapped & (wrapped_ep < 0)] = ep[wrapped & (wrapped_ep < 0)]
        st["frozen"] += int((~live).sum())
        trigger, reset, flush = work_flags(env4, trig, nxt, L, R, consts.calc_degradation, auto)
        assert not (trigger & wrapped).any() and not (flush & wrapped).any(), f"step {s + 1} consumes a wrapped ring"
        st["wrapped_then_eval"] += int((trigger & (wrapped_ep >= 0) & (ep > wrapped_ep)).sum())
        st["one_pending"] += int((trigger & (k + 1 - k_done == 1)).sum())
        st["trig_first"] += int((trigger & (k == 0)).sum())
        st["trig_last"] += int((trigger & (t + 1 == t0 + L)).sum())
        evals_before = n_trig[t + 1] - n_trig[t0 + 1]      # 14:45 rows t0+1 .. t: evaluations already in this episode
        wrap_flush = flush & (k + 1 - k_done >= R - 1)
        st["between_evals"] += int((wrap_flush & ~trigger & (evals_before > 0)).sum())
        only = flush & ~trigger & ~reset
        st["flush_only"] += int(only.sum())
        depth = (p["rf_dc"] & 0xFFFF).astype(np.int64)
        st["slow_ext"] += int(((depth > S) & (p["rf_ext"] >= 0) & (trigger | flush)[:, None]).sum())
        prev.update(k_done=k_done_after(env4, trigger, reset, flush))

    steps = episodes * L if episodes > 2 else 2 * L + 10
    run_vs_oracle(gpu, orc, steps, charge_log=False, dephase=L, hook=hook)
    gpu.close()
    assert st["checked"] > E * (steps - L) // 2, st
    assert st["flush_only"] > 0 and st["one_pending"] > 0 and st["trig_first"] > 0 and st["trig_last"] > 0, st
    assert st["wrapped"] > 0 and (st["wrapped_then_eval"] > 0 or not auto), st
    for k in need:
        assert st[k] > 0, (k, st)


@pytest.mark.gpu
def test_resume_with_wrapped_ring(knobs):
    """export_state() of a capped pf handle at a step where some env's ring has wrapped past k_done (no evaluation left
    in its episode), imported into a dirty pf handle and into a generic-kernel handle: all three continue bit for bit
    (the generic handle's per-env sums to rounding) through the wrapped envs' reset and the next evaluation."""
    import torch
    from oracle.oracle import OracleFleet
    from test_gpu_state import (RESUME_ENV, Outputs, _assert_pf_capped, _capped_envs, _compare_handles, _handle,
                                parse_blob)
    knobs(**RESUME_ENV)
    consts, tables = make_case("resume_wrapped_ring", 20, use_case="ct", two_trips=True)
    E = _capped_envs(consts, tables, 1)
    L = consts.episode_steps
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(5)
    trig, nxt = trigger_rows(tables["hour"], tables["minute"])

    def dirty(h):
        h.reset()
        for _ in range(L + 17):
            h.step(torch.from_numpy(rng.uniform(-1, 1, (E, h.N)).astype(np.float32)).to(dev))
        return h

    knobs(FLEETSTEP_PF_GRID=1)
    a = _handle(consts, tables, E)
    _assert_pf_capped(a, 1)
    b = dirty(_handle(consts, tables, E))
    knobs(FLEETSTEP_KERNEL="generic")
    c = dirty(_handle(consts, tables, E))
    assert c.step_kernel_name == "fleet_step_kernel"
    knobs(FLEETSTEP_KERNEL=None)

    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    st = dict(export_step=None, wrapped=None, reset_after=0, eval_after=0, steps_after=0)
    outs = [(torch.zeros((E, a.D), dtype=torch.float32, device=dev), torch.zeros(E, dtype=torch.float32, device=dev),
             torch.zeros(E, dtype=torch.uint8, device=dev), torch.zeros((E, a.D), dtype=torch.float32, device=dev))
            for _ in range(2)]

    def hook(s, act, obs, rew, done, term):
        if s < L:
            return
        p = parse_blob(a.export_state())
        env4 = p["env4"].astype(np.int64)
        if st["export_step"] is None:
            wrapped = env4[:, 0] - env4[:, 1] - env4[:, 3] > int(p["header"]["R"]) - 1
            if not wrapped.any():
                return
            st.update(export_step=s, wrapped=wrapped, ep=env4[:, 2].copy())
            for h in (b, c):
                h.import_state(a.export_state())
            _compare_handles(a, (b, c), s, [(obs, rew, done, term)] * 3)
            return
        a_t = torch.from_numpy(act).to(dev)
        for h, (o, r, d, t) in zip((b, c), outs):
            h.step(a_t, o, r, d, t)
        _compare_handles(a, (b, c), s, [(obs, rew, done, term)] + outs, other_kernel=(1,))
        st["steps_after"] += 1
        w, new_ep = st["wrapped"], env4[:, 2] > st["ep"]
        st["reset_after"] += int((w & new_ep).sum())
        trigger = work_flags(env4, trig, nxt, L, int(p["header"]["R"]))[0]
        st["eval_after"] += int((w & new_ep & trigger).sum())

    run_vs_oracle(a, orc, 4 * L, charge_log=False, dephase=L, outputs=Outputs(E, a.D, dev), hook=hook)
    assert st["export_step"] is not None and st["reset_after"] > 0 and st["eval_after"] > 0, st
    for h in (b, c):
        assert h.check_errors() == 0
    for h in (a, b, c):
        h.close()
