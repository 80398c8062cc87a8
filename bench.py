#!/usr/bin/env python
"""bench.py — EV-steps/sec of the FleetRL environment step on B200 (BASELINE.json metric), one JSON line.

Workload (BASELINE.json configs[1], SURVEY §8d "cfg2"): last-mile-delivery fleet, 50 EVs x 65,536 parallel envs
per GPU, rainflow/SEI degradation, 15-minute steps, 24-hour episodes, full observer (D = 388), random start
indices, random actions U(-1,1) float32 resident in HBM, SB3-style auto-reset.  Synthetic fleet / price / load /
PV (no network, the reference's multi-EV CSVs are missing blobs) — said so in "data".

A "step" is one fleet_step() call over all envs of the rank (one kernel launch).
  value     : whole-job EV-steps/s with inputs resident in HBM, CUDA-event timed on the launching stream,
              max over ranks (weak scaling: per-GPU work fixed).
  roofline  : algorithmic bytes per launch (SURVEY §8d: B_alg = 52 + (4*D+13)/N bytes per EV-step) / measured
              kernel time, against the measured HBM copy peak (MEASURED_PEAKS.json).
  e2e       : the same metric through fleet_step_host(): host (pinned) action buffer in, host obs/reward/done
              out, H2D + kernel + D2H + stream sync every step.
  cpu_baseline : the C oracle port (oracle/fleet_oracle.c) on all host cores on a bounded sample.
`--impl reference` times the reference arm: the reference is pure Python and cannot travel to the GPU box, so
it is the oracle port of the reference's algorithm on all host threads (kind "port").

Multi-GPU: launched by torchrun, one rank per GPU; envs shard with no data-path collective; the only NCCL call
is one all-reduce of the 10-double episode-statistics vector at the end of the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


# BASELINE.json configs[1..4] (SURVEY §8d).  cfg2 is the metric's configuration; the others are selected with --config.
CONFIGS = {
    "cfg2": dict(use_case="lmd", evs=50, envs=65536, episode_hours=24, minutes=15, over={},
                 label="LMD fleet, 50 EVs, rainflow-SEI degradation, 15-min steps, 24 h episodes, full observer (cfg2)"),
    "cfg3": dict(use_case="ct", evs=20, envs=65536, episode_hours=48, minutes=15, over={},
                 label="caretaker fleet, 20 EVs, building load + PV + grid cap, lunch-break target, rainflow-SEI, 48 h episodes (cfg3)"),
    "cfg4": dict(use_case="ut", evs=50, envs=65536, episode_hours=48, minutes=60, tariff="fixed",
                 over=dict(include_building=False, include_pv=False, spot_markup=10, spot_mul=1.5, feed_in_ded=0.25),
                 label="utility fleet, 50 EVs, V2G, spot price + feed-in tariff, 1-hour resolution, price-only observer (cfg4)"),
    "cfg4full": dict(use_case="ut", evs=50, envs=65536, episode_hours=48, minutes=60, tariff="fixed",
                     over=dict(spot_markup=10, spot_mul=1.5, feed_in_ded=0.25),
                     label="utility fleet, 50 EVs, V2G, 1-hour resolution, full observer (cfg4 variant)"),
    "cfg5": dict(use_case="lmd", evs=50, total_envs=1048576, episode_hours=24, minutes=15, over={},
                 label="LMD fleet, 50 EVs, 1,048,576 envs sharded over the GPUs (cfg5 env step; the PPO-style rollout "
                       "through FleetVecEnv is scripts/rollout_cfg5.py)"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS),
                    help="BASELINE.json workload (cfg2 = configs[1], the one the metric is quoted on)")
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the config's)")
    ap.add_argument("--evs", type=int, default=None)
    ap.add_argument("--use-case", default=None)
    ap.add_argument("--episode-hours", type=int, default=None)
    ap.add_argument("--carry", type=int, default=1, help="carry_degradation_state (1 = reference object semantics)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--ref-envs", type=int, default=2048)
    ap.add_argument("--actions", default="random", choices=["random", "uncontrolled"],
                    help="random: U(-1,1) per (env, EV) and step; uncontrolled: a = 1 everywhere (benchmarking/"
                         "uncontrolled_charging.py:51-54; exercises the overload / overcharging penalty paths, SURVEY 8d cfg2)")
    ap.add_argument("--raw-inputs", action="store_true",
                    help="skip the CSV text round trip of the synthetic inputs (saves ~8 s of start-up; diagnostic runs)")
    ap.add_argument("--settle-episodes", type=int, default=10,
                    help="extra untimed episodes after de-phasing: an env object lives for the whole training run, and its "
                         "RainflowSeiDegradation.rainflow_length (carried across episodes, rainflow_sei_degradation.py:195) converges "
                         "to its running maximum within a few episodes, after which fewer cycles need a stress evaluation; "
                         "without settling a 20-step window runs 5 %% slower than a 960-step one, with it 1.7 %%")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (reward, done, obs, terminal_obs) "
                         "as DIR/<name>.npy, for a fixed, seeded sample of env rows (env_index.npy) of at most 64 MiB in all; "
                         "rank 0's envs when run on several GPUs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours; the reference arm materialises none")
    cf = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.envs is None:
        args.envs = cf["total_envs"] // world if "total_envs" in cf else cf["envs"]
    for k in ("evs", "use_case", "episode_hours"):
        if getattr(args, k) is None:
            setattr(args, k, cf[k])
    args.scaling = "strong" if "total_envs" in cf else "weak"
    args.cfg = cf
    return args


def build_workload(args):
    from fleetrl_b200.config import default_config
    from fleetrl_b200.schedule import generate_schedule, synthetic_series
    from fleetrl_b200.tables import FleetInputs, build_fleet

    sched = generate_schedule(args.use_case, args.evs, seed=42)
    price, tariff, load, pv = synthetic_series(seed=7, tariff=args.cfg.get("tariff", "spot"))
    over = dict(args.cfg["over"])
    if args.cfg["minutes"] == 60:
        over.update(freq="1h", minutes=60, time_steps_per_hour=1)
    cfg = default_config(args.use_case, episode_length=args.episode_hours, seed=0, **over)
    inputs = FleetInputs(sched, price, tariff, load, pv)
    if not getattr(args, "raw_inputs", False):
        # the fleet exactly as the unmodified reference would read it from schedule.write_reference_csvs' files
        # (pandas' CSV float parser moves ~1/8 of the values by one ulp; tests/test_host_logic.py)
        inputs = inputs.csv_round_trip()
    built = build_fleet(cfg, inputs, auto_reset=True,
                        carry_degradation_state=bool(args.carry), seed=0, time_picker="random")
    return built


def b_alg(N, D):
    """SURVEY §8d contract figure: interface + minimal persistent state per EV-step (f64 soc/soc_deg/soh)."""
    return 52.0 + (4.0 * D + 13.0) / N


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(args, D):
    """dram bytes per launch of the step kernel from the committed ncu --set full capture, if it matches."""
    p = os.path.join(ROOT, "profiles", "step_kernel_traffic.json")
    try:
        d = json.load(open(p))
        if d.get("envs") == args.envs and d.get("evs") == args.evs and d.get("obs_dim") == D:
            return float(d["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe), sampled through NVML every
    ~2 ms from a thread (nvidia-smi -lms is too slow to start for a region of tens of milliseconds)."""

    def __init__(self, index):
        self.index, self.rows, self._stop, self.th, self.err = index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.err = f"nvml unavailable: {e}"
            return
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        nv = self.nv
        while not self._stop:
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:
                try:
                    self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                      nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
                except Exception:
                    pass
            time.sleep(0.002)

    def mark(self):
        """samples taken before this point are dropped (call right before the timed region)"""
        self.rows = []

    def stop(self):
        if self.th is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err or "not started"]}
        self._stop = True
        self.th.join(timeout=1)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        sm = [r[0] for r in self.rows]
        reasons = sorted(k for k, bit in names.items() if any(r[1] & bit for r in self.rows))
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.max_sm),
                "reasons": reasons, "samples": len(sm)}


def cpu_baseline(built, seconds, n_envs, steps_cap=96):
    """Oracle port on all host cores on a bounded sample of the same workload."""
    from oracle.oracle import OracleFleet
    cores = len(os.sched_getaffinity(0))
    c, N = built.consts, built.consts.num_evs
    orc = OracleFleet(c, built.tables, n_envs, threads=cores)
    orc.reset()
    rng = np.random.default_rng(1)
    acts = [rng.uniform(-1, 1, (n_envs, N)).astype(np.float32) for _ in range(4)]
    orc.step_noout(acts[0])
    t0 = time.perf_counter()
    n = 0
    while True:
        orc.step_noout(acts[n % 4])
        n += 1
        el = time.perf_counter() - t0
        if el > seconds or n >= steps_cap * 1000:
            break
    orc.close()
    return {"value": n_envs * N * n / el, "unit": "EV-steps/s", "cores": cores, "kind": "port",
            "sample": f"{n_envs} envs x {N} EVs x {n} steps of the same fleet (oracle/fleet_oracle.c, {cores} POSIX threads, {el:.1f} s)"}


def run_reference(args):
    """Reference arm: the reference's CPU algorithm (oracle port; the Python reference cannot travel) on all host
    threads, same config/metric; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    built = build_workload(args)
    from oracle.oracle import OracleFleet
    cores = len(os.sched_getaffinity(0))
    N, E = built.consts.num_evs, args.ref_envs
    orc = OracleFleet(built.consts, built.tables, E, threads=cores)
    orc.reset()
    rng = np.random.default_rng(1)
    acts = [rng.uniform(-1, 1, (E, N)).astype(np.float32) for _ in range(4)]
    for w in range(args.warmup):
        orc.step_noout(acts[w % 4])
    t0 = time.perf_counter()
    for s in range(args.steps):
        orc.step_noout(acts[s % 4])
    el = time.perf_counter() - t0
    value = E * N * args.steps / el
    D = orc.D
    sample = f"each step = {E} envs x {N} EVs of the same synthetic fleet, {cores} POSIX threads"
    line = {
        "impl": "reference", "metric": "EV-steps/sec", "value": value, "unit": "EV-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(workload_config(args, built, D), envs_per_step_timed=E,
                       sample=f"bounded sample: {E} of the {args.envs} envs per step (the per-env work is identical)"),
        "cpu_baseline": {"value": value, "unit": "EV-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "EV-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference FleetEnv is pure Python/pandas (≈35-85 EV-steps/s/core measured in the build container, "
                "BASELINE.md §2) and is not present on the GPU box; this arm times the C port of its algorithm",
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 << 20


def dump_outputs(path, obs, rew, done, term):
    """Write what fleet_step returned to its caller in the last step as float32 / float64 .npy files under `path`.

    All envs' rows would exceed DUMP_BYTES at the benchmark's sizes (obs alone is 100 MB at cfg2), so the same fixed,
    seeded sample of env rows is taken from every per-env output; env_index.npy lists it.  terminal_obs holds the rows
    of the sampled envs that finished in that step, in sample order: the step writes no other row of it."""
    import torch
    E, D = obs.shape
    row_bytes = 8 + 4 * (2 + 2 * D)                  # env_index (f64), reward and done (f32), obs and terminal_obs rows
    rows = min(E, (DUMP_BYTES - (1 << 16)) // row_bytes)     # 64 KiB left for the .npy headers
    idx = np.arange(E) if rows == E else np.sort(np.random.default_rng(0).choice(E, rows, replace=False))
    sel = torch.from_numpy(idx).to(obs.device)
    d = done.index_select(0, sel)
    arrays = {"env_index": idx.astype(np.float64), "reward": rew.index_select(0, sel), "done": d.float(),
              "obs": obs.index_select(0, sel), "terminal_obs": term.index_select(0, sel)[d.bool()]}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy() if torch.is_tensor(a) else a)


def workload_config(args, built, D):
    return {"workload": f"{args.cfg['label']}; {args.envs} envs/GPU", "name": args.config,
            "envs_per_gpu": args.envs, "evs": args.evs, "obs_dim": D, "table_len": int(built.consts.table_len),
            "episode_steps": int(built.consts.episode_steps), "auto_reset": True,
            "carry_degradation_state": bool(args.carry), "actions": getattr(args, "actions", "random"),
            "episode_phase": "de-phased: env e is (e mod episode_steps) steps into its episode when timing starts, so "
                             "every step sees ~E/episode_steps auto-resets and ~E/96 daily evaluations (SB3 steady state); "
                             f"{getattr(args, 'settle_episodes', 0)} untimed episodes per env before timing (rainflow_length settled)",
            "l2_policy": "per-step working set (actions+state+obs ≈ 0.27 GB at cfg2) exceeds the 126 MB L2; "
                         "action tensors rotate through a ring"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from fleetrl_b200._lib import FleetStepHandle

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    built = build_workload(args)
    E, N = args.envs, built.consts.num_evs
    h = FleetStepHandle(built.consts, built.tables, E, device=local_rank, env_id_offset=rank * E)
    D = h.D
    K, W = args.steps, max(args.warmup, 3)

    obs = torch.empty((E, D), dtype=torch.float32, device=dev)
    term = torch.empty((E, D), dtype=torch.float32, device=dev)
    rew = torch.empty(E, dtype=torch.float32, device=dev)
    done = torch.empty(E, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev); gen.manual_seed(1 + rank)
    ring = [torch.empty((E, N), dtype=torch.float32, device=dev).uniform_(-1, 1, generator=gen) for _ in range(8)]
    if args.actions == "uncontrolled":
        for a in ring:
            a.fill_(1.0)
    h.reset(obs=obs)
    torch.cuda.synchronize(dev)

    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream
    ptrs = [a.data_ptr() for a in ring]
    o_p, r_p, d_p, t_p = obs.data_ptr(), rew.data_ptr(), done.data_ptr(), term.data_ptr()

    # clocks / throttle reasons are sampled from here on: the warm-up below is the same load as the timed region, which
    # alone (tens of ms) would be shorter than nvidia-smi's sampling period
    sampler = ClockSampler(local_rank)
    sampler.start()
    # De-phase the envs, then warm up: a synchronous reset would leave all envs at the same episode step (no resets for
    # L-1 steps, then all at once).  Env e is re-reset after step (e mod L) of the first L steps, so that when timing
    # starts the episode ages are uniform over 0..L-1 — what a long SB3 rollout converges to.
    L = int(built.consts.episode_steps)
    phase = torch.arange(E, device=dev, dtype=torch.int64) % L
    for s in range(L):
        h.step_unchecked(ptrs[s % 8], o_p, r_p, d_p, t_p, sp)
        h.reset(mask=(phase == s).to(torch.uint8), obs=obs)
    for s in range(W + args.settle_episodes * L):
        h.step_unchecked(ptrs[s % 8], o_p, r_p, d_p, t_p, sp)
    torch.cuda.synchronize(dev)
    h.reset_stats()

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    sampler.mark()
    l0 = h.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for s in range(K):
        h.step_unchecked(ptrs[s % 8], o_p, r_p, d_p, t_p, sp)
    ev1.record(stream)
    stats = h.stats_tensor()
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)          # the path's only collective (episode statistics)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    launches = h.launch_count - l0
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    ms_per_step = total_ms / K
    value = world * E * N * K / (total_ms * 1e-3)
    err = h.check_errors()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, obs, rew, done, term)   # before the kernel-timing pass below overwrites them

    # roofline of the dominant kernel (the step kernel): algorithmic bytes per launch / its average launch duration,
    # measured live with CUDA events around each launch (fleet_set_timing) in a second pass over the same workload;
    # the whole step (step kernel + post kernel + launch gaps, i.e. ms_per_step of the timed region) is reported next
    # to it as the conservative figure
    peak, peak_src = measured_peak()
    bytes_per_launch = b_alg(N, D) * E * N
    h.set_timing(True)
    KT = min(max(K, 96), 960)
    for s in range(KT):
        h.step_unchecked(ptrs[s % 8], o_p, r_p, d_p, t_p, sp)
    step_ms, post_ms, nt = h.get_timing()
    h.set_timing(False)
    km = torch.tensor([step_ms / max(nt, 1), post_ms / max(nt, 1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(km, op=dist.ReduceOp.MAX)
    step_kernel_ms, post_kernel_ms = (float(x) for x in km.tolist())
    achieved = bytes_per_launch / (step_kernel_ms * 1e-3) / 1e9
    whole = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(args, D), "peak_source": peak_src,
                "algorithmic_bytes_per_ev_step": b_alg(N, D), "kernel": h.step_kernel_name,
                "kernel_ms": step_kernel_ms, "post_kernel_ms": post_kernel_ms, "timed_launches": nt,
                "whole_step": {"achieved": whole, "frac": whole / peak, "ms": ms_per_step,
                               "note": "step kernel + post kernel (rainflow consumption, daily degradation, auto-reset) + launch gaps"}}

    # end to end through the host-buffer C-ABI call
    e2e = None
    if not args.no_e2e:
        a_host = [torch.empty((E, N), dtype=torch.float32).uniform_(-1, 1).pin_memory() for _ in range(2)]
        o_host = torch.empty((E, D), dtype=torch.float32).pin_memory()
        r_host = torch.empty(E, dtype=torch.float32).pin_memory()
        d_host = torch.empty(E, dtype=torch.uint8).pin_memory()
        an = [a.numpy() for a in a_host]
        on, rn, dn = o_host.numpy(), r_host.numpy(), d_host.numpy()
        for s in range(3):
            h.step_host(an[s % 2], on, rn, dn)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for s in range(args.e2e_steps):
            h.step_host(an[s % 2], on, rn, dn)
        el = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(el, op=dist.ReduceOp.MAX)
        e2e = {"value": world * E * N * args.e2e_steps / float(el.item()), "unit": "EV-steps/s",
               "h2d_bytes_per_step": E * N * 4, "d2h_bytes_per_step": E * D * 4 + E * 4 + E,
               "ms_per_step": float(el.item()) / args.e2e_steps * 1e3, "api": "fleet_step_host (pinned host buffers)"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(built, args.cpu_seconds, n_envs=min(2048, E))

    if rank == 0:
        st = dict(zip(["episodes", "ep_return", "steps", "reward", "cashflow", "penalty", "overload_kw", "soc_viol",
                       "n_viol", "degradation"], stats.cpu().tolist()))
        line = {
            "metric": "EV-steps/sec", "value": value, "unit": "EV-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, built, D),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "device_bytes": h.device_bytes, "device_error_flags": err,
            "episode_stats": {"episodes": st["episodes"], "env_steps": st["steps"],
                              "mean_reward_per_env_step": st["reward"] / max(st["steps"], 1),
                              "soh_loss_sum": st["degradation"]},
        }
        print(json.dumps(line), flush=True)
    h.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
