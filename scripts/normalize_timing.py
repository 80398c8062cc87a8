"""Cost of the device VecNormalize (fleet_norm_moments + fleet_norm_apply) at cfg2 (65,536 envs x 50 EVs, D = 388) and
at a cfg5 shard (131,072 envs on one GPU), next to a torch-composed float64 equivalent timed in the same run, alternating.

Prints one JSON line: the card's name and power limit, per config the CUDA-event time of the two normalisation kernels
per step, their algorithmic bytes (two reads and one write of the float32 observation batch plus the per-env reward,
return and done traffic) against the copy peak measured in the same run, the torch baseline, and the env step time
with and without the normaliser (FleetVecEnv.step_raw against FleetVecNormalize.step_raw).

  python scripts/normalize_timing.py [--steps 50] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {"cfg2": 65536, "cfg5_shard": 131072}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, power = (q[0].split(", ") + ["?"])[:2] if q else (torch.cuda.get_device_name(0), "?")
    return {"name": name, "power_limit": power}


def timed(fn, n):
    """ms per call of fn over n calls, CUDA events."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def copy_peak_gbs():
    src = torch.empty(1 << 28, dtype=torch.float32, device="cuda")        # 1 GiB, far beyond L2
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    ms = timed(lambda: dst.copy_(src), 20)
    return 2 * src.numel() * 4 / (ms * 1e-3) / 1e9


class TorchNormalize:
    """The same step as fleet_norm_moments + fleet_norm_apply composed from torch float64 operations."""

    def __init__(self, E, D, dev, gamma=0.99, eps=1e-8, clip=10.0):
        f = dict(dtype=torch.float64, device=dev)
        self.mean, self.var, self.count = torch.zeros(D, **f), torch.ones(D, **f), torch.full((), 1e-4, **f)
        self.rmean, self.rvar, self.rcount = torch.zeros((), **f), torch.ones((), **f), torch.full((), 1e-4, **f)
        self.ret = torch.zeros(E, **f)
        self.gamma, self.eps, self.clip = gamma, eps, clip

    @staticmethod
    def _merge(mean, var, count, bm, bv, n):
        delta = bm - mean
        tot = count + n
        return mean + delta * n / tot, (var * count + bv * n + delta * delta * count * n / tot) / tot, count + n

    def step(self, x, r, done, term, out, rout, tout):
        x64 = x.double()
        n = x.shape[0]
        self.mean, self.var, self.count = self._merge(self.mean, self.var, self.count, x64.mean(0), x64.var(0, unbiased=False), n)
        self.ret = self.ret * self.gamma + r.double()
        self.rmean, self.rvar, self.rcount = self._merge(self.rmean, self.rvar, self.rcount, self.ret.mean(),
                                                         self.ret.var(unbiased=False), n)
        den = torch.sqrt(self.var + self.eps)
        out.copy_(((x64 - self.mean) / den).clamp_(-self.clip, self.clip))
        rout.copy_((r.double() / torch.sqrt(self.rvar + self.eps)).clamp_(-self.clip, self.clip))
        d = done.bool()
        tout.copy_(torch.where(d[:, None], ((term.double() - self.mean) / den).clamp_(-self.clip, self.clip), tout.double()))
        self.ret.masked_fill_(d, 0.0)


def run_config(name, E, args, peak):
    import bench
    from fleetrl_b200 import FleetVecEnv, FleetVecNormalize
    wl = SimpleNamespace(use_case="lmd", evs=50, episode_hours=24, carry=1, cfg=dict(over={}, minutes=15))
    built = bench.build_workload(wl)
    env = FleetVecEnv(None, E, built=built, output="torch")
    vn = FleetVecNormalize(env)
    dev, D, N = env.device, env.obs_dim, env.num_cars
    g = torch.Generator(device=dev).manual_seed(0)
    acts = [torch.rand((E, N), generator=g, device=dev) * 2 - 1 for _ in range(8)]
    vn.reset()
    for s in range(120):                                       # past the first episode ends: done envs every step
        vn.step_raw(acts[s % 8])
    torch.cuda.synchronize()
    x, r, done, term = env._obs, env._rew, env._done, env._term
    h, m = vn.handle, vn._moments
    out, rout, tout = vn._obs_n, vn._rew_n, vn._term_n

    def ours():
        h.moments(x, r, m)
        h.apply(m, x, out, r, rout, done, term, tout)

    tn = TorchNormalize(E, D, dev)
    t_out, t_rout, t_tout = torch.empty_like(out), torch.empty_like(rout), torch.empty_like(tout)
    base = lambda: tn.step(x, r, done, term, t_out, t_rout, t_tout)
    k = [0]

    def env_only():
        env.step_raw(acts[k[0] % 8]); k[0] += 1

    def env_norm():
        vn.step_raw(acts[k[0] % 8]); k[0] += 1

    for f in (ours, base, env_only, env_norm):
        for _ in range(5):
            f()
    res = {"ours": [], "moments": [], "apply": [], "torch_f64": [], "step_env": [], "step_env_norm": []}
    for _ in range(args.rounds):                                # alternate the variants
        res["ours"].append(timed(ours, args.steps))
        res["moments"].append(timed(lambda: h.moments(x, r, m), args.steps))
        res["apply"].append(timed(lambda: h.apply(m, x, out, r, rout, done, term, tout), args.steps))
        res["torch_f64"].append(timed(base, args.steps))
        res["step_env"].append(timed(env_only, args.steps))
        res["step_env_norm"].append(timed(env_norm, args.steps))
    med = {k2: float(np.median(v)) for k2, v in res.items()}
    alg = 3 * E * D * 4 + 37 * E                               # obs: moments read, apply read + write; per env 37 B
    line = {"config": name, "envs": E, "obs_dim": D, "batch_mb": E * D * 4 / 1e6,
            "l2_note": "the 126 MB L2 holds part of the cfg2 batch between the two kernels" if E * D * 4 < 126e6 else
                       "batch exceeds the 126 MB L2",
            "norm_ms": med["ours"], "norm_ms_rounds": res["ours"], "moments_ms": med["moments"], "apply_ms": med["apply"],
            "torch_f64_ms": med["torch_f64"],
            "torch_f64_ms_rounds": res["torch_f64"], "speedup_vs_torch": med["torch_f64"] / med["ours"],
            "alg_bytes": alg, "alg_gbs": alg / (med["ours"] * 1e-3) / 1e9, "frac_copy_peak": alg / (med["ours"] * 1e-3) / 1e9 / peak,
            "floor_ms_at_peak": alg / (peak * 1e9) * 1e3,
            "step_env_ms": med["step_env"], "step_env_norm_ms": med["step_env_norm"],
            "launches_per_step": 2}
    vn.close()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--configs", default="cfg2,cfg5_shard")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("normalize_timing.py measures on a GPU; none is available")
    peak = copy_peak_gbs()
    rec = {"card": card(), "copy_peak_gbs": peak, "configs": []}
    for name in args.configs.split(","):
        rec["configs"].append(run_config(name, CONFIGS[name], args, peak))
        torch.cuda.empty_cache()
    s = json.dumps(rec)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
