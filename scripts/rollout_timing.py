"""Cost of the device RolloutBuffer (fleet_rollout_add / _gae / _gather) at cfg2 (65,536 envs, D = 388, 50 EVs) and at a cfg5
shard (131,072 envs on one GPU), T = 64 steps, next to torch compositions that produce the same outputs, timed in the same
run, alternating.

Prints one JSON line: the card's name and power limit, the copy peak measured in the same run, and per config the
CUDA-event time per call of add, GAE and one epoch of gathers (batch 65,536), each with its algorithmic bytes and share
of the copy peak; the torch baselines (GAE as a T-step loop of float32 ops, the gather as index arithmetic plus
index_select); and the collector's cost per step against policy + FleetVecNormalize.step_raw alone with a trivial
policy.

  python scripts/rollout_timing.py [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from normalize_timing import card, copy_peak_gbs, timed   # noqa: E402

CONFIGS = {"cfg2": 65536, "cfg5_shard": 131072}
T, BATCH = 64, 65536


def torch_gae(buf, last_values, dones):
    """compute_returns_and_advantage as a T-step loop of float32 torch ops in SB3's order (same bits as the kernel)."""
    g, gl = np.float32(buf.gamma).item(), np.float32(buf.gamma * buf.gae_lambda).item()
    lgl = torch.zeros_like(last_values)
    adv = torch.empty_like(buf.advantages)
    for t in reversed(range(buf.buffer_size)):
        if t == buf.buffer_size - 1:
            nnt, nv = 1.0 - dones.float(), last_values
        else:
            nnt, nv = 1.0 - buf.episode_starts[t + 1], buf.values[t + 1]
        delta = buf.rewards[t] + (g * nv) * nnt - buf.values[t]
        lgl = delta + (gl * nnt) * lgl
        adv[t] = lgl
    return adv, adv + buf.values


def torch_gather(buf, idx):
    """_get_samples as index arithmetic plus index_select on the [T*E] views of the storage."""
    T_, E = buf.buffer_size, buf.n_envs
    row = (idx % T_) * E + idx // T_
    return (buf.observations.view(T_ * E, -1).index_select(0, row), buf.actions.view(T_ * E, -1).index_select(0, row),
            *[getattr(buf, n).view(-1).index_select(0, row) for n in ("values", "log_probs", "advantages", "returns")])


class TrivialPolicy:
    def __init__(self, E, N, dev):
        self.a = torch.zeros((E, N), device=dev)
        self.v = torch.zeros((E, 1), device=dev)
        self.lp = torch.zeros(E, device=dev)

    def forward(self, obs):
        return self.a, self.v, self.lp

    def predict_values(self, obs):
        return self.v


def run_config(name, E, args, peak):
    import bench
    from fleetrl_b200 import FleetVecEnv, FleetVecNormalize
    from fleetrl_b200.rollout import FleetRolloutBuffer, collect_rollouts
    wl = SimpleNamespace(use_case="lmd", evs=50, episode_hours=24, carry=1, cfg=dict(over={}, minutes=15))
    built = bench.build_workload(wl)
    env = FleetVecEnv(None, E, built=built, output="torch")
    vn = FleetVecNormalize(env)
    dev, D, N = env.device, env.obs_dim, env.num_cars
    buf = FleetRolloutBuffer(T, E, D, N, dev, gamma=0.99, gae_lambda=0.95)
    pol = TrivialPolicy(E, N, dev)
    obs = vn.reset()
    g = torch.Generator(device=dev).manual_seed(0)
    for s in range(120):                                       # past the first episode ends: done envs every step
        obs, _, _ = vn.step_raw(torch.rand((E, N), generator=g, device=dev) * 2 - 1)
    starts = torch.ones(E, dtype=torch.bool, device=dev)
    obs, starts = collect_rollouts(vn, pol, buf, obs, starts)   # fills the buffer with real transitions
    torch.cuda.synchronize()

    x, a, r, d = env._obs, pol.a, env._rew, env._done
    lv, val = torch.randn(E, generator=g, device=dev), torch.randn(E, generator=g, device=dev)
    slot = [0]

    def add():
        buf._write(slot[0], x, a, r, d, val, val)
        slot[0] = (slot[0] + 1) % T

    def gae():
        buf.compute_returns_and_advantage(lv, d)

    perm = torch.randperm(T * E, device=dev, generator=g)

    def gather_epoch():
        for s in range(0, T * E, BATCH):
            buf._get_samples(perm[s:s + BATCH])

    def torch_gather_epoch():
        for s in range(0, T * E, BATCH):
            torch_gather(buf, perm[s:s + BATCH])

    # same outputs: the torch compositions against the kernels, bit for bit
    adv_t, ret_t = torch_gae(buf, lv, d)
    gae()
    same_gae = bool(torch.equal(adv_t, buf.advantages) and torch.equal(ret_t, buf.returns))
    same_gather = all(torch.equal(p, q) for p, q in zip(buf._get_samples(perm[:BATCH]), torch_gather(buf, perm[:BATCH])))

    def collect():
        nonlocal obs, starts
        obs, starts = collect_rollouts(vn, pol, buf, obs, starts)

    def step_only():
        o = obs
        for _ in range(T):
            pol.forward(o)
            o, _, _ = vn.step_raw(torch.clamp(pol.a, -1.0, 1.0))

    fns = {"add": (add, args.calls), "torch_add": (lambda: (buf.observations[0].copy_(x), buf.actions[0].copy_(a),
                                                           buf.rewards[0].copy_(r), buf.episode_starts[0].copy_(d),
                                                           buf.values[0].copy_(val), buf.log_probs[0].copy_(val)), args.calls),
           "gae": (gae, args.calls), "torch_gae": (lambda: torch_gae(buf, lv, d), max(1, args.calls // 10)),
           "gather_epoch": (gather_epoch, 2), "torch_gather_epoch": (torch_gather_epoch, 2),
           "collect": (collect, 1), "step_only": (step_only, 1)}
    for f, _ in fns.values():
        f()
    res = {k2: [] for k2 in fns}
    for _ in range(args.rounds):                                # alternate the variants
        for k2, (f, n) in fns.items():
            res[k2].append(timed(f, n))
    med = {k2: float(np.median(v)) for k2, v in res.items()}
    B_obs = E * D * 4
    alg = {"add": 2 * (B_obs + E * N * 4) + 7 * E * 4 + E,           # rows read + written; 3 floats + 1 B read, 4 floats written
           "gae": 3 * T * E * 4 + E * 5 + 2 * T * E * 4,                                   # read r, v, starts; write adv, ret
           "gather_epoch": T * E * (2 * (D + N + 4) * 4 + 8)}                              # read + write rows, index
    line = {"config": name, "envs": E, "obs_dim": D, "action_dim": N, "buffer_size": T, "batch": BATCH,
            "storage_gb": (T * E * (D + N + 6) * 4) / 1e9, "same_outputs_gae": same_gae, "same_outputs_gather": same_gather,
            "launches": {"add": 1, "gae": 1, "gather_epoch": -(-T * E // BATCH)}}
    for k2 in ("add", "gae", "gather_epoch"):
        ms = med[k2]
        line[k2] = {"ms": ms, "ms_rounds": res[k2], "alg_bytes": alg[k2], "alg_gbs": alg[k2] / (ms * 1e-3) / 1e9,
                    "frac_copy_peak": alg[k2] / (ms * 1e-3) / 1e9 / peak, "floor_ms_at_peak": alg[k2] / (peak * 1e9) * 1e3,
                    "torch_ms": med["torch_" + k2], "speedup_vs_torch": med["torch_" + k2] / ms}
    line["collector"] = {"collect_ms_per_step": med["collect"] / T, "policy_step_raw_ms_per_step": med["step_only"] / T,
                         "overhead_ms_per_step": (med["collect"] - med["step_only"]) / T,
                         "note": "collect includes the final predict_values and the GAE launch"}
    vn.close()
    del buf
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--configs", default="cfg2,cfg5_shard")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rollout_timing.py measures on a GPU; none is available")
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
