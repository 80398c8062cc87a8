"""Cost of PPO's update on the device at the cfg2 shape (minibatch 65,536, N = 50, D = 388; buffer T = 64 x E = 65,536),
next to the torch float32 composition of SB3's loss, timed in the same run, alternating the variants.

  * loss: ppo_loss forward + backward (fleet_ppo_*, three launches, through torch.autograd) against SB3's loss written
    in torch float32 (Normal.log_prob, advantage normalisation, clipped surrogate, mse, entropy) with autograd, on the
    same tensors; and the three kernels alone, their C entry points called back to back with prepared arguments;
  * epoch: one ppo_train epoch (64 minibatches: gather, MLP, loss, backward, clip_grad_norm_, Adam) against the same
    loop with the torch loss and SB3's five host reads per minibatch (.item() on the three losses and the clip fraction,
    .cpu() on approx_kl).

Prints one JSON line: the card's name and power limit, the copy peak measured in the same run, and the median of
`--rounds` CUDA-event timings of each variant, with the fused loss's algorithmic bytes and share of the copy peak.

  python scripts/ppo_timing.py [--rounds 5] [--out FILE]
"""
import argparse
import json
import math
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from normalize_timing import card, copy_peak_gbs, timed   # noqa: E402

B, N, D, T, E = 65536, 50, 388, 64, 65536


def torch_loss(mean, log_std, values, s, clip_range=0.2, ent_coef=0.0, vf_coef=0.5, sync=False):
    """PPO.train's loss (ppo.py) as SB3 composes it, in float32; sync=True adds SB3's five host reads."""
    dist = torch.distributions.Normal(mean, torch.ones_like(mean) * log_std.exp())
    lp = dist.log_prob(s.actions).sum(dim=1)
    ent = dist.entropy().sum(dim=1)
    adv = s.advantages
    adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    ratio = torch.exp(lp - s.old_log_prob)
    pl = -torch.min(adv * ratio, adv * torch.clamp(ratio, 1 - clip_range, 1 + clip_range)).mean()
    vl = torch.nn.functional.mse_loss(s.returns, values)
    el = -torch.mean(ent)
    loss = pl + ent_coef * el + vf_coef * vl
    if sync:
        pl.item()
        torch.mean((torch.abs(ratio - 1) > clip_range).float()).item()
        vl.item()
        el.item()
        with torch.no_grad():
            lr = lp - s.old_log_prob
            torch.mean((torch.exp(lr) - 1) - lr).cpu().numpy()
    return loss


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ppo_timing.py measures on a CUDA device; none found")
    from fleetrl_b200.ppo import FleetMlpPolicy, ppo_loss, ppo_train
    from fleetrl_b200.rollout import FleetRolloutBuffer, RolloutBufferSamples

    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    peak = copy_peak_gbs()

    # ---- the loss alone, on one minibatch
    mean = torch.randn((B, N), device=dev, generator=g).requires_grad_(True)
    log_std = torch.full((N,), -0.5, device=dev).requires_grad_(True)
    values = torch.randn(B, device=dev, generator=g).requires_grad_(True)
    acts = (mean.detach() + 0.6 * torch.randn((B, N), device=dev, generator=g)).contiguous()
    with torch.no_grad():
        lp = torch.distributions.Normal(mean, torch.ones_like(mean) * log_std.exp()).log_prob(acts).sum(1)
    s = RolloutBufferSamples(None, acts, torch.randn(B, device=dev, generator=g),
                             (lp + 0.2 * torch.randn(B, device=dev, generator=g)).contiguous(),
                             torch.randn(B, device=dev, generator=g), torch.randn(B, device=dev, generator=g))

    def fused():
        ppo_loss(mean, log_std, values, s).backward()

    def composed():
        torch_loss(mean, log_std, values, s).backward()

    # the three kernels alone: the C entry points called back to back with prepared arguments (no autograd, no checks)
    import ctypes as C
    from fleetrl_b200._lib import load_library
    from fleetrl_b200.ppo import _batch, _params, _workspace
    lib = load_library()
    md, ld, vd = mean.detach(), log_std.detach(), values.detach()
    cb = C.byref(_batch(md, ld, s.actions, vd, s.old_log_prob, s.old_values, s.advantages, s.returns))
    cp = C.byref(_params(0.2, None, True, 0.0, 0.5))
    ws = _workspace(lib, dev, B, N)
    out = [torch.empty(B * N, device=dev) for _ in range(2)] + [torch.empty(N, device=dev), torch.empty(B, device=dev)]
    coef, st = torch.empty(2 * B, device=dev), torch.zeros(5, dtype=torch.float64, device=dev)
    one = torch.ones((), device=dev)
    a_loss = [cb, cp, C.c_void_p(one.data_ptr()), C.c_void_p(st.data_ptr()), C.c_void_p(coef.data_ptr()),
              C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(torch.cuda.current_stream().cuda_stream)]
    a_back = [cb, cp, C.c_void_p(one.data_ptr()), C.c_void_p(coef.data_ptr())] + \
             [C.c_void_p(t.data_ptr()) for t in out[1:]] + a_loss[5:]

    def kernels():
        lib.fleet_ppo_loss(*a_loss)
        lib.fleet_ppo_loss_backward(*a_back)

    for _ in range(3):
        fused()
        composed()
        kernels()
    reps = 200
    f_ms, t_ms, k_ms = [], [], []
    for _ in range(args.rounds):
        f_ms.append(timed(fused, reps))
        t_ms.append(timed(composed, reps))
        k_ms.append(timed(kernels, reps))
    # loss forward + backward, algorithmic bytes: mean and actions read twice (forward, backward), grad_mean written
    # once, plus the [B] vectors (5 read, 2 coefficients written and read, grad_values written)
    alg_bytes = 4 * (2 * 2 * B * N + B * N) + 4 * (5 + 4 + 1) * B
    loss_ms = statistics.median(f_ms)
    res = {"card": card(), "copy_peak_gbs": peak,
           "shape": {"minibatch": B, "action_dim": N, "obs_dim": D, "buffer_size": T, "envs": E},
           "loss": {"fused_ms": loss_ms, "fused_ms_rounds": f_ms, "torch_ms": statistics.median(t_ms),
                    "torch_ms_rounds": t_ms, "speedup_vs_torch": statistics.median(t_ms) / loss_ms,
                    "alg_bytes": alg_bytes, "alg_gbs": alg_bytes / (loss_ms * 1e-3) / 1e9,
                    "frac_copy_peak": alg_bytes / (loss_ms * 1e-3) / 1e9 / peak,
                    "floor_ms_at_peak": alg_bytes / (peak * 1e9) * 1e3,
                    "kernels_ms": statistics.median(k_ms), "kernels_ms_rounds": k_ms,
                    "kernels_frac_copy_peak": alg_bytes / (statistics.median(k_ms) * 1e-3) / 1e9 / peak}}
    del mean, values, acts, s

    # ---- one ppo_train epoch against the SB3-style loop
    buf = FleetRolloutBuffer(T, E, D, N, dev)
    buf.observations.normal_(generator=g)
    buf.actions.normal_(generator=g)
    for name in ("values", "advantages", "returns"):
        getattr(buf, name).normal_(generator=g)
    buf.log_probs.normal_(-71.0, 1.0, generator=g)
    buf.pos, buf.full = T, True
    torch.manual_seed(0)
    pol_a = FleetMlpPolicy(D, N, dev)
    pol_b = FleetMlpPolicy(D, N, dev)
    pol_b.load_state_dict(pol_a.state_dict())

    def epoch_fused():
        ppo_train(pol_a, buf, n_epochs=1, batch_size=B)

    def epoch_torch():
        for data in buf.get(B):
            mean_a, ls, v = pol_b.loss_inputs(data.observations)
            loss = torch_loss(mean_a, ls, v, data, sync=True)
            pol_b.optimizer.zero_grad()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(pol_b.parameters(), 0.5)
            pol_b.optimizer.step()

    epoch_fused()
    epoch_torch()
    ef, et = [], []
    for _ in range(args.rounds):
        ef.append(timed(epoch_fused, 1))
        et.append(timed(epoch_torch, 1))
    res["epoch"] = {"minibatches": math.ceil(T * E / B), "fused_ms": statistics.median(ef), "fused_ms_rounds": ef,
                    "torch_sync_ms": statistics.median(et), "torch_sync_ms_rounds": et,
                    "speedup_vs_torch": statistics.median(et) / statistics.median(ef)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
