"""Diagnostic: cycles per phase of the post kernel and per flush unit (needs a -DPOST_TIMING build: `make timing`, run with
FLEETSTEP_LIB=fleetrl_b200/libfleetstep_timing.so)."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from fleetrl_b200._lib import FleetStepHandle, load_library

sys.argv = [sys.argv[0]]
args = bench.parse_args()
built = bench.build_workload(args)
E, N = args.envs, built.consts.num_evs
dev = torch.device("cuda", 0)
h = FleetStepHandle(built.consts, built.tables, E, device=0)
L = load_library()
D = h.D
obs = torch.empty((E, D), dtype=torch.float32, device=dev); term = torch.empty_like(obs)
rew = torch.empty(E, dtype=torch.float32, device=dev); done = torch.empty(E, dtype=torch.uint8, device=dev)
ring = [torch.empty((E, N), dtype=torch.float32, device=dev).uniform_(-1, 1) for _ in range(8)]
h.reset(obs=obs); torch.cuda.synchronize()
sp = torch.cuda.current_stream(dev).cuda_stream
step = lambda s: h.step_unchecked(ring[s % 8].data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), term.data_ptr(), sp)
Lh = int(built.consts.episode_steps)
phase = torch.arange(E, device=dev) % Lh
for s in range(Lh):
    step(s); h.reset(mask=(phase == s).to(torch.uint8), obs=obs)
for s in range(20):
    step(s)
buf = (C.c_ulonglong * 16)()
L.fleet_debug_post_clk(buf, 1)
K = 50
for s in range(K):
    step(s)
L.fleet_debug_post_clk(buf, 1)
v = np.array(list(buf), dtype=np.float64)
ent, deg = v[11] / K, v[12] / K
names = ["-", "stage rows (wait)", "scan", "micro-ops", "stress drains", "evaluation", "write-back", "slow path", "entry total (deg part)",
         "reset + env4"]
print(f"entries per step {ent:.0f}, with rainflow work {deg:.0f}, micro-op iterations per rainflow warp-pass {v[10] / max(v[12], 1):.1f}")
print(f"reset entries per step {v[13] / K:.0f}: reset work of thread 0 {v[14] / max(v[13], 1):.0f} cycles per reset entry (mark 8 -> after post_reset_env)")
for k in range(1, 10):
    print(f"  {names[k]:28s} {v[k] / max(v[11 if k >= 8 else 12], 1):9.0f} cycles per entry")
print(f"flush units (32 vehicles of flush-only entries per warp) per step {v[15] / K:.0f}: "
      f"{v[0] / max(v[15], 1):.0f} cycles per unit (lane 0 of each warp, fetch to end)")
