"""The shape-specialised instance of the persistent step kernel.

A fleet of exactly bench.py's cfg2 shape (N = 50, D = 388, header Ha + Hb = 28 + 10, a 16-row history ring, auxiliary
terms, not normalised) steps on an instance of fleet_step_pf_kernel compiled for that shape; every other fleet, and
that one while EvCharger's charge_log is kept, steps on the generic instance.  Which instance a step launched is read
from the kernel name the CUDA profiler records (template argument PfShape<N, D, Ha, Hb, R>, all zero for the generic
instance).  The specialised instance is checked against the oracle, and bit for bit against the generic instance on
the same fleet.
"""
import json
import re

import numpy as np
import pytest
import torch

from fleetrl_b200._abi import FIELDS
from oracle.oracle import OracleFleet
from parity_util import knobs, make_case, run_vs_oracle  # noqa: F401  (knobs: fixture)
from test_gpu_state import FLIP, MIN_TILES_PER_CTA, _capped_envs, _handle, _soh_writes

pytestmark = pytest.mark.gpu

CFG2 = (50, 388, 28, 10, 16)
GENERIC = (0, 0, 0, 0, 0)


def _launched_shape(consts, tables, tmp_path, charge_log=False):
    """PfShape arguments of the step kernel that one step of a fresh two-tile handle of this fleet launches."""
    h = _handle(consts, tables, 2 * (256 // consts.num_evs))
    h.enable_charge_log(charge_log)
    h.reset()
    a = torch.zeros((h.E, h.N), dtype=torch.float32, device=h.device)
    torch.cuda.synchronize(h.device)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        h.step(a)
        torch.cuda.synchronize(h.device)
    assert h.check_errors() == 0
    h.close()
    trace = tmp_path / "trace.json"
    prof.export_chrome_trace(str(trace))
    names = {e.get("name", "") for e in json.loads(trace.read_text())["traceEvents"]}
    names = [n for n in names if "fleet_step_pf_kernel" in n]
    assert len(names) == 1, names
    m = (re.search(r"PfShape<(\d+), (\d+), (\d+), (\d+), (\d+)\s*>", names[0]) or          # demangled
         re.search(r"PfShapeILi(\d+)ELi(\d+)ELi(\d+)ELi(\d+)ELi(\d+)E", names[0]))           # mangled
    assert m, names[0]
    return tuple(int(x) for x in m.groups())


# name: (N, make_case keywords, diagnostic variables, charge_log, instance expected)
SELECT = {
    "cfg2": (50, {}, {}, False, CFG2),
    "cfg2_charge_log": (50, {}, {}, True, GENERIC),
    "n49": (49, {}, {}, False, GENERIC),
    "price_lookahead7_d386": (50, dict(price_lookahead=7), {}, False, GENERIC),
    # same N and D, other header split: Ha = 31, Hb = 7
    "no_building_ha31_hb7": (50, dict(include_building=0, price_lookahead=12), {}, False, GENERIC),
    "ring32": (50, {}, dict(FLEETSTEP_RF_RING=32), False, GENERIC),
    "normalized": (50, dict(normalize=1), {}, False, GENERIC),
}


@pytest.mark.parametrize("name", sorted(SELECT))
def test_instance_selection(name, knobs, tmp_path):
    """The cfg2 shape gets the specialised instance; a fleet one field away from it gets the generic one."""
    N, over, env, charge_log, want = SELECT[name]
    knobs(**env)
    consts, tables = make_case("pf_shape_" + name, N, days=8, over=over)
    assert _launched_shape(consts, tables, tmp_path, charge_log) == want


def test_cfg2_instance_vs_oracle_and_generic(knobs, tmp_path):
    """The specialised instance, every CTA running >= 24 tiles, over two de-phased 96-step episodes and more with
    auto-reset, terminal observations and target-SOC flips of some vehicles (SOH written at and around 0.9, the others
    starting just above it and crossing it at daily evaluations): checked against the oracle after every step, and a
    twin handle of the same fleet on the generic instance (charge_log kept) returns bit-identical outputs and state."""
    consts, tables = make_case("pf_shape_cfg2_flips", 50, days=8, over=dict(init_soh=FLIP + 3e-5))
    assert _launched_shape(consts, tables, tmp_path) == CFG2
    assert _launched_shape(consts, tables, tmp_path, charge_log=True) == GENERIC
    G = 2
    E = _capped_envs(consts, tables, G)
    knobs(FLEETSTEP_PF_GRID=G)
    gpu, twin = _handle(consts, tables, E), _handle(consts, tables, E)
    twin.enable_charge_log(True)
    for h in (gpu, twin):
        g = h.launch_geometry
        assert (h.N, h.D) == CFG2[:2] and g["step_grid"] == G and g["step_tiles"] // G >= MIN_TILES_PER_CTA, g
    N, D, L = gpu.N, gpu.D, consts.episode_steps
    dev = gpu.device
    orc = OracleFleet(consts, tables, E, env_id_offset=1000, threads=8)
    w = _soh_writes(E, N)
    written = ~np.isnan(w)
    t_obs, t_term = torch.zeros((E, D), dtype=torch.float32, device=dev), torch.zeros((E, D), dtype=torch.float32, device=dev)
    t_rew, t_done = torch.zeros(E, dtype=torch.float32, device=dev), torch.zeros(E, dtype=torch.uint8, device=dev)
    fields = [k for k in FIELDS if k != "charge_log"]

    def hook(s, a, obs, rew, done, term):
        if s == -1:
            twin.reset(obs=t_obs)
            assert torch.equal(t_obs, obs), "reset obs"
            soh = np.where(written, w, orc.get("soh"))
            orc.set("soh", soh)
            for h in (gpu, twin):
                h.set("soh", torch.from_numpy(soh))
            return
        twin.step(torch.from_numpy(a).to(dev), t_obs, t_rew, t_done, t_term)
        if s < L:                                     # run_vs_oracle's de-phasing reset, already applied to gpu
            twin.reset(mask=torch.from_numpy((np.arange(E) % L == s).astype(np.uint8)).to(dev), obs=t_obs)
        d = done.bool()
        assert torch.equal(t_done, done) and torch.equal(t_rew, rew) and torch.equal(t_obs, obs), f"outputs step {s}"
        assert torch.equal(t_term[d], term[d]), f"terminal obs step {s}"
        for k in fields:
            assert torch.equal(twin.get(k), gpu.get(k)), f"{k} step {s}"

    r = run_vs_oracle(gpu, orc, 2 * L + 10, charge_log=False, dephase=L, hook=hook)
    flipped = gpu.get("target_soc").cpu().numpy() == FLIP
    assert r["n_done"] > E and r["mixed_tiles"] > 0, r
    assert flipped.any() and not flipped.all() and (flipped & ~written).any(), int(flipped.sum())
    assert twin.check_errors() == 0
    gpu.close()
    twin.close()
