"""EOM-CCSD sigma in one total-momentum sector against the dense sigma, on the TC-UEG 54e Hamiltonian
at 389 plane waves with the dressed V_abcd as an operator (the set-up of tools/bench_eom.py), one GPU.

Both modes use ONE compiled sigma program and the SAME vectors: random vectors of the sector
K = (1,0,0), once tagged with the sector rule (every product that involves them runs on momentum
groups) and once as plain copies (the dense products).  Per batch size r = 1, 4, 16 the two modes
alternate in the timed loop (CUDA events, ms per right-hand side).  Then one 10-root sector Davidson
run is timed.  The JSON line records the card (name, power limit, max SM clock, read in the same
run), the flops executed per vector in each mode (launch trace, backend.enable_trace) and the largest
difference between sector and dense sigma.
usage: bench_eom_sector.py [cutoff=13] [ccsd_sweeps=3] [davidson_max_iter=40]"""
import json
import os
import subprocess
import sys
import time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import bench
from pymes_b200 import backend as bk, log as plog
from pymes_b200.model import ueg
from pymes_b200.solver import ccsd, eom_ccsd
from pymes_b200.integral.partition import KEYS

cutoff = float(sys.argv[1]) if len(sys.argv) > 1 else 13.0
sweeps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
dav_iter = int(sys.argv[3]) if len(sys.argv) > 3 else 40
torch.cuda.set_device(0)
plog.set_quiet(True)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                       "-i", "0"], capture_output=True, text=True).stdout.strip()
no = bench.N_ELE // 2
m = ueg.UEG(bench.N_ELE, no, no, bench.RS)
m.init_single_basis(cutoff)
m.k_cutoff, m.gamma = bench.K_CUTOFF, None
nv = m.n_orb - no
fock = bk.asdev(bench.build_fock(m, no))
dV = m.eval_2b_blocks(no, list(KEYS), bench.tc_parts(m), virtual=("abcd",))
cc = ccsd.CCSD(no)
cc.setup(fock, dV)
for _ in range(sweeps):
    e = cc.sweep()
T1, T2 = cc._st["T1"], cc._st["T2"]
ft = cc.get_T1_dressed_fock(fock, T1, dV)
dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
dVd = {k: dVd[k] for k in eom_ccsd.V_KEYS_USED}
del dV, cc
sec = ueg.excitation_sector(m, no, (1, 0, 0))
info = {e_["sector"].label: e_ for e_ in ueg.excitation_sectors(m, no)}[sec.label]
solver = eom_ccsd.EOM_CCSD(no, n_excit=10, sector=sec)
t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
t0.record()
plan = solver.plan(ft, dVd, T2)
t1.record()
torch.cuda.synchronize()
out = {"card": card, "n_orb": m.n_orb, "n_occ": no, "n_virt": nv, "E_ccsd_after_sweeps": sum(e[:3]),
       "virtual_abcd": True, "sector_K": list(sec.K), "sector_label": sec.label,
       "sector_singles": info["n_singles"], "sector_doubles": info["n_doubles"],
       "plan_ms": t0.elapsed_time(t1), "flops_per_vector_dense_plan": plan.flops_per_vector, "batches": []}

lo, lv = sec.lin[:no], sec.lin[no:]
m1 = torch.from_numpy(sec.singles_mask()).cuda()
m2 = torch.from_numpy((lv[:, None, None, None] + lv[None, :, None, None] - lo[None, None, :, None]
                       - lo[None, None, None, :]) == sec.label).cuda()
gen = torch.Generator(device="cuda").manual_seed(0)


def vectors(r):
    """r random sector vectors: tagged stacks (after the check every trial vector gets) and copies."""
    u1 = [torch.where(m1, torch.randn(m1.shape, generator=gen, device="cuda", dtype=torch.float64), 0.0)
          for _ in range(r)]
    u2 = [torch.where(m2, torch.randn(m2.shape, generator=gen, device="cuda", dtype=torch.float64), 0.0)
          for _ in range(r)]
    for a, b in zip(u1, u2):
        assert bk.adopt_momentum(a, sec.singles_rule()) and bk.adopt_momentum(b, sec.doubles_rule())
    S1, S2 = bk.stack(u1), bk.stack(u2)
    del u1, u2
    return (S1, S2), (S1.clone(), S2.clone())


def traced_flops(U):
    bk.enable_trace(True)
    plan.apply(*U)
    tr = bk.trace_report()
    bk.enable_trace(False)
    return float(sum(fl for _lab, fl, _ms in tr)), sum(1 for lab, _f, _m in tr if "momentum-blocked" in lab)


sec_U, dense_U = vectors(1)
out["flops_per_vector_executed_sector"], out["group_launches_sector"] = traced_flops(sec_U)
out["flops_per_vector_executed_dense"], out["group_launches_dense"] = traced_flops(dense_U)
del sec_U, dense_U
max_diff, max_rel = 0.0, 0.0
for r in (1, 4, 16):
    sec_U, dense_U = vectors(r)
    res = {}
    for name, U in (("sector", sec_U), ("dense", dense_U)):           # warm-up of both shapes
        res[name] = plan.apply(*U)
    for a, b in zip(res["sector"], res["dense"]):
        d = float((a - b).abs().max())
        max_diff = max(max_diff, d)
        max_rel = max(max_rel, d / float(b.abs().max()))
    del res
    ms = {"sector": [], "dense": []}
    for _rep in range(3):
        for name, U in (("dense", dense_U), ("sector", sec_U)):
            t0.record()
            plan.apply(*U)
            t1.record()
            torch.cuda.synchronize()
            ms[name].append(t0.elapsed_time(t1))
    row = {"r": r}
    for name in ms:
        best = min(ms[name])
        row[name + "_ms"] = ms[name]
        row[name + "_ms_per_rhs"] = best / r
    row["speedup"] = row["dense_ms_per_rhs"] / row["sector_ms_per_rhs"]
    out["batches"].append(row)
    print("r=%2d  dense %9.2f ms/rhs  sector %9.3f ms/rhs" % (r, row["dense_ms_per_rhs"], row["sector_ms_per_rhs"]),
          file=sys.stderr, flush=True)
    del sec_U, dense_U
out["sector_vs_dense_max_abs_diff"] = max_diff
out["sector_vs_dense_max_rel_diff"] = max_rel

solver.max_iter = dav_iter
torch.cuda.synchronize()
w0 = time.perf_counter()
roots = solver.solve(ft, dVd, T2)
torch.cuda.synchronize()
out["davidson"] = {"n_excit": 10, "seconds": time.perf_counter() - w0, "iterations": solver.iterations,
                   "max_iter": dav_iter, "roots": [float(x) for x in np.sort(roots)]}
print(json.dumps(out))
