"""One FEAST-EOM-CCSD iteration in one total-momentum sector (compact Krylov vectors) against the dense
driver, on the TC-UEG 54e Hamiltonian at 203 plane waves with the dressed V_abcd as an operator (the
set-up of tools/bench_eom_sector.py), one GPU.

Both modes solve the same contour (8 nodes, n_trial = 8, e_c / e_r as below) from the SAME two start
vectors: the reference's seeded dense draws (feast:89-91) restricted to the sector K = (1,0,0), given
as ``u_singles`` / ``u_doubles`` (``n_excit = 0``: nothing else is drawn).  The first iteration holds
2 trial vectors, i.e. 16 shifted systems.  Every solve is one GCROT cycle (``ls_max_iter = 1``: the
first cycle's 40 Krylov steps at most) so that the dense mode's time stays bounded; both modes use it.
The sector mode advances all systems together; the dense mode uses the largest ``max_systems`` whose
Krylov vectors fit the free memory.  The JSON line records the card (name, power limit, max SM clock,
read in the same run), seconds and matvecs per mode, ``torch.cuda.max_memory_allocated`` per mode and
the largest difference between a sector Ritz value and the nearest dense one (all of them, and those
inside the contour).
usage: bench_feast_sector.py [cutoff=13] [ccsd_sweeps=3] [e_c=-0.156] [e_r=0.03]"""
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
from pymes_b200.solver import ccsd, eom_ccsd, feast_eom_ccsd
from pymes_b200.integral.partition import KEYS

cutoff = float(sys.argv[1]) if len(sys.argv) > 1 else 13.0
sweeps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
e_c = float(sys.argv[3]) if len(sys.argv) > 3 else -0.156
e_r = float(sys.argv[4]) if len(sys.argv) > 4 else 0.03
N_NODES, N_TRIAL, SEED = 8, 8, 0
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
idx = sec.packed_index()
n_dense = nv * no + nv * nv * no * no

# the two start vectors: seeded dense draws in the reference's order, restricted to the sector
np.random.seed(SEED)
starts = []
for _ in range(2):
    a = 0.5 - np.random.rand(nv, no)
    b = (0.5 - np.random.rand(nv, nv, no, no)) * 0.01
    u = np.zeros(n_dense)
    u[idx] = np.concatenate([a.ravel(), b.ravel()])[idx]
    starts.append((u[:nv * no].reshape(nv, no), u[nv * no:].reshape(nv, nv, no, no)))
    del a, b, u

out = {"card": card, "n_orb": m.n_orb, "n_occ": no, "n_virt": nv, "E_ccsd_after_sweeps": sum(e[:3]),
       "virtual_abcd": True, "sector_K": list(sec.K), "sector_label": sec.label, "sector_elements": len(idx),
       "dense_elements": n_dense, "n_nodes": N_NODES, "n_trial": N_TRIAL, "e_c": e_c, "e_r": e_r,
       "ls_max_iter": 1, "modes": {}}


def run(mode):
    fe = feast_eom_ccsd.FEAST_EOM_CCSD(no, e_c=e_c, e_r=e_r, n_trial=N_TRIAL, max_iter=1,
                                       sector=sec if mode == "sector" else None)
    fe.n_excit, fe.n_nodes, fe.ls_max_iter = 0, N_NODES, 1
    fe.u_singles = [bk.asdev(s[0]) for s in starts]
    fe.u_doubles = [bk.asdev(s[1]) for s in starts]
    if mode == "dense":
        # Krylov memory per system in the first cycle: 41 basis vectors, the preconditioned and the
        # operator-applied directions, x, r and b -- complex, so two real vectors each
        per_sys = (fe.ls_restart + (fe.ls_recycle or fe.ls_restart) + 1 + 5) * 2 * 8 * n_dense
        free, _total = torch.cuda.mem_get_info()
        staging = 3 * fe.max_rhs * 8 * n_dense
        fe.max_systems = max(1, min(N_NODES * 2, int((0.85 * free - staging) // per_sys)))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    w0 = time.perf_counter()
    ev = fe.solve(ft, dVd, T2)
    torch.cuda.synchronize()
    sec_s = time.perf_counter() - w0
    ev = np.asarray(ev)
    res = {"seconds_per_iteration": sec_s, "matvecs": fe.ls_matvecs, "systems": len(fe.ls_residuals),
           "max_systems": fe.max_systems, "max_rel_residual": float(max(fe.ls_residuals)),
           "max_memory_allocated_GB": torch.cuda.max_memory_allocated() / 1e9,
           "max_rhs": fe.max_rhs, "ritz": [[float(x.real), float(x.imag)] for x in np.sort_complex(ev)]}
    print("%s: %.2f s, %d matvecs, peak %.1f GB" % (mode, sec_s, fe.ls_matvecs, res["max_memory_allocated_GB"]),
          file=sys.stderr, flush=True)
    del fe
    torch.cuda.empty_cache()
    return ev, res


evs = {}
for mode in ("sector", "dense"):
    evs[mode], out["modes"][mode] = run(mode)
# each sector Ritz value against the nearest dense one (a complex pair whose real parts differ in the last
# bit sorts in either order, so sorted lists are not paired)
diff = np.array([np.abs(evs["dense"] - x).min() for x in evs["sector"]])
out["ritz_max_abs_diff"] = float(diff.max())
inside = np.abs(evs["sector"] - e_c) < e_r
out["ritz_inside_contour"] = int(inside.sum())
out["ritz_inside_max_abs_diff"] = float(diff[inside].max()) if inside.any() else None
out["speedup"] = out["modes"]["dense"]["seconds_per_iteration"] / out["modes"]["sector"]["seconds_per_iteration"]
print(json.dumps(out))
