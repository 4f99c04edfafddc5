#!/usr/bin/env python
"""Benchmark of the coupled-cluster amplitude-equation hot path on B200.

    python bench.py --gpus N --steps K --warmup W          (N=1: plain python; N>1: torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (outputs of the last timed step)

One "step" = one CCSD iteration with DIIS (dressing -> singles + doubles residual ->
amplitude update -> DIIS -> energy) on the transcorrelated 3D UEG with 54 electrons in 515
plane waves (BASELINE.json configs[1]: o=27, v=488) at EVERY GPU count ("strong" scaling).
V_abcd of that basis would be 454 GB; it is never materialised: the particle-particle
ladder's producer warps evaluate its tiles from the k-vector / pair tables
(pmb_ueg_operand_t, SURVEY 8(f).1), bit-identical to the stored block.  The o.v^3 and
smaller blocks (4 x 25 GB + 6 x 1.4 GB) are generated on the device once and kept in HBM, row
blocks per rank when N > 1.  `--dense-abcd` stores V_abcd instead (then the basis must shrink:
use --cutoff 18 -> 341 orbitals on one GPU).  Data are synthetic in the sense that nothing is
read from disk; it is the physical TC-UEG Hamiltonian.

Products of a UEG integral block with amplitudes run MOMENTUM-BLOCKED by default (`--ladder
blocked`, SURVEY 8(f).1): as a matrix the block is block diagonal in the (linearised) total
momentum, and pmb_blocked_contract visits the diagonal blocks only -- the particle-particle
ladder 2 o^2 nnz(V_abcd) flop instead of 2 o^2 v^4 (5.2e10 instead of 8.3e13 at 515 plane
waves), likewise V_iabc.tau / V_aibc.tau, I_klij and the three ring intermediates built from
the stored V_ijab; the T1 products of the o.v^3 blocks over one summed index read partner
tables instead of the blocks (pmb_gather_expand); same results to round-off.  Products of
amplitudes with intermediates or T1-dressed blocks stay on the dense DMMA kernel (nothing is
assumed about amplitudes).
`--ladder dense` switches the blocked path off altogether: the dense DMMA ladder with the
operand generated in the producer warps (the round-1 / early round-2 configuration; its
roofline is the pp-ladder one).

Printed line: see the contract in the task statement; `value` is FP64 TFLOP/s computed from
the ALGORITHMIC flop count of the doubles residual AS EXECUTED,
F = F_CCD - sum over the blocked products of (2 M K N - 2 nnz N), with
F_CCD = 2o^2v^4 + 20o^3v^3 + 4o^4v^2 + 4o^2v^3 + 4o^3v^2
(SURVEY 8d; T1-dressing flops are executed but not counted; F = F_CCD with `--ladder dense`;
the per-product counts are printed in config.blocked_products),
divided by the measured time of a whole iteration -- so it can never exceed the FP64 peak.
`dense_equivalent_tflops` = F_CCD / time is what the reference's dense einsum formulation would
have to sustain to finish the iteration in the same time.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ELE, RS, K_CUTOFF = 54, 1.0, 2.0
# plane-wave cutoff (units of (2pi/L)^2 / 2 ... ueg.py:128) -> nP for 54 electrons
CUTOFF_FOR_GPUS = {1: 25.0, 2: 25.0, 4: 25.0, 8: 25.0}        # 515 orbitals (18/20/24 -> 341/389/469)
SM_COUNT, DMMA_FMA_PER_CLK_PER_SM = 148, 64


def flops_ccd(o, v, is_dcd=False):
    o, v = float(o), float(v)
    if is_dcd:
        return 2*o**2*v**4 + 10*o**3*v**3 + 2*o**4*v**2 + 4*o**2*v**3 + 4*o**3*v**2
    return 2*o**2*v**4 + 20*o**3*v**3 + 4*o**4*v**2 + 4*o**2*v**3 + 4*o**3*v**2


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_RESULT_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version
    banner at communicator creation, for one), so file descriptor 1 is pointed at stderr for
    the whole run and the result line is written to the original stdout."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


# ----------------------------------------------------------------------------
# clocks / throttle reasons during the timed region
# ----------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz, self.ok = None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:          # noqa: BLE001
            log("clock sampler unavailable:", e)

    def run(self):
        while self.ok and not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:           # noqa: BLE001
                pass
            time.sleep(0.1)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ----------------------------------------------------------------------------
# CPU arm: the oracle's restatement of the reference, in the reference's einsum modes
# ----------------------------------------------------------------------------
CPU_SAMPLES = ((5.0, 57), (6.0, 65), (7.0, 81), (8.0, 93), (9.0, 123))    # 54e: cutoff -> plane waves
CPU_MIN_SAMPLE = 65              # v = 38 > o = 27: the smallest non-degenerate shape


class CpuProblem:
    """TC-UEG 54e in a small plane-wave basis, built by the oracle on the host (the reference's own
    triple loop restated): the bounded sample of the workload that the CPU legs time."""

    def __init__(self, cutoff):
        import numpy as np
        from oracle import cc_oracle as oc, ueg_oracle as uo
        self.no = N_ELE // 2
        m = uo.UEG(N_ELE, RS).init_single_basis(cutoff)
        m.k_cutoff, m.gamma = K_CUTOFF, None
        self.cutoff, self.n_orb = cutoff, m.n_orb
        self.fock, self.V = m.tc_hamiltonian(self.no)
        self.dV = oc.partition(self.no, self.V)
        self.eps_i = self.fock.diagonal()[:self.no].copy()
        self.eps_a = self.fock.diagonal()[self.no:].copy()
        self.np, self.oc = np, oc

    def run(self, sweeps, timed_from=0):
        """`sweeps` CCSD+DIIS sweeps from the MP2 start in the reference's einsum modes (ccd.py
        rows bare np.einsum, ccsd.py rows optimize=True); returns (seconds per sweep over the
        sweeps >= timed_from, energy, T1, T2)."""
        oc, np = self.oc, self.np
        oc.set_ccd_einsum_mode("as_written")
        try:
            _, T2 = oc.mp2(self.eps_i, self.eps_a, self.dV["ijab"], self.dV["abij"])
            T1 = np.zeros((self.n_orb - self.no, self.no))
            d1, d2 = oc.denominators(self.eps_i, self.eps_a)
            mixer = oc.DIIS(6)
            e, t0 = (0.0, 0.0, 0.0), None
            for k in range(sweeps):
                if k == timed_from:
                    t0 = time.perf_counter()
                T1, T2, e, _dt = oc.ccsd_sweep(self.no, self.fock, self.dV, T1, T2, d1, d2, mixer)
            dt = (time.perf_counter() - t0) / max(sweeps - timed_from, 1) if t0 is not None else None
        finally:
            oc.set_ccd_einsum_mode("optimized")
        return dt, float(sum(e)), T1, T2


def pick_cpu_sample(n_sweeps, budget_s):
    """Largest sample basis whose `n_sweeps` sweeps fit `budget_s`, from a MEASURED rate: one
    sweep of the 57-plane-wave problem is timed first and scaled by algorithmic flops."""
    no = N_ELE // 2
    probe = CpuProblem(CPU_SAMPLES[0][0])
    t_probe, _, _, _ = probe.run(1)
    rate = flops_ccd(no, probe.n_orb - no) / t_probe            # flop/s of this host on this code
    pick = None
    for cutoff, nP in CPU_SAMPLES:
        if nP < CPU_MIN_SAMPLE:
            continue
        if pick is None or flops_ccd(no, nP - no) / rate * n_sweeps <= budget_s:
            pick = (cutoff, nP)
    return pick, rate, t_probe


def cpu_sample(steps, warmup, budget_s=150.0, cutoff=None, keep_problem=False):
    """Time `steps` CCSD sweeps (after `warmup`) of the reference algorithm (oracle port) on a
    bounded sample of the workload: the same TC-UEG 54e Hamiltonian in a smaller basis."""
    import numpy as np
    cores = len(os.sched_getaffinity(0))
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    no = N_ELE // 2
    rate = t_probe = None
    if cutoff is None:
        (cutoff, _nP), rate, t_probe = pick_cpu_sample(steps + warmup, budget_s)
    prob = CpuProblem(cutoff)
    nP = prob.n_orb
    dt, e, T1, T2 = prob.run(steps + warmup, timed_from=warmup)
    oc = prob.oc
    # the two pieces SURVEY 8(d) asks for beside the whole iteration: CCD.get_residual alone and the
    # single particle-particle ladder einsum, both as ccd.py writes them (bare np.einsum)
    oc.set_ccd_einsum_mode("as_written")
    dV = prob.dV
    t0 = time.perf_counter()
    oc.doubles_residual(no, prob.fock, T2, dV["klij"], dV["ijab"], dV["abij"], dV["iajb"], dV["iabj"], dV["abcd"])
    t_res = time.perf_counter() - t0
    t0 = time.perf_counter()
    np.einsum("abcd,cdij->abij", dV["abcd"], T2)
    t_pp = time.perf_counter() - t0
    oc.set_ccd_einsum_mode("optimized")
    F = flops_ccd(no, nP - no)
    out = {"value": F / dt / 1e12, "unit": "TFLOP/s", "cores": cores, "kind": "port",
           "sample": "TC-UEG 54e rs=%.1f, %d plane waves (o=27, v=%d): %d CCSD+DIIS sweeps (after %d untimed) of "
                     "the numpy oracle in the reference's einsum modes (ccd.py rows single-threaded c_einsum, "
                     "ccsd.py rows optimize=True/BLAS), %.2f s per sweep" % (RS, nP, nP - no, steps, warmup, dt),
           "seconds_per_step": dt, "n_orb": nP, "n_virt": nP - no, "cutoff": cutoff, "sweeps_total": steps + warmup,
           "energy": e, "flops_per_step": F,
           "doubles_residual_seconds": t_res,
           "pp_ladder_einsum_seconds": t_pp,
           "pp_ladder_einsum_gflops": 2.0 * no ** 2 * float(nP - no) ** 4 / t_pp / 1e9}
    if keep_problem:
        out["_problem"] = prob
    if rate is not None:
        out["sizing"] = "sample chosen from a measured rate: one 57-plane-wave sweep took %.2f s = %.2f GF/s" \
                        % (t_probe, rate / 1e9)
    return out


def run_reference(args):
    """`--impl reference`: the reference's algorithm on the host cores (oracle port), on a bounded
    sample of the workload.  The line's `config` describes WHAT WAS TIMED (n_orb, n_virt of the
    sample) and names the workload it samples; `value` is the FP64 rate of that sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, min(args.warmup, 1)
    base = cpu_sample(steps, warmup, budget_s=150.0)
    no = N_ELE // 2
    nP = base["n_orb"]
    line = {"impl": "reference", "metric": "ccsd_iteration_fp64_tflops", "value": base["value"],
            "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": base["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "TC-UEG 54e rs=%.1f CCSD+DIIS iteration, plane-wave cutoff %g: BOUNDED SAMPLE of the "
                                   "cutoff-%g workload (the reference cannot hold that V: 563 GB)"
                                   % (RS, base["cutoff"], CUTOFF_FOR_GPUS[args.gpus]),
                       "method": "CCSD", "correlator": "trunc k_c=%g" % K_CUTOFF, "n_occ": no, "n_orb": nP,
                       "n_virt": nP - no, "flops_per_step": base["flops_per_step"], "energy": base["energy"],
                       "same_config_as_gpu_arm": False,
                       "note": "the GPU arm times this same %d-orbital problem in its `same_config` field; "
                               "that ratio is measured, the one against the 515-orbital line is a rate ratio" % nP},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "TFLOP/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def synthetic_config(n_gpus, no, nv):
    return {"workload": "synthetic non-hermitian FCIDUMP-like integrals (BASELINE configs[2]): o=%d, v=%d, "
                        "V = eps*N(0,1) with only the (pq)(rs)<->(qp)(sr) symmetry, CCSD+DIIS iteration" % (no, nv),
            "method": "CCSD", "n_occ": no, "n_virt": nv, "n_orb": no + nv,
            "V_abcd": "dense, STORED in HBM as (ab) row blocks (%.1f GB per GPU), streamed by the ladder kernel"
                      % (8.0 * ((nv + n_gpus - 1) // n_gpus) * nv ** 3 / 1e9),
            "generator": "pmb_synth_block: counter-based, each rank writes its own rows on the device",
            "l2_policy": "inputs_exceed_l2 (every operand >> 126 MB L2)",
            "parallelism": "ab-block x%d" % n_gpus}


def workload_config(n_gpus, no, cutoff=None, dense_abcd=False, blocked=False):
    cutoff = cutoff or CUTOFF_FOR_GPUS[n_gpus]
    return {"workload": "TC-UEG 54e rs=%.1f CCSD+DIIS iteration, plane-wave cutoff %g" % (RS, cutoff),
            "method": "CCSD", "correlator": "trunc k_c=%g" % K_CUTOFF, "n_occ": no,
            "V_abcd": "stored in HBM" if dense_abcd else
                      ("never materialised: compressed values (one candidate non-zero per dense row), pp ladder "
                       "on the diagonal momentum blocks only (pmb_blocked_contract)" if blocked else
                       "never materialised (generated in the ladder kernel)"),
            "l2_policy": "inputs_exceed_l2 (every T2-sized operand and o.v^3 block >> 126 MB L2)",
            "parallelism": "ab-block x%d" % n_gpus}


# ----------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------
def tc_parts(m):
    return [("only_2b", m.trunc), ("effect_2b", m.trunc)]


def build_fock(m, no):
    """Host Fock matrix of the TC-UEG Hamiltonian, assembled as in
    pymes/test/test_ueg/test_symmetrised_2body_integral.py:84-160: f = h + 2 V_piqi - V_piiq
    (hf.py:14-18) from the pure two-body part, plus the doubly-contracted 3-body one-body shifts."""
    import numpy as np
    nP = m.n_orb
    W0, W1 = m.pair_tables("only_2b", m.trunc)
    Vd = m.build_block((0, 0, 0, 0), (nP, no, nP, no), W0a=W0, W1a=W1).cpu().numpy()
    Vx = m.build_block((0, 0, 0, 0), (nP, no, no, nP), W0a=W0, W1a=W1).cpu().numpy()
    fock = np.diag(m.kinetic()).astype(np.float64)
    fock += 2.0 * np.einsum("piqi->pq", Vd)
    fock -= np.einsum("piiq->pq", Vx)
    fock += np.diag(m.double_contractions_in_3_body())
    return fock


def calibrate(torch):
    """The two roofline denominators MEASURED_PEAKS.json lacks or that should be re-measured on
    THIS box, with the driver's own recipe (torch library calls, CUDA events, best of 10):
    cuBLAS DGEMM 8192^3 (burst) and a device-to-device copy of 2 GiB (read + write bytes)."""
    out = {}
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    c = torch.empty(n, n, dtype=torch.float64, device="cuda")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.matmul(a, b, out=c)
    best = 1e30
    for _ in range(10):
        ev0.record()
        torch.matmul(a, b, out=c)
        ev1.record()
        torch.cuda.synchronize()
        best = min(best, ev0.elapsed_time(ev1))
    out["dgemm_tflops"] = 2.0 * n ** 3 / (best * 1e-3) / 1e12
    del a, b, c
    x = torch.empty(1 << 28, dtype=torch.float64, device="cuda")      # 2 GiB
    y = torch.empty_like(x)
    x.fill_(1.0)
    y.copy_(x)
    best = 1e30
    for _ in range(10):
        ev0.record()
        y.copy_(x)
        ev1.record()
        torch.cuda.synchronize()
        best = min(best, ev0.elapsed_time(ev1))
    out["d2d_copy_gbs"] = 2.0 * x.numel() * 8 / (best * 1e-3) / 1e9
    out["how"] = "torch.matmul f64 8192^3 and tensor.copy_ over 2 GiB, best of 10, CUDA events, this run"
    del x, y
    torch.cuda.empty_cache()
    return out


def dense_ladder_probe(bk, torch, V_abcd, T2, peak, dgemm=None):
    """One launch of the DENSE particle-particle ladder V_abcd.tau on the FP64 tensor cores (operand
    generated in the producer warps, this rank's rows), timed with CUDA events after one warm-up launch:
    the north_star's pp-ladder roofline target, measured in the same run as the default (momentum-
    blocked) iteration.  Outside the timed region; never part of `value`."""
    old = bk.set_blocked(False)
    try:
        nv, no = int(T2.shape[0]), int(T2.shape[2])
        rows = int(V_abcd.shape[0])
        tau = bk.axpby(1.0, T2, 0.0, bk.empty_even_pitch(nv, nv, no))
        R = bk.zeros(rows, nv, no, no)
        term = [(1.0, "abcd", V_abcd, "cdij", tau)]
        bk.contract_terms("abij", term, out=R, beta=1.0)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record(torch.cuda.current_stream())
        bk.contract_terms("abij", term, out=R, beta=1.0)
        ev1.record(torch.cuda.current_stream())
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        flops = 2.0 * rows * float(nv) ** 3 * no * no
        out = {"kernel": "contract_ws_kernel (dense pp ladder V_abcd.tau, DMMA.8x8x4; V_abcd tiles generated by the "
                         "producer warps): one launch after one warm-up, outside the timed region",
               "ms_per_launch": ms, "flops_per_launch": flops, "achieved": flops / (ms * 1e-3) / 1e12,
               "unit": "TFLOP/s", "peak": peak}
        out["frac"] = out["achieved"] / peak
        if dgemm:
            out["frac_of_measured_dgemm"] = out["achieved"] / dgemm
        return out
    finally:
        bk.set_blocked(old)


DUMP_T2_SAMPLES = 1 << 21          # 16 MiB of T2 values and 16 MiB of their positions


def dump_outputs(path, e, T1, T2):
    """Write what the last timed sweep hands a caller of CCSD.sweep as float64 .npy files under
    `path`: energy (e_1b, e_dir, e_ex), norms (|T2|, |dT2|), t1 [v, o], and T2 [v, v, o, o] at a
    fixed, seeded sample of flat positions (t2_sample, positions in t2_sample_index; every position
    when T2 is smaller than the sample), so that two builds can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    n = T2.numel()
    pick = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_T2_SAMPLES), replace=False))
    idx = torch.from_numpy(pick).to(T2.device)
    out = {"energy": e[:3], "norms": e[3:5], "t1": T1.cpu().numpy(),
           "t2_sample": T2[torch.unravel_index(idx, tuple(T2.shape))].cpu().numpy(), "t2_sample_index": pick}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def same_config_leg(cpu, steps_total, torch):
    """The problem the CPU leg timed (TC-UEG 54e in `cpu['n_orb']` plane waves), through the public
    API with HOST buffers on this GPU: numpy Fock / V_pqrs in, `steps_total` CCSD+DIIS sweeps with the
    amplitudes crossing pinned host memory every sweep (`CCSD.sweep_host`).  Same start (MP2), same
    number of sweeps as the CPU leg, so the energies are directly comparable."""
    from pymes_b200.solver import ccsd
    prob = cpu.pop("_problem", None) or CpuProblem(cpu["cutoff"])    # oracle-built host arrays: shared inputs
    no, nP = prob.no, prob.n_orb
    nv = nP - no
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    cc = ccsd.CCSD(no)
    cc.setup(prob.fock, prob.V)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    t1h = torch.zeros((nv, no), dtype=torch.float64).pin_memory()
    t2h = torch.empty((nv, nv, no, no), dtype=torch.float64).pin_memory()
    t1h.copy_(cc._st["T1"])
    t2h.copy_(cc._st["T2"])
    times = []
    e = None
    for _ in range(steps_total):
        t0 = time.perf_counter()
        e = cc.sweep_host(t1h, t2h)
        times.append(time.perf_counter() - t0)
    e_gpu = e[0] + e[1] + e[2]
    n_timed = max(1, steps_total - 1)
    gpu_s = sum(times[-n_timed:]) / n_timed                # first sweep carries one-time allocations
    return {"n_orb": nP, "n_virt": nv, "n_occ": no, "sweeps": steps_total,
            "gpu_seconds_per_step": gpu_s, "gpu_setup_seconds_incl_h2d_of_V": t_setup,
            "cpu_seconds_per_step": cpu["seconds_per_step"], "cpu_cores": cpu["cores"],
            "speedup_measured": cpu["seconds_per_step"] / gpu_s,
            "energy_gpu": e_gpu, "energy_cpu": cpu["energy"], "abs_energy_diff": abs(e_gpu - cpu["energy"]),
            "h2d_bytes_per_step": (t1h.numel() + t2h.numel()) * 8, "d2h_bytes_per_step": (t1h.numel() + t2h.numel()) * 8 + 64,
            "what": "same inputs, same start, same sweep count on both sides; GPU side through CCSD.sweep_host "
                    "with host buffers (launch-latency bound at this size: ~170 kernels per sweep)"}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from pymes_b200 import backend as bk, log as plog
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    plog.set_quiet(True)
    blocked = args.ladder == "blocked" and args.workload == "ueg" and not args.dense_abcd
    bk.set_blocked(blocked)
    no = N_ELE // 2
    cutoff = args.cutoff if args.cutoff else CUTOFF_FOR_GPUS[args.gpus]
    cal = calibrate(torch) if (rank == 0 and not args.no_calibration) else None
    if world > 1:
        dist.barrier()

    t0 = time.time()
    synthetic_wl = args.workload == "synthetic"
    if synthetic_wl:
        # BASELINE configs[2]: V_abcd is genuinely dense here -- stored as row blocks, streamed from HBM
        from pymes_b200 import parallel
        from pymes_b200.integral.partition import KEYS
        from pymes_b200.util import synthetic
        no, nv = args.occ, args.virt
        nP = no + nv
        args.dense_abcd = True
        fock = synthetic.tc_fock(no, nv, seed=0)
        if world > 1:
            comm = parallel.Comm(dist.group.WORLD)
            shard = parallel.Shard(comm, nv)
            ranges = {k: {d: (no + shard.lo, shard.na)} for k, d in parallel.SHARD_DIMS.items()}
            cc = parallel.ShardedCCSD(no, comm, is_dcsd=args.dcsd)
        else:
            ranges = None
            cc = ccsd.CCSD(no, is_dcsd=args.dcsd)
        dV = synthetic.tc_blocks(no, nv, list(KEYS), seed=0, ranges=ranges, device=True)
    else:
        m = ueg.UEG(N_ELE, no, no, RS)
        m.init_single_basis(cutoff)
        m.k_cutoff, m.gamma = K_CUTOFF, None
        nP, nv = m.n_orb, m.n_orb - no
        virtual = () if args.dense_abcd else ("abcd",)
        fock = build_fock(m, no)
        if world > 1:
            from pymes_b200 import parallel
            comm = parallel.Comm(dist.group.WORLD)
            cc = parallel.ShardedCCSD(no, comm, is_dcsd=args.dcsd)
            dV = parallel.build_sharded_hamiltonian(m, no, comm, tc_parts(m), virtual=virtual)
        else:
            from pymes_b200.integral.partition import KEYS
            cc = ccsd.CCSD(no, is_dcsd=args.dcsd)
            dV = m.eval_2b_blocks(no, list(KEYS), tc_parts(m), virtual=virtual)
    torch.cuda.synchronize()
    t_build = time.time() - t0
    if rank == 0:
        log("%s: nP=%d (o=%d, v=%d), integrals built in %.1f s, %.1f GB allocated"
            % ("synthetic" if synthetic_wl else "TC-UEG 54e", nP, no, nv, t_build, torch.cuda.memory_allocated() / 1e9))
    e_mp2 = cc.setup(fock, dV)
    if rank == 0:
        log("E_MP2 = %.10f" % e_mp2)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for w in range(args.warmup):
        e = cc.sweep()
        if rank == 0:
            log("warmup %d: E = %.10f" % (w, e[0] + e[1] + e[2]))

    sampler = ClockSampler(local)
    bk.enable_timing(True)
    if blocked:
        bk.enable_trace(True)          # an event pair around every contraction launch (no synchronisation)
    launches0 = bk.launch_count()
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()        # `ncu --profile-from-start off` sees the timed steps only
    ev0.record()
    for k in range(args.steps):
        e = cc.sweep()
    ev1.record()
    torch.cuda.profiler.stop()
    barrier()
    clocks = sampler.result()
    launches = bk.launch_count() - launches0
    ms = ev0.elapsed_time(ev1) / args.steps
    regions = bk.timing_report()
    trace = bk.trace_report() if blocked else []
    bk.enable_trace(False)
    bk.enable_timing(False)
    e_final = e[0] + e[1] + e[2]
    if args.dump_outputs and rank == 0:     # before the end-to-end sweeps below move the amplitudes on
        dump_outputs(args.dump_outputs, e, cc._st["T1"], cc._st["T2"])
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    F_dense = flops_ccd(no, nv, is_dcd=args.dcsd)
    F = F_dense
    blocked_products = {}
    if blocked:
        # flops as executed: the products of F_CCD that ran momentum-blocked (known from the labels
        # of rank 0's launches) count 2 nnz N instead of 2 M K N; nnz from the WHOLE problem's groups
        ran = {lab.split(" [")[0] for lab, _f, _t in trace if "[momentum-blocked]" in lab}
        O, Vr = (0, no), (no, nv)                     # (lo, extent) of an occupied / virtual axis
        alg = {"abcd,cdij->abij": ((Vr, Vr, Vr, Vr), (0, 1), (2, 3), no * no),        # pp ladder  ccd.py:187
               "klcd,cdij->klij": ((O, O, Vr, Vr), (0, 1), (2, 3), no * no),          # I_klij     ccd.py:180
               "klcd,dblj->cbkj": ((O, O, Vr, Vr), (0, 2), (1, 3), nv * no),          # Xai        ccd.py:202
               "klcd,adkj->alcj": ((O, O, Vr, Vr), (1, 2), (0, 3), nv * no),          # X1         ccd.py:189
               "klcd,daki->alci": ((O, O, Vr, Vr), (1, 2), (0, 3), nv * no)}          # Xp         ccd.py:238
        for lab, (axes, m_ax, k_ax, ncol) in alg.items():
            if lab not in ran:
                continue
            lo4, ext4 = tuple(a[0] for a in axes), tuple(a[1] for a in axes)
            _ro, _eo, _g0, g_rows, _e0, g_ents = ueg.momentum_groups(m.k_int(), m.imax, lo4, ext4, m_ax, k_ax)
            nnz = float((g_rows * g_ents).sum())
            dense = 2.0 * ext4[0] * ext4[1] * ext4[2] * ext4[3] * ncol
            blocked_products[lab] = {"dense_flops": dense, "executed_flops": 2.0 * nnz * ncol, "nnz": nnz}
            F -= dense - 2.0 * nnz * ncol
    value = F / (ms * 1e-3) / 1e12

    rows = getattr(cc, "local_rows", nv) if world > 1 else nv
    peak = SM_COUNT * DMMA_FMA_PER_CLK_PER_SM * 2 * (clocks.get("sm_max_mhz") or 1965) * 1e6 / 1e12
    pp_ms = regions.get("pp_ladder", [])
    pp_avg = sum(pp_ms) / len(pp_ms) if pp_ms else None
    if blocked:
        # dominant kernel now: contract_ws_kernel on the nine ring-type o^3v^3 contractions of
        # ccd.py:189-204,233-240 (seven launches, one of them three terms wide), this rank's rows
        ring_unit = 2.0 * rows * nv * nv * float(no) ** 3
        ring = [(fl, t) for lab, fl, t in trace
                if "[momentum-blocked]" not in lab and "[gemv]" not in lab and fl >= 0.99 * ring_unit]
        ring_flops, ring_ms = sum(fl for fl, _ in ring), sum(t for _, t in ring)
        n_ring = len(ring)
        roof = {"bound": "tensor",
                "kernel": "contract_ws_kernel (ring-type contractions 2 o^3 v^3 of the doubles residual, DMMA.8x8x4; "
                          "per launch = average over the %d launches of one iteration, the three-term launch "
                          "counting its three products)" % (n_ring // max(args.steps, 1)),
                "achieved": (ring_flops / (ring_ms * 1e-3) / 1e12) if ring_ms else None,
                "peak": peak, "unit": "TFLOP/s",
                "peak_source": "FP64 tensor (DMMA) issue peak: 148 SM x 64 FMA/clk x 2 x sm_max_mhz; "
                               "MEASURED_PEAKS.json has no FP64 entry (its bf16 figure does not apply)",
                "traffic": None, "launches_timed": n_ring, "ms_per_launch": ring_ms / n_ring if n_ring else None,
                "flops_per_launch": ring_flops / n_ring if n_ring else None,
                "share_of_step": ring_ms / (ms * args.steps) if ring_ms else None}
        bl = [(fl, t) for lab, fl, t in trace if lab.endswith("abcd,cdij->abij [momentum-blocked]")]
        if bl:
            roof["pp_ladder_blocked"] = {
                "kernel": "blocked_kernel (pmb_blocked_contract: V_abcd.tau on the diagonal momentum blocks)",
                "ms_per_launch": sum(t for _, t in bl) / len(bl), "flops_per_launch_executed": bl[0][0],
                "tflops_executed": sum(fl for fl, _ in bl) / (sum(t for _, t in bl) * 1e-3) / 1e12,
                "dense_flops_replaced": 2.0 * rows * float(nv) ** 3 * no * no, "launches_timed": len(bl)}
    else:
        # dominant kernel: the particle-particle ladder contraction (this rank's row block)
        pp_flops = 2.0 * rows * nv * nv * nv * no * no
        roof = {"bound": "tensor",
                "kernel": "contract_ws_kernel (pp ladder V_abcd.tau, DMMA.8x8x4%s)"
                          % ("" if args.dense_abcd else "; V_abcd tiles generated by the producer warps"),
                "achieved": (pp_flops / (pp_avg * 1e-3) / 1e12) if pp_avg else None,
                "peak": peak, "unit": "TFLOP/s",
                "peak_source": "FP64 tensor (DMMA) issue peak: 148 SM x 64 FMA/clk x 2 x sm_max_mhz; "
                               "MEASURED_PEAKS.json has no FP64 entry (its bf16 figure does not apply)",
                "traffic": None, "launches_timed": len(pp_ms), "ms_per_launch": pp_avg,
                "flops_per_launch": pp_flops}
    roof["frac"] = roof["achieved"] / peak if roof["achieved"] else None
    if cal is not None:                 # second denominator: a library DGEMM measured in THIS run
        roof["peak_measured_dgemm"] = cal["dgemm_tflops"]
        roof["frac_of_measured_dgemm"] = roof["achieved"] / cal["dgemm_tflops"] if roof["achieved"] else None
        roof["hbm_copy_gbs_measured"] = cal["d2d_copy_gbs"]
        roof["calibration"] = cal["how"]
    if clocks.get("sm_mhz"):
        roof["frac_at_observed_clock"] = (roof["achieved"] / (peak * clocks["sm_mhz"] / (clocks["sm_max_mhz"] or 1965))
                                          if roof["achieved"] else None)
    prof = os.path.join(ROOT, "profiles", "pp_ladder_traffic.json" if args.dense_abcd
                        else "pp_ladder_virtual_traffic.json")
    if blocked:
        prof = os.path.join(ROOT, "profiles", "r2_ring_traffic.json")
    if os.path.exists(prof) and world == 1:
        try:                            # ncu capture of the same launch (same v, whole row range)
            rec = json.load(open(prof))
            if rec.get("n_virt", nv) == nv:
                roof["traffic"] = rec.get("dram_bytes_per_launch")
                if blocked and rec.get("flops_per_launch") and roof.get("flops_per_launch"):
                    # the capture is ONE product (2 o^3 v^3); the average launch here is 1.5 products
                    roof["traffic"] *= roof["flops_per_launch"] / rec["flops_per_launch"]
                roof["traffic_source"] = os.path.relpath(prof, ROOT)
        except Exception:               # noqa: BLE001
            pass

    # end to end: amplitudes in pinned host memory every step, new amplitudes + energies back
    t1h = torch.empty((nv, no), dtype=torch.float64).pin_memory()
    t2_rows = cc.shard.rows(cc._st["T2"], 0) if world > 1 else cc._st["T2"]     # this rank's row block
    t2h = torch.empty(tuple(t2_rows.shape), dtype=torch.float64).pin_memory()
    t1h.copy_(cc._st["T1"])
    t2h.copy_(t2_rows)
    cc.sweep_host(t1h, t2h)
    barrier()
    tw = time.perf_counter()
    for k in range(args.steps):
        cc.sweep_host(t1h, t2h)
    barrier()
    e2e_ms = (time.perf_counter() - tw) / args.steps * 1e3
    if world > 1:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    io_bytes = (t1h.numel() + t2h.numel()) * 8
    e2e = {"value": F / (e2e_ms * 1e-3) / 1e12, "unit": "TFLOP/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": io_bytes, "d2h_bytes_per_step": io_bytes + 8 * 8,
           "api": "CCSD.sweep_host(T1, T2): amplitudes from pinned host memory in (each rank its T2 row "
                  "block), one iteration, amplitudes and energies back; the static operator (Fock, V "
                  "blocks) stays in HBM; bytes are per rank"}

    if blocked and not args.no_dense_ladder:
        # the dense DMMA ladder next to the blocked one, same run (every rank its rows; no collective)
        try:
            roof["pp_ladder_dense"] = dense_ladder_probe(bk, torch, dV["abcd"], cc._st["T2"], peak,
                                                         cal["dgemm_tflops"] if cal is not None else None)
        except Exception as exc:        # noqa: BLE001 -- a diagnostic must not cost the bench line
            roof["pp_ladder_dense"] = {"error": repr(exc)}
        barrier()

    line = {"metric": "ccsd_iteration_fp64_tflops", "value": value, "unit": "TFLOP/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(synthetic_config(args.gpus, no, nv) if synthetic_wl
                           else workload_config(args.gpus, no, cutoff, args.dense_abcd, blocked), n_orb=nP, n_virt=nv,
                           **({"method": "DCSD"} if args.dcsd else {}),
                           flops_per_step=F, energy=e_final, build_seconds=t_build),
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof}
    if blocked:
        line["config"]["flop_convention"] = (
            "flops_per_step = doubles-residual flops AS EXECUTED: SURVEY 8(d) F_CCD = %.4e, with every product "
            "that ran momentum-blocked (blocked_products: integral block x amplitudes, on the diagonal momentum "
            "blocks only) counted as 2 nnz N instead of 2 M K N" % F_dense)
        line["config"]["blocked_products"] = blocked_products
        line["config"]["flops_per_step_dense_convention"] = F_dense
        line["dense_equivalent_tflops"] = F_dense / (ms * 1e-3) / 1e12
        line["e2e"]["dense_equivalent_tflops"] = F_dense / (e2e_ms * 1e-3) / 1e12
    if rank == 0:
        if args.gpus == 1 and not args.no_cpu and not synthetic_wl:
            cores = len(os.sched_getaffinity(0))
            log("timing the CPU oracle on %d host cores ..." % cores)
            line["cpu_baseline"] = cpu_sample(2, 1, budget_s=60.0, keep_problem=True)
            # the reference cannot hold this workload's V (563 GB): its time here is EXTRAPOLATED by
            # algorithmic flops from the sample that did run (SURVEY 8d), not measured
            line["cpu_baseline"]["extrapolated_seconds_per_step_at_workload"] = \
                F_dense / (line["cpu_baseline"]["value"] * 1e12)
            # ... and the MEASURED same-config ratio: the GPU runs the sample problem itself
            del cc, dV
            torch.cuda.empty_cache()
            line["same_config"] = same_config_leg(line["cpu_baseline"], line["cpu_baseline"]["sweeps_total"], torch)
        else:
            line["cpu_baseline"] = None
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cutoff", type=float, default=0.0, help="override the plane-wave cutoff (debug)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and same_config legs")
    ap.add_argument("--no-calibration", action="store_true", help="skip the in-run DGEMM / D2D-copy calibration")
    ap.add_argument("--dcsd", action="store_true",
                    help="time a DCSD iteration (the other method of BASELINE configs[1]) instead of CCSD")
    ap.add_argument("--workload", default="ueg", choices=["ueg", "synthetic"],
                    help="ueg: TC-UEG 54e (BASELINE configs[1], the headline); synthetic: configs[2], o=50 v=500 "
                         "random non-hermitian integrals with a STORED dense V_abcd (fits 8 GPUs)")
    ap.add_argument("--occ", type=int, default=50, help="synthetic workload: occupied orbitals")
    ap.add_argument("--virt", type=int, default=500, help="synthetic workload: virtual orbitals")
    ap.add_argument("--ladder", default="blocked", choices=["blocked", "dense"],
                    help="blocked: V_abcd.tau (and V_iabc.tau, V_aibc.tau) on the diagonal momentum blocks only "
                         "(pmb_blocked_contract); dense: the dense DMMA ladder with the generated operand")
    ap.add_argument("--no-dense-ladder", action="store_true",
                    help="skip the one extra launch of the dense DMMA ladder (roofline.pp_ladder_dense) after the "
                         "timed region of a --ladder blocked run")
    ap.add_argument("--dense-abcd", action="store_true",
                    help="store V_abcd in HBM instead of generating it in the ladder kernel")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the energies, T1 and a seeded sample of T2 of the last "
                         "timed step to DIR/<name>.npy (float64, about 32 MiB)")
    args = ap.parse_args()
    claim_stdout()
    if args.gpus not in CUTOFF_FOR_GPUS:
        raise SystemExit("--gpus must be one of %s" % sorted(CUTOFF_FOR_GPUS))
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        raise SystemExit("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
