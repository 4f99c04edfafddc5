"""Which emulated entry point every product of the 14-electron UEG workloads takes, and what it
computes: a CCSD sweep with tagged amplitudes, a sweep through sharded row blocks, a dense and a
sector EOM sigma batch, and the V_iabc / V_aibc products of the T1 dressing and of the dressed
ladder.  The sequence of ``pmb_*`` calls and the results (bit for bit: the emulator sums in list
order) are compared with a record (tests/golden/routing_ueg14.json / .npz) so that a change to
how stored integral blocks are recognised or how their momentum lists are built cannot move a
product to another kernel or reorder its sums unnoticed.

``python -m tests.test_kernel_routing`` rewrites the record."""
import json
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
RECORD = os.path.join(HERE, "golden", "routing_ueg14")


class _Patch:
    def setattr(self, obj, name, val):
        setattr(obj, name, val)


def _system():
    from pymes_b200.model import ueg
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    no = 7
    eps = np.asarray(m.kinetic(), dtype=np.float64).copy()
    eps[:no] -= 1.0
    return m, no, m.n_orb - no, [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)], np.diag(eps)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))


def _ccsd(m, no, nv, parts, fock, out):
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd
    dV = m.eval_2b_blocks(no, list(KEYS), parts)
    cc = ccsd.CCSD(no)
    cc.setup(fock, dV)
    out["ccsd_e"] = np.array(cc.sweep())
    out["ccsd_t1"], out["ccsd_t2"] = cc._st["T1"].numpy().copy(), cc._st["T2"].numpy().copy()
    return cc, dV


def _sharded(m, no, nv, parts, fock, out, tmp):
    import torch.distributed as dist
    from pymes_b200 import parallel
    from pymes_b200.integral.partition import KEYS
    dist.init_process_group("gloo", init_method="file://" + os.path.join(tmp, "store"), rank=0, world_size=1)
    try:
        comm = parallel.Comm()
        dV = m.eval_2b_blocks(no, list(KEYS), parts)
        cc = parallel.ShardedCCSD(no, comm)
        cc.setup(fock, parallel.shard_blocks(dV, parallel.Shard(comm, nv)))
        out["sharded_e"] = np.array(cc.sweep())
        out["sharded_t1"], out["sharded_t2"] = cc._st["T1"].numpy().copy(), cc._st["T2"].numpy().copy()
    finally:
        dist.destroy_process_group()


def _sigma(cc, dV, m, no, nv, fock, out):
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    from pymes_b200.solver import eom_ccsd
    T1, T2 = cc._st["T1"], cc._st["T2"]
    ft = cc.get_T1_dressed_fock(_t(fock), T1, dV)
    dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
    rng = np.random.default_rng(21)
    S1, S2 = eom_ccsd.SigmaPlan(no, ft, dVd, T2).apply(_t(rng.standard_normal((2, nv, no))),
                                                        _t(rng.standard_normal((2, nv, nv, no, no))))
    out["dense_s1"], out["dense_s2"] = S1.numpy().copy(), S2.numpy().copy()
    sec = ueg.excitation_sector(m, no, (1, 0, 0))
    lin = sec.lin
    lo, lv = lin[:no], lin[no:]
    m1 = (lv[:, None] - lo[None, :]) == sec.label
    m2 = (lv[:, None, None, None] + lv[None, :, None, None] - lo[None, None, :, None] - lo[None, None, None, :]) \
        == sec.label
    U1 = [_t(np.where(m1, rng.standard_normal(m1.shape), 0.0)) for _ in range(2)]
    U2 = [_t(np.where(m2, rng.standard_normal(m2.shape), 0.0)) for _ in range(2)]
    for a, b in zip(U1, U2):
        assert bk.adopt_momentum(a, sec.singles_rule()) and bk.adopt_momentum(b, sec.doubles_rule())
    plan = eom_ccsd.EOM_CCSD(no, sector=sec).plan(ft, dVd, T2)
    S1, S2 = plan.apply(bk.stack(U1), bk.stack(U2))
    out["sector_s1"], out["sector_s2"] = S1.numpy().copy(), S2.numpy().copy()


def _companions(dV, no, nv, out):
    from pymes_b200.solver import ccsd
    rng = np.random.default_rng(22)
    tau = _t(rng.standard_normal((nv, nv, no, no)))
    W1, W2 = ccsd.pair_with_tau(dV["iabc"], dV["aibc"], tau, no)
    out["pair_w1"], out["pair_w2"] = W1.numpy().copy(), W2.numpy().copy()
    lad = ccsd.DressedLadder(dV["abcd"], dV["iabc"], dV["aibc"], dV["ijab"], _t(rng.standard_normal((nv, no))))
    out["ladder"] = lad.apply(_t(rng.standard_normal((2, nv, nv, no, no))), _t(np.zeros((2, nv, nv, no, no)))).numpy()


def _run(fake, tmp):
    """The workloads on the emulated library ``fake``: ``({workload: [[entry point, repeats], ..]},
    {name: result array})``."""
    calls = []
    for name in [n for n in dir(fake) if n.startswith("pmb_")]:
        fn = getattr(fake, name)
        if callable(fn):
            setattr(fake, name, lambda *a, _n=name, _f=fn: (calls.append(_n), _f(*a))[1])
    m, no, nv, parts, fock = _system()
    seq, out = {}, {}

    def step(label, f, *a):
        del calls[:]
        res = f(*a)
        runs = []
        for n in calls:
            if runs and runs[-1][0] == n:
                runs[-1][1] += 1
            else:
                runs.append([n, 1])
        seq[label] = runs
        return res
    cc, dV = step("ccsd_sweep", _ccsd, m, no, nv, parts, fock, out)
    step("sharded_sweep", _sharded, m, no, nv, parts, fock, out, tmp)
    step("eom_sigma", _sigma, cc, dV, m, no, nv, fock, out)
    step("companions", _companions, dV, no, nv, out)
    return seq, out


def test_routing_and_results_match_the_record(cpu_abi, tmp_path):
    from tests import sector_emulator
    seq, out = _run(sector_emulator.extend(cpu_abi), str(tmp_path))
    with open(RECORD + ".json") as f:
        want = json.load(f)
    for label in want:
        assert seq[label] == want[label], label
    assert set(seq) == set(want)
    ref = np.load(RECORD + ".npz")
    assert set(ref.files) == set(out)
    for k in ref.files:
        assert out[k].shape == ref[k].shape and np.array_equal(out[k].view(np.int64), ref[k].view(np.int64)), k


if __name__ == "__main__":
    import sys
    import tempfile
    sys.path.insert(0, os.path.dirname(HERE))
    from tests import abi_emulator, sector_emulator
    from pymes_b200 import log
    log.set_quiet(True)
    fake = sector_emulator.extend(abi_emulator.install(_Patch()))
    with tempfile.TemporaryDirectory() as tmp:
        seq, out = _run(fake, tmp)
    with open(RECORD + ".json", "w") as f:
        json.dump(seq, f, indent=0)
        f.write("\n")
    np.savez_compressed(RECORD + ".npz", **out)
