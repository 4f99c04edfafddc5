"""Momentum rules of amplitudes and intermediates (backend.Momentum) and the block-diagonal x
block-diagonal contraction pmb_group_contract: derivation rules, verification at the boundary,
routing of the ring products, and results against the dense path and numpy."""
import os

import numpy as np
import pytest
import torch

TOL = dict(rtol=0, atol=1e-12)


@pytest.fixture
def abi(cpu_abi):
    """The emulated C ABI with the two entry points of this change (tests/momentum_emulator.py)."""
    from tests import momentum_emulator
    return momentum_emulator.extend(cpu_abi)


def _n(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))


def _ueg14():
    from pymes_b200.model import ueg
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    return m, 7, m.n_orb - 7, [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)]


def _fock(m, no):
    """A diagonal (momentum-conserving) Fock matrix with a gap between occupied and virtual levels."""
    eps = np.asarray(m.kinetic(), dtype=np.float64).copy()
    eps[:no] -= 1.0
    return np.diag(eps)


def _count(lib, name):
    calls = {"n": 0}
    orig = getattr(lib, name)

    def wrapped(*a):
        calls["n"] += 1
        return orig(*a)
    setattr(lib, name, wrapped)
    return calls


def test_group_descriptor_matches_the_c_header(tmp_path):
    import ctypes as C
    import shutil
    import subprocess
    from pymes_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "pymes_b200.h"', "int main(void) {",
             'printf("size %zu\\n", sizeof(pmb_group_t));']
    lines += ['printf("%s %%zu\\n", offsetof(pmb_group_t, %s));' % (f, f) for f, _ in _lib.Group._fields_]
    lines += ["return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(_lib.Group)
    for f, _ in _lib.Group._fields_:
        assert int(got[f]) == getattr(_lib.Group, f).offset, f


def _tagged_t2(bk, m, no, nv, rng, dV):
    """A random T2 with the integrals' momentum structure, tagged through the rules (MP2-like)."""
    mask = _n(dV["abij"]) != 0
    T = _t(np.where(mask, rng.standard_normal(mask.shape), 0.0))
    from pymes_b200.solver import ccd
    assert bk.adopt_momentum(T, ccd.fock_rules(dV["abij"], no, nv)["t2"])
    return T


def test_rules_derivation_and_invalidation(abi):
    from pymes_b200 import backend as bk
    from pymes_b200.solver import ccd
    m, no, nv, parts = _ueg14()
    dV = m.eval_2b_blocks(no, ["ijab", "abij", "iajb", "iabj", "klij"], parts)
    rng = np.random.default_rng(3)
    T = _tagged_t2(bk, m, no, nv, rng, dV)
    rule = ccd.fock_rules(dV["abij"], no, nv)["t2"]
    # every product of the doubles residual derives a rule (ccd.py doubles_residual)
    Tt = bk.tilde(T)
    assert bk.momentum_of(Tt) == rule
    for spec, A, B in [("klcd,dblj->cbkj", dV["ijab"], Tt), ("klcd,adkj->alcj", dV["ijab"], T),
                       ("klcd,daki->alci", dV["ijab"], T), ("klcd,cdij->klij", dV["ijab"], T)]:
        assert bk.momentum_of(bk.contract(spec, A, B)) is not None, spec
    Xai = bk.contract("klcd,dblj->cbkj", dV["ijab"], Tt)
    X1 = bk.contract("klcd,adkj->alcj", dV["ijab"], T)
    Xp = bk.contract("klcd,daki->alci", dV["ijab"], T)
    for spec, A, B in [("acik,cbkj->abij", Tt, Xai), ("alcj,cbil->abij", X1, T),
                       ("kaic,cbkj->abij", dV["iajb"], T), ("acik,kbcj->abij", Tt, dV["iabj"]),
                       ("alci,cblj->abij", Xp, bk.lincomb([1.0, -1.0], [T, Tt])),
                       ("kbic,ackj->abij", dV["iajb"], T), ("abkl,klij->abij", T, dV["klij"])]:
        assert bk.momentum_of(bk.contract(spec, A, B)) == rule, spec
    # an in-place edit outside the backend drops the tag (and the geometry tag of a stored block)
    U = bk.copy(T)
    assert bk.momentum_of(U) == rule
    U.mul_(2.0)
    assert bk.momentum_of(U) is None
    W = bk.copy(dV["ijab"])
    assert bk.geom_of(W) is not None
    W.add_(1.0)
    assert bk.geom_of(W) is None and bk.momentum_of(W) is None
    # accumulating a product with a different rule drops the tag of the output
    R = bk.copy(T)
    bk.contract_terms("abij", [(1.0, "acik", Tt, "cbkj", Xai)], out=R, beta=1.0)
    assert bk.momentum_of(R) == rule
    bk.contract_terms("abij", [(1.0, "ac", _t(rng.standard_normal((nv, nv))), "cbij", T)], out=R, beta=1.0)
    assert bk.momentum_of(R) is None
    # summed axes that do not cancel under one sign: untagged (and the product runs dense)
    Z = _t(np.zeros((nv, nv, no, no)))
    assert bk.adopt_momentum(Z, rule.with_axes([(no, nv, 1), (no, nv, 1), (0, no, 1), (0, no, -1)]))
    bad = bk.contract("acik,cbkj->abij", T, Z)           # c needs sigma = -1, k needs sigma = +1
    assert bk.momentum_of(bad) is None
    # a write through a narrowed view keeps the parent's tag only when it obeys the parent's rule
    F = bk.copy(T)
    view = bk.narrow(F, 0, 1, 3)
    bk.axpby(2.0, bk.narrow(T, 0, 1, 3), 0.0, view)
    assert bk.momentum_of(F) == rule
    bk.axpby(1.0, _t(rng.standard_normal(tuple(view.shape))), 0.0, view)
    assert bk.momentum_of(F) is None


def test_group_contract_matches_einsum_and_dense(abi):
    """The new path against numpy for the ring splits, row blocks, beta in {0, 0.5, 1}; the
    existing blocked path with beta = 0.5 on a narrowed block."""
    from pymes_b200 import backend as bk
    m, no, nv, parts = _ueg14()
    dV = m.eval_2b_blocks(no, ["ijab", "abij", "iajb", "iabj"], parts)
    rng = np.random.default_rng(5)
    T = _tagged_t2(bk, m, no, nv, rng, dV)
    grp = _count(abi, "pmb_group_contract")
    blk = _count(abi, "pmb_blocked_contract")
    lo, na = 2, 4
    for spec, A, B in [("kaic,cbkj->abij", dV["iajb"], T), ("kbic,ackj->abij", dV["iajb"], T),
                       ("acik,kbcj->abij", T, dV["iabj"]), ("cbkj,kaic->abij", T, dV["iajb"]),
                       ("kaic,cbkj->abij", bk.narrow(dV["iajb"], 1, lo, na), T)]:
        ref = np.einsum(spec, _n(A), _n(B))
        for beta in (0.0, 0.5, 1.0):
            n0 = grp["n"]
            R0 = rng.standard_normal(ref.shape)
            R = _t(R0.copy())
            bk.contract(spec, A, B, out=R, alpha=-0.7, beta=beta)
            assert grp["n"] == n0 + 1, spec
            np.testing.assert_allclose(_n(R), beta * R0 - 0.7 * ref, **TOL)
    # the existing blocked path (integral block x untagged amplitudes) with beta = 0.5 on a row block
    Tr = _t(rng.standard_normal((nv, nv, no, no)))
    part = bk.narrow(dV["ijab"], 2, lo, na)
    ref = np.einsum("klcd,dblj->cbkj", _n(part), _n(Tr))
    R0 = rng.standard_normal(ref.shape)
    R = _t(R0.copy())
    n0 = blk["n"]
    bk.contract("klcd,dblj->cbkj", part, Tr, out=R, beta=0.5)
    assert blk["n"] == n0 + 1
    np.testing.assert_allclose(_n(R), 0.5 * R0 + ref, **TOL)
    with pytest.raises(ValueError, match="output shape"):
        bk.contract("klcd,dblj->cbkj", part, Tr, out=_t(np.zeros((nv, nv, no, no))), beta=1.0)


def _ccsd_sweeps(bk, m, no, nv, parts, n, amps=None):
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd
    dV = m.eval_2b_blocks(no, list(KEYS), parts)
    cc = ccsd.CCSD(no)
    cc.setup(_fock(m, no), dV, amps=amps)
    return cc, [cc.sweep() for _ in range(n)]


def test_bench_path_ring_products_run_momentum_blocked(abi):
    """Through a CCSD sweep on tagged UEG blocks, the amplitudes stay tagged from sweep to sweep and
    the six ring products take pmb_group_contract; the energies match the dense path."""
    from pymes_b200 import backend as bk
    m, no, nv, parts = _ueg14()
    grp = _count(abi, "pmb_group_contract")
    cc, e_new = _ccsd_sweeps(bk, m, no, nv, parts, 3)
    per_sweep = grp["n"] / 3
    assert per_sweep >= 6
    assert bk.momentum_of(cc._st["T2"]) is not None and bk.momentum_of(cc._st["T1"]) is not None
    old = bk.set_blocked(False)
    try:
        n0 = grp["n"]
        _cc, e_ref = _ccsd_sweeps(bk, m, no, nv, parts, 3)
        assert grp["n"] == n0
    finally:
        bk.set_blocked(old)
    np.testing.assert_allclose(np.array(e_new)[:, :3], np.array(e_ref)[:, :3], rtol=0, atol=1e-12)


def test_non_conserving_warm_start_runs_dense_and_matches_oracle(abi):
    """Random T1 / T2 that break the momentum rule fail verification: nothing is tagged, the ring
    products run dense, and the sweeps agree with the oracle in lock-step."""
    from pymes_b200 import backend as bk
    from oracle import cc_oracle as oc
    m, no, nv, parts = _ueg14()
    rng = np.random.default_rng(11)
    t1 = 1e-3 * rng.standard_normal((nv, no))
    t2 = 1e-3 * rng.standard_normal((nv, nv, no, no))
    grp = _count(abi, "pmb_group_contract")
    cc, e_dev = _ccsd_sweeps(bk, m, no, nv, parts, 2, amps=(_t(t1.copy()), _t(t2.copy())))
    assert grp["n"] == 0
    assert bk.momentum_of(cc._st["T1"]) is None and bk.momentum_of(cc._st["T2"]) is None
    from pymes_b200.integral.partition import KEYS
    dV = {k: _n(v) for k, v in m.eval_2b_blocks(no, list(KEYS), parts).items()}
    f = _fock(m, no)
    d1, d2 = oc.denominators(np.diag(f)[:no], np.diag(f)[no:])
    mixer = oc.DIIS(6)
    T1, T2 = t1.copy(), t2.copy()
    for k in range(2):
        T1, T2, e, _dt = oc.ccsd_sweep(no, f, dV, T1, T2, d1, d2, mixer)
        np.testing.assert_allclose(np.array(e)[:3], np.array(e_dev[k])[:3], rtol=0, atol=1e-10)


@pytest.mark.gpu
def test_group_contract_on_device_matches_dense_kernel():
    """pmb_group_contract on the B200 against the dense DMMA kernel and torch.einsum for the ring
    splits of the doubles residual, beta in {0, 0.5, 1}, a row block; pmb_momentum_residue accepts
    the structured amplitudes and rejects a perturbed copy."""
    from pymes_b200 import backend as bk
    from pymes_b200.solver import ccd
    assert torch.cuda.is_available()
    m, no, nv, parts = _ueg14()
    dV = m.eval_2b_blocks(no, ["ijab", "abij", "iajb", "iabj"], parts)
    rule = ccd.fock_rules(dV["abij"], no, nv)["t2"]
    g = torch.Generator(device="cuda").manual_seed(4)
    mask = dV["abij"] != 0
    T = torch.where(mask, torch.randn(mask.shape, generator=g, device="cuda", dtype=torch.float64), 0.0)
    assert bk.adopt_momentum(T, rule)
    bad = T.clone()
    bad[0, 0, 0, 1] += 1e-3 if not mask[0, 0, 0, 1] else 0.0
    bad[1, 0, 0, 0] += 1e-3 if not mask[1, 0, 0, 0] else 0.0
    assert not bk.adopt_momentum(bad, rule)
    cases = [("kaic,cbkj->abij", dV["iajb"], T), ("kbic,ackj->abij", dV["iajb"], T),
             ("acik,kbcj->abij", T, dV["iabj"]), ("kaic,cbkj->abij", bk.narrow(dV["iajb"], 1, 2, 4), T)]
    for spec, A, B in cases:
        ref = torch.einsum(spec, A, B)
        for beta in (0.0, 0.5, 1.0):
            R0 = torch.randn(ref.shape, generator=g, device="cuda", dtype=torch.float64)
            got = bk.contract(spec, A, B, out=R0.clone(), alpha=-0.7, beta=beta)
            old = bk.set_blocked(False)
            try:
                dense = bk.contract(spec, A, B, out=R0.clone(), alpha=-0.7, beta=beta)
            finally:
                bk.set_blocked(old)
            want = beta * R0 - 0.7 * ref
            assert torch.allclose(got, want, rtol=0, atol=1e-12), spec
            assert torch.allclose(got, dense, rtol=0, atol=1e-12), spec


def test_non_conserving_fock_starts_untagged(abi):
    """A Fock matrix with off-diagonal noise fails the check on the host: the amplitudes start
    untagged and every sweep runs dense, with the same energies as the blocked-off path."""
    from pymes_b200 import backend as bk
    m, no, nv, parts = _ueg14()
    rng = np.random.default_rng(2)
    f = _fock(m, no) + 1e-3 * rng.standard_normal((m.n_orb, m.n_orb))
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd
    grp = _count(abi, "pmb_group_contract")
    res = _count(abi, "pmb_momentum_residue")
    cc = ccsd.CCSD(no)
    cc.setup(f, m.eval_2b_blocks(no, list(KEYS), parts))
    assert cc._rules is None and bk.momentum_of(cc._st["fock"]) is None
    assert bk.momentum_of(cc._st["T1"]) is None and bk.momentum_of(cc._st["T2"]) is None
    e = [cc.sweep()[:3] for _ in range(2)]
    assert grp["n"] == 0 and res["n"] == 0
    old = bk.set_blocked(False)
    try:
        ref = ccsd.CCSD(no)
        ref.setup(f, m.eval_2b_blocks(no, list(KEYS), parts))
        want = [ref.sweep()[:3] for _ in range(2)]
    finally:
        bk.set_blocked(old)
    np.testing.assert_allclose(np.array(e), np.array(want), rtol=0, atol=1e-12)
