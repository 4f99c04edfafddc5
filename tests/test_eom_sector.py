"""EOM-CCSD in one total-momentum sector of the UEG: momentum rules with a total, the batched group
product pmb_group_contract_batched, the sector description of model.ueg and the sector mode of
solver.eom_ccsd, against numpy and the oracle."""
import numpy as np
import pytest
import torch

REL = 1e-12


@pytest.fixture
def abi(cpu_abi):
    """The emulated C ABI with the momentum entry points and the batched group product."""
    from tests import sector_emulator
    return sector_emulator.extend(cpu_abi)


def _n(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def _ueg14():
    from pymes_b200.model import ueg
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    return m, 7, m.n_orb - 7, [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)]


def _fock(m, no):
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


def _masks(sec):
    lin, no = sec.lin, sec.no
    lo, lv = lin[:no], lin[no:]
    m1 = (lv[:, None] - lo[None, :]) == sec.label
    m2 = (lv[:, None, None, None] + lv[None, :, None, None] - lo[None, None, :, None] - lo[None, None, None, :]) \
        == sec.label
    return m1, m2


def _sector_vectors(sec, rng, r):
    m1, m2 = _masks(sec)
    u1 = np.where(m1, rng.standard_normal((r,) + m1.shape), 0.0)
    u2 = np.where(m2, rng.standard_normal((r,) + m2.shape), 0.0)
    return u1, u2


_SYSTEM = {}


def _system(bk):
    """_ueg14 after two CCSD sweeps: the dressed Fock matrix and blocks (host copies) and T2."""
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd, eom_ccsd
    m, no, nv, parts = _ueg14()
    if "host" not in _SYSTEM:
        dV = m.eval_2b_blocks(no, list(KEYS), parts)
        cc = ccsd.CCSD(no)
        cc.setup(_fock(m, no), dV)
        for _ in range(2):
            cc.sweep()
        T1, T2 = cc._st["T1"], cc._st["T2"]
        ft = cc.get_T1_dressed_fock(_t(_fock(m, no)), T1, dV)
        dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
        _SYSTEM["host"] = (_n(ft).copy(), {k: _n(dVd[k]).copy() for k in eom_ccsd.V_KEYS_USED}, _n(T2).copy())
    f, dVh, T2h = _SYSTEM["host"]
    return m, no, nv, f, dVh, T2h


def _device_operands(f, dVh, T2h):
    return _t(f), {k: _t(v) for k, v in dVh.items()}, _t(T2h)


def test_rule_algebra_with_totals(abi):
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m, no, nv, _parts = _ueg14()
    lin = ueg.linear_momenta(m)
    # normal form: flipping every sign flips the total; equality and hashing see the total
    a = bk.Momentum(lin, [(no, nv, -1), (0, no, 1)], total=5)
    b = bk.Momentum(lin, [(no, nv, 1), (0, no, -1)], total=-5)
    assert a == b and hash(a) == hash(b) and a.total == -5
    assert b != b.with_total(5) and b.with_total(0) == bk.Momentum(lin, b.axes)
    assert bk.Momentum(lin, b.axes).total == 0
    # a product: total_A + sigma total_B; "ai,bj->abij" is an outer product (both sigmas)
    sec = ueg.excitation_sector(m, no, (1, 0, 0))
    k1 = sec.singles_rule()
    keys = bk._term_keys("abij", "ai", k1, "bj", k1)
    assert {k.total for k in keys} == {2 * sec.label, 0}
    (kt,) = bk._term_keys("ai", "abij", sec.rule("abij"), "bj", k1)     # b, j summed: sigma = -1
    assert kt == k1.with_total(-sec.label)
    # tensors: a product, sums with equal and with different totals, an accumulation that mismatches
    rng = np.random.default_rng(1)
    u1, u2 = _sector_vectors(sec, rng, 2)
    U1, V1 = _t(u1[0]), _t(u1[1])
    assert bk.adopt_momentum(U1, k1) and bk.adopt_momentum(V1, k1)
    assert bk.momentum_of(bk.lincomb([1.0, -2.0], [U1, V1])) == k1
    other = ueg.excitation_sector(m, no, (0, 1, 0))
    W1 = _t(_sector_vectors(other, rng, 1)[0][0])
    assert bk.adopt_momentum(W1, other.singles_rule())
    assert bk.momentum_of(bk.lincomb([1.0, 1.0], [U1, W1])) is None
    assert bk.momentum_of(bk.axpby(1.0, W1, 1.0, bk.copy(U1))) is None
    assert bk.momentum_of(bk.axpby(1.0, V1, 1.0, bk.copy(U1))) == k1
    fock = _t(_fock(m, no))
    assert bk.adopt_momentum(fock, sec.fock_rule(), host=_fock(m, no))
    fvv = bk.narrow(bk.narrow(fock, 0, no, nv), 1, no, nv)
    assert bk.momentum_of(bk.contract("ab,bi->ai", fvv, U1)) == k1
    U2 = _t(u2[0])
    assert bk.adopt_momentum(U2, sec.doubles_rule())
    assert bk.momentum_of(bk.sym_baji(U2)) == sec.doubles_rule()
    # adopt_momentum: a sector vector is accepted, one element outside the sector is not (device
    # pass and host check alike)
    m1, _m2 = _masks(sec)
    i, j = np.argwhere(~m1)[0]
    bad = u1[0].copy()
    bad[i, j] = 1e-300
    assert not bk.adopt_momentum(_t(bad), k1)
    assert not bk.adopt_momentum(_t(bad), k1, host=bad)
    assert bk.adopt_momentum(_t(u1[0]), k1, host=u1[0])
    assert not bk.adopt_momentum(_t(u1[0]), other.singles_rule())


def test_group_plan_is_never_shared_between_totals(abi):
    """Two products that differ only in the total of one operand get different plans, each right."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m, no, nv, _parts = _ueg14()
    rng = np.random.default_rng(2)
    f, dVh, T2h = _system(bk)[3:]
    V = _t(dVh["iabj"])
    sectors = [e["sector"] for e in ueg.excitation_sectors(m, no)[1:3]]
    plans = []
    for sec in sectors:
        assert bk.adopt_momentum(V, sec.rule("iabj"))
        u1 = _t(_sector_vectors(sec, rng, 1)[0][0])
        assert bk.adopt_momentum(u1, sec.singles_rule())
        g = bk._group_term("ai", (1.0, "jabi", V, "bj", u1))
        assert g is not None
        out = _t(np.zeros((nv, no)))
        plans.append(bk._group_plan("ai", g, out))
        got = bk.contract("jabi,bj->ai", V, u1)
        np.testing.assert_allclose(_n(got), np.einsum("jabi,bj->ai", dVh["iabj"], _n(u1)), rtol=0, atol=1e-13)
        assert bk.momentum_of(got) == sec.singles_rule()
    assert plans[0] is not plans[1]
    assert not np.array_equal(_n(plans[0]["c_row"]), _n(plans[1]["c_row"]))


@pytest.mark.parametrize("side", ["A", "B", "AB"])
def test_batched_group_product_matches_einsum(abi, side):
    """pmb_group_contract_batched (emulated) through contract_terms: the batch axis on A only, on B
    only, on both (stride 0 on the other operand); beta in {0, 0.5, 1}; against numpy.einsum."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m, no, nv, _parts = _ueg14()
    rng = np.random.default_rng(3)
    sec = ueg.excitation_sector(m, no, (1, 1, 0))
    f, dVh, T2h = _system(bk)[3:]
    V = _t(dVh["ijab"])
    assert bk.adopt_momentum(V, sec.rule("ijab"))
    batched = _count(abi, "pmb_group_contract_batched")
    dense = _count(abi, "pmb_contract")
    for r in (1, 3):
        u1, u2 = _sector_vectors(sec, rng, r)
        us = [_t(x) for x in u2]
        for x in us:
            assert bk.adopt_momentum(x, sec.doubles_rule())
        U = bk.stack(us)
        if side == "B":                   # W[k,l,c,d] u[r,c,d,i,j] -> [r,k,l,i,j]
            spec, A, B, out_sub = "klcd,rcdij->rklij", V, U, "rklij"
        elif side == "A":                 # u[r,c,d,i,j] W[k,l,c,d] with the batch axis on A
            spec, A, B, out_sub = "rcdij,klcd->rijkl", U, V, "rijkl"
        else:                             # both stacked: u1[r,a,i] u1'[r,b,i] -> [r,a,b], i summed
            ys = [_t(x) for x in u1]
            zs = [_t(x) for x in _sector_vectors(sec, rng, r)[0]]
            for y in ys + zs:
                assert bk.adopt_momentum(y, sec.singles_rule())
            spec, A, B, out_sub = "rai,rbi->rab", bk.stack(ys), bk.stack(zs), "rab"
        sa, rest = spec.split(",")
        sb = rest.split("->")[0]
        ref = np.einsum(spec, _n(A), _n(B))
        for beta in (0.0, 0.5, 1.0):
            n0, d0 = batched["n"], dense["n"]
            R0 = rng.standard_normal(ref.shape)
            R = _t(R0.copy())
            bk.contract_terms(out_sub, [(-0.7, sa, A, sb, B)], out=R, beta=beta)
            assert batched["n"] == n0 + 1 and dense["n"] == d0, (side, r, beta)
            np.testing.assert_allclose(_n(R), beta * R0 - 0.7 * ref, rtol=0, atol=1e-12)


def test_batched_descriptor_matches_the_c_header(tmp_path):
    import ctypes as C
    import os
    import shutil
    import subprocess
    from pymes_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "pymes_b200.h"', "int main(void) {",
             'printf("size %zu\\n", sizeof(pmb_group_batched_t));']
    lines += ['printf("%s %%zu\\n", offsetof(pmb_group_batched_t, %s));' % (f, f) for f, _ in _lib.GroupBatched._fields_]
    lines += ["return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True,
                                                   check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(_lib.GroupBatched)
    for f, _ in _lib.GroupBatched._fields_:
        assert int(got[f]) == getattr(_lib.GroupBatched, f).offset, f


def test_excitation_sectors_count_and_order():
    from pymes_b200.model import ueg
    m, no, nv, _parts = _ueg14()
    secs = ueg.excitation_sectors(m, no)
    norms = [sum(x * x for x in e["K"]) for e in secs]
    # k_a != k_i for a != i: no single has K = 0
    assert norms == sorted(norms) and norms[0] == 1
    assert sum(e["n_singles"] for e in secs) == nv * no
    for e in secs[:6]:
        m1, m2 = _masks(e["sector"])
        assert (e["n_singles"], e["n_doubles"]) == (int(m1.sum()), int(m2.sum()))
        assert e["sector"] == ueg.excitation_sector(m, no, e["K"])
    with pytest.raises(ValueError, match="integer 3-vector"):
        ueg.excitation_sector(m, no, (0.5, 0, 0))


def _sector_eom(sec, n_excit=2):
    from pymes_b200.solver import eom_ccsd
    return eom_ccsd.EOM_CCSD(7, n_excit=n_excit, sector=sec)


def test_sector_sigma_matches_oracle_and_stays_in_the_sector(abi):
    """Sector sigma for random sector vectors (a batch of 3) against the oracle's 62-term sigma,
    1e-12 relative, exactly zero outside the sector, the result tagged with the sector rule; every
    u-dependent product runs on momentum groups (no pmb_contract launch), the doubles through the
    batched entry point."""
    from oracle import cc_oracle as oc
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m, no, nv, f, dVh, T2h = _system(bk)
    rng = np.random.default_rng(4)
    sec = ueg.excitation_sector(m, no, (1, 0, 0))
    eom = _sector_eom(sec)
    ft, dV, T2 = _device_operands(f, dVh, T2h)
    plan = eom.plan(ft, dV, T2)
    u1, u2 = _sector_vectors(sec, rng, 3)
    U1 = [_t(x) for x in u1]
    U2 = [_t(x) for x in u2]
    for a, b in zip(U1, U2):
        assert bk.adopt_momentum(a, sec.singles_rule()) and bk.adopt_momentum(b, sec.doubles_rule())
    dense = _count(abi, "pmb_contract")
    batched = _count(abi, "pmb_group_contract_batched")
    S1, S2 = plan.apply(bk.stack(U1), bk.stack(U2))
    assert dense["n"] == 0 and batched["n"] > 0
    assert bk.momentum_of(S1) == bk.momentum_of(bk.stack(U1)) is not None
    assert bk.momentum_of(S2) == bk.momentum_of(bk.stack(U2))
    m1, m2 = _masks(sec)
    for k in range(3):
        s1 = oc.eom_sigma_singles(no, f, dVh, u1[k], u2[k], T2h)
        s2 = oc.eom_sigma_doubles(no, f, dVh, u1[k], u2[k], T2h)
        assert _rel(_n(S1[k]), s1) < REL and _rel(_n(S2[k]), s2) < REL
        assert not _n(S1[k])[~m1].any() and not _n(S2[k])[~m2].any()
    # the same vectors through the dense path
    old = bk.set_blocked(False)
    try:
        from pymes_b200.solver import eom_ccsd
        D1, D2 = eom_ccsd.SigmaPlan(no, _t(f), {k: _t(v) for k, v in dVh.items()}, _t(T2h)).apply(
            _t(u1), _t(u2))
    finally:
        bk.set_blocked(old)
    assert _rel(_n(S1), _n(D1)) < REL and _rel(_n(S2), _n(D2)) < REL


def _oracle_hbar(sec, no, f, dVh, T2h):
    """The oracle H-bar on the sector basis (singles then doubles), built column by column."""
    from oracle import cc_oracle as oc
    m1, m2 = _masks(sec)
    i1, i2 = np.flatnonzero(m1), np.flatnonzero(m2)
    n1 = len(i1)
    H = np.zeros((n1 + len(i2), n1 + len(i2)))
    for c in range(H.shape[0]):
        u1, u2 = np.zeros(m1.size), np.zeros(m2.size)
        if c < n1:
            u1[i1[c]] = 1.0
        else:
            u2[i2[c - n1]] = 1.0
        u1, u2 = u1.reshape(m1.shape), u2.reshape(m2.shape)
        s1 = oc.eom_sigma_singles(no, f, dVh, u1, u2, T2h)
        s2 = oc.eom_sigma_doubles(no, f, dVh, u1, u2, T2h)
        if c < 6:          # H-bar maps a sector vector into its sector
            assert not s1[~m1].any() and not s2[~m2].any()
        H[:n1, c], H[n1:, c] = s1.reshape(-1)[i1], s2.reshape(-1)[i2]
    return H


@pytest.mark.parametrize("pick", [0, 7])
def test_sector_davidson_matches_oracle_hbar(abi, pick):
    """The sector Davidson roots are eigenvalues of the oracle H-bar restricted to the sector (the
    states its singles guesses lead to: this unconverged, gapped test system also has doubles-like
    eigenvalues far below them, which no singles guess reaches)."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m, no, nv, f, dVh, T2h = _system(bk)
    sec = [e["sector"] for e in ueg.excitation_sectors(m, no) if e["n_singles"] >= 2][pick]
    ev = np.linalg.eigvals(_oracle_hbar(sec, no, f, dVh, T2h))
    eom = _sector_eom(sec)
    eom.e_epsilon, eom.max_dim = 1e-12, 16
    e = eom.solve(*_device_operands(f, dVh, T2h))
    assert eom.iterations < eom.max_iter
    for root in e:
        assert np.abs(ev - root).min() < 1e-8, (root, np.sort(ev.real))


def test_sector_mode_rejects_what_it_cannot_solve(abi):
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m, no, nv, f, dVh, T2h = _system(bk)
    sec = ueg.excitation_sector(m, no, (1, 0, 0))
    rng = np.random.default_rng(6)
    noisy = f + 1e-6 * rng.standard_normal(f.shape)
    with pytest.raises(ValueError, match="Fock"):
        _sector_eom(sec).solve(noisy, {k: _t(v) for k, v in dVh.items()}, _t(T2h))
    with pytest.raises(ValueError, match="Fock"):
        _sector_eom(sec).solve(_t(noisy), {k: _t(v) for k, v in dVh.items()}, _t(T2h))
    with pytest.raises(ValueError, match="T2"):
        _sector_eom(sec).solve(_t(f), {k: _t(v) for k, v in dVh.items()}, _t(T2h + 1e-6 * rng.standard_normal(T2h.shape)))
    for K in ((40, 0, 0), (0, 0, 0)):      # K = 0 holds doubles only: k_a != k_i
        with pytest.raises(ValueError, match="no single"):
            _sector_eom(ueg.excitation_sector(m, no, K)).solve(*_device_operands(f, dVh, T2h))
    n1 = int(_masks(sec)[0].sum())
    with pytest.raises(ValueError, match="exceeds"):
        _sector_eom(sec, n_excit=n1 + 1).solve(*_device_operands(f, dVh, T2h))
    eom = _sector_eom(sec)
    eom.preconditioner = "diagonal"
    with pytest.raises(NotImplementedError):
        eom.solve(*_device_operands(f, dVh, T2h))


# --------------------------------------------------------------------------
# on the B200
# --------------------------------------------------------------------------
def _gpu_system(virtual=()):
    """_ueg14 on the device after two CCSD sweeps: dressed Fock matrix, dressed blocks, T2."""
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd, eom_ccsd
    m, no, nv, parts = _ueg14()
    dV = m.eval_2b_blocks(no, list(KEYS), parts, virtual=virtual)
    cc = ccsd.CCSD(no)
    cc.setup(_fock(m, no), dV)
    for _ in range(2):
        cc.sweep()
    T1, T2 = cc._st["T1"], cc._st["T2"]
    ft = cc.get_T1_dressed_fock(bk.asdev(_fock(m, no)), T1, dV)
    dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
    return m, no, nv, ft, {k: dVd[k] for k in eom_ccsd.V_KEYS_USED}, T2


@pytest.mark.gpu
def test_batched_group_kernel_on_device_matches_dense_kernel():
    """pmb_group_contract_batched against the dense DMMA kernel for r in {1, 3, 16}, beta in
    {0, 0.5, 1}, the batch axis on A, on B and on both, 1e-13 relative."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m, no, nv, parts = _ueg14()
    V = m.eval_2b_blocks(no, ["ijab"], parts)["ijab"]
    sec = ueg.excitation_sector(m, no, (1, 1, 0))
    assert bk.adopt_momentum(V, sec.rule("ijab"))
    rng = np.random.default_rng(8)
    n_batched = 0
    for r in (1, 3, 16):
        u1, u2 = _sector_vectors(sec, rng, r)
        v1 = _sector_vectors(sec, rng, r)[0]
        U2 = [bk.asdev(x) for x in u2]
        Y, Z = [bk.asdev(x) for x in u1], [bk.asdev(x) for x in v1]
        for x in U2:
            assert bk.adopt_momentum(x, sec.doubles_rule())
        for x in Y + Z:
            assert bk.adopt_momentum(x, sec.singles_rule())
        S2, SY, SZ = bk.stack(U2), bk.stack(Y), bk.stack(Z)
        for out_sub, sa, A, sb, B in (("rklij", "klcd", V, "rcdij", S2), ("rijkl", "rcdij", S2, "klcd", V),
                                      ("rab", "rai", SY, "rbi", SZ)):
            assert bk._batched_group_term(out_sub, (1.0, sa, A, sb, B)) is not None
            shape = tuple(dict(zip(sa + sb, tuple(A.shape) + tuple(B.shape)))[ch] for ch in out_sub)
            for beta in (0.0, 0.5, 1.0):
                R0 = bk.asdev(rng.standard_normal(shape))
                got = bk.contract_terms(out_sub, [(-0.7, sa, A, sb, B)], out=R0.clone(), beta=beta)
                n_batched += 1
                # the dense kernel takes no index shared by both operands and the output: one launch
                # per right-hand side on its slices
                dense = R0.clone()
                old = bk.set_blocked(False)
                try:
                    for k in range(r):
                        Ak, sak = (A[k], sa[1:]) if sa[0] == "r" else (A, sa)
                        Bk, sbk = (B[k], sb[1:]) if sb[0] == "r" else (B, sb)
                        bk.contract_terms(out_sub[1:], [(-0.7, sak, Ak, sbk, Bk)], out=dense[k], beta=beta)
                finally:
                    bk.set_blocked(old)
                assert _rel(_n(got), _n(dense)) < 1e-13, (out_sub, r, beta)
    assert n_batched == 27


@pytest.mark.gpu
def test_sector_sigma_at_o27_vs_oracle():
    """Sector sigma at the benchmark's o = 27 (TC-UEG 54e / 65 plane waves, amplitudes after 3 CCSD
    sweeps, the path of test_eom_sigma_at_o27_vs_oracle) with the dressed V_abcd stored and as the
    never-materialised operator, against the oracle's sigma, 1e-9 relative; zero outside the sector."""
    import bench
    from oracle import cc_oracle as oc
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd, eom_ccsd
    no = bench.N_ELE // 2
    prob = bench.CpuProblem(6.0)
    m = ueg.UEG(bench.N_ELE, no, no, bench.RS)
    m.init_single_basis(6.0)
    m.k_cutoff, m.gamma = bench.K_CUTOFF, None
    fock = bk.asdev(bench.build_fock(m, no))
    sec = ueg.excitation_sector(m, no, (1, 0, 0))
    m1, m2 = _masks(sec)
    rng = np.random.default_rng(5)
    u1, u2 = _sector_vectors(sec, rng, 2)
    for virtual in ((), ("abcd",)):
        dV = m.eval_2b_blocks(no, list(KEYS), bench.tc_parts(m), virtual=virtual)
        cc = ccsd.CCSD(no)
        cc.setup(fock, dV)
        for _ in range(3):
            cc.sweep()
        T1, T2 = cc._st["T1"], cc._st["T2"]
        ft = cc.get_T1_dressed_fock(fock, T1, dV)
        dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
        plan = eom_ccsd.EOM_CCSD(no, sector=sec).plan(ft, {k: dVd[k] for k in eom_ccsd.V_KEYS_USED}, T2)
        U1, U2 = [bk.asdev(x) for x in u1], [bk.asdev(x) for x in u2]
        for a, b in zip(U1, U2):
            assert bk.adopt_momentum(a, sec.singles_rule()) and bk.adopt_momentum(b, sec.doubles_rule())
        S1, S2 = plan.apply(bk.stack(U1), bk.stack(U2))
        T1h, T2h = _n(T1), _n(T2)
        fto = oc.dressed_fock(no, prob.fock, T1h, prob.dV)
        dVo = oc.dressed_V(T1h, prob.dV)
        for k in range(2):
            s1 = oc.eom_sigma_singles(no, fto, dVo, u1[k], u2[k], T2h)
            s2 = oc.eom_sigma_doubles(no, fto, dVo, u1[k], u2[k], T2h)
            assert _rel(_n(S1[k]), s1) < 1e-9 and _rel(_n(S2[k]), s2) < 1e-9, virtual
            assert not _n(S1[k])[~m1].any() and not _n(S2[k])[~m2].any()


@pytest.mark.gpu
def test_sector_davidson_on_device_matches_oracle_roots():
    """Sector Davidson on the B200 (_ueg14, two sectors): every root is an eigenvalue of the oracle
    H-bar of the sector, built on the host from the same dressed operators."""
    from pymes_b200.model import ueg
    m, no, nv, ft, dVd, T2 = _gpu_system()
    f, dVh, T2h = _n(ft), {k: _n(v) for k, v in dVd.items()}, _n(T2)
    for pick in (0, 7):
        sec = [e["sector"] for e in ueg.excitation_sectors(m, no) if e["n_singles"] >= 2][pick]
        ev = np.linalg.eigvals(_oracle_hbar(sec, no, f, dVh, T2h))
        eom = _sector_eom(sec)
        eom.e_epsilon, eom.max_dim = 1e-12, 16
        e = eom.solve(ft, dVd, T2)
        assert eom.iterations < eom.max_iter
        for root in e:
            assert np.abs(ev - root).min() < 1e-8, (root, np.sort(ev.real))
