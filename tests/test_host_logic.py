"""Host logic of pymes_b200 (einsum front end, term tables, DIIS, solver drivers, UEG
tables) checked on the CPU against the reference-generated goldens.  The C ABI is
emulated in numpy by tests/abi_emulator.py (test infrastructure, see its header);
the CUDA kernels themselves are checked in the -m gpu tests."""
import os

import numpy as np
import pytest
import torch

from tests.conftest import golden

TOL = dict(rtol=1e-10, atol=1e-11)


DEVICE = "cpu"      # tests/test_gpu_parity.py re-runs these bodies with DEVICE = "cuda"


def _t(x):
    x = np.asarray(x, dtype=np.float64)
    t = torch.from_numpy(np.ascontiguousarray(x)) if x.ndim else torch.tensor(float(x), dtype=torch.float64)
    return t.to(DEVICE)


def _n(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def test_library_exports_every_declared_symbol():
    """The built .so loads and exports each function include/pymes_b200.h declares."""
    import ctypes
    import re
    from pymes_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "run python -m pymes_b200.build"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "pymes_b200.h")).read()
    declared = set(re.findall(r"\b(pmb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.pmb_version() == 100


def test_ctypes_structs_match_the_c_header(tmp_path):
    """Size and field offsets of every struct of include/pymes_b200.h as gcc lays them out ==
    the ctypes mirrors in pymes_b200/_lib.py (the descriptors cross the C ABI by pointer)."""
    import ctypes as C
    import shutil
    import subprocess
    from pymes_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    pairs = {"pmb_term_t": _lib.Term, "pmb_contract_t": _lib.Contract, "pmb_bdot_t": _lib.Bdot,
             "pmb_gemv_t": _lib.Gemv, "pmb_ueg_t": _lib.Ueg, "pmb_ueg_operand_t": _lib.UegOperand,
             "pmb_blocked_t": _lib.Blocked, "pmb_gather_t": _lib.Gather}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "pymes_b200.h"', "int main(void) {"]
    for cname, cls in pairs.items():
        lines.append('printf("%s size %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ["return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = {}
    for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines():
        cname, fname, val = ln.split()
        got[(cname, fname)] = int(val)
    for cname, cls in pairs.items():
        assert got[(cname, "size")] == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)


def test_missing_cuda_fails_loudly():
    from pymes_b200 import backend as bk
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        bk.asdev(np.zeros(3))


@pytest.mark.parametrize("spec,shapes", [
    ("abcd,cdij->abij", [(5, 5, 5, 5), (5, 5, 3, 3)]),
    ("klij,abkl->abij", [(3, 3, 3, 3), (5, 5, 3, 3)]),
    ("klcd,adkj->alcj", [(3, 3, 5, 5), (5, 5, 3, 3)]),
    ("alcj,cbil->abij", [(5, 3, 5, 3), (5, 5, 3, 3)]),
    ("kbic,ackj->abij", [(3, 5, 3, 5), (5, 5, 3, 3)]),
    ("adkl,lkdc->ac", [(5, 5, 3, 3), (3, 3, 5, 5)]),
    ("cdil,lkdc->ki", [(5, 5, 3, 3), (3, 3, 5, 5)]),
    ("ki,abkj->abij", [(3, 3), (5, 5, 3, 3)]),
    ("ia,ai->", [(3, 5), (5, 3)]),
    ("bj,jabi->ia", [(5, 3), (3, 5, 5, 3)]),
    ("ai,bj->abij", [(5, 3), (5, 3)]),
])
def test_contract_matches_einsum(cpu_abi, spec, shapes):
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(1)
    A, B = (rng.standard_normal(s) for s in shapes)
    ref = np.einsum(spec, A, B)
    got = bk.contract(spec, A, B, alpha=0.7)
    np.testing.assert_allclose(_n(got), 0.7 * ref, **TOL)
    out = _t(rng.standard_normal(ref.shape))
    keep = _n(out).copy()
    bk.contract(spec, A, B, out=out, alpha=-1.5, beta=0.25)
    np.testing.assert_allclose(_n(out), 0.25 * keep - 1.5 * ref, **TOL)


def test_contract_on_strided_views_and_multi_term(cpu_abi):
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import part_2_body_int
    rng = np.random.default_rng(2)
    no, nv = 2, 4
    V = rng.standard_normal((no + nv,) * 4)
    T = rng.standard_normal((nv, nv, no, no))
    dV = part_2_body_int(no, _t(V))
    dVn = part_2_body_int(no, V)
    got = bk.contract("abcd,cdij->abij", dV["abcd"], _t(T))
    np.testing.assert_allclose(_n(got), np.einsum("abcd,cdij->abij", dVn["abcd"], T), **TOL)
    I = rng.standard_normal((no,) * 4)
    R = _t(dVn["abij"].copy())
    bk.contract_terms("abij", [(1.0, "abkl", _t(T), "klij", _t(I)),
                               (2.0, "cdij", _t(T), "abcd", dV["abcd"])], out=R, beta=1.0)
    ref = dVn["abij"] + np.einsum("abkl,klij->abij", T, I) + 2 * np.einsum("abcd,cdij->abij", dVn["abcd"], T)
    np.testing.assert_allclose(_n(R), ref, **TOL)
    # output into a strided view
    F = _t(np.zeros((no + nv, no + nv)))
    bk.contract("bj,jabi->ia", _t(rng.standard_normal((nv, no))), dV["iabj"], out=F[:no, no:])
    assert np.abs(_n(F)[no:, :]).max() == 0 and np.abs(_n(F)[:no, no:]).max() > 0


def test_multi_operand_einsum(cpu_abi):
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(3)
    no, nv = 3, 4
    t = rng.standard_normal((nv, no))
    V = rng.standard_normal((no, no, nv, nv))
    for spec, ops in (("bj,jkbc,ci,ak->ai", (t, V, t, t)),
                      ("klcd,ak,ci,bl,dj->abij", (V, t, t, t, t)),
                      ("baij->abij", (rng.standard_normal((nv, nv, no, no)),))):
        np.testing.assert_allclose(_n(bk.einsum(spec, *ops)), np.einsum(spec, *ops, optimize=True), **TOL)
    with pytest.raises(ValueError):
        bk.einsum("ab,ab->ab", t, t)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_ccd_residual_energy_mp2(cpu_abi, tag):
    from pymes_b200.solver import ccd, mp2
    g = golden("residual_random_" + tag)
    no = int(g["no"])
    args = [g[k] for k in ("klij", "ijab", "abij", "iajb", "iabj", "abcd")]
    for name, flag in (("R_ccd", False), ("R_dcd", True)):
        R = ccd.CCD(no, is_dcd=flag).get_residual(g["fock"], g["T2"], *args)
        np.testing.assert_allclose(R, g[name], **TOL)
    ed, ex = ccd.CCD(no).get_energy(g["T2"], g["ijab"])
    np.testing.assert_allclose([ed, ex], [g["e_dir"], g["e_ex"]], rtol=1e-12)
    e, t = mp2.solve(g["eps_i"], g["eps_a"], g["ijab"], g["abij"], float(g["mp2_shift"]))
    assert np.isclose(e, g["mp2_e"], rtol=1e-12)
    np.testing.assert_allclose(t, g["mp2_t2"], **TOL)
    e2, _ = mp2.solve(g["eps_i"], g["eps_a"], t_V_abij=g["abij"], t_V_ijab=g["ijab"], leve_shift=0.3)
    assert np.isclose(e2, e)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_ccsd_dressing_singles_doubles(cpu_abi, tag):
    from pymes_b200.solver import ccsd, ccd
    from pymes_b200.integral.partition import part_2_body_int
    from pymes_b200 import backend as bk
    g = golden("dressing_random_" + tag)
    no = int(g["no"])
    cc = ccsd.CCSD(no)
    dV = part_2_body_int(no, g["V"])
    assert len(dV) == 16
    ft = cc.get_T1_dressed_fock(g["fock"], g["T1"], dV)
    np.testing.assert_allclose(ft, g["fock_dressed"], **TOL)
    dVt = cc.get_T1_dressed_V(g["T1"], dV)
    assert sorted(k for k, v in dVt.items() if v is None) == sorted(g["none_keys"].tolist())
    for k, v in dVt.items():
        if v is not None:
            np.testing.assert_allclose(v, g["dressed_" + k], **TOL)
    np.testing.assert_allclose(cc.get_singles_residual(ft, g["T1"], g["T2"], dV), g["R1"], **TOL)
    np.testing.assert_allclose(cc.get_doubles_residual(ft, g["T2"], dVt), g["R2"], **TOL)
    np.testing.assert_allclose(cc.get_energy(g["fock"][:no, no:], g["T1"], g["T2"], dV["ijab"]),
                               [g["e_1b"], g["e_dir"], g["e_ex"]], rtol=1e-12)
    # the lean path of solve(): tau ladder, dressed V_abcd never formed
    dVd = {k: _t(v) for k, v in part_2_body_int(no, g["V"]).items()}
    T1, T2, ftd = _t(g["T1"]), _t(g["T2"]), _t(ft)
    R2 = ccd.doubles_residual(no, ftd, T2, ccsd.dressed_block("klij", T1, dVd), dVd["ijab"],
                              ccsd.dressed_block("abij", T1, dVd, skip_tau=True),
                              ccsd.dressed_block("iajb", T1, dVd), ccsd.dressed_block("iabj", T1, dVd),
                              None, pp_ladder=ccsd.tau_ladder(T1, dVd))
    np.testing.assert_allclose(_n(R2), g["R2"], **TOL)
    # requesting a subset of keys
    sub = cc.get_T1_dressed_V(g["T1"], dV, {"klij": None, "iabc": None})
    assert set(sub) == {"klij", "iabc"}
    np.testing.assert_allclose(sub["iabc"], g["dressed_iabc"], **TOL)


def test_diis_matches_reference_sequence(cpu_abi):
    from pymes_b200.mixer.diis import DIIS
    g = golden("diis_sequence")
    mixer = DIIS(int(g["dim_space"]))
    for n in range(int(g["n_calls"])):
        out = mixer.mix([_t(g[f"e1_{n}"]), _t(g[f"e2_{n}"])], [_t(g[f"a1_{n}"]), _t(g[f"a2_{n}"])])
        np.testing.assert_allclose(mixer.L, g[f"L_{n}"], rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(_n(out[0]), g[f"o1_{n}"], rtol=1e-9, atol=1e-11)
        np.testing.assert_allclose(_n(out[1]), g[f"o2_{n}"], rtol=1e-9, atol=1e-11)


@pytest.mark.parametrize("tag", ["LiH_321g", "LiH_tc"])
def test_solvers_follow_reference_iteration_by_iteration(cpu_abi, tag, capsys):
    from pymes_b200.solver import ccd, dcd, ccsd
    from pymes_b200.mean_field import hf
    g = golden("mol_" + tag)
    no = int(g["n_elec"]) // 2
    assert np.isclose(hf.calc_hf_e(no, float(g["e_core"]), g["h"], g["V"]), g["hf_e"], rtol=1e-13)
    fock = hf.construct_hf_matrix(no, g["h"], g["V"])
    np.testing.assert_allclose(fock, g["fock"], rtol=1e-13, atol=1e-14)
    r = ccd.CCD(no).solve(fock, g["V"], delta_e=1e-12, max_iter=200)
    assert set(r) == {"ccd e", "t2 amp", "hole e", "particle e", "dE"}
    assert abs(r["ccd e"] - g["ccd_e"]) < 1e-11
    np.testing.assert_allclose(r["t2 amp"], g["ccd_t2"], rtol=1e-8, atol=1e-11)
    r = dcd.DCD(no).solve(fock, g["V"], delta_e=1e-12, max_iter=200)
    assert abs(r["ccd e"] - g["dcd_e"]) < 1e-11
    for name, flag in (("ccsd", False), ("dcsd", True)):
        cc = ccsd.CCSD(no, is_dcsd=flag)
        r = cc.solve(fock, g["V"], delta_e=1e-12, max_iter=200)
        assert set(r) == {"ccsd e", "t1", "t2", "hole e", "particle e", "dE"}
        assert abs(r["ccsd e"] - g[name + "_e"]) < 1e-11
        assert cc.iterations == len(g[name + "_trace"])
        np.testing.assert_allclose(r["t1"], g[name + "_t1"], rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(r["t2"], g[name + "_t2"], rtol=1e-8, atol=1e-11)
        assert cc.t_T_abij is r["t2"]


def test_amps_warm_start_aliasing(cpu_abi):
    """`amps` is updated in place on the first sweep, as in ccd.py:78,124."""
    from pymes_b200.solver import ccd
    g = golden("mol_LiH_321g")
    no = int(g["n_elec"]) // 2
    amps = g["ccd_t2"].copy()
    start = amps.copy()
    r = ccd.CCD(no).solve(g["fock"], g["V"], amps=amps, delta_e=1e-9)
    assert abs(r["ccd e"] - g["ccd_e"]) < 1e-8
    assert not np.array_equal(amps, start) and np.allclose(amps, start, atol=1e-6)


def test_fcidump_roundtrip(tmp_path):
    from pymes_b200.util import fcidump
    for tag, is_tc in (("LiH_tc", True), ("H2_321g", False)):
        g = golden("mol_" + tag)
        path = str(tmp_path / ("FCIDUMP." + tag))
        fcidump.write(path, int(g["n_elec"]), g["h"], g["V"], float(g["e_core"]), is_tc=is_tc)
        n_elec, n_orb, e_core, eps, h, V = fcidump.read(path, is_tc=is_tc)
        assert (n_elec, n_orb) == (int(g["n_elec"]), g["h"].shape[0])
        assert e_core == float(g["e_core"])
        np.testing.assert_array_equal(h, g["h"])
        np.testing.assert_array_equal(V, g["V"])


@pytest.mark.parametrize("tag,is_tc", [("LiH_321g", False), ("LiH_tc", True)])
def test_fcidump_read_blocks_equals_partition_of_dense_read(tmp_path, tag, is_tc):
    """fcidump.read_blocks fills the 16 partition blocks (optionally only one rank's rows of the
    v^4 / o.v^3 blocks) exactly as slicing the dense tensor of fcidump.read does."""
    from pymes_b200.integral.partition import part_2_body_int, KEYS
    from pymes_b200.parallel import SHARD_DIMS
    from pymes_b200.util import fcidump
    g = golden("mol_" + tag)
    path = str(tmp_path / "FCIDUMP")
    fcidump.write(path, int(g["n_elec"]), g["h"], g["V"], e_core=float(g["e_core"]), is_tc=is_tc)
    n_elec, n_orb, e_core, eps, h, V = fcidump.read(path, is_tc=is_tc)
    np.testing.assert_allclose(V, g["V"], rtol=0, atol=1e-15)
    no = n_elec // 2
    dense = part_2_body_int(no, V)
    got = fcidump.read_blocks(path, is_tc=is_tc)
    assert got[:3] == (n_elec, n_orb, e_core) and sorted(got[5]) == sorted(KEYS)
    np.testing.assert_array_equal(got[4], h)
    for key in KEYS:
        np.testing.assert_array_equal(got[5][key], dense[key])
    lo, n = 1, (n_orb - no) // 2
    part = fcidump.read_blocks(path, is_tc=is_tc, rows=(lo, n), sharded_dims=SHARD_DIMS)[5]
    for key in KEYS:
        want = dense[key]
        if key in SHARD_DIMS:
            want = np.take(want, range(lo, lo + n), axis=SHARD_DIMS[key])
        np.testing.assert_array_equal(part[key], want)


def test_ueg_basis_matches_reference():
    from pymes_b200.model import ueg
    g = golden("ueg_coulomb")
    for nel, cut, nP in g["basis_sizes"]:
        m = ueg.UEG(int(nel), int(nel) // 2, int(nel) // 2, 1.0)
        m.init_single_basis(float(cut))
        assert m.n_orb == int(nP)
        np.testing.assert_array_equal(m.k_int(), g[f"basis_{int(nel)}_{int(cut)}_kint"])
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(5.0)
    np.testing.assert_array_equal(m.basis_indices_map, g["rs05_map"])
    np.testing.assert_array_equal(m.kinetic(), g["rs05_kin"])
    assert m.L == float(g["rs05_L"]) and m.imax == int(g["rs05_imax"])


def _dense(idx, val, nP):
    V = np.zeros(nP ** 4)
    V[idx] = val
    return V.reshape((nP,) * 4)


def test_ueg_coulomb_integrals_and_ccd(cpu_abi):
    from pymes_b200.model import ueg
    from pymes_b200.mean_field import hf
    from pymes_b200.solver import ccd
    g = golden("ueg_coulomb")
    m = ueg.UEG(14, 7, 7, 1.0)
    m.init_single_basis(5.0)
    V = m.eval_2b_integrals(sp=0)
    ref = _dense(g["rs1_V_idx"], g["rs1_V_val"], m.n_orb)
    np.testing.assert_allclose(V, ref, rtol=1e-13, atol=0)
    fock = hf.construct_hf_matrix(7, np.diag(m.kinetic()), V)
    np.testing.assert_allclose(fock, g["rs1_fock"], rtol=1e-12, atol=1e-13)
    blocks = m.eval_2b_blocks(7, ["abij", "iajb"], [("coulomb", None)])
    np.testing.assert_array_equal(_n(blocks["iajb"]), V[:7, 7:, :7, 7:])


@pytest.mark.slow
def test_ueg_ccd_trace(cpu_abi):
    from pymes_b200.solver import ccd
    g = golden("ueg_coulomb")
    nP = 57
    V = _dense(g["rs1_V_idx"], g["rs1_V_val"], nP)
    cc = ccd.CCD(7)
    r = cc.solve(g["rs1_fock"], V, max_iter=2)
    np.testing.assert_allclose(r["ccd e"], g["rs1_ccd_trace"][2], rtol=0, atol=1e-10)


def test_ueg_tc_tables_small(cpu_abi):
    """TC pair tables / u_mat / symmetrised effective 2-body against the reference goldens
    (subset of rows, the full build is checked on the GPU)."""
    from pymes_b200.model import ueg
    g = golden("ueg_tc")
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(5.0)
    m.gamma = None
    m.k_cutoff = 1.0
    nP = m.n_orb
    np.testing.assert_array_equal(m.k_int(), g["kint"])
    # u_mat on a few q with a reduced lattice cutoff is checked separately below;
    # here: effective two-body block (no u_mat needed)
    W0, _ = m.pair_tables("effect_2b", m.trunc)
    # eval_2b_integrals(is_effect_2b=True) returns the (pq)(rs)<->(qp)(sr) symmetrised tensor
    blk = m.build_block((0, 0, 0, 0), (3, nP, 3, nP), W0s=W0)
    ref = _dense(g["Veff_idx"], g["Veff_val"], nP)[:3, :, :3, :]
    np.testing.assert_allclose(_n(blk), ref, rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(m.double_contractions_in_3_body(), g["one_body"], rtol=1e-11)
    np.testing.assert_allclose(m.triple_contractions_in_3_body(), g["zero_body"], rtol=1e-11)


def test_contract_realigns_conflicting_unit_strides(cpu_abi, monkeypatch):
    """``abjk,jkcb->ac`` (dressed Fock, ccsd.py:264) and ``ajbc,bcij->ai`` (singles residual,
    ccsd.py:433): the operands are unit-stride along different contracted indices; the
    smaller one is re-laid out so that both stream along K -- same numbers."""
    from pymes_b200 import backend as bk
    monkeypatch.setattr(bk, "ALIGN_K_MIN_ELEMENTS", 0)
    rng = np.random.default_rng(11)
    no, nv = 3, 5
    T2 = rng.standard_normal((nv, nv, no, no))
    V = rng.standard_normal((no, no, nv, nv))
    W = rng.standard_normal((nv, no, nv, nv))
    for spec, A, B in (("abjk,jkcb->ac", T2, V), ("ajbc,bcij->ai", W, T2)):
        sa, sb = spec.split("->")[0].split(",")
        a2, A2, b2, B2 = bk._align_k(sa, _t(A), sb, _t(B))
        assert (a2, b2) != (sa, sb)                       # one operand was re-laid out
        ks = set(sa) & set(sb)
        assert bk._unit_index(a2, A2) == bk._unit_index(b2, B2) and bk._unit_index(a2, A2) in ks
        np.testing.assert_allclose(_n(bk.contract(spec, _t(A), _t(B))), np.einsum(spec, A, B), **TOL)
    # nothing to do when one operand's unit-stride index is an output index
    assert bk._align_k("abcd", _t(rng.standard_normal((4, 4, 4, 4))), "cdij", _t(T2[:4, :4]))[0] == "abcd"


def test_matrix_vector_contractions_go_to_gemv(cpu_abi, monkeypatch):
    """The T1 dressing einsums with an o.v^3 block and no output index on T1 (ccsd.py:257-286:
    ``ci,iabc->ab``, ``ci,iacb->ab``, ``jacb,bj->ac``, ``jabc,bj->ac``; singles ``bj,jaib->ai``)
    take the pmb_gemv route: both unit-stride cases, views, alpha/beta accumulation."""
    from pymes_b200 import backend as bk
    monkeypatch.setattr(bk, "GEMV_MIN_ELEMENTS", 0)
    monkeypatch.setattr(bk, "GEMV_MIN_OUTPUTS", 0)
    monkeypatch.setattr(bk, "GEMV_MIN_WARP_OUTPUTS", 0)
    rng = np.random.default_rng(5)
    no, nv = 3, 37
    t1 = rng.standard_normal((nv, no))
    Viabc = rng.standard_normal((no, nv, nv, nv))
    Vfull = rng.standard_normal((no + nv,) * 4)
    called = []
    lib = bk._lib.load()
    orig = lib.pmb_gemv
    monkeypatch.setattr(lib, "pmb_gemv", lambda d, s: (called.append(1), orig(d, s))[1], raising=False)
    for spec, A, B in (("ci,iabc->ab", t1, Viabc), ("ci,iacb->ab", t1, Viabc), ("jacb,bj->ac", Viabc, t1),
                       ("jabc,bj->ac", Viabc, t1), ("bj,jaib->ai", t1, Vfull[:no, no:, :no, no:])):
        n0 = len(called)
        got = bk.contract(spec, _t(A), _t(B))
        assert len(called) == n0 + 1, spec
        np.testing.assert_allclose(_n(got), np.einsum(spec, A, B), **TOL)
    out = _t(rng.standard_normal((nv, nv)))
    want = 0.5 * _n(out) - 2.0 * np.einsum("ci,iabc->ab", t1, Viabc)
    bk.contract("ci,iabc->ab", _t(t1), _t(Viabc), out=out, alpha=-2.0, beta=0.5)
    np.testing.assert_allclose(_n(out), want, **TOL)
    # transposed output view
    outT = _t(np.zeros((nv, nv)))
    bk.contract("ci,iabc->ab", _t(t1), _t(Viabc), out=outT.t())
    np.testing.assert_allclose(_n(outT).T, np.einsum("ci,iabc->ab", t1, Viabc), **TOL)
    # ordinary matrix products are not diverted
    n0 = len(called)
    bk.contract("ab,bc->ac", _t(rng.standard_normal((40, 50))), _t(rng.standard_normal((50, 30))))
    assert len(called) == n0


def test_small_output_side_can_go_to_the_column_group(cpu_abi, monkeypatch):
    """Operand-role swap for contractions whose one output side is a single occupied index (the
    default since round 2; PYMES_B200_SMALL_SIDE_TO_N=0 switches it off)."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(6)
    t1 = rng.standard_normal((17, 5))
    V = rng.standard_normal((17, 17, 17, 5))                 # V_abci-like: a, b, c, j
    want = np.einsum("ci,abcj->abij", t1, V)
    monkeypatch.setattr(bk, "SMALL_SIDE_TO_N", False)
    base, _, _ = bk.describe_contraction("abij", [(1.0, "ci", _t(t1), "abcj", _t(V))])
    assert (base.nm, base.nn) == (1, 3)                      # without it: the unit-stride output index on N
    np.testing.assert_allclose(_n(bk.contract("ci,abcj->abij", _t(t1), _t(V))), want, **TOL)
    monkeypatch.setattr(bk, "SMALL_SIDE_TO_N", True)
    d, _, _ = bk.describe_contraction("abij", [(1.0, "ci", _t(t1), "abcj", _t(V))])
    assert (d.nm, d.nn) == (3, 1)
    np.testing.assert_allclose(_n(bk.contract("ci,abcj->abij", _t(t1), _t(V))), want, **TOL)


def test_ueg_virtual_block_descriptor(cpu_abi):
    """Never-materialised V block as the row operand of a contraction (pmb_term_t.a_gen):
    the descriptor's axis assignment for the pp ladder, a permuted o.v^3 pattern and a row
    block reproduce the contraction with the dense block."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    nP, no = m.n_orb, 7
    nv = nP - no
    W0a, W1a = m.pair_tables("only_non_hermi_2b", m.trunc)
    W0s, _ = m.pair_tables("effect_2b", m.trunc)
    rng = np.random.default_rng(3)
    tau = _t(rng.standard_normal((nv, nv, no, no)))
    virt = m.virtual_block((no,) * 4, (nv,) * 4, W0a=W0a, W1a=W1a, W0s=W0s)
    dense = virt.materialise()
    assert float(dense.abs().max()) > 0
    ref = bk.contract("abcd,cdij->abij", dense, tau)
    got = bk.contract("abcd,cdij->abij", virt, tau)
    np.testing.assert_allclose(_n(got), _n(ref), rtol=0, atol=1e-13)
    d, _, _ = bk.describe_contraction("abij", [(1.0, "abcd", virt, "cdij", tau)])
    g = d._keep[0]
    assert [g.m_axis[i] for i in range(2)] == [1, 0] and [g.k_axis[i] for i in range(2)] == [3, 2]
    # row block of a (what one rank of a sharded run owns), accumulated into an existing R
    part = virt.rows(0, 2, 3)
    R = _t(rng.standard_normal((3, nv, no, no)))
    want = _n(R) + np.einsum("abcd,cdij->abij", _n(dense)[2:5], _n(tau))
    bk.contract_terms("abij", [(1.0, "abcd", part, "cdij", tau)], out=R, beta=1.0)
    np.testing.assert_allclose(_n(R), want, rtol=0, atol=1e-13)
    # o.v^3 block with the occupied index in the row group: "kbcd,cdij->kbij"
    v2 = m.virtual_block((0, no, no, no), (no, nv, nv, nv), W0a=W0a, W1a=W1a, W0s=W0s)
    got = bk.contract("kbcd,cdij->kbij", v2, tau)
    np.testing.assert_allclose(_n(got), np.einsum("kbcd,cdij->kbij", _n(v2.materialise()), _n(tau)),
                               rtol=0, atol=1e-13)
    # formula-evaluating variant (no compressed value table) gives the same numbers
    raw = m.virtual_block((no,) * 4, (nv,) * 4, W0a=W0a, W1a=W1a, W0s=W0s, compressed=False)
    assert raw.nz is None and virt.nz is not None
    np.testing.assert_allclose(_n(bk.contract("abcd,cdij->abij", raw, tau)), _n(ref), rtol=0, atol=1e-13)
    # an output layout that would put the generated operand on the column side: the roles
    # are swapped back (it can only be produced as the row operand)
    outp = bk.empty(no, no, nv, nv).permute(2, 3, 0, 1)
    bk.contract("abcd,cdij->abij", virt, tau, out=outp)
    np.testing.assert_allclose(_n(outp), _n(ref), rtol=0, atol=1e-13)
    # contraction over ONE index of V with a small matrix (T1 dressing "abdc,di->abic")
    t1 = _t(rng.standard_normal((nv, no)))
    np.testing.assert_allclose(_n(bk.contract("abdc,di->abic", virt, t1)),
                               np.einsum("abdc,di->abic", _n(dense), _n(t1)), rtol=0, atol=1e-13)
    np.testing.assert_allclose(_n(bk.einsum("abcd,ci,dj->abij", virt, t1, t1)),
                               np.einsum("abcd,ci,dj->abij", _n(dense), _n(t1), _n(t1)), rtol=0, atol=1e-13)


def test_eom_with_never_materialised_abcd(cpu_abi):
    """EOM-CCSD on a TC-UEG Hamiltonian whose V_abcd exists only as a generated operand: the
    T1-dressed V_abcd becomes an operator (ccsd.DressedLadder) that sigma applies and whose
    (abab) diagonal the FEAST preconditioner reads -- same numbers as with dense blocks."""
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd, eom_ccsd
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    no, nP = 7, m.n_orb
    nv = nP - no
    parts = [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)]
    rng = np.random.default_rng(12)
    fock = _t(np.diag(m.kinetic()) + 1e-3 * rng.standard_normal((nP, nP)))
    dV = m.eval_2b_blocks(no, list(KEYS), parts)
    dVv = dict(dV)
    dVv["abcd"] = m.eval_2b_blocks(no, ["abcd"], parts, virtual=("abcd",))["abcd"]
    T1 = _t(0.05 * rng.standard_normal((nv, no)))
    T2 = _t(0.05 * rng.standard_normal((nv, nv, no, no)))
    cc = ccsd.CCSD(no)
    ft = cc.get_T1_dressed_fock(fock, T1, dV)
    dense = cc.get_T1_dressed_V(T1, dV)
    virt = cc.get_T1_dressed_V(T1, dVv)
    op = virt["abcd"]
    assert isinstance(op, ccsd.DressedLadder)
    for k in dense:                                  # every other block is the same tensor
        if k != "abcd" and dense[k] is not None:
            np.testing.assert_array_equal(_n(virt[k]), _n(dense[k]))
    np.testing.assert_allclose(_n(op.dense()), _n(dense["abcd"]), rtol=0, atol=1e-14)
    np.testing.assert_allclose(_n(op.diag_abab()), np.einsum("abab->ab", _n(dense["abcd"])), rtol=0, atol=1e-14)
    # operator application, single vector and batch, with accumulation
    U = _t(rng.standard_normal((3, nv, nv, no, no)))
    out = _t(rng.standard_normal((3, nv, nv, no, no)))
    want = _n(out) - 0.5 * np.einsum("abcd,rcdij->rabij", _n(dense["abcd"]), _n(U))
    op.apply(U, out, coef=-0.5)
    np.testing.assert_allclose(_n(out), want, rtol=0, atol=1e-12)
    # the whole sigma and the diagonals through the EOM class
    a, b = eom_ccsd.EOM_CCSD(no, n_excit=2), eom_ccsd.EOM_CCSD(no, n_excit=2)
    u1, u2 = _t(rng.standard_normal((nv, no))), _t(rng.standard_normal((nv, nv, no, no)))
    np.testing.assert_allclose(_n(b.update_doubles(ft, virt, u1, u2, T2)), _n(a.update_doubles(ft, dense, u1, u2, T2)),
                               rtol=0, atol=1e-11)
    np.testing.assert_allclose(_n(b.update_singles(ft, virt, u1, u2, T2)), _n(a.update_singles(ft, dense, u1, u2, T2)),
                               rtol=0, atol=1e-11)
    np.testing.assert_allclose(_n(b.get_diag_doubles(ft, virt, T2)), _n(a.get_diag_doubles(ft, dense, T2)),
                               rtol=0, atol=1e-12)
    U1 = _t(rng.standard_normal((2, nv, no)))
    S1a, S2a = a.sigma_batched(ft, dense, U1, U[:2], T2)
    S1b, S2b = b.sigma_batched(ft, virt, U1, U[:2], T2)
    np.testing.assert_allclose(_n(S2b), _n(S2a), rtol=0, atol=1e-11)
    np.testing.assert_allclose(_n(S1b), _n(S1a), rtol=0, atol=1e-11)


# --------------------------------------------------------------------------
# EOM-CCSD: compiled sigma program, batching, diagonals, Davidson
# --------------------------------------------------------------------------
def _dressed(g):
    return {k[8:]: g[k] for k in g.keys() if k.startswith("dressed_")}


@pytest.mark.parametrize("tag", ["a", "b"])
def test_eom_sigma_diag_and_batching(cpu_abi, tag):
    from pymes_b200.solver import eom_ccsd
    from oracle import cc_oracle as oc
    g = golden("dressing_random_" + tag)
    no = int(g["no"])
    dVt, ft, T2 = _dressed(g), g["fock_dressed"], g["T2"]
    eom = eom_ccsd.EOM_CCSD(no, n_excit=2)
    np.testing.assert_allclose(eom.update_singles(ft, dVt, g["u1"], g["u2"], T2), g["sigma1"], **TOL)
    np.testing.assert_allclose(eom.update_doubles(ft, dVt, g["u1"], g["u2"], T2), g["sigma2"], **TOL)
    np.testing.assert_allclose(eom.get_diag_singles(ft, dVt, T2), g["diag1"], **TOL)
    np.testing.assert_allclose(eom.get_diag_doubles(ft, dVt, T2), g["diag2"], **TOL)
    # a batch of right-hand sides in one pass == the oracle vector by vector
    rng = np.random.default_rng(4)
    U1 = rng.standard_normal((3,) + g["u1"].shape)
    U2 = rng.standard_normal((3,) + g["u2"].shape)
    S1, S2 = eom.sigma_batched(ft, dVt, _t(U1), _t(U2), T2)
    for r in range(3):
        np.testing.assert_allclose(_n(S1[r]), oc.eom_sigma_singles(no, ft, dVt, U1[r], U2[r], T2), **TOL)
        np.testing.assert_allclose(_n(S2[r]), oc.eom_sigma_doubles(no, ft, dVt, U1[r], U2[r], T2), **TOL)
    # fewer contractions than the 62 einsum terms of the reference
    plan = eom._plan
    n_groups = sum(len(p["direct"]) + len(p["twostep"]) for p in plan.programs.values())
    assert n_groups <= 30


@pytest.mark.parametrize("tag", ["H2_321g", "LiH_321g"])
def test_eom_davidson_roots(cpu_abi, tag):
    """LiH roots are the constants of pymes/test/test_eom_ccsd/test_eom_ccsd.py:9."""
    from pymes_b200.solver import eom_ccsd, ccsd
    from pymes_b200.integral.partition import part_2_body_int
    g = golden("mol_" + tag)
    no = int(g["n_elec"]) // 2
    cc = ccsd.CCSD(no)
    dV = part_2_body_int(no, g["V"])
    ft = cc.get_T1_dressed_fock(g["fock"], g["ccsd_t1"], dV)
    dVt = cc.get_T1_dressed_V(g["ccsd_t1"], dV)
    eom = eom_ccsd.EOM_CCSD(no, n_excit=len(g["eom_e"]))
    eom.max_iter = 1000
    e = eom.solve(ft, dVt, g["ccsd_t2"])
    np.testing.assert_allclose(e, g["eom_e"], rtol=0, atol=1e-8)
    if tag == "LiH_321g":
        assert np.allclose(e, [0.1180867117168979, 0.154376205595602])
    q1, q2 = eom.QR([g["ccsd_t1"], 2 * g["ccsd_t1"] + 1.0], [g["ccsd_t2"], g["ccsd_t2"] ** 2])
    gram = [[np.vdot(q1[a], q1[b]) + np.vdot(q2[a], q2[b]) for b in range(2)] for a in range(2)]
    np.testing.assert_allclose(gram, np.eye(2), atol=1e-13)


# --------------------------------------------------------------------------
# FEAST-EOM-CCSD: batched shifted linear solves and the contour iteration
# --------------------------------------------------------------------------
def _feast_inputs():
    from pymes_b200.solver import ccsd
    from pymes_b200.integral.partition import part_2_body_int
    g, m = golden("feast_LiH"), golden("mol_LiH_321g")
    no = 2
    cc = ccsd.CCSD(no)
    dV = part_2_body_int(no, m["V"])
    ft = cc.get_T1_dressed_fock(m["fock"], g["t1"], dV)
    dVt = cc.get_T1_dressed_V(g["t1"], dV)
    return g, no, ft, dVt


def test_feast_linear_solve_matches_reference_gcrot(cpu_abi):
    """One (z - H-bar) Q = u solve against the reference's scipy GCROT(m,k) result
    (feast_eom_ccsd.py:293-350, tol 1e-4): the lock-step GCROT(m,k) runs the same first cycle of
    m + k = 40 flexible-GMRES steps -> the same iterate, to rounding."""
    from pymes_b200.solver import feast_eom_ccsd
    g, no, ft, dVt = _feast_inputs()
    fe = feast_eom_ccsd.FEAST_EOM_CCSD(no, e_c=float(g["e_c"]), e_r=float(g["e_r"]), n_trial=2, max_iter=3)
    d1, d2 = fe.get_diag_singles(ft, dVt, g["t2"]), fe.get_diag_doubles(ft, dVt, g["t2"])
    np.testing.assert_allclose(d1, g["diag1"], **TOL)
    np.testing.assert_allclose(d2, g["diag2"], **TOL)
    fe.u_singles, fe.u_doubles = [g["u1"].copy()], [g["u2"].copy()]
    q1, q2 = fe._gcrotmk(0, complex(g["z"]), d1, d2, ft, dVt, g["t2"])
    assert fe.ls_residuals[0] < 1e-4
    nrm = np.sqrt(np.sum(abs(g["q1"]) ** 2) + np.sum(abs(g["q2"]) ** 2))
    err = np.sqrt(np.sum(abs(q1 - g["q1"]) ** 2) + np.sum(abs(q2 - g["q2"]) ** 2)) / nrm
    assert err < 1e-10, err


def test_feast_gcrot_matches_scipy_over_many_cycles(cpu_abi):
    """The lock-step GCROT(m,k) of ``FEAST_EOM_CCSD._solve_group`` against scipy's ``gcrotmk`` (the
    solver the reference calls, feast_eom_ccsd.py:346; scipy is the checker here) on systems that
    need MANY outer cycles (m = k = 3 and 5: recycling of (c, u) pairs, truncation of the oldest,
    projection off C inside the inner cycles): same iterate to 1e-10 relative, same number of
    operator applications; two systems advanced together."""
    from scipy.sparse import diags
    from scipy.sparse.linalg import LinearOperator, gcrotmk
    from pymes_b200.solver import feast_eom_ccsd
    g, no, ft, dVt = _feast_inputs()
    fe = feast_eom_ccsd.FEAST_EOM_CCSD(no, e_c=0.13, e_r=0.05, n_trial=2, max_iter=3)
    plan = fe.plan(ft, dVt, g["t2"])
    diag = np.concatenate([g["diag1"].ravel(), g["diag2"].ravel()])
    n = diag.size
    Hb = np.zeros((n, n))                       # dense H-bar: sigma of the unit vectors
    for lo in range(0, n, 64):
        E = np.zeros((min(64, n - lo), n))
        E[np.arange(E.shape[0]), lo + np.arange(E.shape[0])] = 1.0
        Hb[:, lo:lo + E.shape[0]] = _n(plan.apply_packed(_t(E))).T
    rng = np.random.default_rng(3)
    for m, tol, z in ((3, 1e-9, 0.13 + 0.05j), (5, 1e-8, 0.15 + 0.02j), (20, 1e-4, 0.13 + 0.05 * np.exp(0.7j))):
        b1, b2 = rng.standard_normal(n), rng.standard_normal(n)
        fe.ls_restart, fe.ls_tol, fe.ls_max_iter, fe.ls_matvecs = m, tol, 200, 0
        sol = fe.solve_shifted_systems(plan, _t(diag), [z, z.conjugate()], [_t(b1), _t(b2)])
        assert max(fe.ls_residuals) <= tol
        count = [0]
        for zz, b, s_ in ((z, b1, sol[0]), (z.conjugate(), b2, sol[1])):
            def mv(v, zz=zz):
                count[0] += 1
                return zz * v - Hb @ v
            A = LinearOperator((n, n), matvec=mv, dtype=complex)
            xs, info = gcrotmk(A, b.astype(complex), x0=np.zeros(n, dtype=complex), M=diags(1.0 / (zz - diag + 0.01)),
                               maxiter=200, rtol=tol, m=m)
            assert info == 0
            x = _n(s_.re) + 1j * _n(s_.im)
            assert np.linalg.norm(x - xs) < 1e-10 * np.linalg.norm(xs), (m, tol)
        # scipy applies the operator once more per system: r0 = b - A x0 with x0 = 0
        assert fe.ls_matvecs == count[0] - 2, (fe.ls_matvecs, count[0])


def test_feast_batched_systems_and_seeded_iteration(cpu_abi):
    from pymes_b200.solver import feast_eom_ccsd
    from pymes_b200 import backend as bk
    from oracle import cc_oracle as oc
    g, no, ft, dVt = _feast_inputs()
    fe = feast_eom_ccsd.FEAST_EOM_CCSD(no, e_c=0.13, e_r=0.05, n_trial=2, max_iter=3)
    plan = fe.plan(ft, dVt, g["t2"])
    nv = plan.nv
    diag = np.concatenate([g["diag1"].ravel(), g["diag2"].ravel()])
    rng = np.random.default_rng(2)
    zs = [0.13 + 0.05 * np.exp(1j * t) for t in (0.3, 1.1, 2.5)] * 2
    rhs = [rng.standard_normal(diag.size) for _ in range(6)]
    fe.ls_tol = 1e-9
    sol = fe.solve_shifted_systems(plan, _t(diag), zs, [_t(b) for b in rhs])
    n1 = nv * no
    dVn = {k: np.asarray(v) for k, v in dVt.items() if v is not None}
    for z, b, s in zip(zs, rhs, sol):
        x = _n(s.re) + 1j * _n(s.im)
        x1, x2 = x[:n1].reshape(nv, no), x[n1:].reshape(nv, nv, no, no)
        hx = np.concatenate([oc.eom_sigma_singles(no, ft, dVn, x1, x2, g["t2"]).ravel(),
                             oc.eom_sigma_doubles(no, ft, dVn, x1, x2, g["t2"]).ravel()])
        assert np.linalg.norm(z * x - hx - b) < 1e-8 * np.linalg.norm(b)
    # seeded 3-iteration FEAST run of the golden generator (np.random.seed(5), feast:89-91)
    np.random.seed(5)
    fe2 = feast_eom_ccsd.FEAST_EOM_CCSD(no, e_c=0.13, e_r=0.05, n_trial=2, max_iter=3)
    ev = fe2.solve(ft, dVt, g["t2"])
    # EOM eigenvalues within 1e-8 Eh of the reference's (north_star); measured: 5e-14
    np.testing.assert_allclose(np.sort(ev.real), np.sort(g["eigvals"].real), rtol=0, atol=1e-9)
    assert np.abs(ev.imag).max() < 1e-8
    x, w = feast_eom_ccsd.get_gauss_legendre_quadrature(8)
    assert abs(w.sum() - 2.0) < 1e-14


# --------------------------------------------------------------------------
# RT-EOM-CCSD: one contour-integral propagation step (SURVEY 8(f).3)
# --------------------------------------------------------------------------
def test_rt_eom_step_matches_reference(cpu_abi):
    """Two consecutive RT-EOM-CCSD steps (real start state, then the complex result) against the
    reference run of tests/golden/make_golden.py::sec_rt.  Both sides stop their linear solves at
    a relative residual of 1e-4 (gcrotmk tol, feast_eom_ccsd.py:346) -- and, since the lock-step
    solver is the same GCROT(m,k), at the same iterate: the propagated states agree to round-off
    (measured 7e-15), far inside the solver tolerance."""
    from pymes_b200.integral.partition import part_2_body_int
    from pymes_b200.solver import ccsd, rt_eom_ccsd
    g, m = golden("rt_LiH"), golden("mol_LiH_321g")
    no = int(m["n_elec"]) // 2
    cc = ccsd.CCSD(no)
    dV = part_2_body_int(no, m["V"])
    ft = cc.get_T1_dressed_fock(m["fock"], g["t1"], dV)
    dVt = cc.get_T1_dressed_V(g["t1"], dV)
    rt = rt_eom_ccsd.RT_EOM_CCSD(no, e_c=float(g["e_c"]), e_r=float(g["e_r"]), dt=float(g["dt"]))

    def err(a1, a2, b1, b2):
        return np.sqrt(np.sum(abs(a1 - b1) ** 2) + np.sum(abs(a2 - b2) ** 2))   # states have norm 1

    q1, q2 = rt.solve(ft, dVt, g["t2"], dt=float(g["dt"]), u_singles=g["u1"].copy(), u_doubles=g["u2"].copy())
    assert max(rt.ls_residuals) < 1e-4
    assert abs(np.sum(abs(q1) ** 2) + np.sum(abs(q2) ** 2) - 1.0) < 1e-12
    assert err(q1, q2, g["q1"], g["q2"]) < 1e-10
    p1, p2 = rt.solve(ft, dVt, g["t2"], dt=float(g["dt"]), u_singles=g["q1"].copy(), u_doubles=g["q2"].copy())
    assert err(p1, p2, g["p1"], g["p2"]) < 1e-10
    # independent check: the contour integral is exp(i H dt) restricted to the eigenvalues of H-bar
    # inside |lambda - e_c| < e_r (an 8-node quadrature of the Cauchy formula); with converged linear
    # solves the step must reproduce the quadrature of the dense resolvent exactly
    nv = g["t2"].shape[0]
    n = nv * no + nv * nv * no * no
    plan = rt.plan(ft, dVt, g["t2"])
    H = _n(plan.apply_packed(_t(np.eye(n)))).T
    y = np.concatenate([g["u1"].ravel(), g["u2"].ravel()])
    dt, e_c, e_r = float(g["dt"]), float(g["e_c"]), float(g["e_r"])
    x, w = np.polynomial.legendre.leggauss(8)
    theta = -np.pi * x
    z = (e_c * 1j + e_r * np.exp(1j * theta)) * dt
    dense = np.zeros(n, dtype=complex)
    for e in range(8):
        dense -= w[e] / 2 * e_r * dt * np.exp(1j * theta[e]) * np.linalg.solve(z[e] * np.eye(n) - 1j * dt * H,
                                                                               np.exp(z[e]) * y)
    dense /= np.linalg.norm(dense)
    got = np.concatenate([q1.ravel(), q2.ravel()])
    ref = np.concatenate([g["q1"].ravel(), g["q2"].ravel()])
    print("RT step vs dense resolvent quadrature: ours %.2e, reference %.2e; ours - reference %.2e"
          % (np.linalg.norm(got - dense), np.linalg.norm(ref - dense), np.linalg.norm(got - ref)))
    assert np.linalg.norm(got - dense) < 5e-4
    rt.ls_tol, rt.ls_restart = 1e-11, 200        # (restarted GMRES(20) stagnates on the node nearest an eigenvalue)
    t1, t2 = rt.solve(ft, dVt, g["t2"], dt=dt, u_singles=g["u1"].copy(), u_doubles=g["u2"].copy())
    tight = np.concatenate([t1.ravel(), t2.ravel()])
    print("RT step, converged solves, vs dense resolvent quadrature: %.2e" % np.linalg.norm(tight - dense))
    assert np.linalg.norm(tight - dense) < 1e-8


# --------------------------------------------------------------------------
# synthetic non-hermitian integrals (BASELINE configs[2]) -- counter-based, block-wise
# --------------------------------------------------------------------------
def test_synthetic_tc_integrals_blockwise_and_ccsd(cpu_abi):
    """util.synthetic: only the (pq)(rs)<->(qp)(sr) symmetry, N(0,1) statistics, any block equals
    the slice of the dense tensor, and CCSD / DCSD on the generated blocks follow the oracle
    sweep by sweep (non-hermitian: V != V^T, no hermiticity shortcut survives)."""
    from pymes_b200.integral.partition import KEYS, part_2_body_int
    from pymes_b200.solver import ccsd
    from pymes_b200.util import synthetic
    from oracle import cc_oracle as oc
    no, nv = 4, 9
    n = no + nv
    V = synthetic.tc_integrals(n, seed=0)
    np.testing.assert_array_equal(V, V.transpose(1, 0, 3, 2))
    assert np.abs(V - V.transpose(2, 3, 0, 1)).max() > 1e-4          # not hermitian
    assert np.abs(V - V.transpose(0, 1, 3, 2)).max() > 1e-4
    big = synthetic.normal_from_index(7, np.arange(200000))
    assert abs(big.mean()) < 0.01 and abs(big.std() - 1.0) < 0.01 and np.abs(big).max() < 6.5
    assert not np.array_equal(synthetic.tc_integrals(n, seed=1), V)
    blocks = synthetic.tc_blocks(no, nv, KEYS, seed=0)
    dense = part_2_body_int(no, V)
    for key in KEYS:
        np.testing.assert_array_equal(blocks[key], dense[key])
    rows = synthetic.tc_blocks(no, nv, ["abcd"], seed=0, ranges={"abcd": {0: (no + 2, 3)}})["abcd"]
    np.testing.assert_array_equal(rows, dense["abcd"][2:5])
    # the device writer (pmb_synth_block) produces the very same doubles, block by block
    dev = synthetic.tc_blocks(no, nv, KEYS, seed=0, device=True)
    for key in KEYS:
        assert np.array_equal(_n(dev[key]), dense[key]), key
    drows = synthetic.tc_blocks(no, nv, ["iabc"], seed=3, ranges={"iabc": {1: (no + 1, 4)}}, device=True)["iabc"]
    assert np.array_equal(_n(drows), synthetic.tc_blocks(no, nv, ["iabc"], seed=3)["iabc"][:, 1:5])
    fock = synthetic.tc_fock(no, nv, seed=0)
    assert np.abs(fock - fock.T).max() > 1e-5
    for is_dcsd in (False, True):
        cc = ccsd.CCSD(no, is_dcsd=is_dcsd)
        cc.setup(fock, {k: _t(v) for k, v in blocks.items()})
        dVo = oc.partition(no, V)
        eps_i, eps_a = fock.diagonal()[:no].copy(), fock.diagonal()[no:].copy()
        _, T2 = oc.mp2(eps_i, eps_a, dVo["ijab"], dVo["abij"])
        T1 = np.zeros((nv, no))
        d1, d2 = oc.denominators(eps_i, eps_a)
        mixer = oc.DIIS(6)
        for _ in range(6):
            T1, T2, eo, _dt = oc.ccsd_sweep(no, fock, dVo, T1, T2, d1, d2, mixer, is_dcsd=is_dcsd)
            e = cc.sweep()
            assert abs(sum(e[:3]) - sum(eo)) < 1e-12
            assert np.abs(_n(cc._st["T2"]) - T2).max() < 1e-9 * np.abs(T2).max()
            assert np.abs(_n(cc._st["T1"]) - T1).max() < 1e-9 * np.abs(T1).max()


# --------------------------------------------------------------------------
# SURVEY 8(f).2: the is_dr_ccd / is_bruekner branches, reproduced as the reference executes them
# (fixtures: tests/golden/ccd_variants.npz, made by running the reference)
# --------------------------------------------------------------------------
VARIANTS = [("drccd", dict(is_dr_ccd=True), 4), ("drccd_nodiis", dict(is_dr_ccd=True, is_diis=False), 4),
            ("bruekner", dict(is_bruekner=True), 2), ("bruekner_nodiis", dict(is_bruekner=True, is_diis=False), 2),
            ("bruekner_dcd", dict(is_bruekner=True, is_dcd=True), 2)]


def test_drccd_residual_matches_reference(cpu_abi):
    from pymes_b200.solver import drccd
    g = golden("ccd_variants")
    R = drccd.get_residual(g["rnd_eps_i"], g["rnd_eps_a"], g["rnd_T2"], g["rnd_abij"], g["rnd_aijb"],
                           g["rnd_iabj"], g["rnd_ijab"])
    np.testing.assert_allclose(R, g["rnd_R_drccd"], rtol=1e-12, atol=1e-12)
    e = drccd.getEnergy(g["rnd_T2"], g["rnd_ijab"])
    assert abs(e[0] - 2.0 * np.einsum("abij,ijab->", g["rnd_T2"], g["rnd_ijab"])) < 1e-12 and e[1] == 0.


@pytest.mark.parametrize("tag", ["LiH", "LiHtc"])
@pytest.mark.parametrize("name,kw,sweeps", VARIANTS)
def test_ccd_variants_match_reference(cpu_abi, tag, name, kw, sweeps):
    """Energies, amplitudes, quasi-particle energies and -- for is_bruekner -- the Fock matrix the
    reference leaves modified, after the same number of sweeps (relative: the Brueckner branch
    diverges to O(10) Eh in the reference itself)."""
    from pymes_b200.solver import ccd
    g = golden("ccd_variants")
    no, V, key = int(g[tag + "_no"]), g[tag + "_V"], tag + "_" + name
    fock = g[tag + "_fock"].copy()
    cc = ccd.CCD(no, **kw)
    r = cc.solve(fock, V, max_iter=sweeps - 1, delta_e=1e-14)
    assert cc.iterations == sweeps
    assert abs(r["ccd e"] - g[key + "_e"]) <= 1e-10 * max(1.0, abs(g[key + "_e"]))
    scale = np.abs(g[key + "_t2"]).max()
    assert np.abs(r["t2 amp"] - g[key + "_t2"]).max() <= 1e-9 * scale
    np.testing.assert_allclose(r["hole e"], g[key + "_hole"], rtol=1e-10, atol=1e-11)
    np.testing.assert_allclose(r["particle e"], g[key + "_particle"], rtol=1e-10, atol=1e-11)
    np.testing.assert_allclose(fock, g[key + "_fock_after"], rtol=1e-10, atol=1e-11)
    assert abs(r["dE"] - g[key + "_dE"]) <= 1e-10 * max(1.0, abs(g[key + "_dE"]))


def test_ccd_rejects_non_contiguous_amps(cpu_abi):
    from pymes_b200.solver import ccd
    g = golden("ccd_variants")
    no, V, fock = int(g["LiH_no"]), g["LiH_V"], g["LiH_fock"]
    nv = fock.shape[0] - no
    amps = _t(np.zeros((nv, nv, no, no))).permute(1, 0, 2, 3)[:, :, :, ::1].transpose(2, 3)
    with pytest.raises(ValueError, match="contiguous"):
        ccd.CCD(no).solve(_t(fock), _t(V), amps=amps, max_iter=0)


def test_dots_and_lincomb_beyond_16_vectors(cpu_abi):
    """The C entry points take at most 16 vectors per call (a 10-root Davidson subspace holds 40):
    the wrappers split longer lists."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(2)
    X = rng.standard_normal((37, 50))
    y = rng.standard_normal(50)
    c = rng.standard_normal(37)
    xs = [_t(x) for x in X]
    np.testing.assert_allclose(_n(bk.dots(xs, _t(y))), X @ y, rtol=1e-13)
    np.testing.assert_allclose(_n(bk.lincomb(list(c), xs)), c @ X, rtol=1e-13, atol=1e-13)


# --------------------------------------------------------------------------
# eval_2b_integrals: the remaining branches and every correlator (fixtures: ueg_modes*.npz)
# --------------------------------------------------------------------------
UEG_FLAGS = ["is_rpa_approx", "is_only_hermi_2b", "is_only_non_hermi_2b", "is_exchange_1", "is_exchange_2",
             "is_exchange_3"]
UEG_CORRELATORS = [("trunc", None, 1.0), ("coulomb", None, None), ("smooth", None, 1.0), ("yukawa", None, None),
                   ("yukawa", 0.7, 1.0), ("stg", None, None), ("stg", 1.3, 1.0), ("yukawa_coulomb", None, None),
                   ("yukawa_coulomb", 1.1, 1.0), ("gaskell", None, None), ("gaskell", 0.9, 2.0),
                   ("gaskell_modified", None, None), ("gaskell_modified", None, 1.0)]


@pytest.mark.parametrize("flag", UEG_FLAGS)
def test_ueg_remaining_branches_match_reference(cpu_abi, flag):
    """ueg.py:416-423, 440-457, 478-504 with `trunc` at 14e / 57 plane waves against the reference's
    triple loop.  On the CPU emulator a slab of rows, on the GPU the whole tensor."""
    from pymes_b200.model import ueg
    g = golden("ueg_modes_branches")
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(5.0)
    m.gamma, m.k_cutoff = None, 1.0
    nP = m.n_orb
    np.testing.assert_array_equal(m.k_int(), g["big_kint"])
    ref = _dense(g["big_" + flag + "_idx"], g["big_" + flag + "_val"], nP)
    scale = np.abs(ref).max()
    if DEVICE == "cuda":
        V = m.eval_2b_integrals(correlator=m.trunc, sp=0, **{flag: True})
        assert np.abs(V - ref).max() <= 1e-11 * scale
        zero = m.eval_2b_integrals(correlator=m.trunc, sp=0)            # no branch selected: zeros
        assert np.abs(zero).max() == 0.0 == float(g["big_noflag_absmax"])
    else:
        mode = "rpa" if flag == "is_rpa_approx" else flag[3:]
        W0, W1 = m.pair_tables(mode, m.trunc)
        blk = m.build_block((2, 0, 11, 0), (3, nP, 4, nP), W0a=W0, W1a=W1)
        assert np.abs(_n(blk) - ref[2:5, :, 11:15, :]).max() <= 1e-11 * scale


# Correlators that compare k^2 with a cutoff WITHOUT a guard band (yukawa / stg / yukawa_coulomb with
# k_cutoff, gaskell, gaskell_modified): when the cutoff is exactly the squared length of a lattice
# shell ((2 pi/L)^2 for k_cutoff = 1; 4 k_F^2 = 8 (2 pi/L)^2 for gaskell at 14 electrons) the reference's
# answer is decided by the rounding of ITS k-vector differences.  For these the pair tables are
# formed with the reference's own floating-point arguments (UEG._pair_tables_exact); a table over
# the integer |k|^2 -- what `trunc` (guard band 1 + 1e-5, ueg.py:793) may use -- would put a whole
# shell on one side (seen before the exact path existed: 1e-3 relative in u_mat for yukawa / stg).


@pytest.mark.parametrize("name,gamma,k_cutoff", UEG_CORRELATORS)
def test_ueg_every_correlator_matches_reference(cpu_abi, name, gamma, k_cutoff):
    """Each correlator of ueg.py:740-956 (default and explicit gamma / k_cutoff) through the
    `only_2b` and `effect_2b` branches at 14e / 19 plane waves, whole tensor, and the values the
    correlator leaves in ``gamma`` / ``k_cutoff``."""
    from pymes_b200.model import ueg
    g = golden("ueg_modes")
    tag = "c_%s_g%s_k%s" % (name, gamma, k_cutoff)
    for flag in ("is_only_2b", "is_effect_2b"):
        m = ueg.UEG(14, 7, 7, 1.0)
        m.init_single_basis(2.0)
        m.gamma, m.k_cutoff = gamma, k_cutoff
        nP = m.n_orb
        np.testing.assert_array_equal(m.k_int(), g["small_kint"])
        V = m.eval_2b_integrals(correlator=getattr(m, name), sp=0, **{flag: True})
        ref = _dense(g[tag + "_" + flag + "_idx"], g[tag + "_" + flag + "_val"], nP)
        assert np.abs(V - ref).max() <= 1e-10 * max(np.abs(ref).max(), 1e-300), flag
    ga, kc = float(g[tag + "_gamma_after"]), float(g[tag + "_kc_after"])
    assert (m.gamma is None and np.isnan(ga)) or m.gamma == ga
    assert (m.k_cutoff is None and np.isnan(kc)) or m.k_cutoff == kc


def test_trunc_mutates_its_array_argument_like_the_reference():
    """ueg.py:797 zeroes the small entries of the caller's array in place."""
    from pymes_b200.model import ueg
    g = golden("ueg_modes")
    m = ueg.UEG(14, 7, 7, 1.0)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    arg = np.linspace(0.0, 3.0, 13)
    res = m.trunc(arg)
    np.testing.assert_array_equal(arg, g["trunc_arg_after"])
    np.testing.assert_allclose(res, g["trunc_res"], rtol=1e-15)
    assert m.trunc(0.2) == 0.0 and m.trunc(10.0) == -4.0 * np.pi / 100.0


def test_davidson_diagonal_preconditioner_finds_eigenvalues(cpu_abi):
    """Extension: EOM_CCSD.preconditioner = "diagonal" (r / (e - diag(H-bar) + 1e-5) instead of the
    reference's one-number-per-root scaling, eom_ccsd.py:140).  Its roots are eigenvalues of the dense
    H-bar (built column by column through the same sigma), the lowest one is the reference's, and it
    may find LOWER further roots than the reference's iteration does (H2/3-21G: 0.4801 instead of 1.1646,
    both eigenvalues: the singles-only start vectors of eom_ccsd.py:76-82 never reach the state)."""
    from pymes_b200.integral.partition import part_2_body_int
    from pymes_b200.solver import ccsd, eom_ccsd
    for tag in ("LiH_321g", "H2_321g"):
        g = golden("mol_" + tag)
        no = int(g["n_elec"]) // 2
        dV = part_2_body_int(no, _t(g["V"]))
        cc = ccsd.CCSD(no)
        T1, T2, fock = _t(g["ccsd_t1"]), _t(g["ccsd_t2"]), _t(g["fock"])
        ft = cc.get_T1_dressed_fock(fock, T1, dV)
        dVt = cc.get_T1_dressed_V(T1, dV)
        roots = {}
        for kind in ("scalar", "diagonal"):
            eom = eom_ccsd.EOM_CCSD(no, n_excit=len(g["eom_e"]))
            eom.preconditioner = kind
            roots[kind] = np.sort(eom.solve(ft, dVt, T2))
        np.testing.assert_allclose(roots["scalar"], np.sort(g["eom_e"]), rtol=0, atol=1e-8)
        plan = eom.plan(ft, dVt, T2)
        nv = T2.shape[0]
        n = nv * no + nv * nv * no * no
        H = _n(plan.apply_packed(_t(np.eye(n)))).T
        ev = np.linalg.eigvals(H)
        for r in roots["diagonal"]:
            assert np.abs(ev - r).min() < 1e-7, (tag, r)
        assert abs(roots["diagonal"][0] - roots["scalar"][0]) < 1e-7
        assert np.all(roots["diagonal"] <= roots["scalar"] + 1e-7)


def test_stacked_rows_and_even_pitch_helpers(cpu_abi):
    """backend.empty_stacked / stacked_rows (two blocks as one operand) and empty_even_pitch (16-byte
    aligned (i,j) rows): the views alias the right memory, and the negative cases are refused."""
    from pymes_b200 import backend as bk
    no, nb, nv = 3, 4, 5
    A, B = bk.empty_stacked((no, nb, nv, nv), (nb, no, nv, nv))
    A.copy_(_t(np.arange(A.numel(), dtype=float).reshape(A.shape)))
    B.copy_(_t(-np.arange(B.numel(), dtype=float).reshape(B.shape)))
    st = bk.stacked_rows(A, B, (nv, nv))
    assert tuple(st.shape) == (2, no * nb, nv, nv)
    assert torch.equal(st[0].reshape(-1), A.reshape(-1)) and torch.equal(st[1].reshape(-1), B.reshape(-1))
    tau = _t(np.random.default_rng(0).standard_normal((nv, nv, 2, 2)))
    W = bk.contract("grcd,cdij->grij", st, tau)
    np.testing.assert_allclose(_n(W[0]).reshape(no, nb, 2, 2), np.einsum("kbcd,cdij->kbij", _n(A), _n(tau)), **TOL)
    np.testing.assert_allclose(_n(W[1]).reshape(nb, no, 2, 2), np.einsum("alcd,cdij->alij", _n(B), _n(tau)), **TOL)
    assert bk.stacked_rows(A, B.clone(), (nv, nv)) is None              # not adjacent
    assert bk.stacked_rows(B, A, (nv, nv)) is None                      # wrong order
    assert bk.stacked_rows(A, B, (nv, nv + 1)) is None                  # other contracted shape
    with pytest.raises(ValueError):
        bk.empty_stacked((2, 3), (4, 2))
    for o in (3, 4):                                                   # o^2 odd -> one pad double; even -> none
        t = bk.empty_even_pitch(5, 6, o)
        assert tuple(t.shape) == (5, 6, o, o) and t.stride(1) % 2 == 0 and t.stride(3) == 1 and t.stride(2) == o
        assert t.stride(1) == o * o + (o * o) % 2


def test_momentum_blocked_contraction_host_logic(cpu_abi):
    """``pmb_blocked_contract`` dispatch (SURVEY 8(f).1, the momentum-blocked path): the group /
    tile lists of a VirtualBlock, the offset tables for several operand layouts (even-pitch tau,
    batched right-hand sides, a row block, the o.v^3 pattern), the mixed call with a dense term,
    beta = 0 on rows without any group, and the switch back to the dense generated-operand path."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    nP, no = m.n_orb, 7
    nv = nP - no
    W0a, W1a = m.pair_tables("only_non_hermi_2b", m.trunc)
    W0s, _ = m.pair_tables("effect_2b", m.trunc)
    rng = np.random.default_rng(5)
    virt = m.virtual_block((no,) * 4, (nv,) * 4, W0a=W0a, W1a=W1a, W0s=W0s)
    dense = _n(virt.materialise())
    L = virt.blocked_lists()
    # the lists describe exactly the non-zero structure of the dense block
    assert L["nnz"] >= np.count_nonzero(dense) > 0
    tiles = _n(L["tiles"])
    assert tiles[:, 1].max() <= 64 and (np.diff(tiles[:, 3]) <= 0).all()
    covered = np.zeros((nv * nv, nv * nv), dtype=bool)
    rows = L["row_i0"] * nv + L["row_i1"]
    ents = L["ent_j0"] * nv + L["ent_j1"]
    for m0, mn, k0, kn in tiles:
        covered[np.ix_(rows[m0:m0 + mn], ents[k0:k0 + kn])] = True
    assert not (dense.reshape(nv * nv, -1) != 0)[~covered].any()
    assert covered.sum() == L["nnz"]

    calls = {"blocked": 0, "dense": 0}
    blocked0, dense0 = cpu_abi.pmb_blocked_contract, cpu_abi.pmb_contract
    cpu_abi.pmb_blocked_contract = lambda *a: (calls.__setitem__("blocked", calls["blocked"] + 1), blocked0(*a))[1]
    cpu_abi.pmb_contract = lambda *a: (calls.__setitem__("dense", calls["dense"] + 1), dense0(*a))[1]

    # even-pitch tau (the ladder's operand in ccsd.tau_ladder), accumulate into R
    tau = bk.empty_even_pitch(nv, nv, no)
    tau.copy_(_t(rng.standard_normal((nv, nv, no, no))))
    R0 = rng.standard_normal((nv, nv, no, no))
    R = _t(R0.copy())
    bk.contract_terms("abij", [(0.7, "abcd", virt, "cdij", tau)], out=R, beta=1.0)
    np.testing.assert_allclose(_n(R), R0 + 0.7 * np.einsum("abcd,cdij->abij", dense, _n(tau)), rtol=0, atol=1e-13)
    assert calls == {"blocked": 1, "dense": 0}
    # fresh output (beta = 0): rows of momentum groups without entries come out as zeros
    got = bk.contract("abcd,cdij->abij", virt, tau)
    np.testing.assert_allclose(_n(got), np.einsum("abcd,cdij->abij", dense, _n(tau)), rtol=0, atol=1e-13)
    junk = _t(rng.standard_normal((nv, nv, no, no)))
    bk.contract("abcd,cdij->abij", virt, tau, out=junk)
    np.testing.assert_allclose(_n(junk), _n(got), rtol=0, atol=0)
    assert calls == {"blocked": 3, "dense": 0}
    # batched right-hand sides (EOM sigma, ccsd.DressedLadder.apply)
    U = _t(rng.standard_normal((3, nv, nv, no, no)))
    S = _t(np.zeros((3, nv, nv, no, no)))
    bk.contract_terms("rabij", [(-1.0, "abcd", virt, "rcdij", U)], out=S, beta=1.0)
    np.testing.assert_allclose(_n(S), -np.einsum("abcd,rcdij->rabij", dense, _n(U)), rtol=0, atol=1e-13)
    assert calls == {"blocked": 4, "dense": 0}
    # a row block (one rank of a sharded run) and the o.v^3 pattern with an occupied row index
    part = virt.rows(0, 2, 3)
    got = bk.contract("abcd,cdij->abij", part, tau)
    np.testing.assert_allclose(_n(got), np.einsum("abcd,cdij->abij", dense[2:5], _n(tau)), rtol=0, atol=1e-13)
    v2 = m.virtual_block((0, no, no, no), (no, nv, nv, nv), W0a=W0a, W1a=W1a, W0s=W0s)
    got = bk.contract("kbcd,cdij->kbij", v2, tau)
    np.testing.assert_allclose(_n(got), np.einsum("kbcd,cdij->kbij", _n(v2.materialise()), _n(tau)),
                               rtol=0, atol=1e-13)
    v3 = m.virtual_block((no, 0, no, no), (nv, no, nv, nv), W0a=W0a, W1a=W1a, W0s=W0s)
    got = bk.contract("alcd,cdij->alij", v3, tau)
    np.testing.assert_allclose(_n(got), np.einsum("alcd,cdij->alij", _n(v3.materialise()), _n(tau)),
                               rtol=0, atol=1e-13)
    assert calls == {"blocked": 7, "dense": 0}
    # mixed call: the hole-hole ladder keeps the dense kernel, the pp ladder is blocked (ccd.py:185-187)
    I = _t(rng.standard_normal((no, no, no, no)))
    T2 = _t(rng.standard_normal((nv, nv, no, no)))
    R = _t(R0.copy())
    bk.contract_terms("abij", [(1.0, "abkl", T2, "klij", I), (1.0, "abcd", virt, "cdij", T2)], out=R, beta=1.0)
    want = R0 + np.einsum("abkl,klij->abij", _n(T2), _n(I)) + np.einsum("abcd,cdij->abij", dense, _n(T2))
    np.testing.assert_allclose(_n(R), want, rtol=0, atol=1e-13)
    assert calls == {"blocked": 8, "dense": 1}
    # a column layout the blocked kernel does not take (output with (i,j) outermost): dense path
    outp = bk.empty(no, no, nv, nv).permute(2, 3, 0, 1)
    bk.contract("abcd,cdij->abij", virt, tau, out=outp)
    np.testing.assert_allclose(_n(outp), np.einsum("abcd,cdij->abij", dense, _n(tau)), rtol=0, atol=1e-13)
    assert calls == {"blocked": 8, "dense": 2}
    # switched off: the generated-operand path of pmb_contract
    old = bk.set_blocked(False)
    try:
        got = bk.contract("abcd,cdij->abij", virt, tau)
    finally:
        bk.set_blocked(old)
    np.testing.assert_allclose(_n(got), np.einsum("abcd,cdij->abij", dense, _n(tau)), rtol=0, atol=1e-13)
    assert calls == {"blocked": 8, "dense": 3} and bk.blocked_enabled()
    # an operand without compressed values has no lists
    raw = m.virtual_block((no,) * 4, (nv,) * 4, W0a=W0a, W1a=W1a, W0s=W0s, compressed=False)
    assert raw.blocked_lists() is None
    bk.contract("abcd,cdij->abij", raw, tau)
    assert calls == {"blocked": 8, "dense": 4}


def test_momentum_groups_follow_the_reference_index_lookup():
    """The groups of ``momentum_groups`` are exactly the (p,q,r,s) the reference's index lookup can
    hit (ueg.py:395-404), ALIASED vectors included: at 54e / 147 plane waves k_p + k_q - k_r has
    components beyond imax whose linearisation lands on another basis vector, and the reference's
    V is non-zero there too (it only range-checks the linear index)."""
    from pymes_b200.model import ueg
    m = ueg.UEG(54, 27, 27, 0.5)
    m.init_single_basis(10.0)
    no, nP = 27, m.n_orb
    nv = nP - no
    k = m.k_int().astype(np.int64)
    n = 2 * m.imax + 1
    for lo, ext in (((no,) * 4, (nv,) * 4), ((0, no, no, no), (no, nv, nv, nv)), ((no + 5, 0, no, no), (40, no, nv, nv))):
        row_ord, ent_ord, g_r0, g_rn, g_e0, g_en = ueg.momentum_groups(k, m.imax, lo, ext)
        # the reference's lookup, vectorised: s*(p,q,r) or -1
        P, Q, R = (np.arange(lo[d], lo[d] + ext[d]) for d in range(3))
        v = k[Q][None, :, None, :] - (k[R][None, None, :, :] - k[P][:, None, None, :]) + m.imax
        loc = n * n * v[..., 0] + n * v[..., 1] + v[..., 2]
        ok = (loc >= 0) & (loc < n ** 3)
        s = np.where(ok, m.basis_indices_map[np.clip(loc, 0, n ** 3 - 1)], -1)
        s = np.where((s >= lo[3]) & (s < lo[3] + ext[3]), s - lo[3], -1)
        true_momentum = (np.abs(v - m.imax).max(axis=-1) <= m.imax) | (s < 0)
        if lo == (no,) * 4:
            assert not true_momentum.all()            # this basis does have aliased hits
        # group id of every row / entry (-1: group absent on the other side)
        row_gid = -np.ones(ext[0] * ext[1], dtype=np.int64)
        ent_gid = -np.ones(ext[2] * ext[3], dtype=np.int64)
        for g in range(len(g_rn)):
            row_gid[row_ord[g_r0[g]:g_r0[g] + g_rn[g]]] = g
            ent_gid[ent_ord[g_e0[g]:g_e0[g] + g_en[g]]] = g
        hit = s >= 0
        pi, qi, ri = np.nonzero(hit)
        rows = pi * ext[1] + qi
        ents = ri * ext[3] + s[hit]
        assert (row_gid[rows] >= 0).all() and (row_gid[rows] == ent_gid[ents]).all()
        assert int((g_rn * g_en).sum()) == int(hit.sum())      # and nothing else is visited


def test_momentum_blocked_stored_blocks_host_logic(cpu_abi):
    """Stored integral blocks carry a geometry tag (``UEG.eval_2b_blocks``): contractions that split
    their four indices 2 + 2 between output and sum run on the diagonal momentum blocks for ANY
    such split (the ring-type products of ccd.py:189-204,233-240 with V_ijab / V_iajb), including
    narrowed row blocks; patterns the blocked kernel cannot take stay on the dense kernel."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    nP, no = m.n_orb, 7
    nv = nP - no
    parts = [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)]
    dV = m.eval_2b_blocks(no, ["ijab", "iajb", "iabj", "klij", "abic"], parts)
    assert all(bk.geom_of(v) is not None for v in dV.values())
    rng = np.random.default_rng(9)
    T = _t(rng.standard_normal((nv, nv, no, no)))
    calls = {"blocked": 0, "dense": 0}
    blocked0, dense0 = cpu_abi.pmb_blocked_contract, cpu_abi.pmb_contract
    cpu_abi.pmb_blocked_contract = lambda *a: (calls.__setitem__("blocked", calls["blocked"] + 1), blocked0(*a))[1]
    cpu_abi.pmb_contract = lambda *a: (calls.__setitem__("dense", calls["dense"] + 1), dense0(*a))[1]

    def check(spec, A, B, want_blocked, **kw):
        b0, d0 = calls["blocked"], calls["dense"]
        got = bk.contract(spec, A, B, **kw)
        np.testing.assert_allclose(_n(got), kw.get("alpha", 1.0) * np.einsum(spec, _n(A), _n(B)), rtol=0, atol=1e-12)
        assert (calls["blocked"] - b0, calls["dense"] - d0) == ((1, 0) if want_blocked else (0, 1)), spec

    V_ijab, V_iajb, V_iabj = dV["ijab"], dV["iajb"], dV["iabj"]
    check("klcd,dblj->cbkj", V_ijab, T, True)                 # Xai            ccd.py:202
    check("klcd,adkj->alcj", V_ijab, T, True)                 # X1             ccd.py:189
    check("klcd,daki->alci", V_ijab, T, True)                 # Xp             ccd.py:238
    check("klcd,cdij->klij", V_ijab, T, True)                 # I_klij         ccd.py:180
    check("kaic,cbkj->abij", V_iajb, T, True, alpha=-1.0)     # ring           ccd.py:233
    check("kbic,ackj->abij", V_iajb, T, True)                 # ring           ccd.py:234
    check("cbkj,kaic->abij", T, V_iajb, True)                 # structured operand given second
    # column index (a,i) with i not unit-stride in T[a,c,i,k]: the blocked kernel does not take it
    check("acik,kbcj->abij", T, V_iabj, False)
    # one or three output indices on the integral block: not a 2 + 2 split
    check("adkl,lkdc->ac", T, V_ijab, False)
    old_gather = bk.set_gather(False)      # (with it on, this one-summed-index product goes to pmb_gather_expand)
    try:
        check("abid,dj->abij", dV["abic"], _t(rng.standard_normal((nv, no))), False)
    finally:
        bk.set_gather(old_gather)
    # row blocks keep their tag through backend.narrow (parallel.Shard.rows)
    part = bk.narrow(V_ijab, 2, 2, 3)
    assert bk.geom_of(part).lo[2] == no + 2 and bk.geom_of(part).ext[2] == 3
    b0 = calls["blocked"]
    got = bk.contract("klcd,dblj->cbkj", part, T)
    np.testing.assert_allclose(_n(got), np.einsum("klcd,dblj->cbkj", _n(V_ijab)[:, :, 2:5], _n(T)), rtol=0, atol=1e-12)
    assert calls["blocked"] == b0 + 1
    # the undressed V_ijab "dressed" is a tagged copy; dressed blocks with T1 terms are not tagged
    T1 = _t(rng.standard_normal((nv, no)))
    full = m.eval_2b_blocks(no, ["ijab", "ijka", "ijak", "iajb", "iacb"] if False else ["ijab", "ijka"], parts)
    assert bk.geom_of(ccsd.dressed_block("ijab", T1, full)) is not None
    assert bk.geom_of(ccsd.dressed_block("ijka", T1, full)) is None
    # accumulate into an existing tensor with a coefficient, multi-term call with a dense term
    R0 = rng.standard_normal((nv, nv, no, no))
    R = _t(R0.copy())
    X = _t(rng.standard_normal((nv, no, nv, no)))
    bk.contract_terms("abij", [(-1.0, "kaic", V_iajb, "cbkj", T), (1.0, "alci", X, "cblj", T)], out=R, beta=1.0)
    want = R0 - np.einsum("kaic,cbkj->abij", _n(V_iajb), _n(T)) + np.einsum("alci,cblj->abij", _n(X), _n(T))
    np.testing.assert_allclose(_n(R), want, rtol=0, atol=1e-12)


def test_momentum_gather_t1_products_host_logic(cpu_abi):
    """``pmb_gather_expand``: the T1 dressing products of a stored UEG block with ONE summed index
    (ccsd.py:322-419: "abid,dj->abij", "abcj,ci->abij", "iabc,cj->iabj", "iacb,cj->iajb") through
    the partner tables (one candidate orbital per (x0,x1,x2), ueg.py:395-404), against the dense
    kernel and numpy, with a RANDOM T1 (in the UEG itself T1 vanishes identically, so the UEG
    lock-step tests cannot see these values); row blocks of a sharded run; the dressed V_abij and
    the shared X3 / X4 of a CCSD sweep with the path on and off."""
    from pymes_b200 import backend as bk
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd
    from pymes_b200.integral.partition import KEYS
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    nP, no = m.n_orb, 7
    nv = nP - no
    parts = [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)]
    dV = m.eval_2b_blocks(no, list(KEYS), parts)
    rng = np.random.default_rng(12)
    T1 = _t(rng.standard_normal((nv, no)))
    calls = {"gather": 0, "dense": 0}
    g0, d0 = cpu_abi.pmb_gather_expand, cpu_abi.pmb_contract
    cpu_abi.pmb_gather_expand = lambda *a: (calls.__setitem__("gather", calls["gather"] + 1), g0(*a))[1]
    cpu_abi.pmb_contract = lambda *a: (calls.__setitem__("dense", calls["dense"] + 1), d0(*a))[1]
    old = bk.set_gather(True)
    try:
        cases = [("abid,dj->abij", "abic"), ("abcj,ci->abij", "abci"), ("iabc,cj->iabj", "iabc"),
                 ("iacb,cj->iajb", "iabc"), ("dj,abid->abij", "abic")]
        for spec, key in cases:
            first_is_v = spec.split(",")[0] != "dj"
            A, B = (dV[key], T1) if first_is_v else (T1, dV[key])
            n0 = calls["gather"]
            got = bk.contract(spec, A, B)
            assert calls["gather"] == n0 + 1, spec
            np.testing.assert_allclose(_n(got), np.einsum(spec, _n(A), _n(B)), rtol=0, atol=1e-13)
        # the tables hold exactly the non-zero structure of the block
        tab = bk.geom_of(dV["abic"]).partner_tables(dV["abic"], 3)
        assert tab["n_hit"] >= np.count_nonzero(_n(dV["abic"])) > 0
        # coefficient + accumulation into an existing tensor (a row of the dressed V_abij)
        R0 = rng.standard_normal((nv, nv, no, no))
        R = _t(R0.copy())
        bk.contract_terms("abij", [(-0.5, "abcj", dV["abci"], "ci", T1)], out=R, beta=1.0)
        np.testing.assert_allclose(_n(R), R0 - 0.5 * np.einsum("abcj,ci->abij", _n(dV["abci"]), _n(T1)),
                                   rtol=0, atol=1e-13)
        # local row blocks as one rank of a sharded run builds them
        loc = m.eval_2b_blocks(no, ["abic", "iabc"], parts,
                               ranges={"abic": {0: (no + 2, 3)}, "iabc": {1: (no + 2, 3)}})
        got = bk.contract("abid,dj->abij", loc["abic"], T1)
        np.testing.assert_allclose(_n(got), np.einsum("abid,dj->abij", _n(dV["abic"])[2:5], _n(T1)), rtol=0, atol=1e-13)
        got = bk.contract("iacb,cj->iajb", loc["iabc"], T1)
        np.testing.assert_allclose(_n(got), np.einsum("iacb,cj->iajb", _n(dV["iabc"])[:, 2:5], _n(T1)), rtol=0, atol=1e-13)
        # not the pattern: two summed indices, a non-contiguous output -> other kernels
        n0 = calls["gather"]
        bk.contract("abid,dj->abij", dV["abic"], T1, out=bk.empty(no, no, nv, nv).permute(2, 3, 0, 1))
        assert calls["gather"] == n0
        # the CCSD building blocks that issue these products, path on vs off
        on = (ccsd.t1_shared(T1, dV), ccsd.dressed_block("abij", T1, dV, skip_tau=True))
        n_on = calls["gather"]
        bk.set_gather(False)
        off = (ccsd.t1_shared(T1, dV), ccsd.dressed_block("abij", T1, dV, skip_tau=True))
        assert calls["gather"] == n_on and n_on >= n0 + 4
        for k in ("X3", "X4", "G3", "G4"):
            np.testing.assert_allclose(_n(on[0][k]), _n(off[0][k]), rtol=0, atol=1e-12)
        np.testing.assert_allclose(_n(on[1]), _n(off[1]), rtol=0, atol=1e-12)
    finally:
        bk.set_gather(old)


def test_momentum_groups_cover_every_nonzero_for_every_split():
    """Every non-zero of the oracle-built TC-UEG V_pqrs (the reference's triple loop restated,
    oracle/ueg_oracle.py) lies inside the groups of ``momentum_groups`` -- for all six ways of
    splitting (p,q,r,s) into two row and two entry axes and for random sub-blocks (what the geometry
    tags of stored blocks and their narrowed row blocks rely on) -- and the partner tables of
    ``pmb_gather_expand`` name exactly the non-zero's position for each of the four summed axes."""
    import itertools
    from oracle import ueg_oracle as uo
    from pymes_b200.model import ueg
    mo = uo.UEG(14, 1.0).init_single_basis(3.0)
    mo.k_cutoff, mo.gamma = 2.0, None
    _fock, V = mo.tc_hamiltonian(7)
    nP = V.shape[0]
    m = ueg.UEG(14, 7, 7, 1.0)
    m.init_single_basis(3.0)
    assert m.n_orb == nP and np.array_equal(m.k_int(), mo.kint)
    k, imax = m.k_int(), m.imax
    rng = np.random.default_rng(0)
    blocks = [((0,) * 4, (nP,) * 4)]
    for _ in range(4):
        lo = rng.integers(0, nP - 3, size=4)
        ext = [int(rng.integers(2, nP - l + 1)) for l in lo]
        blocks.append((tuple(int(x) for x in lo), tuple(ext)))
    n_checked = 0
    for lo, ext in blocks:
        blk = V[lo[0]:lo[0] + ext[0], lo[1]:lo[1] + ext[1], lo[2]:lo[2] + ext[2], lo[3]:lo[3] + ext[3]]
        nz = np.argwhere(blk != 0)
        for m_axes in itertools.combinations(range(4), 2):
            k_axes = tuple(ax for ax in range(4) if ax not in m_axes)
            row_ord, ent_ord, g_r0, g_rn, g_e0, g_en = ueg.momentum_groups(k, imax, lo, ext, m_axes, k_axes)
            row_gid = -np.ones(ext[m_axes[0]] * ext[m_axes[1]], dtype=np.int64)
            ent_gid = -np.ones(ext[k_axes[0]] * ext[k_axes[1]], dtype=np.int64)
            for g in range(len(g_rn)):
                row_gid[row_ord[g_r0[g]:g_r0[g] + g_rn[g]]] = g
                ent_gid[ent_ord[g_e0[g]:g_e0[g] + g_en[g]]] = g
            rows = nz[:, m_axes[0]] * ext[m_axes[1]] + nz[:, m_axes[1]]
            ents = nz[:, k_axes[0]] * ext[k_axes[1]] + nz[:, k_axes[1]]
            assert (row_gid[rows] >= 0).all() and (row_gid[rows] == ent_gid[ents]).all(), (lo, ext, m_axes)
            n_checked += len(nz)
        # one candidate partner per triple, on every axis
        n = 2 * imax + 1
        lin = (n * n * k[:, 0] + n * k[:, 1] + k[:, 2]).astype(np.int64)
        for y in range(4):
            others = [ax for ax in range(4) if ax != y]
            l = [ueg.SIGNS[ax] * lin[lo[ax]:lo[ax] + ext[ax]] for ax in range(4)]
            want = -ueg.SIGNS[y] * (l[others[0]][nz[:, others[0]]] + l[others[1]][nz[:, others[1]]]
                                    + l[others[2]][nz[:, others[2]]])
            assert np.array_equal(ueg.SIGNS[y] * l[y][nz[:, y]], want), (lo, ext, y)     # raw l(k_y)
    assert n_checked > 10000
