"""Parity of the CUDA path (through the C ABI in libpymes_b200.so) with the CPU oracle
and the reference-generated goldens.  Needs a B200: run with ``-m gpu``.

Tolerances (north_star): correlation energy 1e-10 Eh, amplitudes 1e-9 relative."""
import numpy as np
import pytest
import torch

from tests.conftest import golden
from tests import test_host_logic as host

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, scope="module")
def _native_library_loaded():
    """Fail loudly (not skip) if the CUDA extension is not what runs."""
    assert torch.cuda.is_available(), "the -m gpu tests need a CUDA device"
    from pymes_b200 import _lib, backend as bk
    lib = _lib.load()
    import ctypes as C
    sm, cc, mem = C.c_int(), C.c_int(), C.c_size_t()
    _lib.check(lib.pmb_device_info(C.byref(sm), C.byref(cc), C.byref(mem)))
    assert cc.value >= 100, "libpymes_b200.so is built for sm_100a"
    before = bk.launch_count()
    host.DEVICE = "cuda"
    yield
    host.DEVICE = "cpu"
    assert bk.launch_count() > before, "no kernel of libpymes_b200.so was launched"


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


# --------------------------------------------------------------------------
# the host-logic checks, now on the real kernels (cpu_abi=None -> CUDA path)
# --------------------------------------------------------------------------
@pytest.mark.parametrize("spec,shapes", host.test_contract_matches_einsum.pytestmark[0].args[1])
def test_contract_small(spec, shapes):
    host.test_contract_matches_einsum(None, spec, shapes)


def test_contract_views_multi_term():
    host.test_contract_on_strided_views_and_multi_term(None)


def test_multi_operand_einsum():
    host.test_multi_operand_einsum(None)


def test_matrix_vector_contractions_go_to_gemv(monkeypatch):
    host.test_matrix_vector_contractions_go_to_gemv(None, monkeypatch)


def test_gemv_medium_both_mappings(monkeypatch):
    """pmb_gemv at o=9, v=83 (ragged against the 32-lane / 8-row unrolling) vs numpy."""
    from pymes_b200 import backend as bk
    monkeypatch.setattr(bk, "GEMV_MIN_OUTPUTS", 0)
    monkeypatch.setattr(bk, "GEMV_MIN_WARP_OUTPUTS", 0)
    rng = np.random.default_rng(8)
    no, nv = 9, 83
    t1 = rng.standard_normal((nv, no))
    V = rng.standard_normal((no, nv, nv, nv))
    assert V.size >= bk.GEMV_MIN_ELEMENTS
    before = bk.launch_count()
    for spec, A, B in (("ci,iabc->ab", t1, V), ("ci,iacb->ab", t1, V), ("jacb,bj->ac", V, t1),
                       ("jabc,bj->ac", V, t1)):
        got = bk.contract(spec, host._t(A), host._t(B))
        assert _rel(got.cpu().numpy(), np.einsum(spec, A, B)) < 1e-13
    assert bk.launch_count() - before == 4          # one kernel each: no split-K second stage


def test_contract_realigns_conflicting_unit_strides(monkeypatch):
    host.test_contract_realigns_conflicting_unit_strides(None, monkeypatch)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_ccd_residual_energy_mp2(tag):
    host.test_ccd_residual_energy_mp2(None, tag)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_ccsd_dressing_singles_doubles(tag):
    host.test_ccsd_dressing_singles_doubles(None, tag)


def test_diis_sequence():
    host.test_diis_matches_reference_sequence(None)


@pytest.mark.parametrize("tag", ["LiH_321g", "LiH_tc"])
def test_molecule_solvers_iteration_parity(tag, capsys):
    host.test_solvers_follow_reference_iteration_by_iteration(None, tag, capsys)


def test_amps_aliasing():
    host.test_amps_warm_start_aliasing(None)


def test_ueg_coulomb_build_and_fock():
    host.test_ueg_coulomb_integrals_and_ccd(None)


def test_ueg_tc_tables():
    host.test_ueg_tc_tables_small(None)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_eom_sigma_diag_and_batching(tag):
    host.test_eom_sigma_diag_and_batching(None, tag)


@pytest.mark.parametrize("tag", ["H2_321g", "LiH_321g"])
def test_eom_davidson_roots(tag):
    host.test_eom_davidson_roots(None, tag)


def test_feast_linear_solve_matches_reference_gcrot():
    host.test_feast_linear_solve_matches_reference_gcrot(None)


def test_feast_batched_systems_and_seeded_iteration():
    host.test_feast_batched_systems_and_seeded_iteration(None)


def test_feast_gcrot_matches_scipy_over_many_cycles():
    host.test_feast_gcrot_matches_scipy_over_many_cycles(None)


# --------------------------------------------------------------------------
# contraction engine: every tile configuration, both load mappings, ragged edges,
# split-K, multi-term accumulation, strided views
# --------------------------------------------------------------------------
CASES = [
    # pp ladder shapes (M=v^2, K=v^2, N=o^2); N=49 is the hostile 14-electron case
    ("abcd,cdij->abij", [(50, 50, 50, 50), (50, 50, 7, 7)]),
    ("abcd,cdij->abij", [(23, 23, 23, 23), (23, 23, 13, 13)]),
    # hh ladder / I build: tiny K or tiny M -> split-K path
    ("klij,abkl->abij", [(7, 7, 7, 7), (40, 40, 7, 7)]),
    ("klcd,cdij->klij", [(6, 6, 45, 45), (45, 45, 6, 6)]),
    # ring-type, interleaved M/K/N groups
    ("klcd,adkj->alcj", [(9, 9, 31, 31), (31, 31, 9, 9)]),
    ("alcj,cbil->abij", [(31, 9, 31, 9), (31, 31, 9, 9)]),
    ("acik,cbkj->abij", [(33, 33, 8, 8), (33, 33, 8, 8)]),
    ("kbic,ackj->abij", [(8, 33, 8, 33), (33, 33, 8, 8)]),
    ("acik,kbcj->abij", [(33, 33, 8, 8), (8, 33, 33, 8)]),
    # Fock-like
    ("adkl,lkdc->ac", [(37, 37, 6, 6), (6, 6, 37, 37)]),
    ("cdil,lkdc->ki", [(37, 37, 6, 6), (6, 6, 37, 37)]),
    ("ac,cbij->abij", [(41, 41), (41, 41, 5, 5)]),
    ("ki,abkj->abij", [(5, 5), (41, 41, 5, 5)]),
    # T1-dressing shapes
    ("kbcd,cdij->kbij", [(5, 29, 29, 29), (29, 29, 5, 5)]),
    ("ak,kbij->abij", [(29, 5), (5, 29, 5, 5)]),
    ("ai,bj->abij", [(17, 4), (17, 4)]),
    ("ia,ai->", [(6, 300), (300, 6)]),
    # plain big GEMM crossing many tiles in both directions
    ("mk,kn->mn", [(517, 301), (301, 389)]),
]


@pytest.mark.parametrize("cfg", [-1, 0, 1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("spec,shapes", CASES)
def test_contract_engine(spec, shapes, cfg):
    from pymes_b200 import _lib, backend as bk
    import zlib
    rng = np.random.default_rng(zlib.crc32(spec.encode()) + len(shapes[0]))      # same data every run
    A, B = (rng.standard_normal(s) for s in shapes)
    ref = np.einsum(spec, A, B, optimize=True)
    # error scale of a sum with cancellation: sum_k |a||b|, not |sum_k a b|
    scale = np.einsum(spec, np.abs(A), np.abs(B), optimize=True).max()
    _lib.load().pmb_contract_set_tuning(cfg, 0)
    try:
        got = bk.contract(spec, A, B, alpha=-0.75)
        assert np.abs(got.cpu().numpy() + 0.75 * ref).max() < 2e-14 * scale
        out = bk.asdev(rng.standard_normal(ref.shape))
        keep = out.cpu().numpy().copy()
        bk.contract(spec, A, B, out=out, alpha=1.25, beta=-0.5)
        assert np.abs(out.cpu().numpy() - (-0.5 * keep + 1.25 * ref)).max() < 2e-14 * (scale + 1.0)
    finally:
        _lib.load().pmb_contract_set_tuning(-1, 0)


@pytest.mark.parametrize("cfg", [-1, 5])
@pytest.mark.parametrize("split", [1, 2, 3, 7, 16])
def test_contract_split_k(split, cfg):
    from pymes_b200 import _lib, backend as bk
    rng = np.random.default_rng(split)
    A = rng.standard_normal((6, 6, 41, 41))
    B = rng.standard_normal((41, 41, 6, 6))
    ref = np.einsum("klcd,cdij->klij", A, B, optimize=True)
    _lib.load().pmb_contract_set_tuning(cfg, split)
    try:
        out = bk.asdev(np.ones_like(ref))
        bk.contract("klcd,cdij->klij", A, B, out=out, beta=2.0)
        assert _rel(out.cpu().numpy(), 2.0 + ref) < 1e-13
    finally:
        _lib.load().pmb_contract_set_tuning(-1, 0)


@pytest.mark.parametrize("cfg", [0, 2, 5])
def test_contract_k_windows(cfg):
    """K-window launches (L2 residency of the smaller operand) accumulate in C in fixed order."""
    from pymes_b200 import _lib, backend as bk
    lib = _lib.load()
    rng = np.random.default_rng(17)
    nv, no = 52, 7                                   # K = 2704 -> 169 k-tiles -> 3 windows of >= 64
    V, T = rng.standard_normal((nv,) * 4), rng.standard_normal((nv, nv, no, no))
    Xa, Xb = rng.standard_normal((nv, nv, no, no)), rng.standard_normal((no, no, no, no))
    ref = np.einsum("abcd,cdij->abij", V, T, optimize=True) - 0.5 * np.einsum("abkl,klij->abij", Xa, Xb, optimize=True)
    lib.pmb_contract_set_tuning(cfg, 1)              # no split-K: windows apply to unsplit launches
    lib.pmb_contract_set_panel_bytes(1)
    try:
        before = bk.launch_count()
        out = bk.asdev(np.ones_like(ref))
        bk.contract_terms("abij", [(1.0, "abcd", bk.asdev(V), "cdij", bk.asdev(T)),
                                   (-0.5, "abkl", bk.asdev(Xa), "klij", bk.asdev(Xb))], out=out, beta=3.0)
        assert bk.launch_count() - before >= 3
        assert _rel(out.cpu().numpy(), 3.0 + ref) < 1e-13
        got = bk.contract("abcd,cdij->abij", V, T)          # beta = 0: C is never read
        assert _rel(got.cpu().numpy(), np.einsum("abcd,cdij->abij", V, T, optimize=True)) < 1e-13
    finally:
        lib.pmb_contract_set_tuning(-1, 0)
        lib.pmb_contract_set_panel_bytes(-1)


def test_contract_views_of_V_pqrs_no_symmetry():
    """Operands are strided views of one V_pqrs with NO permutational symmetry."""
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import part_2_body_int
    rng = np.random.default_rng(11)
    no, nv = 5, 21
    n = no + nv
    V = rng.standard_normal((n, n, n, n))
    T = rng.standard_normal((nv, nv, no, no))
    dV, dVn = part_2_body_int(no, bk.asdev(V)), part_2_body_int(no, V)
    Td = bk.asdev(T)
    for spec, key in (("abcd,cdij->abij", "abcd"), ("klcd,cdij->klij", "ijab"),
                      ("kaic,cbkj->abij", "iajb"), ("kbcj,acik->abij", "iabj"),
                      ("kbcd,cdij->kbij", "iabc"), ("alcd,cdij->alij", "aibc")):
        got = bk.contract(spec, dV[key], Td).cpu().numpy()
        assert _rel(got, np.einsum(spec, dVn[key], T, optimize=True)) < 1e-13, spec


def test_contract_eight_terms_one_launch():
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(5)
    nv, no = 19, 6
    Ts = [rng.standard_normal((nv, nv, no, no)) for _ in range(8)]
    Xs = [rng.standard_normal((nv, nv, no, no)) for _ in range(8)]
    before = bk.launch_count()
    got = bk.contract_terms("abij", [(0.1 * (k + 1), "acik", bk.asdev(Ts[k]), "cbkj", bk.asdev(Xs[k]))
                                     for k in range(8)])
    assert bk.launch_count() - before <= 2      # one contraction launch (+ split-K reduce)
    ref = sum(0.1 * (k + 1) * np.einsum("acik,cbkj->abij", Ts[k], Xs[k]) for k in range(8))
    assert _rel(got.cpu().numpy(), ref) < 1e-13


def test_contract_bad_arguments():
    from pymes_b200 import _lib
    import ctypes as C
    lib = _lib.load()
    d = _lib.Contract()
    d.nterms = 0
    assert lib.pmb_contract(C.byref(d), None, 0, None) == -1
    with pytest.raises(RuntimeError, match="bad argument"):
        _lib.check(-1, "x")


# --------------------------------------------------------------------------
# elementwise kernels against plain numpy
# --------------------------------------------------------------------------
def test_elementwise_kernels():
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(3)
    no, nv = 6, 17
    ei, ea = np.sort(rng.uniform(-2, -1, no)), np.sort(rng.uniform(1, 3, nv))
    T = rng.standard_normal((nv, nv, no, no))
    R = rng.standard_normal((nv, nv, no, no))
    V = rng.standard_normal((no, no, nv, nv))
    T1 = rng.standard_normal((nv, no))
    D = (ei[None, None, :, None] + ei[None, None, None, :] - ea[:, None, None, None]
         - ea[None, :, None, None] + 0.25)
    Td, scal = bk.asdev(T.copy()), bk.zeros(8)
    dT = bk.update_doubles(bk.asdev(ei), bk.asdev(ea), 0.25, 1.0, bk.asdev(R), Td, scal[3:4])
    assert _rel(dT.cpu().numpy(), R / D) < 1e-14
    assert _rel(Td.cpu().numpy(), T + R / D) < 1e-14
    assert abs(scal[3].item() - np.sum((R / D) ** 2)) < 1e-10 * np.sum((R / D) ** 2)
    bk.energy_doubles(bk.asdev(T), bk.asdev(V), scal, T1=bk.asdev(T1))
    tau = T + np.einsum("ai,bj->abij", T1, T1)
    s = scal.cpu().numpy()
    assert abs(s[0] - 2 * np.einsum("abij,ijab->", tau, V)) < 1e-10
    assert abs(s[1] + np.einsum("abij,ijba->", tau, V)) < 1e-10
    assert abs(s[2] - np.sum(T * T)) < 1e-10
    assert _rel(bk.tilde(bk.asdev(T)).cpu().numpy(), 2 * T - T.transpose(1, 0, 2, 3)) == 0
    assert _rel(bk.tilde(bk.asdev(T), swap_ij=True).cpu().numpy(), 2 * T - T.transpose(0, 1, 3, 2)) == 0
    Rd = bk.asdev(R.copy())
    bk.sym_baji(bk.asdev(T), Rd, accumulate=True)
    assert _rel(Rd.cpu().numpy(), R + T + T.transpose(1, 0, 3, 2)) < 1e-15
    xs = [rng.standard_normal(1000003) for _ in range(7)]
    y = rng.standard_normal(1000003)
    got = bk.dots([bk.asdev(x) for x in xs], bk.asdev(y)).cpu().numpy()
    np.testing.assert_allclose(got, [x @ y for x in xs], rtol=1e-11, atol=1e-9)
    c = rng.standard_normal(7)
    got = bk.lincomb(c, [bk.asdev(x) for x in xs]).cpu().numpy()
    np.testing.assert_allclose(got, sum(ci * x for ci, x in zip(c, xs)), rtol=1e-13, atol=1e-13)
    src = bk.asdev(V)
    got = bk.axpby(2.0, src.permute(2, 3, 0, 1)).cpu().numpy()
    assert _rel(got, 2 * V.transpose(2, 3, 0, 1)) == 0


# --------------------------------------------------------------------------
# solvers against goldens that only make sense at GPU speed
# --------------------------------------------------------------------------
def test_hf_augccpvdz_ccsd_diis_full_subspace():
    """HF / aug-cc-pVDZ (o=5, v=27): DIIS subspace overflows -> bug-compatible bookkeeping.

    Sweep-by-sweep lock-step with the oracle.  Amplitudes agree to 1e-9 relative (in practice
    1e-14) while the DIIS system is well conditioned; from sweep 11 on the residual overlaps
    reach 1e-16 and DIIS amplifies ANY round-off difference to ~1e-9..1e-8: the reference
    deviates from ITSELF by 6e-9 (T1) / 1e-9 (T2) there when only the einsum summation order
    changes (oracle "as_written" vs "optimized" mode, see DESIGN.md "DIIS noise floor").  So
    the late sweeps are held to 2e-8, the energy to 1e-10 throughout."""
    from pymes_b200.solver import ccsd
    from oracle import cc_oracle as oc
    g = golden("mol_HF_augccpvdz")
    no = int(g["n_elec"]) // 2
    for name, flag in (("ccsd", False), ("dcsd", True)):
        trace = []
        oc.ccsd_solve(no, g["fock"], g["V"], is_dcsd=flag, delta_e=1e-8, max_iter=50, trace=trace)
        assert len(trace) == len(g[name + "_trace"])
        cc = ccsd.CCSD(no, is_dcsd=flag)
        cc.setup(g["fock"], g["V"])
        for n, ref in enumerate(trace):
            e1, ed, ex, _, _ = cc.sweep()
            d2 = _rel(cc._st["T2"].cpu().numpy(), ref["t2"])
            d1 = _rel(cc._st["T1"].cpu().numpy(), ref["t1"])
            assert abs(e1 + ed + ex - ref["e"]) < 1e-10, (n, e1 + ed + ex - ref["e"])
            tol = 1e-9 if n < 10 else 2e-8
            assert d2 < tol and d1 < tol, (name, n, d2, d1)
        cc = ccsd.CCSD(no, is_dcsd=flag)
        r = cc.solve(g["fock"], g["V"], delta_e=1e-8, max_iter=50)
        assert cc.iterations == len(g[name + "_trace"])
        assert abs(r["ccsd e"] - g[name + "_e"]) < 1e-10
        assert _rel(r["t2"], g[name + "_t2"]) < 2e-8 and _rel(r["t1"], g[name + "_t1"]) < 2e-8


def test_ueg_14e_ccd_dcd_reference_goldens():
    """UEG 14e / 57 PW (config 1): rs=1.0 to convergence and the rs=0.5, shift -1 constants of
    pymes/test/test_ueg/test_ccd_dcd.py:208-209."""
    from pymes_b200.model import ueg
    from pymes_b200.mean_field import hf
    from pymes_b200.solver import ccd, dcd
    g = golden("ueg_coulomb")
    for rs, tag, shift in ((1.0, "rs1", 0.0), (0.5, "rs05", -1.0)):
        m = ueg.UEG(14, 7, 7, rs)
        m.init_single_basis(5.0)
        V = m.eval_2b_integrals(device=True)
        assert V.is_cuda
        fock = hf.construct_hf_matrix(7, np.diag(m.kinetic()), V)
        np.testing.assert_allclose(fock.cpu().numpy() if isinstance(fock, torch.Tensor) else fock,
                                   g[tag + "_fock"], rtol=1e-12, atol=1e-13)
        cc = ccd.CCD(7)
        r = cc.solve(g[tag + "_fock"], V, level_shift=shift)
        assert cc.iterations == len(g[tag + "_ccd_trace"])
        assert abs(r["ccd e"] - g[tag + "_ccd_e"]) < 1e-10
        dd = dcd.DCD(7)
        # test_ccd_dcd.py:176-181 warm-starts the rs=0.5 DCD from the CCD amplitudes
        amps = r["t2 amp"].clone() if tag == "rs05" else None
        r = dd.solve(g[tag + "_fock"], V, level_shift=shift, amps=amps)
        assert dd.iterations == len(g[tag + "_dcd_trace"])
        assert abs(r["ccd e"] - g[tag + "_dcd_e"]) < 1e-10
    assert abs(g["rs05_ccd_e"] - (-0.5120153512190824)) < 1e-6       # test_ccd_dcd.py:208
    assert abs(g["rs05_dcd_e"] - (-0.515296499349519)) < 1e-6        # test_ccd_dcd.py:209


def test_ueg_tc_full_build_and_ccd():
    """TC-UEG 14e rs=0.5 (test_symmetrised_2body_integral.py:205-220): u_mat, both TC integral
    kinds, TC-CCD energy -0.256670836708 (1e-8 there, 1e-10 against the regenerated golden)."""
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccd
    from pymes_b200 import backend as bk
    g = golden("ueg_tc")
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(5.0)
    m.k_cutoff = float(g["k_cutoff"])
    m.gamma = None
    nP = m.n_orb
    V2 = m.eval_2b_integrals(correlator=m.trunc, is_only_2b=True, device=True)
    assert _rel(V2.cpu().numpy(), host._dense(g["V2_idx"], g["V2_val"], nP)) < 1e-11
    Veff = m.eval_2b_integrals(correlator=m.trunc, is_effect_2b=True, device=True)
    assert _rel(Veff.cpu().numpy(), host._dense(g["Veff_idx"], g["Veff_val"], nP)) < 1e-11
    V = bk.lincomb([1.0, 1.0], [V2, Veff])
    r = ccd.CCD(7).solve(g["fock"], V)
    assert abs(r["ccd e"] - g["ccd_e"]) < 1e-10
    assert abs(r["ccd e"] - (-0.256670836708)) < 1e-8
    # blocks built directly == slices of the dense tensor
    blocks = m.eval_2b_blocks(7, ["abcd", "iajb", "klij"], [("only_2b", m.trunc), ("effect_2b", m.trunc)])
    Vn = V.cpu().numpy()
    assert _rel(blocks["abcd"].cpu().numpy(), Vn[7:, 7:, 7:, 7:]) < 1e-13
    assert _rel(blocks["iajb"].cpu().numpy(), Vn[:7, 7:, :7, 7:]) < 1e-13


def test_ueg_virtual_block_host_cases():
    host.test_ueg_virtual_block_descriptor(None)


def test_eom_with_never_materialised_abcd():
    """Dressed V_abcd as an operator (ccsd.DressedLadder) over a generated V_abcd: sigma, batches
    and diagonals equal the dense path (first passed on a B200 at the end of round 1)."""
    host.test_eom_with_never_materialised_abcd(None)


def _tc_model(n_ele, cutoff, rs=0.5):
    from pymes_b200.model import ueg
    m = ueg.UEG(n_ele, n_ele // 2, n_ele // 2, rs)
    m.init_single_basis(cutoff)
    m.k_cutoff, m.gamma = 1.0, None
    return m


@pytest.mark.parametrize("n_ele,cutoff", [(14, 5.0), (14, 9.0), (54, 7.0), (54, 8.0)])   # 54/8.0: 210 tiles -> tail launch
def test_ueg_virtual_pp_ladder_bit_identical(n_ele, cutoff):
    """Never-materialised V_abcd (SURVEY 8(f).1): the pp ladder with the operand generated in
    the kernel's producer warps equals the ladder on the block pmb_ueg_build_block wrote --
    bit for bit when both run the same (warp-specialised) kernel, because the generated tile
    holds the very same doubles.  TC integrals (non-hermitian W1 term + symmetrised W0s)."""
    from pymes_b200 import _lib, backend as bk
    m = _tc_model(n_ele, cutoff)
    no, nP = n_ele // 2, m.n_orb
    nv = nP - no
    parts = [("only_2b", m.trunc), ("effect_2b", m.trunc)]
    virt = m.eval_2b_blocks(no, ["abcd"], parts, virtual=("abcd",))["abcd"]
    dense = m.eval_2b_blocks(no, ["abcd"], parts)["abcd"]
    assert torch.equal(virt.materialise(), dense) and float(dense.abs().max()) > 0
    g = torch.Generator(device="cuda").manual_seed(1)
    tau = torch.randn(nv, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
    lib = _lib.load()
    blocked_was = bk.set_blocked(False)      # this test is about the DENSE generated-operand path
    # +64: the tail wave is left alone.  A generated operand rasters the tiles m-fastest, a stored one
    # n-fastest, so a tail launch (54e / 93 plane waves: 210 tiles = 148 + 62) would k-split DIFFERENT
    # tiles in the two runs: equal to round-off then, not bit for bit (checked right below)
    NT = 64
    try:
        lib.pmb_contract_set_tuning(5, 0)
        n0 = bk.launch_count()
        with_tail = bk.contract("abcd,cdij->abij", virt, tau)
        tiles = ((nv * nv + 127) // 128) * ((no * no + 127) // 128)
        tail_expected = tiles > 148 and 0 < tiles % 148 <= 74
        assert (bk.launch_count() - n0 == 3) if tail_expected else (bk.launch_count() - n0 <= 2)
        assert _rel(with_tail.cpu().numpy(), bk.contract("abcd,cdij->abij", dense, tau).cpu().numpy()) < 1e-13
        lib.pmb_contract_set_tuning(5 + NT, 0)
        ref = bk.contract("abcd,cdij->abij", dense, tau)
        got = bk.contract("abcd,cdij->abij", virt, tau)
        assert torch.equal(got, ref)
        lib.pmb_contract_set_tuning(6 + NT, 0)                 # 6-stage ring
        assert torch.equal(bk.contract("abcd,cdij->abij", virt, tau), bk.contract("abcd,cdij->abij", dense, tau))
        # split-K: partial sums of the generated operand
        lib.pmb_contract_set_tuning(5 + NT, 3)
        assert torch.equal(bk.contract("abcd,cdij->abij", virt, tau), bk.contract("abcd,cdij->abij", dense, tau))
        # +16: the scanning producer instead of the non-zero walker (what patterns whose
        # contracted indices are not (r, s) use), alone and with split-K
        for split in (0, 5):
            lib.pmb_contract_set_tuning(5 + 16 + NT, split)
            assert torch.equal(bk.contract("abcd,cdij->abij", virt, tau), ref if split == 0 else
                               bk.contract("abcd,cdij->abij", dense, tau))
        # contraction over (p, q): the solved index s sits in the row group -> scanning producer
        lib.pmb_contract_set_tuning(5 + NT, 0)
        assert torch.equal(bk.contract("abcd,abij->cdij", virt, tau), bk.contract("abcd,abij->cdij", dense, tau))
        # without the compressed value table the producers evaluate the integral formula in
        # place (walker and scanning variants): still the very same doubles
        raw = m.virtual_block(virt.lo, virt.shape, *virt.tables, compressed=False)
        assert virt.nz is not None and raw.nz is None
        for cfg in (5, 5 + 16):
            lib.pmb_contract_set_tuning(cfg + NT, 0)
            assert torch.equal(bk.contract("abcd,cdij->abij", raw, tau), ref)
        assert torch.equal(bk.contract("abcd,abij->cdij", raw, tau), bk.contract("abcd,abij->cdij", dense, tau))
    finally:
        lib.pmb_contract_set_tuning(-1, 0)
        bk.set_blocked(blocked_was)
    _virtual_ladder_default_checks(m, no, nv, virt, dense, tau, g, blocked=False)
    _virtual_ladder_default_checks(m, no, nv, virt, dense, tau, g, blocked=True)


def _virtual_ladder_default_checks(m, no, nv, virt, dense, tau, g, blocked):
    """Default heuristics, dense generated operand (blocked=False) or the momentum-blocked kernel."""
    from pymes_b200 import backend as bk
    blocked_was = bk.set_blocked(blocked)
    try:
        _virtual_ladder_default_checks_body(m, no, nv, virt, dense, tau, g)
    finally:
        bk.set_blocked(blocked_was)


def _virtual_ladder_default_checks_body(m, no, nv, virt, dense, tau, g):
    from pymes_b200 import backend as bk
    # default heuristics (the dense block may pick another tile shape): round-off only
    ref = bk.contract("abcd,cdij->abij", dense, tau)
    got = bk.contract("abcd,cdij->abij", virt, tau)
    assert _rel(got.cpu().numpy(), ref.cpu().numpy()) < 1e-13
    # against numpy on the host
    want = dense.cpu().numpy().reshape(nv * nv, -1) @ tau.cpu().numpy().reshape(nv * nv, -1)
    assert _rel(got.cpu().numpy().reshape(nv * nv, -1), want) < 1e-13
    # one launch with the hh ladder as a second (memory) term, accumulated into R; row block
    I = torch.randn(no, no, no, no, dtype=torch.float64, device="cuda", generator=g)
    lo, na = nv // 3, nv - nv // 3 - 1
    R0 = torch.randn(na, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
    Ra, Rb = R0.clone(), R0.clone()
    taul = tau[lo:lo + na]
    bk.contract_terms("abij", [(1.0, "klij", I, "abkl", taul), (0.5, "abcd", virt.rows(0, lo, na), "cdij", tau)],
                      out=Ra, beta=1.0)
    bk.contract_terms("abij", [(1.0, "klij", I, "abkl", taul), (0.5, "abcd", dense[lo:lo + na], "cdij", tau)],
                      out=Rb, beta=1.0)
    assert _rel(Ra.cpu().numpy(), Rb.cpu().numpy()) < 1e-13


@pytest.mark.parametrize("n_ele,cutoff", [(14, 5.0), (14, 9.0), (54, 7.0), (54, 10.0)])
def test_momentum_blocked_contractions(n_ele, cutoff):
    """pmb_blocked_contract (SURVEY 8(f).1, momentum-blocked path): the pp ladder and the two o.v^3
    products of the T1 dressing on the diagonal momentum blocks only, against (i) the dense
    generated-operand kernel, (ii) numpy on the materialised block; even-pitch tau, accumulation,
    fresh output (rows without a group are zeros), batched right-hand sides, a row block, and the
    executed flop count 2 nnz o^2.  54e / 147 plane waves: groups of up to 120 rows (two tiles)."""
    from pymes_b200 import backend as bk
    m = _tc_model(n_ele, cutoff)
    no, nP = n_ele // 2, m.n_orb
    nv = nP - no
    parts = [("only_2b", m.trunc), ("effect_2b", m.trunc)]
    blocks = m.eval_2b_blocks(no, ["abcd", "iabc", "aibc"], parts, virtual=("abcd",))
    virt = blocks["abcd"]
    L = virt.blocked_lists()
    dense = virt.materialise()
    assert L["nnz"] >= int((dense != 0).sum()) > 0 and L["nnz"] < dense.numel() // 4
    g = torch.Generator(device="cuda").manual_seed(2)
    rnd = lambda *s: torch.randn(*s, dtype=torch.float64, device="cuda", generator=g)
    tau = bk.empty_even_pitch(nv, nv, no)
    tau.copy_(rnd(nv, nv, no, no))
    assert bk.blocked_enabled()
    n0 = bk.launch_count()
    got = bk.contract("abcd,cdij->abij", virt, tau)
    assert bk.launch_count() - n0 == 1
    old = bk.set_blocked(False)
    try:
        ref = bk.contract("abcd,cdij->abij", virt, tau)
    finally:
        bk.set_blocked(old)
    assert _rel(got.cpu().numpy(), ref.cpu().numpy()) < 1e-13
    # (the checker's products run as cuBLAS DGEMMs through torch: 3e11 flop each at 147 plane waves)
    D2 = dense.reshape(nv * nv, nv * nv)
    want = (D2 @ tau.reshape(nv * nv, -1)).cpu().numpy()
    assert _rel(got.cpu().numpy().reshape(nv * nv, -1), want) < 1e-13
    # fresh output over junk; accumulation with a coefficient
    junk = rnd(nv, nv, no, no)
    bk.contract("abcd,cdij->abij", virt, tau, out=junk)
    assert torch.equal(junk, got)
    R0 = rnd(nv, nv, no, no)
    R = R0.clone()
    bk.contract_terms("abij", [(-0.3, "abcd", virt, "cdij", tau)], out=R, beta=1.0)
    assert _rel(R.cpu().numpy(), R0.cpu().numpy() - 0.3 * want.reshape(nv, nv, no, no)) < 1e-13
    # batched right-hand sides (EOM sigma), row block
    r = 3
    U = rnd(r, nv, nv, no, no)
    S = bk.contract_terms("rabij", [(1.0, "abcd", virt, "rcdij", U)])
    wantU = torch.stack([D2 @ U[k].reshape(nv * nv, -1) for k in range(r)]).cpu().numpy()
    assert _rel(S.cpu().numpy().reshape(r, nv * nv, -1), wantU) < 1e-13
    lo, na = nv // 3, nv - nv // 3 - 1
    part = bk.contract("abcd,cdij->abij", virt.rows(0, lo, na), tau)
    assert torch.equal(part, got[lo:lo + na])
    # the stored o.v^3 blocks carry a never-materialised twin: V_iabc.tau / V_aibc.tau
    from pymes_b200.solver import ccsd
    assert bk.blocked_companion(blocks["iabc"]) is not None and bk.blocked_companion(blocks["aibc"]) is not None
    n0 = bk.launch_count()
    W1, W2 = ccsd.pair_with_tau(blocks["iabc"], blocks["aibc"], tau, no)
    assert bk.launch_count() - n0 == 2
    old = bk.set_blocked(False)
    try:
        W1d, W2d = ccsd.pair_with_tau(blocks["iabc"], blocks["aibc"], tau, no)
    finally:
        bk.set_blocked(old)
    assert _rel(W1.cpu().numpy(), W1d.cpu().numpy()) < 1e-13 and _rel(W2.cpu().numpy(), W2d.cpu().numpy()) < 1e-13
    w1 = (blocks["iabc"].reshape(no * nv, -1) @ tau.reshape(nv * nv, -1)).cpu().numpy()
    assert _rel(W1.cpu().numpy().reshape(no * nv, -1), w1) < 1e-13


@pytest.mark.parametrize("n_ele,cutoff", [(14, 5.0), (54, 7.0), (54, 10.0)])
def test_momentum_blocked_stored_blocks(n_ele, cutoff):
    """Stored integral blocks with a geometry tag: every 2 + 2 split of the ring-type products of the
    doubles residual (ccd.py:180,189,202,233,234,238) runs on the diagonal momentum blocks and equals
    the dense kernel and a cuBLAS product of the same operands; narrowed row blocks (sharded runs);
    fresh outputs whose rows are not all covered."""
    from pymes_b200 import backend as bk
    m = _tc_model(n_ele, cutoff)
    no, nP = n_ele // 2, m.n_orb
    nv = nP - no
    parts = [("only_2b", m.trunc), ("effect_2b", m.trunc)]
    dV = m.eval_2b_blocks(no, ["ijab", "iajb"], parts)
    g = torch.Generator(device="cuda").manual_seed(3)
    T = torch.randn(nv, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
    lo, na = nv // 3, nv - nv // 3 - 1
    cases = [("klcd,dblj->cbkj", dV["ijab"], T), ("klcd,adkj->alcj", dV["ijab"], T),
             ("klcd,daki->alci", dV["ijab"], T), ("klcd,cdij->klij", dV["ijab"], T),
             ("kaic,cbkj->abij", dV["iajb"], T), ("kbic,ackj->abij", dV["iajb"], T),
             # row blocks as one rank of a sharded run sees them (parallel.Shard.rows)
             ("klcd,dblj->cbkj", bk.narrow(dV["ijab"], 2, lo, na), T),
             ("klcd,adkj->alcj", dV["ijab"], T[lo:lo + na]),
             ("klcd,daki->alci", dV["ijab"], T[:, lo:lo + na]),
             ("kaic,cbkj->abij", bk.narrow(dV["iajb"], 1, lo, na), T)]
    for spec, A, B in cases:
        bk.enable_trace(True)
        got = bk.contract(spec, A, B)
        labels = [lab for lab, _f, _t in bk.trace_report()]
        bk.enable_trace(False)
        assert len(labels) == 1 and labels[0].endswith("[momentum-blocked]"), (spec, labels)
        old = bk.set_blocked(False)
        try:
            ref = bk.contract(spec, A, B)
        finally:
            bk.set_blocked(old)
        want = torch.einsum(spec, A, B)
        assert _rel(got.cpu().numpy(), ref.cpu().numpy()) < 1e-13, spec
        assert _rel(got.cpu().numpy(), want.cpu().numpy()) < 1e-13, spec
    # accumulation with a coefficient into the ring sum, next to a dense term
    X = torch.randn(nv, no, nv, no, dtype=torch.float64, device="cuda", generator=g)
    R0 = torch.randn(nv, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
    R = R0.clone()
    bk.contract_terms("abij", [(-1.0, "kaic", dV["iajb"], "cbkj", T), (1.0, "alci", X, "cblj", T)], out=R, beta=1.0)
    want = R0 - torch.einsum("kaic,cbkj->abij", dV["iajb"], T) + torch.einsum("alci,cblj->abij", X, T)
    assert _rel(R.cpu().numpy(), want.cpu().numpy()) < 1e-13


@pytest.mark.parametrize("n_ele,cutoff", [(14, 5.0), (54, 7.0), (54, 10.0)])
def test_momentum_gather_t1_products(n_ele, cutoff):
    """pmb_gather_expand: products of a stored UEG o.v^3 block with T1 over ONE summed index, through
    the partner tables, against the dense kernel and a torch einsum of the same operands -- with a
    RANDOM T1 (T1 vanishes identically in the UEG, so the lock-step tests cannot see these values)."""
    from pymes_b200 import backend as bk
    m = _tc_model(n_ele, cutoff)
    no, nP = n_ele // 2, m.n_orb
    nv = nP - no
    parts = [("only_2b", m.trunc), ("effect_2b", m.trunc)]
    lo, na = nv // 3, nv - nv // 3 - 1
    dV = m.eval_2b_blocks(no, ["abic", "abci", "iabc"], parts)
    loc = m.eval_2b_blocks(no, ["abic", "abci", "iabc"], parts,
                           ranges={"abic": {0: (no + lo, na)}, "abci": {0: (no + lo, na)}, "iabc": {1: (no + lo, na)}})
    g = torch.Generator(device="cuda").manual_seed(4)
    T1 = torch.randn(nv, no, dtype=torch.float64, device="cuda", generator=g)
    old = bk.set_gather(True)
    try:
        for blocks in (dV, loc):
            for spec, key in (("abid,dj->abij", "abic"), ("abcj,ci->abij", "abci"), ("iabc,cj->iabj", "iabc"),
                              ("iacb,cj->iajb", "iabc")):
                A = blocks[key]
                bk.enable_trace(True)
                got = bk.contract(spec, A, T1)
                labels = [lab for lab, _f, _t in bk.trace_report()]
                bk.enable_trace(False)
                assert len(labels) == 1 and labels[0].endswith("[momentum-gather]"), (spec, labels)
                bk.set_gather(False)
                ref = bk.contract(spec, A, T1)
                bk.set_gather(True)
                want = torch.einsum(spec, A, T1)
                assert float(want.abs().max()) > 0
                assert _rel(got.cpu().numpy(), ref.cpu().numpy()) < 1e-13, spec
                assert _rel(got.cpu().numpy(), want.cpu().numpy()) < 1e-13, spec
        R0 = torch.randn(nv, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
        R = R0.clone()
        bk.contract_terms("abij", [(-0.5, "abcj", dV["abci"], "ci", T1)], out=R, beta=1.0)
        want = R0 - 0.5 * torch.einsum("abcj,ci->abij", dV["abci"], T1)
        assert _rel(R.cpu().numpy(), want.cpu().numpy()) < 1e-13
    finally:
        bk.set_gather(old)


def test_momentum_blocked_ladder_long_groups():
    """A group longer than the kernel's 512-entry offset window (several table refills per CTA) and
    more than 64 rows per group: a synthetic block-diagonal operand driven through the C ABI
    directly, against numpy."""
    import ctypes as C
    from pymes_b200 import _lib, backend as bk
    rng = np.random.default_rng(11)
    groups = [(130, 1100), (64, 513), (1, 1), (7, 40), (65, 16)]          # (rows, entries)
    n0e, n1e = 45, 3
    n_rows, n_ent = sum(g[0] for g in groups), sum(g[1] for g in groups)
    A = rng.standard_normal((n_rows, 1100))                                 # A[row, local entry]
    B = rng.standard_normal((n_ent, n1e, n0e + 3))                          # padded pitch
    Cm = rng.standard_normal((n_rows, n1e, n0e))
    perm = rng.permutation(n_rows)                                          # rows scattered in C
    tiles, want = [], Cm.copy()
    a_koff, r0, e0 = np.zeros(n_ent, dtype=np.int64), 0, 0
    for nr, ne in groups:
        a_koff[e0:e0 + ne] = np.arange(ne)
        for t in range(0, nr, 64):
            tiles.append((r0 + t, min(64, nr - t), e0, ne))
        blk = A[r0:r0 + nr, :ne] @ B[e0:e0 + ne, :, :n0e].reshape(ne, -1)
        want[perm[r0:r0 + nr]] = 0.5 * want[perm[r0:r0 + nr]] - 1.5 * blk.reshape(nr, n1e, n0e)
        r0, e0 = r0 + nr, e0 + ne
    dev = bk.device()
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    Ad, Bd, Cd = tt(A), tt(B), tt(Cm)
    tabs = [tt(np.arange(n_rows, dtype=np.int64) * 1100), tt(perm.astype(np.int64) * n1e * n0e), tt(a_koff),
            tt(np.arange(n_ent, dtype=np.int64) * n1e * (n0e + 3)), tt(np.array(tiles, dtype=np.int32))]
    d = _lib.Blocked()
    d.A, d.B, d.C = Ad.data_ptr(), Bd.data_ptr(), Cd.data_ptr()
    d.a_moff, d.c_moff, d.a_koff, d.b_koff, d.tiles = (t.data_ptr() for t in tabs)
    d.n_tiles, d.n0_ext, d.n1_ext, d.b_n1str, d.c_n1str = len(tiles), n0e, n1e, n0e + 3, n0e
    d.alpha, d.beta = -1.5, 0.5
    _lib.check(_lib.load().pmb_blocked_contract(C.byref(d), bk._stream()), "pmb_blocked_contract")
    torch.cuda.synchronize()
    assert _rel(Cd.cpu().numpy(), want) < 1e-13


def test_ueg_virtual_abcd_ccsd_matches_dense():
    """TC-UEG 14e CCSD with V_abcd never materialised == the same solve on dense blocks,
    sweep by sweep (energies 1e-12, amplitudes 1e-11 relative)."""
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd
    g = golden("ueg_tc")
    m = _tc_model(14, 5.0)
    m.k_cutoff = float(g["k_cutoff"])
    parts = [("only_2b", m.trunc), ("effect_2b", m.trunc)]
    dV = m.eval_2b_blocks(7, list(KEYS), parts)
    dVv = dict(dV)
    dVv["abcd"] = m.eval_2b_blocks(7, ["abcd"], parts, virtual=("abcd",))["abcd"]
    a, b = ccsd.CCSD(7), ccsd.CCSD(7)
    a.setup(g["fock"], dV)
    b.setup(g["fock"], dVv)
    for _ in range(6):
        ea, eb = a.sweep(), b.sweep()
        assert abs(sum(ea[:3]) - sum(eb[:3])) < 1e-12
        assert _rel(b._st["T2"].cpu().numpy(), a._st["T2"].cpu().numpy()) < 1e-11
        assert _rel(b._st["T1"].cpu().numpy(), a._st["T1"].cpu().numpy()) < 1e-11


def test_umat_golden():
    from pymes_b200.model import ueg
    g = golden("ueg_tc")
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(5.0)
    m.k_cutoff = float(g["k_cutoff"])
    m.gamma = None
    got = m.umat(g["umat_q"], m.trunc)
    np.testing.assert_allclose(got, g["umat"], rtol=1e-11)


# --------------------------------------------------------------------------
# size-independent properties at a size the oracle cannot reach quickly
# --------------------------------------------------------------------------
def test_pp_ladder_linearity_and_blas_crosscheck_large():
    """o=27, v=96: linearity in T and agreement with numpy's BLAS matmul on the same data."""
    from pymes_b200 import backend as bk
    no, nv = 27, 96
    g = torch.Generator(device="cuda").manual_seed(0)
    V = torch.randn(nv, nv, nv, nv, dtype=torch.float64, device="cuda", generator=g)
    T1 = torch.randn(nv, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
    T2 = torch.randn(nv, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
    R1 = bk.contract("abcd,cdij->abij", V, T1)
    R2 = bk.contract("abcd,cdij->abij", V, T2)
    R12 = bk.contract("abcd,cdij->abij", V, bk.lincomb([1.0, -2.5], [T1, T2]))
    lin = (R12 - (R1 - 2.5 * R2)).abs().max().item() / R12.abs().max().item()
    assert lin < 1e-13
    ref = V.cpu().numpy().reshape(nv * nv, nv * nv) @ T1.cpu().numpy().reshape(nv * nv, no * no)
    assert _rel(R1.cpu().numpy().reshape(nv * nv, no * no), ref) < 1e-13


def test_residual_no_symmetry_shortcut_medium():
    """Random blocks with no symmetry at o=6, v=30 against the oracle."""
    from pymes_b200.solver import ccd
    from oracle import cc_oracle as oc
    rng = np.random.default_rng(99)
    no, nv = 6, 30
    f = rng.standard_normal((no + nv, no + nv))
    T = 0.1 * rng.standard_normal((nv, nv, no, no))
    blk = dict(klij=(no,) * 4, ijab=(no, no, nv, nv), abij=(nv, nv, no, no), iajb=(no, nv, no, nv),
               iabj=(no, nv, nv, no), abcd=(nv,) * 4)
    args = [rng.standard_normal(blk[k]) for k in ("klij", "ijab", "abij", "iajb", "iabj", "abcd")]
    for flag in (False, True):
        got = ccd.CCD(no, is_dcd=flag).get_residual(f, T, *args)
        ref = oc.doubles_residual(no, f, T, *args, is_dcd=flag)
        assert _rel(got, ref) < 1e-12


def test_bdot_and_views():
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(0)
    V, T = rng.standard_normal((6, 6, 19, 19)), rng.standard_normal((19, 19, 6, 6))
    for spec in ["kica,caki->ai", "kjab,abkj->abj", "ijcd,cdij->ij", "kiab,abkj->abij", "klca,cakl->a",
                 "ijca,cbij->abij", "klab,abkl->ab"]:
        assert _rel(bk.bdot(spec, V, T).cpu().numpy(), np.einsum(spec, V, T)) < 1e-13, spec
    Vx = bk.asdev(rng.standard_normal((6, 19, 19, 6)))
    assert _rel(bk.diag_view(Vx, "iaai", "ai").cpu().numpy(), np.einsum("iaai->ai", Vx.cpu().numpy())) == 0


def test_eom_sigma_medium_random_vs_oracle():
    """o=5, v=14 random non-symmetric operands, 4 right-hand sides in one batch."""
    from pymes_b200.solver import eom_ccsd
    from oracle import cc_oracle as oc
    rng = np.random.default_rng(21)
    no, nv = 5, 14
    n = no + nv
    V = rng.standard_normal((n, n, n, n))
    dV = oc.partition(no, V)
    f = rng.standard_normal((n, n))
    T2 = 0.2 * rng.standard_normal((nv, nv, no, no))
    U1, U2 = rng.standard_normal((4, nv, no)), rng.standard_normal((4, nv, nv, no, no))
    eom = eom_ccsd.EOM_CCSD(no)
    S1, S2 = eom.sigma_batched(f, dV, U1, U2, T2)
    for r in range(4):
        assert _rel(S1[r].cpu().numpy(), oc.eom_sigma_singles(no, f, dV, U1[r], U2[r], T2)) < 1e-12
        assert _rel(S2[r].cpu().numpy(), oc.eom_sigma_doubles(no, f, dV, U1[r], U2[r], T2)) < 1e-12
    assert _rel(eom.get_diag_doubles(f, dV, T2), oc.eom_diag_doubles(no, f, dV, T2)) < 1e-12
    assert _rel(eom.get_diag_singles(f, dV, T2), oc.eom_diag_singles(no, f, dV, T2)) < 1e-12


# --------------------------------------------------------------------------
# SURVEY 8(f).2 / 8(f).3 on the CUDA path
# --------------------------------------------------------------------------
def test_drccd_residual_matches_reference():
    host.test_drccd_residual_matches_reference(None)


@pytest.mark.parametrize("tag", ["LiH", "LiHtc"])
@pytest.mark.parametrize("name,kw,sweeps", host.VARIANTS)
def test_ccd_variants_match_reference(tag, name, kw, sweeps):
    host.test_ccd_variants_match_reference(None, tag, name, kw, sweeps)


def test_ccd_rejects_non_contiguous_amps():
    host.test_ccd_rejects_non_contiguous_amps(None)


def test_rt_eom_step_matches_reference():
    """One real-time propagation step through the lock-step GMRES on the CUDA kernels (passed on a
    B200 in round 2's first GPU session as tests/test_gpu_next.py)."""
    host.test_rt_eom_step_matches_reference(None)


# --------------------------------------------------------------------------
# parity AT THE BENCHMARK'S OWN SHAPE: o = 27, the bench's own Hamiltonian path
# --------------------------------------------------------------------------
@pytest.mark.parametrize("virtual", [(), ("abcd",)], ids=["dense", "generated_abcd"])
@pytest.mark.parametrize("is_dcsd", [False, True], ids=["ccsd", "dcsd"])
def test_bench_path_54e_lockstep_with_oracle(virtual, is_dcsd):
    """TC-UEG 54 electrons / 65 plane waves (o = 27, v = 38) through exactly what bench.py runs --
    ``bench.build_fock`` + ``UEG.eval_2b_blocks(..., virtual=)`` + ``CCSD.setup / sweep`` -- in
    lock-step with the oracle's ``ccsd_sweep`` on the oracle-built Hamiltonian (the reference's
    triple loop restated, ueg_oracle.tc_hamiltonian): energy 1e-10 Eh, amplitudes 1e-9 relative,
    after every one of 3 sweeps."""
    import bench
    from oracle import cc_oracle as oc
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd
    no = bench.N_ELE // 2
    prob = bench.CpuProblem(6.0)
    assert prob.n_orb == 65
    m = ueg.UEG(bench.N_ELE, no, no, bench.RS)
    m.init_single_basis(6.0)
    m.k_cutoff, m.gamma = bench.K_CUTOFF, None
    fock = bench.build_fock(m, no)
    np.testing.assert_allclose(fock, prob.fock, rtol=1e-11, atol=1e-12)
    dV = m.eval_2b_blocks(no, list(KEYS), bench.tc_parts(m), virtual=virtual)
    for key in ("ijab", "abij", "iabc", "klij"):
        assert _rel(dV[key].cpu().numpy(), prob.dV[key]) < 1e-11, key
    cc = ccsd.CCSD(no, is_dcsd=is_dcsd)
    e_mp2 = cc.setup(fock, dV)
    e_ref, T2 = oc.mp2(prob.eps_i, prob.eps_a, prob.dV["ijab"], prob.dV["abij"])
    assert abs(e_mp2 - e_ref) < 1e-10
    T1 = np.zeros((prob.n_orb - no, no))
    d1, d2 = oc.denominators(prob.eps_i, prob.eps_a)
    mixer = oc.DIIS(6)
    for sweep in range(3):
        T1, T2, e, _ = oc.ccsd_sweep(no, prob.fock, prob.dV, T1, T2, d1, d2, mixer, is_dcsd=is_dcsd)
        got = cc.sweep()
        assert abs(sum(got[:3]) - sum(e)) < 1e-10, sweep
        assert _rel(cc._st["T2"].cpu().numpy(), T2) < 1e-9, sweep
        assert _rel(cc._st["T1"].cpu().numpy(), T1) < 1e-9, sweep


def test_two_rank_nccl_parity(tmp_path):
    """Two processes, one per GPU, NCCL: sharded CCSD/DCSD (LiH-TC, TC-UEG 14e with per-rank
    generated rows), row-sharded EOM sigma at o = 27, vector-parallel Davidson and system-parallel
    FEAST, each checked against the oracle / goldens inside tests/nccl_worker.py.  Skipped where
    fewer than two GPUs are visible."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from pymes_b200 import backend as bk
    assert float(bk.copy(torch.ones(3, 3, dtype=torch.float64, device="cuda")).sum()) == 9.0    # library loaded here too
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "nccl_parity.json"
    port = 29700 + os.getpid() % 200
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(root, "tests", "nccl_worker.py"), str(out)],
                         capture_output=True, text=True, timeout=1200, cwd=root)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "NCCL_PARITY_OK" in res.stdout


@pytest.mark.parametrize("M,N,K", [(1280, 1920, 1100), (1250, 1900, 1031), (128 * 149, 128, 2048), (2000, 9500, 1030)])
def test_tail_wave_split(M, N, K):
    """Grids of the warp-specialised kernel whose last wave is nearly empty are cut into full
    waves + a k-split tail launch (cc_contract.cu: tail_plan).  Result == numpy and == the same
    kernel with the tail left alone (tuning bit 64) to round-off; accumulation into C (beta = 1)
    and a strided C included."""
    from pymes_b200 import _lib, backend as bk
    g = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn(M, K, dtype=torch.float64, device="cuda", generator=g)
    B = torch.randn(K, N, dtype=torch.float64, device="cuda", generator=g)
    C0 = torch.randn(N, M, dtype=torch.float64, device="cuda", generator=g)
    lib = _lib.load()
    try:
        lib.pmb_contract_set_tuning(5, 0)
        before = bk.launch_count()
        got = bk.contract("mk,kn->mn", A, B)
        launches = bk.launch_count() - before
        acc = C0.clone()
        bk.contract("mk,kn->mn", A, B, out=acc.t(), alpha=0.5, beta=1.0)          # C stored transposed
        lib.pmb_contract_set_tuning(5 + 64, 0)
        before = bk.launch_count()
        plain = bk.contract("mk,kn->mn", A, B)
        assert bk.launch_count() - before == 1
    finally:
        lib.pmb_contract_set_tuning(-1, 0)
    tiles = ((M + 127) // 128) * ((N + 127) // 128)
    rest = tiles % 148
    assert launches == (3 if (tiles > 148 and 0 < rest <= 74) else 1)
    want = A.cpu().numpy() @ B.cpu().numpy()
    assert _rel(got.cpu().numpy(), want) < 1e-13
    assert _rel(plain.cpu().numpy(), got.cpu().numpy()) < 1e-13
    assert _rel(acc.t().cpu().numpy(), C0.t().cpu().numpy() + 0.5 * want) < 1e-13


def test_dots_and_lincomb_beyond_16_vectors():
    host.test_dots_and_lincomb_beyond_16_vectors(None)


# --------------------------------------------------------------------------
# BASELINE configs[2]: synthetic non-hermitian FCIDUMP-like integrals, generated on the device
# --------------------------------------------------------------------------
def test_synthetic_blocks_device_equals_host_and_ccsd():
    host.test_synthetic_tc_integrals_blockwise_and_ccsd(None)


@pytest.mark.parametrize("is_dcsd", [False, True], ids=["ccsd", "dcsd"])
def test_synthetic_o10_v60_lockstep_with_oracle(is_dcsd):
    """o = 10, v = 60 (the parity size the survey's C3 recipe names): every partition block written by
    pmb_synth_block is bit-identical to the host generator, V_abcd is STORED (dense operand of the
    ladder), and CCSD / DCSD follow the oracle sweep by sweep on the non-hermitian tensor."""
    from oracle import cc_oracle as oc
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd
    from pymes_b200.util import synthetic
    no, nv = 10, 60
    n = no + nv
    V = synthetic.tc_integrals(n, seed=0)
    assert np.abs(V - V.transpose(2, 3, 0, 1)).max() > 1e-5
    fock = synthetic.tc_fock(no, nv, seed=0)
    dV = synthetic.tc_blocks(no, nv, KEYS, seed=0, device=True)
    dVo = oc.partition(no, V)
    for key in KEYS:
        assert np.array_equal(dV[key].cpu().numpy(), dVo[key]), key
    cc = ccsd.CCSD(no, is_dcsd=is_dcsd)
    cc.setup(fock, dV)
    eps_i, eps_a = fock.diagonal()[:no].copy(), fock.diagonal()[no:].copy()
    _, T2 = oc.mp2(eps_i, eps_a, dVo["ijab"], dVo["abij"])
    T1 = np.zeros((nv, no))
    d1, d2 = oc.denominators(eps_i, eps_a)
    mixer = oc.DIIS(6)
    for sweep in range(4):
        T1, T2, e, _ = oc.ccsd_sweep(no, fock, dVo, T1, T2, d1, d2, mixer, is_dcsd=is_dcsd)
        got = cc.sweep()
        assert abs(sum(got[:3]) - sum(e)) < 1e-10, sweep
        assert _rel(cc._st["T2"].cpu().numpy(), T2) < 1e-9, sweep
        assert _rel(cc._st["T1"].cpu().numpy(), T1) < 1e-9, sweep


def test_synth_block_large_rows_statistics():
    """A 0.5 GB row block at the full problem's orbital count (n = 550): bit-identical to the host on a
    sampled sub-block, the (pq)(rs)<->(qp)(sr) symmetry holds across separately generated blocks, and the
    values are N(0,1)-distributed (size-independent checks for the block that is 500 GB at full size)."""
    from pymes_b200.util import synthetic
    n, no = 550, 50
    blk = synthetic.tc_block_device(n, (no + 7, no, no, no), (1, 500, 250, 500), seed=0, eps=1.0)
    sub = synthetic.tc_block(n, (no + 7, no + 100, no + 20, no + 3), (1, 5, 6, 7), seed=0, eps=1.0)
    assert np.array_equal(blk[:, 100:105, 20:26, 3:10].cpu().numpy(), sub)
    # V[p,q,r,s] = V[q,p,s,r]: rows generated as (q,p,s,r) from another block
    other = synthetic.tc_block_device(n, (no + 100, no + 7, no + 3, no + 20), (5, 1, 7, 6), seed=0, eps=1.0)
    assert torch.equal(other.permute(1, 0, 3, 2), blk[:, 100:105, 20:26, 3:10])
    assert abs(float(blk.mean())) < 1e-3 and abs(float(blk.std()) - 1.0) < 1e-3 and float(blk.abs().max()) < 4.5


@pytest.mark.parametrize("no,nv", [(6, 17), (27, 40), (50, 21)])
def test_elementwise_kernels_pair_rows_and_streams(no, nv):
    """Round-2 forms of the HBM-bound kernels: T-tilde and Ex + Ex^{baji} by row PAIRS (a,b),(b,a),
    the energy streaming an [a,b,i,j]-stored V_ijab (whole tensor and a row block), the strided copy
    with its 32-bit inner index split -- all against numpy, bit for bit where no sum is involved.
    Every o here runs the row-pair kernels: o = 50 still fits the two shared-memory rows of
    sym_baji (40000 of 49152 bytes).  The element-per-thread fallbacks (o >= 56 for sym_baji,
    o >= 65 for T-tilde) are covered in test_elementwise_edges.py."""
    from pymes_b200 import backend as bk
    from pymes_b200.solver import ccsd
    rng = np.random.default_rng(no * 100 + nv)
    T = rng.standard_normal((nv, nv, no, no))
    R = rng.standard_normal((nv, nv, no, no))
    V = rng.standard_normal((no, no, nv, nv))
    T1 = rng.standard_normal((nv, no))
    Td = bk.asdev(T)
    assert _rel(bk.tilde(Td).cpu().numpy(), 2 * T - T.transpose(1, 0, 2, 3)) == 0
    assert _rel(bk.tilde(Td, swap_ij=True).cpu().numpy(), 2 * T - T.transpose(0, 1, 3, 2)) == 0
    Rd = bk.asdev(R.copy())
    bk.sym_baji(Td, Rd, accumulate=True)
    assert _rel(Rd.cpu().numpy(), R + (T + T.transpose(1, 0, 3, 2))) < 1e-15
    assert _rel(bk.sym_baji(Td).cpu().numpy(), T + T.transpose(1, 0, 3, 2)) == 0
    Ve = ccsd.energy_layout(bk.asdev(V))
    assert tuple(Ve.shape) == (no, no, nv, nv) and Ve.stride(1) == 1 and torch.equal(Ve, bk.asdev(V))
    tau = T + np.einsum("ai,bj->abij", T1, T1)
    want = (2 * np.einsum("abij,ijab->", tau, V), -np.einsum("abij,ijba->", tau, V), np.sum(T * T))
    for Vdev in (Ve, bk.asdev(V)):                       # streamed rows / tiled gather: same sums
        scal = bk.zeros(8)
        bk.energy_doubles(Td, Vdev, scal, T1=bk.asdev(T1))
        s = scal.cpu().numpy()
        assert np.allclose(s[:3], want, rtol=1e-12, atol=1e-10)
    lo, na = nv // 3, nv - nv // 3 - 2
    scal = bk.zeros(8)
    bk.energy_doubles(bk.asdev(T[lo:lo + na].copy()), Ve, scal, T1=bk.asdev(T1), rows=(lo, na))
    part = (2 * np.einsum("abij,ijab->", tau[lo:lo + na], V[:, :, lo:lo + na]),
            -np.einsum("abij,ijba->", tau[lo:lo + na], V[:, :, :, lo:lo + na]), np.sum(T[lo:lo + na] ** 2))
    assert np.allclose(scal.cpu().numpy()[:3], part, rtol=1e-12, atol=1e-10)
    # strided copies: permuted source, strided destination, accumulation
    src = bk.asdev(V)
    assert _rel(bk.axpby(2.0, src.permute(2, 3, 0, 1)).cpu().numpy(), 2 * V.transpose(2, 3, 0, 1)) == 0
    big = bk.asdev(rng.standard_normal((nv + 3, no + 2, nv + 1, no + 5)))
    view = big[2:2 + nv, 1:1 + no, :nv, 3:3 + no]
    got = bk.axpby(-0.5, view.permute(0, 2, 1, 3), 1.0, Rd.clone())
    assert _rel(got.cpu().numpy(), Rd.cpu().numpy() - 0.5 * view.permute(0, 2, 1, 3).cpu().numpy()) < 1e-15
    out = bk.zeros(nv + 3, no + 2, nv + 1, no + 5)
    bk.axpby(1.0, Td.permute(0, 2, 1, 3), 0.0, out[2:2 + nv, 1:1 + no, :nv, 3:3 + no])
    assert torch.equal(out[2:2 + nv, 1:1 + no, :nv, 3:3 + no], Td.permute(0, 2, 1, 3)) and float(out[0].abs().max()) == 0


# --------------------------------------------------------------------------
# eval_2b_integrals: every branch and every correlator against the reference's triple loop
# --------------------------------------------------------------------------
@pytest.mark.parametrize("flag", host.UEG_FLAGS)
def test_ueg_remaining_branches_match_reference(flag):
    host.test_ueg_remaining_branches_match_reference(None, flag)


@pytest.mark.parametrize("name,gamma,k_cutoff", host.UEG_CORRELATORS)
def test_ueg_every_correlator_matches_reference(name, gamma, k_cutoff):
    host.test_ueg_every_correlator_matches_reference(None, name, gamma, k_cutoff)


@pytest.mark.parametrize("no,nv", [(27, 40), (7, 50), (10, 33)])
def test_sixteen_byte_operand_copies(no, nv):
    """An [.,.,o,o] operand in an even-pitch buffer (backend.empty_even_pitch: o^2 = 729 -> pitch 730) is
    copied into the tiles 16 bytes at a time by the warp-specialised kernel (b_vec2).  Same arithmetic
    as the 8-byte copies: results are bit-identical to the run with tuning bit 128 (8-byte copies), to the
    contiguous operand, and equal numpy to round-off; ragged last column tile, split-K and a second
    (8-byte) term in the same launch included."""
    from pymes_b200 import _lib, backend as bk
    g = torch.Generator(device="cuda").manual_seed(5)
    V = torch.randn(nv, nv, nv, nv, dtype=torch.float64, device="cuda", generator=g)
    T = torch.randn(nv, nv, no, no, dtype=torch.float64, device="cuda", generator=g)
    I = torch.randn(no, no, no, no, dtype=torch.float64, device="cuda", generator=g)
    Tp = bk.axpby(1.0, T, 0.0, bk.empty_even_pitch(nv, nv, no))
    assert torch.equal(Tp, T) and Tp.stride(1) % 2 == 0 and Tp.data_ptr() % 16 == 0
    lib = _lib.load()
    try:
        lib.pmb_contract_set_tuning(5, 0)
        plain = bk.contract("abcd,cdij->abij", V, T)
        vec = bk.contract("abcd,cdij->abij", V, Tp)
        two = bk.contract_terms("abij", [(0.5, "abcd", V, "cdij", Tp), (2.0, "abkl", T, "klij", I)])
        lib.pmb_contract_set_tuning(5, 3)
        vec_split = bk.contract("abcd,cdij->abij", V, Tp)
        lib.pmb_contract_set_tuning(5 + 128, 0)
        novec = bk.contract("abcd,cdij->abij", V, Tp)
        two_novec = bk.contract_terms("abij", [(0.5, "abcd", V, "cdij", Tp), (2.0, "abkl", T, "klij", I)])
        lib.pmb_contract_set_tuning(5 + 128, 3)
        novec_split = bk.contract("abcd,cdij->abij", V, Tp)
    finally:
        lib.pmb_contract_set_tuning(-1, 0)
    assert torch.equal(vec, novec) and torch.equal(vec, plain) and torch.equal(two, two_novec)
    assert torch.equal(vec_split, novec_split)
    want = V.cpu().numpy().reshape(nv * nv, -1) @ T.cpu().numpy().reshape(nv * nv, -1)
    assert _rel(vec.cpu().numpy().reshape(nv * nv, -1), want) < 1e-13


def test_eom_sigma_at_o27_vs_oracle():
    """Batched EOM-CCSD sigma at the benchmark's o = 27 (TC-UEG 54e / 65 plane waves, amplitudes after
    3 CCSD sweeps): with the dressed V_abcd stored AND with it as the never-materialised operator
    (ccsd.DressedLadder over the generated V_abcd), against the oracle's 62-term sigma, 1e-9 relative."""
    import bench
    from oracle import cc_oracle as oc
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd, eom_ccsd
    no = bench.N_ELE // 2
    prob = bench.CpuProblem(6.0)
    nv = prob.n_orb - no
    m = ueg.UEG(bench.N_ELE, no, no, bench.RS)
    m.init_single_basis(6.0)
    m.k_cutoff, m.gamma = bench.K_CUTOFF, None
    fock = bk.asdev(bench.build_fock(m, no))
    rng = np.random.default_rng(4)
    U1, U2 = rng.standard_normal((2, nv, no)), rng.standard_normal((2, nv, nv, no, no))
    results = []
    for virtual in ((), ("abcd",)):
        dV = m.eval_2b_blocks(no, list(KEYS), bench.tc_parts(m), virtual=virtual)
        cc = ccsd.CCSD(no)
        cc.setup(fock, dV)
        for _ in range(3):
            cc.sweep()
        T1, T2 = cc._st["T1"], cc._st["T2"]
        ft = cc.get_T1_dressed_fock(fock, T1, dV)
        dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
        assert isinstance(dVd["abcd"], bk.LinearOperator) == bool(virtual)
        plan = eom_ccsd.SigmaPlan(no, ft, {k: dVd[k] for k in eom_ccsd.V_KEYS_USED}, T2)
        S1, S2 = plan.apply(bk.asdev(U1), bk.asdev(U2))
        results.append((T1.cpu().numpy(), T2.cpu().numpy(), S1.cpu().numpy(), S2.cpu().numpy()))
    T1h, T2h = results[0][0], results[0][1]
    assert _rel(results[1][1], T2h) < 1e-11
    fto = oc.dressed_fock(no, prob.fock, T1h, prob.dV)
    dVo = oc.dressed_V(T1h, prob.dV)
    for k in range(2):
        s1 = oc.eom_sigma_singles(no, fto, dVo, U1[k], U2[k], T2h)
        s2 = oc.eom_sigma_doubles(no, fto, dVo, U1[k], U2[k], T2h)
        for _t1, _t2, S1, S2 in results:
            assert _rel(S1[k], s1) < 1e-9 and _rel(S2[k], s2) < 1e-9
