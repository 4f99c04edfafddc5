#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ by RUNNING THE REFERENCE.

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py [section ...]

The unmodified reference (nickirk/pymes @ 734974a) is imported from
/root/reference with the three shims SURVEY.md 8(c) lists (none touches
arithmetic): a dummy ``ctf`` module (pymes/solver/dcd.py:4 imports it and never
uses it), ``gcrotmk(tol=)`` -> ``rtol=`` for scipy >= 1.14, and a seeded
``np.random``.  The ``rt`` section needs two more, also outside the arithmetic
(see ``sec_rt``): ``RT_EOM_CCSD`` never sets ``ls_max_iter`` and still calls the
ctf-era ``.to_nparray()`` on numpy arrays.  Outputs are small ``.npz`` files; the
tests never need the reference itself.
"""
import io
import os
import sys
import types
import contextlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
sys.dont_write_bytecode = True
sys.modules["ctf"] = types.ModuleType("ctf")
sys.path.insert(0, REF)

import scipy.sparse.linalg as _sla  # noqa: E402

_gcrotmk = _sla.gcrotmk


def _gcrotmk_compat(A, b, x0=None, *, tol=None, rtol=1e-5, **kw):
    return _gcrotmk(A, b, x0=x0, rtol=(tol if tol is not None else rtol), **kw)


_sla.gcrotmk = _gcrotmk_compat

from pymes.solver import ccd, ccsd, dcd, mp2, eom_ccsd, feast_eom_ccsd  # noqa: E402
from pymes.mixer import diis  # noqa: E402
from pymes.mean_field import hf  # noqa: E402
from pymes.model import ueg  # noqa: E402
from pymes.util import fcidump  # noqa: E402
from pymes.integral.partition import part_2_body_int  # noqa: E402

TESTDIR = os.path.join(REF, "pymes", "test")


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


class Tracer:
    """Record the energy printed at every sweep by wrapping get_energy."""

    def __init__(self, solver):
        self.e = []
        self._inner = solver.get_energy
        solver.get_energy = self

    def __call__(self, *a):
        out = self._inner(*a)
        self.e.append(float(np.real(sum(out))))
        return out


def pack_integrals(V):
    """V[p,q,r,s] of a real FCIDUMP is exactly invariant under p<->r and under q<->s: keep the
    non-zeros with p <= r and q <= s.  tests/conftest.py::golden rebuilds V from them exactly."""
    p, q, r, s = np.indices(V.shape)
    keep = (p <= r) & (q <= s) & (V != 0)
    for perm in ((2, 1, 0, 3), (0, 3, 2, 1)):
        assert np.array_equal(V, V.transpose(perm))
    return dict(n=V.shape[0], mask=np.packbits(keep.ravel()), val=V[keep])


def molecule(tag, path, is_tc=False, eom_roots=0, delta_e=1e-12, max_iter=200, pack_V=False):
    n_elec, nb, e_core, eps, h, V = quiet(fcidump.read, path, is_tc)
    no = n_elec // 2
    out = dict(n_elec=n_elec, e_core=e_core, h=h, V=V, is_tc=is_tc)
    if pack_V:          # a dense V of 32 orbitals alone would be 3.7 MB compressed
        save("mol_" + tag + "_V", **pack_integrals(out.pop("V")))
    out["hf_e"] = hf.calc_hf_e(no, e_core, h, V)
    fock = hf.construct_hf_matrix(no, h, V)
    out["fock"] = fock
    for name, is_dcd in (("ccd", False), ("dcd", True)):
        cc = ccd.CCD(no, is_dcd=is_dcd)
        tr = Tracer(cc)
        r = quiet(cc.solve, fock, V, delta_e=delta_e, max_iter=max_iter)
        out[name + "_e"] = r["ccd e"]
        out[name + "_trace"] = np.array(tr.e)
        out[name + "_t2"] = r["t2 amp"]
    for name, is_dcsd in (("ccsd", False), ("dcsd", True)):
        cc = ccsd.CCSD(no, is_dcsd=is_dcsd)
        tr = Tracer(cc)
        r = quiet(cc.solve, fock, V, delta_e=delta_e, max_iter=max_iter)
        out[name + "_e"] = r["ccsd e"]
        out[name + "_trace"] = np.array(tr.e)
        out[name + "_t1"] = r["t1"]
        out[name + "_t2"] = r["t2"]
        if name == "ccsd" and eom_roots:
            dV = part_2_body_int(no, V)
            ft = cc.get_T1_dressed_fock(fock, r["t1"].copy(), dV)
            dVt = cc.get_T1_dressed_V(r["t1"].copy(), dV)
            eom = eom_ccsd.EOM_CCSD(no, n_excit=eom_roots)
            eom.max_iter = 1000
            out["eom_e"] = quiet(eom.solve, ft, dVt, r["t2"].copy())
    save("mol_" + tag, **out)


def sec_molecules():
    molecule("LiH_321g", os.path.join(TESTDIR, "test_ccsd/FCIDUMP.LiH.321g"),
             eom_roots=2)
    molecule("LiH_tc", os.path.join(TESTDIR, "test_tc_ccsd/FCIDUMP.LiH.tc"),
             is_tc=True)
    molecule("H2_321g", os.path.join(TESTDIR, "test_eom_ccsd/FCIDUMP.H2.321g"),
             eom_roots=2)


def sec_hf_molecule():
    # 32 orbitals, 43 CCSD sweeps: exercises the DIIS-full bookkeeping path
    molecule("HF_augccpvdz",
             os.path.join(TESTDIR, "test_eom_ccsd/FCIDUMP.HF.augccpvdz"),
             delta_e=1e-8, max_iter=50, pack_V=True)


def sec_residual_random():
    rng = np.random.default_rng(7)
    for tag, no, nv in (("a", 3, 5), ("b", 4, 9)):
        nP = no + nv
        fock = rng.standard_normal((nP, nP))
        T2 = rng.standard_normal((nv, nv, no, no)) * 0.3
        blocks = dict(
            klij=rng.standard_normal((no,) * 4),
            ijab=rng.standard_normal((no, no, nv, nv)),
            abij=rng.standard_normal((nv, nv, no, no)),
            iajb=rng.standard_normal((no, nv, no, nv)),
            iabj=rng.standard_normal((no, nv, nv, no)),
            abcd=rng.standard_normal((nv,) * 4))
        out = dict(no=no, fock=fock, T2=T2, **blocks)
        for name, flag in (("R_ccd", False), ("R_dcd", True)):
            out[name] = ccd.CCD(no, is_dcd=flag).get_residual(
                fock, T2, blocks["klij"], blocks["ijab"], blocks["abij"],
                blocks["iajb"], blocks["iabj"], blocks["abcd"])
        ed, ex = ccd.CCD(no).get_energy(T2, blocks["ijab"])
        out["e_dir"], out["e_ex"] = ed, ex
        eps_i = -1.0 - rng.random(no)
        eps_a = 1.0 + rng.random(nv)
        e, t = mp2.solve(eps_i, eps_a, blocks["ijab"], blocks["abij"], 0.3)
        out.update(eps_i=eps_i, eps_a=eps_a, mp2_e=e, mp2_t2=t, mp2_shift=0.3)
        save("residual_random_" + tag, **out)


def sec_dressing_random():
    rng = np.random.default_rng(11)
    for tag, no, nv in (("a", 2, 3), ("b", 3, 6)):
        nP = no + nv
        V = rng.standard_normal((nP,) * 4)          # no symmetry at all
        fock = rng.standard_normal((nP, nP))
        T1 = rng.standard_normal((nv, no)) * 0.4
        T2 = rng.standard_normal((nv, nv, no, no)) * 0.3
        cc = ccsd.CCSD(no)
        dV = part_2_body_int(no, V)
        ft = cc.get_T1_dressed_fock(fock, T1, dV)
        dVt = cc.get_T1_dressed_V(T1, dV)
        out = dict(no=no, V=V, fock=fock, T1=T1, T2=T2, fock_dressed=ft,
                   R1=cc.get_singles_residual(ft, T1, T2, dV),
                   R2=cc.get_doubles_residual(ft, T2, dVt))
        e1, ed, ex = cc.get_energy(fock[:no, no:], T1, T2, dV["ijab"])
        out.update(e_1b=e1, e_dir=ed, e_ex=ex)
        none_keys = []
        for k, v in dVt.items():
            if v is None:
                none_keys.append(k)
            else:
                out["dressed_" + k] = v
        out["none_keys"] = np.array(none_keys)
        # EOM sigma / diagonals on the same dressed quantities
        eom = eom_ccsd.EOM_CCSD(no, n_excit=2)
        u1 = rng.standard_normal((nv, no))
        u2 = rng.standard_normal((nv, nv, no, no))
        out.update(u1=u1, u2=u2,
                   sigma1=eom.update_singles(ft, dVt, u1, u2, T2),
                   sigma2=eom.update_doubles(ft, dVt, u1, u2, T2),
                   diag1=eom.get_diag_singles(ft, dVt, T2),
                   diag2=eom.get_diag_doubles(ft, dVt, T2))
        save("dressing_random_" + tag, **out)


def sec_diis():
    rng = np.random.default_rng(3)
    mixer = diis.DIIS(dim_space=4)
    errs, amps, outs, Ls = [], [], [], []
    for it in range(9):                      # passes the full-subspace branch 5x
        e = [rng.standard_normal((3, 2)) * 0.5 ** it,
             rng.standard_normal((3, 3, 2, 2)) * 0.5 ** it]
        a = [rng.standard_normal((3, 2)), rng.standard_normal((3, 3, 2, 2))]
        o = quiet(mixer.mix, e, a)
        errs.append(e), amps.append(a), outs.append(o), Ls.append(mixer.L.copy())
    out = {}
    for n, (e, a, o, L) in enumerate(zip(errs, amps, outs, Ls)):
        out.update({f"e1_{n}": e[0], f"e2_{n}": e[1], f"a1_{n}": a[0],
                    f"a2_{n}": a[1], f"o1_{n}": o[0], f"o2_{n}": o[1],
                    f"L_{n}": L})
    save("diis_sequence", dim_space=4, n_calls=9, **out)


def _ueg_setup(nel, rs, cutoff):
    m = ueg.UEG(nel, nel // 2, nel // 2, rs)
    quiet(m.init_single_basis, cutoff)
    nP = len(m.basis_fns) // 2
    kint = np.array([m.basis_fns[2 * i].k for i in range(nP)])
    kin = np.array([m.basis_fns[2 * i].kinetic for i in range(nP)])
    return m, nP, kint, kin


def _sparse(V):
    idx = np.flatnonzero(V)
    return idx.astype(np.int64), V.ravel()[idx]


def sec_ueg_coulomb():
    out = {}
    for tag, rs, shift in (("rs1", 1.0, 0.0), ("rs05", 0.5, -1.0)):
        m, nP, kint, kin = _ueg_setup(14, rs, 5.0)
        V = quiet(m.eval_2b_integrals, sp=0)
        no = 7
        fock = hf.construct_hf_matrix(no, np.diag(kin), V)
        idx, val = _sparse(V)
        out.update({tag + "_kint": kint, tag + "_kin": kin, tag + "_L": m.L,
                    tag + "_imax": m.imax, tag + "_V_idx": idx,
                    tag + "_V_val": val, tag + "_fock": fock,
                    tag + "_map": m.basis_indices_map})
        cc = ccd.CCD(no)
        tr = Tracer(cc)
        r = quiet(cc.solve, fock, V, level_shift=shift)
        out[tag + "_ccd_e"], out[tag + "_ccd_trace"] = r["ccd e"], np.array(tr.e)
        t2 = r["t2 amp"]
        cc = dcd.DCD(no)
        tr = Tracer(cc)
        if tag == "rs05":      # test_ccd_dcd.py:176-181 warm-starts DCD from CCD
            r = quiet(cc.solve, fock, V, level_shift=shift, amps=t2.copy())
        else:
            r = quiet(cc.solve, fock, V, level_shift=shift)
        out[tag + "_dcd_e"], out[tag + "_dcd_trace"] = r["ccd e"], np.array(tr.e)
    # basis sizes of the closed shells the benchmark uses (SURVEY appendix B)
    sizes = []
    for nel, cut in ((14, 2.0), (14, 5.0), (14, 9.0), (54, 3.0), (54, 6.0),
                     (54, 10.0), (54, 13.0)):
        m, nP, kint, kin = _ueg_setup(nel, 1.0, cut)
        sizes.append((nel, cut, nP))
        out[f"basis_{nel}_{int(cut)}_kint"] = kint
    out["basis_sizes"] = np.array(sizes)
    save("ueg_coulomb", **out)


def sec_ueg_tc():
    """TC-UEG following test_symmetrised_2body_integral.py:41-220 (14e, rs 0.5)."""
    nel, rs, cutoff, no = 14, 0.5, 5.0, 7
    m, nP, kint, kin = _ueg_setup(nel, rs, cutoff)
    m.gamma = None
    m.k_cutoff = 1.0
    V2 = quiet(m.eval_2b_integrals, correlator=m.trunc, is_only_2b=True, sp=0)
    eps_i = hf.calcOccupiedOrbE(kin, V2[:no, :no, :no, :no], no)
    eps_a = hf.calcVirtualOrbE(kin, V2[no:, :no, no:, :no], V2[no:, :no, :no, no:],
                               no, nP - no)
    occ = V2[:no, :no, :no, :no]
    e_hf = 2 * np.sum(eps_i) - (2.0 * np.einsum("jiji->", occ)
                                - np.einsum("ijji->", occ))
    fock = hf.construct_hf_matrix(no, np.diag(kin), V2)
    Veff = quiet(m.eval_2b_integrals, correlator=m.trunc, is_effect_2b=True, sp=0)
    V = V2 + 0.5 * (Veff + Veff.transpose(1, 0, 3, 2))
    one_body = quiet(m.double_contractions_in_3_body)
    zero_body = quiet(m.triple_contractions_in_3_body)
    eps_i = eps_i + one_body[:no]
    eps_a = eps_a + one_body[no:]
    fock = fock + np.diag(one_body)
    e_mp2, _ = mp2.solve(eps_i, eps_a, t_V_abij=V[no:, no:, :no, :no],
                         t_V_ijab=V[:no, :no, no:, no:])
    cc = ccd.CCD(no)
    tr = Tracer(cc)
    r = quiet(cc.solve, fock, V)
    i2, v2 = _sparse(V2)
    ie, ve = _sparse(Veff)
    # u_mat(q) table for every distinct q the build needs
    qs = sorted({tuple(kint[r_] - kint[p]) for p in range(nP) for r_ in range(nP)})
    qs = np.array(qs)
    umat = np.array([m.sumNablaUSquare(2 * np.pi / m.L * q.astype(float))
                     for q in qs[::37]])
    save("ueg_tc", kint=kint, kin=kin, L=m.L, Omega=m.Omega, imax=m.imax,
         k_cutoff=m.k_cutoff, gamma=m.gamma, V2_idx=i2, V2_val=v2, Veff_idx=ie,
         Veff_val=ve, e_hf=e_hf, fock=fock, one_body=one_body,
         zero_body=zero_body, e_mp2=e_mp2, ccd_e=r["ccd e"],
         ccd_trace=np.array(tr.e), umat_q=qs[::37], umat=umat)


def sec_feast():
    """One seeded FEAST linear solve + sigma on complex vectors (LiH)."""
    path = os.path.join(TESTDIR, "test_ccsd/FCIDUMP.LiH.321g")
    n_elec, nb, e_core, eps, h, V = quiet(fcidump.read, path)
    no = n_elec // 2
    fock = hf.construct_hf_matrix(no, h, V)
    cc = ccsd.CCSD(no)
    r = quiet(cc.solve, fock, V, delta_e=1e-12, max_iter=200)
    dV = part_2_body_int(no, V)
    ft = cc.get_T1_dressed_fock(fock, r["t1"].copy(), dV)
    dVt = cc.get_T1_dressed_V(r["t1"].copy(), dV)
    T2 = r["t2"].copy()
    np.random.seed(5)
    fe = feast_eom_ccsd.FEAST_EOM_CCSD(no, e_c=0.13, e_r=0.05, n_trial=2,
                                       max_iter=3)
    d1 = fe.get_diag_singles(ft, dVt, T2)
    d2 = fe.get_diag_doubles(ft, dVt, T2)
    u1 = 0.5 - np.random.rand(*d1.shape)
    u2 = (0.5 - np.random.rand(*d2.shape)) * 0.01
    u1, u2 = feast_eom_ccsd.normalize_amps(u1, u2)
    fe.u_singles, fe.u_doubles = [u1.copy()], [u2.copy()]
    z = 0.13 + 0.05 * np.exp(1j * 0.7)
    q1, q2 = quiet(fe._gcrotmk, 0, z, d1, d2, ft, dVt, T2)
    # seeded full solve
    np.random.seed(5)
    fe2 = feast_eom_ccsd.FEAST_EOM_CCSD(no, e_c=0.13, e_r=0.05, n_trial=2,
                                        max_iter=3)
    eig = quiet(fe2.solve, ft, dVt, T2)
    save("feast_LiH", u1=u1, u2=u2, z=z, q1=q1, q2=q2, diag1=d1, diag2=d2,
         eigvals=np.asarray(eig), t1=r["t1"], t2=T2, e_c=0.13, e_r=0.05)


class _NdWithToNparray(np.ndarray):
    """numpy array that also answers the ctf-era ``.to_nparray()`` the reference still calls in
    rt_eom_ccsd.py:84-85 (returns itself: no arithmetic is touched)."""

    def to_nparray(self):
        return np.asarray(self)


def sec_rt():
    """One RT-EOM-CCSD propagation step (rt_eom_ccsd.py:64-133) on LiH.  Two more shims, both
    outside the arithmetic: the class never calls its parent's __init__, so ``ls_max_iter``
    (read by ``_gcrotmk``) is set by hand to the parent's default 20, and the diagonals are
    handed back as ndarray subclasses that accept ``.to_nparray()``."""
    from pymes.solver import rt_eom_ccsd
    path = os.path.join(TESTDIR, "test_ccsd/FCIDUMP.LiH.321g")
    n_elec, nb, e_core, eps, h, V = quiet(fcidump.read, path)
    no = n_elec // 2
    fock = hf.construct_hf_matrix(no, h, V)
    cc = ccsd.CCSD(no)
    r = quiet(cc.solve, fock, V, delta_e=1e-12, max_iter=200)
    dV = part_2_body_int(no, V)
    ft = cc.get_T1_dressed_fock(fock, r["t1"].copy(), dV)
    dVt = cc.get_T1_dressed_V(r["t1"].copy(), dV)
    T2 = r["t2"].copy()
    rt = rt_eom_ccsd.RT_EOM_CCSD(no, e_c=0.2, e_r=0.6, dt=0.1)
    rt.ls_max_iter = 20
    for name in ("get_diag_singles", "get_diag_doubles"):
        orig = getattr(rt, name)
        setattr(rt, name, (lambda f: lambda *a: np.asarray(f(*a)).view(_NdWithToNparray))(orig))
    rng = np.random.default_rng(3)
    nv = T2.shape[0]
    u1 = rng.standard_normal((nv, no))
    u2 = 0.1 * rng.standard_normal((nv, nv, no, no))
    u1, u2 = feast_eom_ccsd.normalize_amps(u1, u2)
    q1, q2 = quiet(rt.solve, ft, dVt, T2, dt=0.1, u_singles=u1.copy(), u_doubles=u2.copy())
    # second step from the (complex) result of the first
    p1, p2 = quiet(rt.solve, ft, dVt, T2, dt=0.1, u_singles=q1.copy(), u_doubles=q2.copy())
    save("rt_LiH", u1=u1, u2=u2, q1=q1, q2=q2, p1=p1, p2=p2, e_c=0.2, e_r=0.6, dt=0.1, t1=r["t1"], t2=T2)

def sec_variants():
    """The two CCD variants SURVEY 8(f).2 lists, exactly as the reference EXECUTES them:
    ``is_dr_ccd`` (drccd.py:10-39; its einsum strings sum k over V alone and carry j as a
    batch index) and ``is_bruekner`` (ccd.py:104-121, 207-221: product denominator, and the
    Fock matrix is modified in place through the views t_X_ac / t_X_ki)."""
    from pymes.solver import drccd
    rng = np.random.default_rng(23)
    out = {}
    no, nv = 3, 5
    eps_i = -1.0 - rng.random(no)
    eps_a = 1.0 + rng.random(nv)
    T2 = rng.standard_normal((nv, nv, no, no)) * 0.3
    blk = dict(abij=rng.standard_normal((nv, nv, no, no)), aijb=rng.standard_normal((nv, no, no, nv)),
               iabj=rng.standard_normal((no, nv, nv, no)), ijab=rng.standard_normal((no, no, nv, nv)))
    out.update(rnd_no=no, rnd_eps_i=eps_i, rnd_eps_a=eps_a, rnd_T2=T2,
               **{"rnd_" + k: v for k, v in blk.items()})
    out["rnd_R_drccd"] = drccd.get_residual(eps_i, eps_a, T2, blk["abij"], blk["aijb"], blk["iabj"], blk["ijab"])
    for tag, path, is_tc in (("LiH", "test_ccsd/FCIDUMP.LiH.321g", False),
                             ("LiHtc", "test_tc_ccsd/FCIDUMP.LiH.tc", True)):
        n_elec, nb, e_core, eps, h, V = quiet(fcidump.read, os.path.join(TESTDIR, path), is_tc)
        no = n_elec // 2
        fock = hf.construct_hf_matrix(no, h, V)
        out.update({tag + "_no": no, tag + "_V": V, tag + "_fock": fock})
        for name, kw, sweeps in (("drccd", dict(is_dr_ccd=True), 4), ("drccd_nodiis", dict(is_dr_ccd=True, is_diis=False), 4),
                                 ("bruekner", dict(is_bruekner=True), 2),
                                 ("bruekner_nodiis", dict(is_bruekner=True, is_diis=False), 2),
                                 ("bruekner_dcd", dict(is_bruekner=True, is_dcd=True), 2)):
            cc = ccd.CCD(no, **kw)
            tr = Tracer(cc)
            f = fock.copy()
            r = quiet(cc.solve, f, V, max_iter=sweeps - 1, delta_e=1e-14)
            key = tag + "_" + name
            out.update({key + "_e": r["ccd e"], key + "_trace": np.array(tr.e), key + "_t2": r["t2 amp"],
                        key + "_hole": np.array(r["hole e"]), key + "_particle": np.array(r["particle e"]),
                        key + "_fock_after": f, key + "_dE": r["dE"]})
    save("ccd_variants", **out)

def sec_ueg_modes():
    """Every branch of eval_2b_integrals that ueg_tc does not cover (ueg.py:416-423, 440-457,
    478-504) with the `trunc` correlator at 14e / 57 plane waves, and every correlator of
    ueg.py:740-956 through the `only_2b` (array arguments via sumNablaUSquare, scalar ones via
    the loop) and `effect_2b` branches at 14e / 19 plane waves.  One shim outside the
    arithmetic: sumNablaUSquare is MEMOISED on its argument (the reference recomputes the same
    226 981-term lattice sum for every (p, r) pair: 190 s per build at 57 plane waves)."""
    out = {}

    def memoised(m):
        inner, cache = m.sumNablaUSquare, {}

        def wrapped(k, cutoff=30):
            key = tuple(np.round(np.asarray(k, dtype=float) * m.L / (2 * np.pi)).astype(int))
            if key not in cache:
                cache[key] = inner(k, cutoff)
            return cache[key]
        m.sumNablaUSquare = wrapped

    m, nP, kint, kin = _ueg_setup(14, 0.5, 5.0)
    m.gamma, m.k_cutoff = None, 1.0
    memoised(m)
    out.update(big_kint=kint, big_L=m.L, big_k_cutoff=1.0)
    for flag in ("is_rpa_approx", "is_only_hermi_2b", "is_only_non_hermi_2b", "is_exchange_1",
                 "is_exchange_2", "is_exchange_3"):
        V = quiet(m.eval_2b_integrals, correlator=m.trunc, sp=0, **{flag: True})
        idx, val = _sparse(V)
        out["big_" + flag + "_idx"], out["big_" + flag + "_val"] = idx, val
        print(flag, len(idx), "non-zeros")
    # a correlator given without any branch flag: all zeros (the elif chain falls through)
    V = quiet(m.eval_2b_integrals, correlator=m.trunc, sp=0)
    out["big_noflag_absmax"] = np.abs(V).max()
    save("ueg_modes_branches", **out)       # kept apart: together with the rest it exceeds 1 MB
    out = {}
    for name, gamma, k_cutoff in (("trunc", None, 1.0), ("coulomb", None, None), ("smooth", None, 1.0),
                                  ("yukawa", None, None), ("yukawa", 0.7, 1.0), ("stg", None, None), ("stg", 1.3, 1.0),
                                  ("yukawa_coulomb", None, None), ("yukawa_coulomb", 1.1, 1.0),
                                  ("gaskell", None, None), ("gaskell", 0.9, 2.0),
                                  ("gaskell_modified", None, None), ("gaskell_modified", None, 1.0)):
        m, nP, kint, kin = _ueg_setup(14, 1.0, 2.0)
        m.gamma, m.k_cutoff = gamma, k_cutoff
        memoised(m)
        corr = getattr(m, name)
        tag = "%s_g%s_k%s" % (name, gamma, k_cutoff)
        try:
            for flag in ("is_only_2b", "is_effect_2b"):
                V = quiet(m.eval_2b_integrals, correlator=corr, sp=0, **{flag: True})
                idx, val = _sparse(V)
                out["c_" + tag + "_" + flag + "_idx"], out["c_" + tag + "_" + flag + "_val"] = idx, val
            out["c_" + tag + "_gamma_after"] = np.nan if m.gamma is None else m.gamma
            out["c_" + tag + "_kc_after"] = np.nan if m.k_cutoff is None else m.k_cutoff
            print(tag, "ok")
        except Exception as exc:                                  # noqa: BLE001
            out["c_" + tag + "_raises"] = np.array(type(exc).__name__)
            print(tag, "raises", type(exc).__name__, exc)
    out["small_kint"] = kint
    out["small_L"] = m.L
    # trunc mutates an ndarray argument in place (ueg.py:797)
    m, nP, kint, kin = _ueg_setup(14, 1.0, 2.0)
    m.gamma, m.k_cutoff = None, 1.0
    arg = np.linspace(0.0, 3.0, 13)
    res = m.trunc(arg)
    out["trunc_arg_after"], out["trunc_res"] = arg, res
    save("ueg_modes", **out)


SECTIONS = dict(molecules=sec_molecules, hf_molecule=sec_hf_molecule,
                residual_random=sec_residual_random,
                dressing_random=sec_dressing_random, diis=sec_diis,
                ueg_coulomb=sec_ueg_coulomb, ueg_tc=sec_ueg_tc, feast=sec_feast, rt=sec_rt, variants=sec_variants, ueg_modes=sec_ueg_modes)

if __name__ == "__main__":
    for name in (sys.argv[1:] or list(SECTIONS)):
        print("==", name)
        SECTIONS[name]()
