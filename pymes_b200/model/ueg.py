"""3D uniform electron gas: plane-wave basis and momentum-conserving integrals.

Call surface of the reference ``pymes.model.ueg.UEG`` (pymes/model/ueg.py:12-516):
``UEG(n_ele, n_alpha, n_beta, rs)``, ``init_single_basis(cutoff, k_shift)``,
``eval_2b_integrals(correlator, is_*..., dtype, sp)``, the attributes ``basis_fns, L,
Omega, gamma, k_cutoff, imax, basis_indices_map, correlator`` and the correlators
as bound methods.

The basis is generated on the host in the reference's floating-point arithmetic
(shell membership at the cutoff and the order inside degenerate shells depend
on it, SURVEY 7.3).  The integral build runs on the device in three steps
(``pmb_ueg_umat`` -> ``pmb_ueg_pair_tables`` -> ``pmb_ueg_build_block``), see
include/pymes_b200.h; ``eval_2b_blocks`` builds named sub-blocks directly so that
V_pqrs never has to exist for systems where it would not fit.
"""
import ctypes as C
import time
import warnings

import numpy as np
import torch
from scipy import special

from .. import _lib
from .. import backend as bk
from ..basis_set import planewave
from ..integral.partition import OCCUPIED
from ..log import print_logging_info

MODES = {"coulomb": 0, "rpa": 1, "only_2b": 2, "only_hermi_2b": 3, "only_non_hermi_2b": 4,
         "effect_2b": 5, "exchange_1": 6, "exchange_2": 7, "exchange_3": 8}


class UEG:
    def __init__(self, n_ele, n_alpha, n_beta, rs):
        if n_ele % 2 != 0 or int(n_alpha) != int(n_beta):
            warnings.warn("The number of electrons is not even, currently only "
                          "closed shell systems are supported!")
        self.n_ele = int(n_ele)
        self.n_alpha = int(n_alpha)
        self.n_beta = int(n_beta)
        self.rs = rs
        self.L = self.rs * ((4 * np.pi * self.n_ele) / 3) ** (1.0 / 3.0)     # ueg.py:66
        self.Omega = self.L ** 3
        self.basis_fns = None
        self.imax = 0
        self.cutoff = 0.
        self.basis_indices_map = None
        self.kPrime = None
        self.correlator = None
        self.k_cutoff = None
        self.gamma = None
        self._dev = None

    # ------------------------------------------------------------------ basis
    def is_k_in_basis(self, ke):
        return bool(ke <= self.cutoff * (2 * np.pi / self.L) ** 2 / 2.)      # ueg.py:100-103

    def init_basis_indices_map(self):
        n = self.imax * 2 + 1
        table = -1 * np.ones(n ** 3).astype(int)
        for i in range(len(self.basis_fns) // 2):
            k = self.basis_fns[2 * i].k
            table[n * n * (k[0] + self.imax) + n * (k[1] + self.imax) + k[2] + self.imax] = i
        self.basis_indices_map = table

    def init_single_basis(self, cutoff, k_shift=[0., 0., 0.]):
        k_shift = np.array(k_shift)
        imax = int(np.ceil(np.sqrt(cutoff + k_shift.dot(k_shift)))) + 1      # ueg.py:153
        self.cutoff = cutoff
        self.imax = imax
        fns = []
        rng = range(-imax, imax + 1)
        for i in rng:
            for j in rng:
                for k in rng:
                    up = planewave.BasisFunc(i, j, k, self.L, 1, k_shift)
                    if self.is_k_in_basis(up.kinetic):
                        fns.append(up)
                        fns.append(planewave.BasisFunc(i, j, k, self.L, -1, k_shift))
        fns.sort()                                   # stable, key = kinetic (planewave.py:25-26)
        self.basis_fns = tuple(fns)
        self.init_basis_indices_map()
        self._dev = None
        return self.basis_fns

    @property
    def n_orb(self):
        return len(self.basis_fns) // 2

    def k_int(self):
        return np.array([self.basis_fns[2 * i].k for i in range(self.n_orb)], dtype=np.int32)

    def k_float(self):
        return np.array([self.basis_fns[2 * i].kp for i in range(self.n_orb)], dtype=np.float64)

    def kinetic(self):
        return np.array([self.basis_fns[2 * i].kinetic for i in range(self.n_orb)])

    # --------------------------------------------------------- device build
    def _device_state(self):
        if self._dev is None:
            dev = bk.device()
            self._dev = dict(
                kvec=torch.from_numpy(self.k_int().reshape(-1)).to(dev),
                kp=torch.from_numpy(self.k_float().reshape(-1)).to(dev),
                imap=torch.from_numpy(self.basis_indices_map.astype(np.int32)).to(dev))
        return self._dev

    def _descriptor(self, u_table=None):
        st = self._device_state()
        d = _lib.Ueg()
        d.n_orb, d.imax, d.n_occ, d.n_ele = self.n_orb, self.imax, self.n_ele // 2, self.n_ele
        d.omega = self.Omega
        d.u_table = u_table.data_ptr() if u_table is not None else None
        d.u_table_len = u_table.numel() if u_table is not None else 0
        d.kvec, d.kp, d.index_map = st["kvec"].data_ptr(), st["kp"].data_ptr(), st["imap"].data_ptr()
        return d

    def _correlator_table(self, correlator, lattice_cutoff):
        """u(n2 (2 pi/L)^2) for every integer n2 = |k|^2 the build can ask for."""
        kmax = int(np.abs(self.k_int()).max())
        # largest |component| any kernel asks for: lattice vector +- transfer vectors in the
        # u_mat sum, and sums of up to four basis vectors in contract_exchange_3_body /
        # contractP_KWithQ (ueg.py:518-573) -- the latter wins for kmax > lattice_cutoff + 1
        reach = max(lattice_cutoff + 3 * kmax, 4 * kmax) + 1
        n2 = np.arange(3 * reach * reach + 1, dtype=np.float64)
        vals = np.asarray(correlator(n2 * (2 * np.pi / self.L) ** 2), dtype=np.float64)
        return torch.from_numpy(np.ascontiguousarray(vals)).to(bk.device())

    def _umat_device(self, desc, q_int, lattice_cutoff):
        lib = _lib.load()
        q_int = np.ascontiguousarray(np.asarray(q_int).reshape(-1, 3).astype(np.int32))
        qdev = torch.from_numpy(q_int.reshape(-1)).to(bk.device())
        out = bk.empty(len(q_int))
        _lib.check(lib.pmb_ueg_umat(C.byref(desc), float(self.L), int(lattice_cutoff), len(q_int),
                                    bk._ptr(qdev), bk._ptr(out), bk._stream()), "pmb_ueg_umat")
        return out

    def umat(self, q_int, correlator, lattice_cutoff=30):
        """u_mat(q) = sum_k' (k'.(q-k')) u(k'^2) u((q-k')^2) / Omega over the [-30,30]^3 lattice
        (``sumNablaUSquare``, ueg.py:581-596) for integer transfer vectors ``q_int`` [nq,3]."""
        self.correlator = correlator
        u_table = self._correlator_table(correlator, lattice_cutoff)
        desc = self._descriptor(u_table)
        return self._umat_device(desc, q_int, lattice_cutoff).cpu().numpy()

    # Correlators whose value at every lattice point is insensitive to the last bits of the
    # argument (continuous there, or switched with a guard band like trunc's 1 + 1e-5): for these
    # the device kernels may look the correlator up in a table over the integer |k|^2.
    _TABLE_SAFE = ("trunc", "coulomb", "smooth")

    def _wants_exact_arguments(self, correlator):
        """Must the correlator be evaluated at the reference's own floating-point arguments?
        ``self.exact_correlator_arguments`` = True / False forces it; None (default) decides by the
        correlator: yukawa, stg, yukawa_coulomb, gaskell, gaskell_modified and user callables compare
        k^2 with a cutoff without a guard band, and when that cutoff is exactly the squared length of
        a lattice shell the reference's answer depends on the rounding of its k-vector differences
        (e.g. 3x - 2x against 2x - x), pair by pair and lattice term by lattice term."""
        flag = getattr(self, "exact_correlator_arguments", None)
        if flag is not None:
            return bool(flag)
        func = getattr(correlator, "__func__", None)
        return not (getattr(correlator, "__self__", None) is self and func is not None
                    and func.__name__ in self._TABLE_SAFE)

    def _pair_tables_exact(self, mode, correlator, lattice_cutoff):
        """W0 / W1 of one branch of ueg.py:411-504 with every correlator argument formed exactly as
        the reference forms it (same numpy calls, same order, one (p, r) pair at a time) -- O(nP^2 n_occ)
        host work on the nP x nP tables; the dense block is still written by the device."""
        from functools import partial
        einsum = partial(np.einsum, optimize=True)                          # ueg.py:10
        nP, nocc = self.n_orb, self.n_ele // 2
        kp, kint = self.k_float(), self.k_int().astype(np.int64)
        occ = np.array([kp[i] for i in range(nocc)])
        omega, n_ele = self.Omega, self.n_ele
        lattice = np.array([[i, j, k] for i in range(-lattice_cutoff, lattice_cutoff + 1)
                            for j in range(-lattice_cutoff, lattice_cutoff + 1)
                            for k in range(-lattice_cutoff, lattice_cutoff + 1)])
        umat_cache = {}

        def u_mat(q_int, k):                                                # ueg.py:581-596
            key = tuple(int(x) for x in q_int)
            if key not in umat_cache:
                k1 = 2 * np.pi * lattice / self.L
                k2 = k - k1
                res = einsum("ni,ni->n", k1, k2) * correlator(einsum("ni,ni->n", k1, k1)) \
                    * correlator(einsum("ni,ni->n", k2, k2))
                umat_cache[key] = einsum("n->", res) / omega
            return umat_cache[key]

        def ex3(p_vec, kvec):                                               # ueg.py:518-542
            pv = p_vec - occ
            res = einsum("ni,i->n", pv, kvec) * correlator(einsum("i,i->", kvec, kvec)) \
                * correlator(einsum("ni,ni->n", pv, pv))
            return einsum("n->", res) / omega

        def pk(p_vec, kvec):                                                # ueg.py:544-573
            v1, v2 = p_vec - kvec - occ, p_vec - occ
            res = einsum("ni,ni->n", v1, v2) * correlator(einsum("ni,ni->n", v1, v1)) \
                * correlator(einsum("ni,ni->n", v2, v2))
            return einsum("n->", res) / omega

        W0, W1 = np.zeros((nP, nP)), np.zeros((nP, nP))
        need_umat = mode in ("only_2b", "only_hermi_2b")
        for p in range(nP):
            for r in range(nP):
                d = kp[r] - kp[p]
                d2 = d.dot(d)
                nz = np.abs(d2) > 0.
                um = u_mat(kint[r] - kint[p], d) if need_umat else 0.
                if mode == "rpa":
                    if nz:
                        W0[p, r] = (-n_ele * d2 * correlator(d2) ** 2 / omega) / omega
                elif mode in ("only_2b", "only_hermi_2b"):
                    W0[p, r] = (4. * np.pi / d2 + um + d2 * correlator(d2)) / omega if nz else um / omega
                    if nz and mode == "only_2b":
                        W1[p, r] = -correlator(d2) / omega
                elif mode == "only_non_hermi_2b":
                    if nz:
                        W0[p, r] = (4. * np.pi / d2) / omega
                        W1[p, r] = -correlator(d2) / omega
                elif mode == "effect_2b":
                    if nz:
                        w = -n_ele * d2 * correlator(d2) ** 2 / omega + 2. * ex3(kp[r], d) - 2. * ex3(kp[p], d) \
                            + 2. * pk(kp[r], d)
                    else:
                        w = 2. * pk(kp[r], d)
                    W0[p, r] = w / omega
                elif mode == "exchange_1":
                    if nz:
                        W0[p, r] = 2. * ex3(kp[r], d) / omega
                elif mode == "exchange_2":
                    if nz:
                        W0[p, r] = -2. * ex3(kp[p], d) / omega
                elif mode == "exchange_3":
                    W0[p, r] = 2. * pk(kp[r], d) / omega
                else:
                    raise ValueError(mode)
        return bk.asdev(W0.reshape(-1)), bk.asdev(W1.reshape(-1))

    def pair_tables(self, mode, correlator=None, lattice_cutoff=30):
        """(W0, W1) for one branch of ueg.py:411-504: nP x nP tables of the (p, r)-only factors."""
        lib = _lib.load()
        nP = self.n_orb
        if mode != "coulomb" and correlator is not None and self._wants_exact_arguments(correlator):
            self.correlator = correlator
            return self._pair_tables_exact(mode, correlator, lattice_cutoff)
        u_table = None
        if mode != "coulomb":
            if correlator is None:
                raise ValueError("mode %s needs a correlator" % mode)
            self.correlator = correlator
            u_table = self._correlator_table(correlator, lattice_cutoff)
        desc = self._descriptor(u_table)
        umat_pr = None
        if mode in ("only_2b", "only_hermi_2b"):
            k = self.k_int().astype(np.int64)
            q = (k[None, :, :] - k[:, None, :]).reshape(-1, 3)          # q[p*nP+r] = k_r - k_p
            uniq, inverse = np.unique(q, axis=0, return_inverse=True)
            umat_q = self._umat_device(desc, uniq, lattice_cutoff)
            idx = torch.from_numpy(inverse.reshape(-1).astype(np.int64)).to(bk.device())
            umat_pr = umat_q[idx].contiguous()
        W0, W1 = bk.empty(nP * nP), bk.empty(nP * nP)
        _lib.check(lib.pmb_ueg_pair_tables(C.byref(desc), MODES[mode],
                                           bk._ptr(umat_pr) if umat_pr is not None else None,
                                           bk._ptr(W0), bk._ptr(W1), bk._stream()), "pmb_ueg_pair_tables")
        return W0, W1

    def build_block(self, lo, ext, W0a=None, W1a=None, W0s=None, out=None):
        """Dense block V[lo:lo+ext] from pair tables (device tensor [ext0,ext1,ext2,ext3])."""
        lib = _lib.load()
        if out is None:
            out = bk.empty(*ext)
        desc = self._descriptor()
        p = lambda t: bk._ptr(t) if t is not None else None
        _lib.check(lib.pmb_ueg_build_block(C.byref(desc), p(W0a), p(W1a), p(W0s), _lib.I32x4(*lo),
                                           _lib.I32x4(*ext), bk._ptr(out), bk._stream()),
                   "pmb_ueg_build_block")
        return out

    def build_nz(self, lo, ext, W0a=None, W1a=None, W0s=None):
        """Momentum-compressed block [ext0,ext1,ext2]: V[p,q,r,s*(p,q,r)] where s* falls into the
        block's s range, else 0 (``pmb_ueg_build_nz``) -- the one candidate non-zero per dense row."""
        lib = _lib.load()
        out = bk.empty(*ext[:3])
        desc = self._descriptor()
        p = lambda t: bk._ptr(t) if t is not None else None
        _lib.check(lib.pmb_ueg_build_nz(C.byref(desc), p(W0a), p(W1a), p(W0s), _lib.I32x4(*lo),
                                        _lib.I32x4(*ext), bk._ptr(out), bk._stream()), "pmb_ueg_build_nz")
        return out

    def _mode_of(self, correlator, is_rpa_approx, is_only_2b, is_only_non_hermi_2b, is_only_hermi_2b,
                 is_effect_2b, is_exchange_1, is_exchange_2, is_exchange_3):
        if correlator is None:
            return "coulomb"
        for flag, name in ((is_rpa_approx, "rpa"), (is_only_2b, "only_2b"),
                           (is_only_hermi_2b, "only_hermi_2b"),
                           (is_only_non_hermi_2b, "only_non_hermi_2b"), (is_effect_2b, "effect_2b"),
                           (is_exchange_1, "exchange_1"), (is_exchange_2, "exchange_2"),
                           (is_exchange_3, "exchange_3")):
            if flag:                       # same precedence as the elif chain ueg.py:411-504
                return name
        return None

    def eval_2b_integrals(self, correlator=None, is_rpa_approx=False, is_only_2b=False,
                          is_only_non_hermi_2b=False, is_only_hermi_2b=False, is_effect_2b=False,
                          is_exchange_1=False, is_exchange_2=False, is_exchange_3=False,
                          dtype=np.float64, sp=1, device=False):
        """Dense V_pqrs [nP,nP,nP,nP] (numpy by default, CUDA tensor with ``device=True``)."""
        t0 = time.time()
        print_logging_info(__name__, level=0)
        if self.basis_fns is None:
            raise ValueError("Basis functions not initialized!")
        if correlator is not None:
            self.correlator = correlator
            print_logging_info("Using TC method", level=1)
            print_logging_info("Using correlator: ", correlator.__name__, level=1)
        mode = self._mode_of(correlator, is_rpa_approx, is_only_2b, is_only_non_hermi_2b,
                             is_only_hermi_2b, is_effect_2b, is_exchange_1, is_exchange_2, is_exchange_3)
        nP = self.n_orb
        if mode is None:                   # correlator given but no branch selected: all zeros
            V = bk.zeros(nP, nP, nP, nP)
        else:
            W0, W1 = self.pair_tables(mode, correlator)
            if mode == "effect_2b":        # symmetrised under (pq)(rs)<->(qp)(sr), ueg.py:509-513
                V = self.build_block((0,) * 4, (nP,) * 4, W0s=W0)
            else:
                V = self.build_block((0,) * 4, (nP,) * 4, W0a=W0, W1a=W1)
        if correlator is not None:
            if self.k_cutoff is not None:
                print_logging_info("k_cutoff in correlator = {:.8f}".format(self.k_cutoff), level=1)
            if self.gamma is not None:
                print_logging_info("Gamma in correlator = {:.8f}".format(self.gamma), level=1)
        out = V if device else V.cpu().numpy().astype(dtype, copy=False)
        print_logging_info("{:.3f} s spent on ".format(time.time() - t0) + __name__, level=1)
        return out

    def virtual_block(self, lo, ext, W0a=None, W1a=None, W0s=None, compressed=True):
        """The block ``build_block`` would write, as a never-materialised operand (SURVEY 8(f).1):
        handed to ``backend.contract_terms`` in place of a tensor, its tiles are produced by the
        contraction kernel's producer warps, bit-identical to the dense block.  ``compressed``:
        the non-zero values (one per dense row, ``build_nz``) are stored and looked up; otherwise
        the producers evaluate the integral formula in place."""
        return VirtualBlock(self, lo, ext, W0a, W1a, W0s, compressed=compressed)

    def eval_2b_blocks(self, no, keys, parts, ranges=None, virtual=()):
        """Named sub-blocks (partition.py keys, e.g. "abcd") of a SUM of integral kinds,
        built directly on the device: ``parts`` is a list of ``(mode, correlator)``;
        ``effect_2b`` parts enter symmetrised exactly as in
        test_symmetrised_2body_integral.py:141-145.  ``ranges`` = ``{key: {dim: (lo, n)}}`` restricts
        a dimension of a block to absolute orbital indices [lo, lo+n) (the row block one rank of
        a sharded run owns).  Keys listed in ``virtual`` (e.g. ``("abcd",)``) come back as
        :class:`VirtualBlock` operands instead of tensors.  Returns ``{key: cuda tensor}``."""
        nP = self.n_orb
        tabs = []
        for mode, corr in parts:
            W0, W1 = self.pair_tables(mode, corr)
            tabs.append((mode, W0, W1))
        plain = [t for t in tabs if t[0] != "effect_2b"]
        sym = [t for t in tabs if t[0] == "effect_2b"]
        W0a = W1a = W0s = None
        if plain:
            W0a = plain[0][1] if len(plain) == 1 else bk.lincomb([1.0] * len(plain), [t[1] for t in plain])
            W1a = plain[0][2] if len(plain) == 1 else bk.lincomb([1.0] * len(plain), [t[2] for t in plain])
        if sym:
            W0s = sym[0][1] if len(sym) == 1 else bk.lincomb([1.0] * len(sym), [t[1] for t in sym])
        out, geom = {}, {}
        for key in keys:
            lo = [0 if ch in OCCUPIED else no for ch in key]
            ext = [no if ch in OCCUPIED else nP - no for ch in key]
            for dim, (r_lo, r_n) in (ranges or {}).get(key, {}).items():
                lo[dim], ext[dim] = int(r_lo), int(r_n)
            geom[key] = (tuple(lo), tuple(ext))
        # V_iabc and V_aibc meet the same tau in every sweep: allocated back to back they are one
        # operand of one launch (solver.ccsd.pair_with_tau)
        pre = {}
        if "iabc" in geom and "aibc" in geom and not {"iabc", "aibc"} & set(virtual) and \
                int(np.prod(geom["iabc"][1])) == int(np.prod(geom["aibc"][1])):
            pre["iabc"], pre["aibc"] = bk.empty_stacked(geom["iabc"][1], geom["aibc"][1])
        for key in keys:
            lo, ext = geom[key]
            if key in virtual:
                out[key] = self.virtual_block(lo, ext, W0a=W0a, W1a=W1a, W0s=W0s)
            else:
                out[key] = bk.tag_block(self.build_block(lo, ext, W0a=W0a, W1a=W1a, W0s=W0s, out=pre.get(key)),
                                        momentum_rule(self, lo, ext))
                if key in BLOCKED_COMPANIONS:
                    # stored AND available as compressed values (1/v of the block): V.tau of the
                    # T1 dressing runs momentum-blocked (solver.ccsd.pair_with_tau)
                    out[key]._pmb_blocked = self.virtual_block(lo, ext, W0a=W0a, W1a=W1a, W0s=W0s)
        return out

    # ------------------------------------------------- 3-body mean-field parts
    def _occupied_k(self):
        return self.k_float()[: self.n_ele // 2]

    def triple_contractions_in_3_body(self):
        """Scalar mean-field energy of the 3-body operator (ueg.py:598-630).  The correlator (a host
        callable) is evaluated on the |k_i - k_j|^2 table; the contractions run on the device
        (``pmb_bdot`` / ``pmb_dots``: batch-index products, not matrix products)."""
        ki = self._occupied_k()
        d = ki[:, None, :] - ki[None, :, :]
        d2 = np.einsum("pqi,pqi->pq", d, d)
        u = bk.asdev(self.correlator(d2.copy()))
        dd, d2d = bk.asdev(d), bk.asdev(d2)
        u2 = bk.bdot("pq,pq->pq", u, u)
        direct = float(bk.dots([u2.reshape(-1)], d2d.reshape(-1)).item()) * self.n_ele / 2 / self.Omega ** 2 * 2
        # sum_{pqo} (d_po . d_pq) u_pq u_po = sum_p | sum_q u_pq d_pq |^2
        Y = bk.bdot("pqi,pq->pi", dd, u)
        exch = -2 * 2 * float(bk.dots([Y.reshape(-1)], Y.reshape(-1)).item()) / 2. / self.Omega ** 2
        return direct + exch

    def double_contractions_in_3_body(self):
        """One-body energies from doubly contracted 3-body terms (ueg.py:632-733), contractions on the
        device as above; returns a numpy array like the reference."""
        kp, ki = self.k_float(), self._occupied_k()
        dpi = kp[:, None, :] - ki[None, :, :]                    # p - i
        dpi2 = np.einsum("pij,pij->pi", dpi, dpi)
        upi = bk.asdev(self.correlator(dpi2.copy()))
        dij = ki[:, None, :] - ki[None, :, :]
        dij2 = np.einsum("ijk,ijk->ij", dij, dij)
        uij = bk.asdev(self.correlator(dij2.copy()))
        dpi_d, dpi2_d, dij_d, dij2_d = bk.asdev(dpi), bk.asdev(dpi2), bk.asdev(dij), bk.asdev(dij2)
        om2 = self.Omega ** 2
        upi2 = bk.bdot("pi,pi->pi", upi, upi)
        perl = bk.bdot("pi,pi->p", upi2, dpi2_d, alpha=2.0 * self.n_ele / om2 / 2)
        Y = bk.bdot("pik,pi->pk", dpi_d, upi)                    # sum_i u_pi (p - i)
        wave = bk.bdot("pk,pk->p", Y, Y, alpha=-2.0 / om2 / 2)
        uij2 = bk.bdot("ij,ij->ij", uij, uij)
        shield = float(bk.dots([uij2.reshape(-1)], dij2_d.reshape(-1)).item()) * 2 / 2 / om2
        Z = bk.bdot("ijk,ij->ik", dij_d, uij)                    # sum_j u_ij (i - j)
        W = bk.bdot("pik,pi->pik", dpi_d, upi)
        frog = bk.bdot("pik,ik->p", W, Z, alpha=4.0 / om2 / 2)   # -(...)(-dpi) of ueg.py:725-731
        out = bk.lincomb([1.0, 1.0, 1.0], [perl, wave, frog])
        return bk.tonumpy(out) + shield

    # ------------------------------------------------------------ correlators
    # u(k^2); scalar or array argument.  ueg.py:740-956
    def _defaults(self, gamma):
        if self.k_cutoff is None:
            self.k_cutoff = int(np.ceil(np.sqrt(self.cutoff)))
        if self.gamma is None:
            self.gamma = gamma

    def trunc(self, kSquare):
        """-4 pi gamma / k^4 for k > k_c, else 0 (ueg.py:772-800)."""
        self._defaults(1.0)
        kc2 = (self.k_cutoff * 2 * np.pi / self.L) ** 2
        if isinstance(kSquare, np.ndarray):
            # the reference zeroes the small entries of ITS ARGUMENT in place (ueg.py:797): an
            # observable side effect on the caller's array, kept
            kSquare[kSquare <= kc2 * (1 + 0.00001)] = 0.
            k2 = np.asarray(kSquare, dtype=np.float64)
        else:
            k2 = np.array(0. if kSquare <= kc2 * (1 + 0.00001) else kSquare, dtype=np.float64)
        res = np.divide(-4. * np.pi, k2 ** 2, out=np.zeros_like(k2), where=(k2 > 1e-12)) * self.gamma
        return res if isinstance(kSquare, np.ndarray) else float(res)

    def coulomb(self, kSquare, multiply_by_k_square=False):
        g = 1. if self.gamma is None else self.gamma
        k2 = np.asarray(kSquare, dtype=np.float64)
        return np.divide(-4. * np.pi * g, k2, out=np.zeros_like(k2), where=k2 > 1e-12)

    def smooth(self, kSquare, multiply_by_k_square=False):
        self._defaults(0.01)
        kc = np.sqrt((self.k_cutoff * 2 * np.pi / self.L) ** 2)
        k2 = np.asarray(kSquare, dtype=np.float64)
        num = -4. * np.pi * (1. + special.erf((np.sqrt(k2) - kc) / (kc * self.gamma))) / 2.
        return np.divide(num, k2 ** 2, out=np.zeros_like(k2), where=k2 > (kc * self.gamma) ** 2)

    def yukawa(self, kSquare, multiply_by_k_square=False):
        g0 = np.sqrt(self.n_ele / self.Omega / 4. * np.pi)
        g = g0 if self.gamma is None else self.gamma * g0
        floor = 1e-12 if self.k_cutoff is None else self.k_cutoff * (2 * np.pi / self.L) ** 2 + g
        b = np.asarray(kSquare, dtype=np.float64) + g
        return np.divide(-4. * np.pi, b, out=np.zeros_like(b), where=np.abs(b) > floor)

    def stg(self, kSquare, multiply_by_k_square=False):
        g = np.sqrt(4. * np.pi * self.n_ele / self.Omega) if self.gamma is None else self.gamma
        floor = 1e-12 if self.k_cutoff is None else (self.k_cutoff * (2 * np.pi / self.L) ** 2 + g ** 2) ** 2
        b = (np.asarray(kSquare, dtype=np.float64) + g ** 2) ** 2
        return np.divide(-4. * np.pi / g, b, out=np.zeros_like(b), where=np.abs(b) > floor)

    def yukawa_coulomb(self, kSquare, multiply_by_k_square=False):
        g = 1.5 if self.gamma is None else self.gamma
        A = g / np.sqrt(self.Omega / (4.0 * np.pi * self.n_ele))
        floor = 1e-12 if self.k_cutoff is None else self.k_cutoff * (2 * np.pi / self.L) ** 2 + A
        k2 = np.asarray(kSquare, dtype=np.float64)
        b = (k2 + A) * k2
        return np.divide(-4. * np.pi, b, out=np.zeros_like(b), where=np.abs(b) > floor)

    def gaskell(self, kSquare, multiply_by_k_square=False):
        mu = np.sqrt(4. * np.pi * self.Omega / self.n_ele) * (1. if self.gamma is None else self.gamma)
        kf = self.basis_fns[(self.n_ele // 2) * 2].kp
        kf2 = kf.dot(kf)
        kc2 = 4. * kf2 if self.k_cutoff is None else self.k_cutoff ** 2 * kf2
        # the reference branches on isinstance(kSquare, np.ndarray): a 0-d ARRAY (what
        # einsum(..., optimize=True) returns for "i,i->") takes the array branch, whose cutoff test
        # is `>` while the scalar branch's is `<` -- they differ exactly at k^2 == cutoff
        if not isinstance(kSquare, np.ndarray):
            return -(mu / kSquare) if (1e-12 < kSquare < kc2) else -0.0
        k2 = np.asarray(kSquare, dtype=np.float64)
        res = np.divide(mu, k2, out=np.zeros_like(k2), where=(k2 > 1e-12))
        res[k2 > kc2] = 0.
        return -res

    def gaskell_modified(self, kSquare, multiply_by_k_square=False):
        kc2 = 2 if self.k_cutoff is None else (self.k_cutoff * (2 * np.pi / self.L)) ** 2
        if not isinstance(kSquare, np.ndarray):          # same dispatch as the reference (see gaskell)
            return -0.0 if (1e-12 < kSquare < kc2) else -(4 * np.pi / kSquare ** 2)
        k2 = np.asarray(kSquare, dtype=np.float64)
        return -np.divide(4 * np.pi, k2 ** 2, out=np.zeros_like(k2), where=(k2 >= kc2))


SIGNS = (1, 1, -1, -1)            # <pq|rs>: l(k_p) + l(k_q) - l(k_r) - l(k_s) = 0


def momentum_groups(k_int, imax, lo, ext, m_axes=(0, 1), k_axes=(2, 3)):
    """Block-diagonal structure of V[lo:lo+ext] as the matrix [rows, entries], rows = the two
    axes ``m_axes`` of (p,q,r,s), entries = the other two (``k_axes``).  The reference finds
    the one s of a (p,q,r) by looking up the LINEARISED vector k_q - (k_r - k_p) in its index map
    (ueg.py:395-404: loc = n^2 (x + imax) + n (y + imax) + z + imax, n = 2 imax + 1, only the range
    of loc is checked, not that of the components), so an element can be non-zero exactly where
    l(k_p) + l(k_q) = l(k_r) + l(k_s) with l(k) = n^2 x + n y + z: the momentum-conserving
    elements and the few aliased ones the reference produces as well (a component beyond imax
    carries into the next digit).  With signs (+,+,-,-) for (p,q,r,s), a row and an entry can
    meet where  sum_rows sign.l = - sum_entries sign.l ; rows and entries with the same key form a
    group.  Returns ``(row_ord, ent_ord, g_row0, g_rows, g_ent0, g_ents)``: the rows i0*ext[m1]+i1 /
    the entries j0*ext[k1]+j1 of the groups present on BOTH sides, sorted by group (index order
    inside a group), and per group its first position and length in the two lists
    (``backend.block_groups``).  ``(g_rows * g_ents).sum()`` is the number of candidate non-zeros
    (54e / 515 plane waves, V_abcd: 3.3e7 of 5.7e10)."""
    if sorted(tuple(m_axes) + tuple(k_axes)) != [0, 1, 2, 3]:
        raise ValueError("row and entry axes must split (p,q,r,s)")
    return bk.block_groups(bk.Momentum(linearise(k_int, imax), zip(lo, ext, SIGNS)), m_axes, k_axes)


def linearise(k, imax):
    """l(k) = n^2 x + n y + z (n = 2 imax + 1) of integer momenta ``k[..., 3]``: the label the
    reference's index lookup conserves (see :func:`momentum_groups`)."""
    k = np.asarray(k).astype(np.int64)
    n = 2 * int(imax) + 1
    return n * n * k[..., 0] + n * k[..., 1] + k[..., 2]


def linear_momenta(model):
    """:func:`linearise` of every orbital's momentum; cached on the model."""
    lin = model.__dict__.get("_pmb_lin")
    if lin is None:
        lin = model.__dict__["_pmb_lin"] = linearise(model.k_int(), model.imax)
    return lin


class ExcitationSector:
    """One total-momentum sector of the excitations of a UEG reference: the singles a <- i with
    l(k_a) - l(k_i) = l(K) and the doubles ab <- ij with l(k_a) + l(k_b) - l(k_i) - l(k_j) = l(K).
    Made by :func:`excitation_sector`; it hands out the momentum rules (``backend.Momentum``) of
    the tensors an EOM solve in the sector meets, so that the solver never sees the linearised
    labels themselves."""

    def __init__(self, lin, no, label, K=None):
        self.lin, self.no, self.label = lin, int(no), int(label)
        self.nv = len(lin) - self.no
        self.K = None if K is None else tuple(int(x) for x in K)

    def __repr__(self):
        return "ExcitationSector(K=%s, l(K)=%d)" % (self.K, self.label)

    def __eq__(self, other):
        return isinstance(other, ExcitationSector) and self.no == other.no and self.label == other.label \
            and np.array_equal(self.lin, other.lin)

    def __hash__(self):
        return hash((self.no, self.label, len(self.lin)))

    def rule(self, key, total=0):
        """Rule of a tensor indexed like ``key`` (occupied letters i-l, virtual a-h; two indices
        signed (+,-), four (+,+,-,-), the integral blocks' <pq|rs> convention) with ``total``."""
        if len(key) not in (2, 4):
            raise ValueError("a rule for 2 or 4 indices, not %r" % key)
        signs = (1, -1) if len(key) == 2 else SIGNS
        axes = [((0, self.no) if ch in "ijkl" else (self.no, self.nv)) + (sg,) for ch, sg in zip(key, signs)]
        return bk.Momentum(self.lin, axes, total=total)

    def fock_rule(self):
        """Rule of the (dressed) Fock matrix over all orbitals: momentum-diagonal."""
        n = self.no + self.nv
        return bk.Momentum(self.lin, [(0, n, 1), (0, n, -1)])

    def singles_rule(self):
        return self.rule("ai", self.label)

    def doubles_rule(self):
        return self.rule("abij", self.label)

    def singles_mask(self):
        """[v, o] booleans: the singles of the sector."""
        lo, lv = self.lin[:self.no], self.lin[self.no:]
        return (lv[:, None] - lo[None, :]) == self.label

    def packed_index(self):
        """Sorted int64 offsets of the sector's elements in the packed [singles | doubles] layout of
        length v.o + v^2.o^2 (``SigmaPlan.apply_packed``): the singles a,i with l_a - l_i = l(K), then
        v.o + the doubles a,b,i,j with l_a + l_b - l_i - l_j = l(K).  Built one virtual a at a time
        (one [v, o^2] mask), cached on the sector."""
        if getattr(self, "_packed", None) is None:
            no, nv = self.no, self.nv
            lo, lv = np.asarray(self.lin[:no], dtype=np.int64), np.asarray(self.lin[no:], dtype=np.int64)
            n1, blk = nv * no, nv * no * no
            lij = (lo[:, None] + lo[None, :]).reshape(-1)
            parts = [np.flatnonzero(self.singles_mask())]
            for a in range(nv):
                hit = np.flatnonzero((lv[:, None] - lij[None, :]) == self.label - lv[a])
                parts.append(n1 + a * blk + hit)
            self._packed = np.concatenate(parts).astype(np.int64)
        return self._packed


def excitation_sector(model, no, K):
    """The sector of total momentum ``K`` (an integer 3-vector, in units of the reciprocal lattice of
    the box) of the excitations of ``model`` with ``no`` occupied orbitals.

    The sector is defined by the LINEAR label l(K) = n^2 K_x + n K_y + K_z, n = 2 imax + 1, and not
    by the vector K: that label is what the reference's integrals conserve, including the aliased
    elements described in :func:`momentum_groups` (a component beyond imax carries into the next
    digit).  H-bar built from them therefore couples exactly the excitations with equal l(K).  Where
    two different vectors K and K' have l(K) = l(K') -- a difference k_a - k_i has components up to
    2 imax, so it can -- they are ONE sector here, and its states are not sorted by vector K."""
    K = np.asarray(K)
    if K.shape != (3,) or not np.issubdtype(K.dtype, np.integer):
        raise ValueError("K must be an integer 3-vector")
    return ExcitationSector(linear_momenta(model), no, int(linearise(K, model.imax)), K)


def excitation_sectors(model, no):
    """Every sector that holds at least one single (a, i): a list of dicts ``{"K", "sector",
    "n_singles", "n_doubles", "aliases"}`` sorted by |K| (then by K).  ``K`` is the shortest
    k_a - k_i of the sector; ``aliases`` lists the other vectors k_a - k_i with the same linear label
    (see :func:`excitation_sector`)."""
    k = model.k_int().astype(np.int64)
    lin = linear_momenta(model)
    lo, lv = lin[:no], lin[no:]
    dk = (k[no:][:, None, :] - k[:no][None, :, :]).reshape(-1, 3)
    lab = (lv[:, None] - lo[None, :]).reshape(-1)
    # doubles per label: histogram of l_a + l_b against that of l_i + l_j
    pv, cv = np.unique(np.add.outer(lv, lv).reshape(-1), return_counts=True)
    po, co = np.unique(np.add.outer(lo, lo).reshape(-1), return_counts=True)
    out = []
    for l_ in np.unique(lab):
        vecs = np.unique(dk[lab == l_], axis=0)
        vecs = vecs[np.lexsort((vecs[:, 2], vecs[:, 1], vecs[:, 0], (vecs ** 2).sum(axis=1)))]
        want = po + l_
        hit = np.isin(want, pv)
        n_dbl = int((co[hit] * cv[np.searchsorted(pv, want[hit])]).sum())
        out.append({"K": tuple(int(x) for x in vecs[0]), "aliases": [tuple(int(x) for x in v) for v in vecs[1:]],
                    "sector": ExcitationSector(lin, no, int(l_), vecs[0]), "n_singles": int((lab == l_).sum()),
                    "n_doubles": n_dbl})
    out.sort(key=lambda e: (sum(x * x for x in e["K"]), e["K"]))
    return out


def momentum_rule(model, lo, ext, signs=SIGNS):
    """``backend.Momentum`` of a tensor over the orbital ranges ``lo`` / ``ext`` with the given signs
    (an integral block: (+,+,-,-); the Fock matrix: (+,-))."""
    return bk.Momentum(linear_momenta(model), zip(lo, ext, signs))


# stored blocks that also get a never-materialised twin (``backend.blocked_companion``)
BLOCKED_COMPANIONS = ("iabc", "aibc")


class VirtualBlock(bk.GeneratedOperand):
    """Sub-block ``V[lo:lo+ext]`` of the UEG integrals that exists only as its pair tables
    (``include/pymes_b200.h: pmb_ueg_operand_t``).  Usable as the row operand of a
    contraction, e.g. the particle-particle ladder ``abcd,cdij->abij`` (ccd.py:187)."""

    def __init__(self, model, lo, ext, W0a=None, W1a=None, W0s=None, compressed=True, _packed=False):
        if W0a is None and W0s is None:
            raise ValueError("a virtual block needs pair tables (W0a and/or W0s)")
        if model.n_orb > 2047 or model.imax > 27:
            raise ValueError("generated operands support n_orb <= 2047 and imax <= 27")
        self.model, self.lo, self.shape = model, tuple(int(x) for x in lo), tuple(int(x) for x in ext)
        if not _packed:
            # the tables side by side in one allocation: one L2 access-policy window covers them
            given = [t for t in (W0a, W1a, W0s) if t is not None]
            pack = bk.empty(len(given), model.n_orb * model.n_orb)
            for row, t in zip(pack, given):
                row.copy_(t.reshape(-1))
            rows = iter(pack)
            W0a, W1a, W0s = (next(rows) if t is not None else None for t in (W0a, W1a, W0s))
        self.tables = (W0a, W1a, W0s)
        self.compressed = bool(compressed)
        self.nz = model.build_nz(self.lo, self.shape, *self.tables) if self.compressed else None
        st = model._device_state()
        if "lin" not in st:
            st["lin"] = torch.from_numpy(linearise(model.k_int(), model.imax).astype(np.int32)).to(bk.device())
        self.lin = st["lin"]

    def rows(self, dim, lo, n):
        """The same block restricted along ``dim`` to LOCAL indices [lo, lo+n) (cached: a sharded
        sigma asks for the same row block on every application)."""
        key = (int(dim), int(lo), int(n))
        cache = self.__dict__.setdefault("_rows_cache", {})
        if key not in cache:
            new_lo, new_ext = list(self.lo), list(self.shape)
            new_lo[dim] += int(lo)
            new_ext[dim] = int(n)
            cache[key] = VirtualBlock(self.model, new_lo, new_ext, *self.tables, compressed=self.compressed,
                                      _packed=True)
        return cache[key]

    def momentum(self):
        return momentum_rule(self.model, self.lo, self.shape)

    def blocked_lists(self):
        """The block as the matrix [(p,q),(r,s)] is block diagonal in the (linearised) total
        momentum, see :func:`momentum_groups` (ueg.py:395-404).  Returns the lists of
        ``backend.block_lists`` plus the operand side of ``pmb_blocked_contract``: the compressed
        values ``nz[p,q,r]`` and the row / entry offsets into them (the s index is implied by the
        group).  Needs the compressed values; None otherwise."""
        if self.nz is None:
            return None
        L = self.__dict__.get("_blocked")
        if L is None:
            L = dict(bk.block_lists(self.momentum()))
            ext, dev = self.shape, bk.device()
            L["values"] = self.nz
            L["a_moff"] = torch.from_numpy((L["row_i0"] * ext[1] + L["row_i1"]) * ext[2]).to(dev)
            L["a_koff"] = torch.from_numpy(L["ent_j0"].copy()).to(dev)
            self.__dict__["_blocked"] = L
        return L

    def diag_pqpq(self):
        """D[p,q] = V[p,q,p,q] (the ``einsum("abab->ab")`` of eom_ccsd.py:262) without the dense
        block: for r = p the momentum-conserving s is q itself, so the element is the stored
        candidate ``nz[p,q,p]``.  Needs equal p/r and q/s ranges and the compressed values."""
        if self.nz is None:
            raise ValueError("diag_pqpq needs the compressed values (compressed=True)")
        if self.lo[0] != self.lo[2] or self.shape[0] != self.shape[2] or \
                self.lo[1] != self.lo[3] or self.shape[1] != self.shape[3]:
            raise ValueError("diag_pqpq needs a block with equal (p, r) and (q, s) ranges")
        return torch.diagonal(self.nz, dim1=0, dim2=2).t()          # [q,p] view -> [p,q]

    def materialise(self):
        """The dense tensor (tests / small systems)."""
        W0a, W1a, W0s = self.tables
        return self.model.build_block(self.lo, self.shape, W0a=W0a, W1a=W1a, W0s=W0s)

    def gen_descriptor(self, sub, m_ord, k_ord):
        g = _lib.UegOperand()
        g.ueg = self.model._descriptor()
        p = lambda t: t.data_ptr() if t is not None else None
        g.W0a, g.W1a, g.W0s = (p(t) for t in self.tables)
        g.lin = self.lin.data_ptr()
        g.nz = self.nz.data_ptr() if self.nz is not None else None
        axis = {ch: i for i, ch in enumerate(sub)}
        for i in range(4):
            g.lo[i] = self.lo[i]
            g.m_axis[i] = axis[m_ord[i]] if i < len(m_ord) else -1
            g.k_axis[i] = axis[k_ord[i]] if i < len(k_ord) else -1
        g._keep = (self.tables, self.lin, self.nz, self.model._dev)
        return g
