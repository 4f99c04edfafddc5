"""CCSD / DCSD through the T1-dressed Hamiltonian, on the B200 contraction engine.

Call surface of the reference ``pymes.solver.ccsd.CCSD`` (pymes/solver/ccsd.py:22-466):
constructor, ``solve``, ``get_T1_dressed_fock``, ``get_T1_dressed_V``,
``get_singles_residual``, ``get_doubles_residual``, ``get_energy``, the returned
dict keys, ``self.t_T_ai`` / ``self.t_T_abij`` and the log lines.

Design differences (results agree to round-off: tests/test_gpu_parity.py, lock-step with the oracle
sweep by sweep on LiH, LiH-TC, HF/aug-cc-pVDZ, TC-UEG 14e and 54e, synthetic o=10 v=60):

* Every dressing product (ccsd.py:257-286, 322-419) is a row of a term table that
  is evaluated pairwise on the DMMA engine (``backend.einsum``); sources are always
  the undressed blocks, exactly as in the reference.
* ``solve`` never forms the dressed V_abcd (a v^4 copy plus three o.v^4
  contractions per sweep in the reference, ccsd.py:414-419).  All terms in which
  V_abcd, V_iabc, V_aibc or V_ijab meet two virtual-contracted amplitudes collapse
  onto one particle-particle ladder applied to tau = T2 + T1 (x) T1:

      W  = V_abcd.tau                       W1 = V_iabc.tau   (k b i j)
      W2 = V_aibc.tau  (a l i j)            W3 = V_ijab.tau   (k l i j)
      R += W - t_ak W1_kbij - t_bl (W2 - t_ak W3)_alij

  which reproduces the four tau-type rows of the dressed V_abij (ccsd.py:334-343)
  together with the dressed-V_abcd ladder of ccd.py:187.  The public
  ``get_T1_dressed_V`` still returns every dressed block (EOM-CCSD consumes them).
"""
import time

import numpy as np
import torch

from .. import backend as bk
from ..integral.partition import part_2_body_int
from ..log import print_logging_info
from ..mixer import diis
from . import ccd, mp2

# (coef, subscripts, operand names); "t" = T1, "foo"/"fvv"/"fov" = Fock blocks,
# anything else = key of the undressed integral dictionary.
FOCK_TERMS = {
    "ov": [(+2.0, "bj,jabi->ia", "t iabj"), (-1.0, "bj,jiab->ia", "t ijab")],
    "vo": [(-1.0, "ji,aj->ai", "foo t"), (+1.0, "ab,bi->ai", "fvv t"),
           (-1.0, "jb,bi,aj->ai", "fov t t"),
           (+2.0, "bj,jabi->ai", "t iabj"), (-2.0, "bj,jkbi,ak->ai", "t ijak t"),
           (+2.0, "ac,ci->ai", "G3 t"), (-2.0, "bj,jkbc,ci,ak->ai", "t ijab t t"),      # "bj,jabc,ci->ai"
           (-1.0, "bj,jaib->ai", "t iajb"), (+1.0, "bj,jkib,ak->ai", "t ijka t"),
           (-1.0, "ac,ci->ai", "G4 t"), (+1.0, "bj,jkcb,ci,ak->ai", "t ijab t t")],      # "bj,jacb,ci->ai"
    "oo": [(+2.0, "ck,kicj->ij", "t ijak"), (-1.0, "ck,kijc->ij", "t ijka"),
           (+1.0, "ib,bj->ij", "fov t"),
           (+2.0, "ck,kicb,bj->ij", "t ijab t"), (-1.0, "ck,kibc,bj->ij", "t ijab t")],
    "vv": [(+2.0, "ab->ab", "G3"), (-1.0, "ab->ab", "G4"),                                 # "ci,iacb->ab", "ci,iabc->ab"
           (-1.0, "ib,ai->ab", "fov t"),
           (-2.0, "ck,klcb,al->ab", "t ijab t"), (+1.0, "ck,kibc,ai->ab", "t ijab t")],
}

# Products of the o.v^3 block V_iabc with T1 that several rows share (each is one HBM pass over the
# block, 25 GB at v = 488, so each is evaluated ONCE per sweep, `t1_shared`):
#   X3[i,a,j,b] = sum_c V_iabc[i,a,c,b] t[c,j]      the row "iacb,cj->iajb" of the dressed V_iajb (ccsd.py:379)
#   X4[i,a,b,j] = sum_c V_iabc[i,a,b,c] t[c,j]      the row "iabc,cj->iabj" of the dressed V_iabj (ccsd.py:387)
# and the four Fock rows that read V_iabc (ccsd.py:266,270,282,283) are partial traces of them:
#   G3[a,b] = sum_i X3[i,a,i,b]:  "bj,jabc,ci->ai" = (G3.t)_ai,  "ci,iacb->ab" = G3_ab
#   G4[a,b] = sum_i X4[i,a,b,i]:  "bj,jacb,ci->ai" = (G4.t)_ai,  "ci,iabc->ab" = G4_ab
SHARED_PRODUCTS = {"X3": ("iacb,cj->iajb", "iabc t"), "X4": ("iabc,cj->iabj", "iabc t")}
SHARED_TRACES = {"G3": ("X3", "iaib", "iab"), "G4": ("X4", "iabi", "iab")}
FOCK_SHARED = ("G3", "G4")


def t1_shared(T1, dV):
    """{"X3", "X4", "G3", "G4"} for these amplitudes (device tensors; with a row-sharded V_iabc
    [i, a in A, b, c] every entry holds the local rows a in A)."""
    src = dict(dV)
    src["t"] = T1
    out = {}
    for name, (spec, names) in SHARED_PRODUCTS.items():
        out[name] = bk.einsum(spec, *[src[n] for n in names.split()])
    ones = bk.ones(T1.shape[1])
    for name, (source, sub, view_sub) in SHARED_TRACES.items():
        out[name] = bk.einsum(view_sub + ",i->ab", bk.diag_view(out[source], sub, view_sub), ones)
    return out


# rows marked True are the tau-type terms folded into the pp ladder by `solve`
V_TERMS = {
    "abij": [(-1.0, "kbij,ak->abij", "iajk", False), (+1.0, "abcj,ci->abij", "abci", False),
             (-1.0, "kbcj,ak,ci->abij", "iabj", False), (-1.0, "alij,bl->abij", "aijk", False),
             (+1.0, "klij,ak,bl->abij", "klij", False), (-1.0, "alcj,ci,bl->abij", "aibj", False),
             (+1.0, "klcj,ak,ci,bl->abij", "ijak", False), (+1.0, "abid,dj->abij", "abic", False),
             (-1.0, "kbid,ak,dj->abij", "iajb", False), (+1.0, "abcd,ci,dj->abij", "abcd", True),
             (-1.0, "kbcd,ak,ci,dj->abij", "iabc", True), (-1.0, "alid,bl,dj->abij", "aijb", False),
             (+1.0, "klid,ak,bl,dj->abij", "ijka", False), (-1.0, "alcd,ci,bl,dj->abij", "aibc", True),
             (+1.0, "klcd,ak,ci,bl,dj->abij", "ijab", True)],
    "klij": [(+1.0, "klaj,ai->klij", "ijak", False), (+1.0, "klib,bj->klij", "ijka", False),
             (+1.0, "klab,ai,bj->klij", "ijab", False)],
    "ijab": [],
    "ijka": [(+1.0, "ijba,bk->ijka", "ijab", False)],
    "ijak": [(+1.0, "ijab,bk->ijak", "ijab", False)],
    "iajb": [(+1.0, "iajb->iajb", "X3", False), (-1.0, "ikjb,ak->iajb", "ijka", False),        # "iacb,cj->iajb"
             (-1.0, "ikcb,cj,ak->iajb", "ijab", False)],
    "iabj": [(-1.0, "ikbj,ak->iabj", "ijak", False), (+1.0, "iabj->iabj", "X4", False),        # "iabc,cj->iabj"
             (-1.0, "ikbc,ak,cj->iabj", "ijab", False)],
    "iabc": [(-1.0, "ijbc,aj->iabc", "ijab", False)],
    "abic": [(-1.0, "jbic,aj->abic", "iajb", False), (+1.0, "abdc,di->abic", "abcd", False),
             (-1.0, "jbdc,aj,di->abic", "iabc", False), (-1.0, "ajic,bj->abic", "aijb", False),
             (+1.0, "kjic,ak,bj->abic", "ijka", False), (-1.0, "ajdc,di,bj->abic", "aibc", False),
             (+1.0, "kjdc,ak,di,bj->abic", "ijab", False)],
    "iajk": [(-1.0, "iljk,al->iajk", "klij", False), (+1.0, "iajb,bk->iajk", "iajb", False),
             (-1.0, "iljb,al,bk->iajk", "ijka", False), (+1.0, "iabk,bj->iajk", "iabj", False),
             (-1.0, "ilbk,bj,al->iajk", "ijak", False), (+1.0, "iabc,bj,ck->iajk", "iabc", False),
             (-1.0, "ilbc,bj,al,ck->iajk", "ijab", False)],
    "abcd": [(-1.0, "jbcd,aj->abcd", "iabc", False), (-1.0, "aicd,bi->abcd", "aibc", False),
             (+1.0, "jicd,aj,bi->abcd", "ijab", False)],
}

SINGLES_TERMS = [(+1.0, "jb,abij->ai", "fov Tt"), (+1.0, "ajbc,bcij->ai", "aibc Tt"),
                 (-1.0, "kjbc,ak,bcij->ai", "ijab t Tt"), (-1.0, "jkib,abjk->ai", "ijka Tt"),
                 (-1.0, "jkcb,ci,abjk->ai", "ijab t Tt")]


def _dev_dict(dict_t_V):
    return {k: (bk.asdev(v) if v is not None else None) for k, v in dict_t_V.items()}


def dressed_fock(no, fock, T1, dV, shared=None):
    """Device tensors in, dressed Fock (new tensor) out.  ccsd.py:226-288.  ``shared``: the
    result of :func:`t1_shared` for these amplitudes (computed here when not given)."""
    src = dict(dV)
    nv = fock.shape[0] - no
    src.update(t=T1, foo=ccd.block2(fock, 0, no, 0, no), fvv=ccd.block2(fock, no, nv, no, nv),
               fov=ccd.block2(fock, 0, no, no, nv))
    src.update(shared if shared is not None else t1_shared(T1, dV))
    out = bk.copy(fock)
    views = {"ov": ccd.block2(out, 0, no, no, nv), "vo": ccd.block2(out, no, nv, 0, no),
             "oo": ccd.block2(out, 0, no, 0, no), "vv": ccd.block2(out, no, nv, no, nv)}
    for blk, rows in FOCK_TERMS.items():
        for coef, spec, names in rows:
            bk.einsum(spec, *[src[n] for n in names.split()], out=views[blk], alpha=coef, beta=1.0)
    return out


def dressed_block(key, T1, dV, skip_tau=False, shared=None):
    """One T1-dressed V block from the undressed dictionary.  ccsd.py:322-419.  ``shared``: the
    result of :func:`t1_shared` (needed by "iajb" / "iabj"; computed here when not given)."""
    blk = bk.copy(dV[key])
    for coef, spec, source, is_tau in V_TERMS[key]:
        if skip_tau and is_tau:
            continue
        nt = spec.split("->")[0].count(",")
        if source in SHARED_PRODUCTS:
            if shared is None:
                shared = t1_shared(T1, dV)
            bk.einsum(spec, shared[source], out=blk, alpha=coef, beta=1.0)
            continue
        bk.einsum(spec, dV[source], *([T1] * nt), out=blk, alpha=coef, beta=1.0)
    return blk


def singles_residual(no, fock_dressed, T1, T2, dV):
    """R_ai from the dressed Fock matrix and the UNDRESSED integrals (ccsd.py:167-168, 423-438)."""
    Tt = bk.tilde(T2, swap_ij=True)
    src = dict(dV)
    nv = fock_dressed.shape[0] - no
    src.update(t=T1, Tt=Tt, fov=ccd.block2(fock_dressed, 0, no, no, nv))
    R1 = bk.copy(ccd.block2(fock_dressed, no, nv, 0, no))
    for coef, spec, names in SINGLES_TERMS:
        bk.einsum(spec, *[src[n] for n in names.split()], out=R1, alpha=coef, beta=1.0)
    return R1


def energy_layout(V_ijab):
    """V_ijab re-stored as [a,b,i,j] and handed back as an (i,j,a,b)-indexed VIEW of that storage.
    The block is static, the energy is evaluated every sweep: with this layout ``pmb_energy_doubles``
    streams row (a,b) for the direct and row (b,a) for the exchange term next to the same row of T2
    (coalesced, 24 B per amplitude) instead of gathering V[i,j,.,.] at stride v^2."""
    return bk.copy(V_ijab.permute(2, 3, 0, 1)).permute(2, 3, 0, 1)


def pair_with_tau(V_iabc, V_aibc, tau, no):
    """(W1, W2) = (V_iabc.tau [k,b,i,j], V_aibc.tau [a,l,i,j]) with V_iabc = [o, nb, v, v] and V_aibc =
    [nb, o, v, v] (nb = v, or the local rows of a sharded run).  When the two blocks were allocated
    back to back (``UEG.eval_2b_blocks`` / ``synthetic.tc_blocks`` do that) they are ONE operand of
    2.o.nb rows: a single launch whose sparse last wave is split over k, instead of two grids of
    4.2 waves each (N = 1) or of 78 tiles on 148 SMs each (N = 8).  Otherwise two launches side by
    side on two streams."""
    ct = bk.contract_terms
    nv = tau.shape[0]
    nb = V_iabc.shape[1]
    ca, cb = bk.blocked_companion(V_iabc), bk.blocked_companion(V_aibc)
    if ca is not None and cb is not None:
        # momentum-conserving blocks: only the diagonal blocks of [(k,b),(c,d)] / [(a,l),(c,d)]
        # are visited (pmb_blocked_contract), from 1/v of the stored values
        return (ct("kbij", [(1.0, "kbcd", ca, "cdij", tau)]), ct("alij", [(1.0, "alcd", cb, "cdij", tau)]))
    st = bk.stacked_rows(V_iabc, V_aibc, (nv, nv))
    if st is not None:
        W = bk.empty(2, no * nb, no, no)
        ct("grij", [(1.0, "grcd", st, "cdij", tau)], out=W)
        return W[0].view(no, nb, no, no), W[1].view(nb, no, no, no)
    W1, W2 = bk.empty(no, nb, no, no), bk.empty(nb, no, no, no)
    with bk.side_by_side() as side:
        ct("kbij", [(1.0, "kbcd", V_iabc, "cdij", tau)], out=W1)
        side(lambda: ct("alij", [(1.0, "alcd", V_aibc, "cdij", tau)], out=W2))
    return W1, W2


def tau_ladder(T1, dV):
    """Returns the ``pp_ladder(T2, R)`` callback described in the module docstring."""
    def apply(T2, R):
        ct = bk.contract_terms
        tau = bk.axpby(1.0, T2, 0.0, bk.empty_even_pitch(T2.shape[0], T2.shape[1], T2.shape[2]))
        ct("abij", [(1.0, "ai", T1, "bj", T1)], out=tau, beta=1.0)
        with bk.timed("pp_ladder"):
            ct("abij", [(1.0, "abcd", dV["abcd"], "cdij", tau)], out=R, beta=1.0)
        nv, no = T1.shape
        W1, W2 = pair_with_tau(dV["iabc"], dV["aibc"], tau, no)
        ct("abij", [(-1.0, "ak", T1, "kbij", W1)], out=R, beta=1.0)
        W3 = ct("klij", [(1.0, "klcd", dV["ijab"], "cdij", tau)])
        ct("alij", [(-1.0, "ak", T1, "klij", W3)], out=W2, beta=1.0)
        ct("abij", [(-1.0, "bl", T1, "alij", W2)], out=R, beta=1.0)
    return apply


class DressedLadder(bk.LinearOperator):
    """The T1-dressed V_abcd (ccsd.py:405-419)

        Vd[a,b,c,d] = V[a,b,c,d] - t[a,k] V_iabc[k,b,c,d] - t[b,l] V_aibc[a,l,c,d]
                                 + t[a,k] t[b,l] V_ijab[k,l,c,d]

    as an operator: it is never formed (a v^4 array), only applied to amplitude-shaped
    vectors and asked for its (abab) diagonal -- the two things EOM-CCSD does with it
    (eom_ccsd.py:262,383).  ``V_abcd`` may be a dense tensor or a never-materialised
    ``model.ueg.VirtualBlock``; the blocks are the UNDRESSED ones."""

    def __init__(self, V_abcd, V_iabc, V_aibc, V_ijab, T1):
        self.V_abcd, self.V_iabc, self.V_aibc, self.V_ijab, self.T1 = V_abcd, V_iabc, V_aibc, V_ijab, T1
        nv = T1.shape[0]
        self.shape = (nv, nv, nv, nv)

    def apply(self, U, out, coef=1.0, shard=None):
        """out[(r,)a,b,i,j] += coef * sum_cd Vd[a,b,c,d] U[(r,)c,d,i,j]; U of shape [v,v,o,o] or
        batched [r,v,v,o,o].  Same factorisation as ``tau_ladder``.  With ``shard``, ``out`` holds
        the rows a in A only: V_abcd and V_aibc are restricted to those rows, W1 / W3 (no index
        a) are replicated."""
        ct, T1 = bk.contract_terms, self.T1
        r = "r" if U.dim() == 5 else ""
        if shard is None:
            Va, Vaibc, T1a = self.V_abcd, self.V_aibc, T1
        else:
            V = self.V_abcd
            Va = V.rows(0, shard.lo, shard.na) if isinstance(V, bk.GeneratedOperand) else shard.rows(V, 0)
            Vaibc, T1a = shard.rows(self.V_aibc, 0), shard.rows(T1, 0)
        # stored o.v^3 blocks with a never-materialised twin go momentum-blocked as well
        ca, cb = bk.blocked_companion(self.V_iabc), bk.blocked_companion(self.V_aibc)
        if cb is not None:
            Vaibc = cb if shard is None else cb.rows(0, shard.lo, shard.na)
        ct(r + "abij", [(coef, "abcd", Va, r + "cdij", U)], out=out, beta=1.0)
        W1 = ct(r + "kbij", [(1.0, "kbcd", self.V_iabc if ca is None else ca, r + "cdij", U)])
        ct(r + "abij", [(-coef, "ak", T1a, r + "kbij", W1)], out=out, beta=1.0)
        del W1
        W2 = ct(r + "alij", [(1.0, "alcd", Vaibc, r + "cdij", U)])
        W3 = ct(r + "klij", [(1.0, "klcd", self.V_ijab, r + "cdij", U)])
        ct(r + "alij", [(-1.0, "ak", T1a, r + "klij", W3)], out=W2, beta=1.0)
        ct(r + "abij", [(-coef, "bl", T1, r + "alij", W2)], out=out, beta=1.0)
        return out

    def diag_abab(self):
        """D[a,b] = Vd[a,b,a,b] as a [v,v] tensor."""
        T1, V = self.T1, self.V_abcd
        if isinstance(V, bk.GeneratedOperand):
            D = bk.copy(V.diag_pqpq())
        else:
            D = bk.copy(bk.diag_view(V, "abab", "ab"))
        X = bk.diag_view(self.V_iabc, "kbab", "kab")
        bk.bdot("ak,kab->ab", T1, X, out=D, alpha=-1.0, beta=1.0)
        Y = bk.diag_view(self.V_aibc, "alab", "alb")
        bk.bdot("bl,alb->ab", T1, Y, out=D, alpha=-1.0, beta=1.0)
        Z = bk.bdot("ak,klab->lab", T1, self.V_ijab)
        bk.bdot("bl,lab->ab", T1, Z, out=D, alpha=1.0, beta=1.0)
        return D

    def adopt_momentum(self, rule_of):
        """Check (and tag) the operator's parts under their momentum rules ``rule_of(key)`` (key:
        "abcd", "iabc", "aibc", "ijab", "ai"); True when every part conserves momentum."""
        V = self.V_abcd
        ok = V.momentum() == rule_of("abcd") if isinstance(V, bk.GeneratedOperand) else \
            bk.adopt_momentum(V, rule_of("abcd"))
        return ok and all(bk.adopt_momentum(t, rule_of(k)) for k, t in
                          (("iabc", self.V_iabc), ("aibc", self.V_aibc), ("ijab", self.V_ijab), ("ai", self.T1)))

    def dense(self):
        """The dressed block itself (tests / small systems)."""
        V = self.V_abcd.materialise() if isinstance(self.V_abcd, bk.GeneratedOperand) else self.V_abcd
        return dressed_block("abcd", self.T1, {"abcd": V, "iabc": self.V_iabc, "aibc": self.V_aibc,
                                               "ijab": self.V_ijab})


class CCSD(ccd.CCD):
    def __init__(self, no, is_diis=True, delta_e=1.e-8, is_non_canonical=False, is_dcsd=False):
        self.t_T_ai = None
        self.t_T_abij = None
        self.is_dcd = is_dcsd
        self.is_diis = is_diis
        self.is_bruekner = False
        self.is_dr_ccd = False
        self.no = no
        self.max_iter = 50
        self.delta = 1.0
        self.delta_e = delta_e
        self.debug_level = 1
        if self.is_diis:
            self.mixer = diis.DIIS(dim_space=6)

    def write_logging_info(self):
        return

    # ---- public building blocks (numpy or CUDA tensors in, same kind out) ----
    def get_T1_dressed_fock(self, t_fock_pq, t_T_ai, dict_t_V):
        want_numpy = not isinstance(t_fock_pq, torch.Tensor)
        out = dressed_fock(self.no, bk.asdev(t_fock_pq), bk.asdev(t_T_ai), _dev_dict(dict_t_V))
        return bk.tonumpy(out) if want_numpy else out

    def get_T1_dressed_V(self, t_T_ai, dict_t_V, dict_t_V_dressed=None):
        """All (or the requested) dressed blocks; blocks the reference leaves
        undressed stay ``None`` (``dict.fromkeys``, ccsd.py:316-317)."""
        want_numpy = not isinstance(t_T_ai, torch.Tensor)
        if dict_t_V_dressed is None or len(dict_t_V_dressed) == 0:
            dict_t_V_dressed = {}.fromkeys(dict_t_V, None)
        dV, T1 = _dev_dict(dict_t_V), bk.asdev(t_T_ai)
        shared = t1_shared(T1, dV) if any(k in dict_t_V_dressed for k in ("iajb", "iabj")) else None
        for key in V_TERMS:
            if key in dict_t_V_dressed:
                if key == "abcd" and isinstance(dV["abcd"], bk.GeneratedOperand):
                    # V_abcd is never materialised: its dressed form is an operator as well
                    dict_t_V_dressed[key] = DressedLadder(dV["abcd"], dV["iabc"], dV["aibc"], dV["ijab"], T1)
                    continue
                blk = dressed_block(key, T1, dV, shared=shared)
                dict_t_V_dressed[key] = bk.tonumpy(blk) if want_numpy else blk
        return dict_t_V_dressed

    def get_singles_residual(self, t_fock_pq, t_T_ai, t_T_abij, dict_t_V):
        want_numpy = not isinstance(t_T_abij, torch.Tensor)
        R1 = singles_residual(self.no, bk.asdev(t_fock_pq), bk.asdev(t_T_ai),
                              bk.asdev(t_T_abij).contiguous(), _dev_dict(dict_t_V))
        return bk.tonumpy(R1) if want_numpy else R1

    def get_doubles_residual(self, t_fock_pq, t_T_abij, dict_t_V_dressed):
        d = dict_t_V_dressed
        return self.get_residual(t_fock_pq, t_T_abij, d["klij"], d["ijab"], d["abij"], d["iajb"],
                                 d["iabj"], d["abcd"])

    def get_energy(self, t_fock_ia, t_T_ai, t_T_abij, t_V_ijab):
        """[one-body, direct, exchange], ccsd.py:458-466."""
        T1, T2 = bk.asdev(t_T_ai).contiguous(), bk.asdev(t_T_abij).contiguous()
        scal = bk.zeros(8)
        bk.energy_doubles(T2, bk.asdev(t_V_ijab), scal, T1=T1)
        bk.contract_terms("", [(2.0, "ia", bk.asdev(t_fock_ia), "ai", T1)], out=scal[4])
        s = scal.cpu().numpy()
        return [float(s[4]), float(s[0]), float(s[1])]

    # ------------------------------------------------------------------
    def setup(self, t_fock_pq, t_V_pqrs, level_shift=0., amps=None):
        """Upload the static operator (Fock, V blocks), MP2 start amplitudes (ccsd.py:118-156).
        ``t_V_pqrs`` is V_pqrs (numpy / CUDA tensor) or -- extension for systems whose V_pqrs
        cannot exist as one array -- a dict of the 16 partition blocks as CUDA tensors."""
        no = self.no
        blocks_given = isinstance(t_V_pqrs, dict)
        fock_host = bk.tonumpy(t_fock_pq)
        nv = fock_host.shape[0] - no
        st = self._st = {}
        st["want_numpy"] = not (blocks_given or isinstance(t_V_pqrs, torch.Tensor))
        st["eps_i"] = bk.asdev(fock_host.diagonal()[:no].copy())
        st["eps_a"] = bk.asdev(fock_host.diagonal()[no:].copy())
        st["fock"] = bk.asdev(fock_host)
        if blocks_given:
            st["dV"] = _dev_dict(t_V_pqrs)
            st["dtype_name"] = "float64"
        else:
            V = bk.asdev(t_V_pqrs)
            st["dV"] = part_2_body_int(no, V)
            st["dtype_name"] = str(V.dtype).replace("torch.", "")
        st["shift"] = level_shift
        e_mp2, T2 = mp2.solve_device(st["eps_i"], st["eps_a"], st["dV"]["ijab"], st["dV"]["abij"],
                                     level_shift)
        # Structure from outside is verified, never assumed.  The Fock matrix is checked on the host,
        # where it already is.  The amplitudes start tagged only under a Hamiltonian that conserves
        # momentum as a whole: with a one-body part that breaks the rule they break it from the first
        # update on, and the sweeps then run dense from the start instead of switching after one.
        rule = ccd.fock_rules(st["dV"]["abij"], no, nv)
        if rule is not None and not bk.adopt_momentum(st["fock"], rule["fock"], host=fock_host):
            rule = None
        self._rules = rule
        T1 = bk.zeros(nv, no, rule=rule["t1"] if rule is not None else None)
        st["amps_host"] = None
        if amps is not None:
            if isinstance(amps[0], torch.Tensor):
                T1, T2 = bk.asdev(amps[0]), bk.asdev(amps[1])        # aliased: updated in place
                if not (T1.is_contiguous() and T2.is_contiguous()):  # the elementwise kernels index them flat
                    raise ValueError("amps given as tensors must be contiguous [nv,no] / [nv,nv,no,no]")
            else:
                st["amps_host"] = amps
                T1, T2 = bk.asdev(amps[0]).contiguous(), bk.asdev(amps[1]).contiguous()
        st["T1"], st["T2"] = T1, T2
        if rule is None:
            bk.drop_momentum(T2)              # MP2 amplitudes of tagged integrals carry a derived rule
        elif amps is not None:
            bk.adopt_momentum(T1, rule["t1"])
            bk.adopt_momentum(T2, rule["t2"])
        st["scal"] = bk.zeros(8)
        st["e_mp2"] = e_mp2
        st["iteration"] = 0
        st["V_ijab_e"] = energy_layout(st["dV"]["ijab"])
        return e_mp2

    def sweep(self):
        """One CCSD/DCSD iteration (loop body ccsd.py:159-197) on the device-resident state:
        dressing -> singles + doubles residual -> update -> DIIS -> energy.
        Returns (e_1b, e_dir, e_ex, |T2|, |dT2|)."""
        st = self._st
        no, dV, fock = self.no, st["dV"], st["fock"]
        T1, T2, scal = st["T1"], st["T2"], st["scal"]
        eps_i, eps_a, shift = st["eps_i"], st["eps_a"], st["shift"]
        st["iteration"] += 1
        shared = t1_shared(T1, dV)              # the V_iabc.T1 products: one pass each per sweep
        ft = dressed_fock(no, fock, T1, dV, shared=shared)
        R1 = singles_residual(no, ft, T1, T2, dV)
        V_iajb = dressed_block("iajb", T1, dV, shared=shared)
        V_iabj = dressed_block("iabj", T1, dV, shared=shared)
        del shared
        R2 = ccd.doubles_residual(
            no, ft, T2, dressed_block("klij", T1, dV), dV["ijab"],
            dressed_block("abij", T1, dV, skip_tau=True), V_iajb, V_iabj, None, is_dcd=self.is_dcd,
            pp_ladder=tau_ladder(T1, dV))
        del V_iajb, V_iabj
        dT1 = bk.update_singles(eps_i, eps_a, shift, self.delta, R1, T1)
        dT2 = bk.update_doubles(eps_i, eps_a, shift, self.delta, R2, T2, scal[3:4])
        del R1, R2
        amps_host = st["amps_host"]
        if amps_host is not None and (st["iteration"] == 1 or not self.is_diis):
            amps_host[0][...] = bk.tonumpy(T1)          # the reference mutates `amps` in place
            amps_host[1][...] = bk.tonumpy(T2)
        if self.is_diis:
            T1, T2 = self.mixer.mix([dT1, dT2], [T1, T2])
        st["T1"], st["T2"] = T1, T2
        bk.energy_doubles(T2, st["V_ijab_e"], scal, T1=T1)
        bk.contract_terms("", [(2.0, "ia", ccd.block2(fock, 0, no, no, T1.shape[0]), "ai", T1)], out=scal[4])
        s = scal.cpu().numpy()
        return float(s[4]), float(s[0]), float(s[1]), float(np.sqrt(s[2])), float(np.sqrt(s[3]))

    def sweep_host(self, t1_host, t2_host):
        """Host-buffer form of :meth:`sweep`: amplitudes come in as host tensors / arrays
        (pinned memory makes the copy asynchronous), one iteration runs on the device, and the
        new amplitudes are copied back into the same host buffers.  Returns the energies and
        norms of :meth:`sweep`.  The static operator (Fock, V blocks) stays device-resident."""
        st = self._st
        t1 = t1_host if isinstance(t1_host, torch.Tensor) else torch.from_numpy(t1_host)
        t2 = t2_host if isinstance(t2_host, torch.Tensor) else torch.from_numpy(t2_host)
        st["T1"] = t1.to(bk.device(), non_blocking=True)
        st["T2"] = t2.to(bk.device(), non_blocking=True)
        rule = getattr(self, "_rules", None)
        if rule is not None:
            bk.adopt_momentum(st["T1"], rule["t1"])
            bk.adopt_momentum(st["T2"], rule["t2"])
        out = self.sweep()
        t1.copy_(st["T1"], non_blocking=True)
        t2.copy_(st["T2"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out

    def solve(self, t_fock_pq, t_V_pqrs, level_shift=0., amps=None, sp=0, **kwargs):
        algo_name = "ccsd.solve"
        t_start = time.time()
        max_iter = kwargs.get("max_iter", self.max_iter)
        delta_e = kwargs.get("delta_e", self.delta_e)

        print_logging_info(algo_name)
        print_logging_info("Using dcsd: ", self.is_dcd, level=1)
        print_logging_info("Solving doubles amplitude equation", level=1)
        e_mp2 = self.setup(t_fock_pq, t_V_pqrs, level_shift, amps)
        st = self._st
        print_logging_info("Using data type %s" % st["dtype_name"], level=1)
        print_logging_info("Using DIIS mixer: ", self.is_diis, level=1)
        print_logging_info("Iteration = 0", level=1)

        dE = abs(e_mp2)
        iteration = 0
        e_last = e_mp2
        e_ccsd = e_1b = e_dir = e_ex = 0.0
        while abs(dE) > delta_e and iteration <= max_iter:
            iteration += 1
            e_1b, e_dir, e_ex, t2_norm, res_norm = self.sweep()
            e_ccsd = e_1b + e_dir + e_ex
            dE = e_ccsd - e_last
            e_last = e_ccsd
            if iteration <= max_iter:
                print_logging_info("Iteration = ", iteration, level=1)
                print_logging_info("Correlation Energy = {:.14f}".format(e_ccsd), level=2)
                print_logging_info("dE = {:.12e}".format(dE), level=2)
                print_logging_info("L1 Norm of T2 = {:.14f}".format(t2_norm), level=2)
                print_logging_info("Norm Residual = {:.14f}".format(res_norm), level=2)
            else:
                print_logging_info("A converged solution is not found!", level=1)

        print_logging_info("Fock contribution = {:.12f}".format(e_1b), level=1)
        print_logging_info("Direct contribution = {:.12f}".format(e_dir), level=1)
        print_logging_info("Exchange contribution = {:.12f}".format(e_ex), level=1)
        print_logging_info("CCSD correlation energy = {:.12f}".format(e_ccsd), level=1)
        print_logging_info("{:.3f} seconds spent on ccsd".format(time.time() - t_start), level=1)
        self.iterations = iteration
        T1, T2, eps_i, eps_a = st["T1"], st["T2"], st["eps_i"], st["eps_a"]
        if st["want_numpy"]:
            T1, T2, eps_i, eps_a = (bk.tonumpy(x) for x in (T1, T2, eps_i, eps_a))
        self.t_T_ai = T1
        self.t_T_abij = T2
        return {"ccsd e": e_ccsd, "t1": T1, "t2": T2, "hole e": eps_i, "particle e": eps_a, "dE": dE}
