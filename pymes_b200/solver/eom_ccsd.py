"""EOM-EE-CCSD for non-hermitian (transcorrelated) Hamiltonians on the B200 contraction engine.

Call surface of the reference ``pymes.solver.eom_ccsd.EOM_CCSD`` (pymes/solver/eom_ccsd.py:30-541):
``EOM_CCSD(no, n_excit=3)``, ``solve(fock_dressed, dictV_dressed, T2) -> e_excit``,
``update_singles / update_doubles(fock, dictV, u1, u2, T2)``, ``get_diag_singles / get_diag_doubles``,
``QR``, the attributes ``u_singles, u_doubles, e_excit, max_dim, e_epsilon, max_iter``.

How the sigma product H-bar.R is evaluated here
-----------------------------------------------
The reference types the sigma equations as 18 (singles) + 44 (doubles) einsum terms, most of
them three-operand products V.T2.u evaluated pairwise on every call (``optimize=True``).
:class:`SigmaPlan` reads the SAME term tables (transcribed below with their reference lines)
and, once per (fock, V, T2):

* picks for every three-operand term the pairing with the fewest per-vector flops:
  either the u-independent pair V.T2 is contracted ONCE into an H-bar intermediate
  ("hoisted"), or the small pair X.u is formed first and the result meets the other
  static operand ("two-step");
* renames indices canonically so that terms with the same final contraction pattern are
  merged (their intermediates are summed), leaving ~25 contractions per sigma instead of 62;
* evaluates every contraction for a BATCH of right-hand sides at once: trial vectors are
  stacked along a leading index ``r`` which simply joins the N index group of the strided
  DMMA contraction (``u2[r,a,b,i,j]``), so V_abcd is streamed once per batch -- this is what
  the FEAST contour (nodes x trial vectors) and the Davidson block use.

Nothing is symmetrised: V_klij != V_ijkl, the ``+ baji`` permutation is applied explicitly
(eom_ccsd.py:377) and left/right vectors are never assumed equal.
"""
import time

import numpy as np
import torch

from .. import backend as bk
from ..log import print_logging_info, print_title

# --------------------------------------------------------------------------
# term tables: (coefficient, einsum string, operand names)
#   fov/foo/fvv = blocks of the (dressed) Fock matrix, T = ground-state T2,
#   u1/u2 = trial vector, anything else = key of the (dressed) integral dictionary
# --------------------------------------------------------------------------
SIGMA1_TERMS = [                                                       # eom_ccsd.py:288-308
    (+2., "jb,baji->ai", "fov u2"), (-1., "ji,aj->ai", "foo u1"),
    (-1., "jb,abji->ai", "fov u2"), (+1., "ab,bi->ai", "fvv u1"),
    (+2., "jabi,bj->ai", "iabj u1"), (-1., "jaib,bj->ai", "iajb u1"),
    (-2., "jkib,abjk->ai", "ijka u2"), (+2., "jabc,bcji->ai", "iabc u2"),
    (+1., "jkib,bajk->ai", "ijka u2"), (-1., "jacb,bcji->ai", "iabc u2"),
    (+4., "jkbc,baji,ck->ai", "ijab T u1"), (-2., "jkbc,bajk,ci->ai", "ijab T u1"),
    (-2., "jkbc,bcji,ak->ai", "ijab T u1"), (-2., "jkbc,abji,ck->ai", "ijab T u1"),
    (-2., "jkcb,baji,ck->ai", "ijab T u1"), (+1., "jkbc,abjk,ci->ai", "ijab T u1"),
    (+1., "jkcb,bcji,ak->ai", "ijab T u1"), (+1., "jkcb,abji,ck->ai", "ijab T u1"),
]

SIGMA2_P_TERMS = [                                                     # eom_ccsd.py:332-373
    (-2., "klid,abkj,dl->abij", "ijka T u1"), (-2., "klci,cbkj,al->abij", "ijak T u1"),
    (+2., "kacd,cbkj,di->abij", "iabc T u1"), (+2., "ladc,cbij,dl->abij", "iabc T u1"),
    (-1., "kd,abkj,di->abij", "fov T u1"), (-1., "lc,cbij,al->abij", "fov T u1"),
    (+1., "klid,abkl,dj->abij", "ijka T u1"), (+1., "klic,cbkj,al->abij", "ijka T u1"),
    (+1., "klid,adkj,bl->abij", "ijka T u1"), (-1., "kbij,ak->abij", "iajk u1"),
    (+1., "kldi,bdkj,al->abij", "ijak T u1"), (-1., "kacd,bckj,di->abij", "iabc T u1"),
    (+1., "kldi,abkj,dl->abij", "ijak T u1"), (-1., "kadc,cbkj,di->abij", "iabc T u1"),
    (-1., "kadc,bcki,dj->abij", "iabc T u1"), (-1., "lacd,cdji,bl->abij", "iabc T u1"),
    (-1., "lacd,cbij,dl->abij", "iabc T u1"), (+1., "abic,cj->abij", "abic u1"),
    (+4., "klcd,caki,dblj->abij", "ijab T u2"), (-2., "klcd,cakl,dbij->abij", "ijab T u2"),
    (-2., "klcd,cdki,ablj->abij", "ijab T u2"), (-2., "klcd,caki,bdlj->abij", "ijab T u2"),
    (+2., "kaci,cbkj->abij", "iabj u2"), (-2., "klcd,acki,dblj->abij", "ijab T u2"),
    (-2., "kldc,caki,dblj->abij", "ijab T u2"), (-2., "kldc,abkj,dcil->abij", "ijab T u2"),
    (-2., "lkcd,cbij,adlk->abij", "ijab T u2"), (-1., "ki,abkj->abij", "foo u2"),
    (+1., "ac,cbij->abij", "fvv u2"), (-1., "kaic,cbkj->abij", "iajb u2"),
    (-1., "kbic,ackj->abij", "iajb u2"), (+1., "klcd,ackl,dbij->abij", "ijab T u2"),
    (+1., "kldc,cdki,ablj->abij", "ijab T u2"), (+1., "klcd,acki,bdlj->abij", "ijab T u2"),
    (-1., "kaci,bckj->abij", "iabj u2"), (+1., "kldc,acki,dblj->abij", "ijab T u2"),
    (+1., "kldc,abkj,dcli->abij", "ijab T u2"), (+1., "kldc,caki,dbjl->abij", "ijab T u2"),
    (+1., "kldc,ackj,dbil->abij", "ijab T u2"), (+1., "lkcd,cbij,dalk->abij", "ijab T u2"),
]

SIGMA2_NP_TERMS = [                                                    # eom_ccsd.py:380-383
    (+1., "klij,abkl->abij", "klij u2"), (+1., "kldc,abkl,dcij->abij", "ijab T u2"),
    (+1., "lkcd,cdij,ablk->abij", "ijab T u2"), (+1., "abcd,cdij->abij", "abcd u2"),
]

V_KEYS_USED = ("ijka", "ijak", "iabc", "iajk", "abic", "ijab", "iabj", "iajb", "klij", "abcd")
_U_CANON = {"u1": "em", "u2": "efmn"}
_Z_CANON = "wxyz"


def _prod(ext, idx):
    n = 1
    for ch in idx:
        n *= ext[ch]
    return n


def _rename(sub, table):
    return "".join(table.get(ch, ch) for ch in sub)


class SigmaPlan:
    """Compiled sigma program for one (fock, V blocks, T2); see the module docstring."""

    def __init__(self, no, fock, dV, T2, hoist_cap=None, shard=None):
        """``shard`` (``pymes_b200.parallel.Shard``): this rank evaluates the rows a in
        [lo, lo+na) of sigma1[r,a,i] and sigma2[r,a,b,i,j] -- the output index ``a`` of every
        contraction is restricted on whichever operand carries it -- and the row blocks are
        all-gathered at the end of ``apply``; trial vectors and intermediates that do not carry
        ``a`` stay replicated.  The only other exchange is the all-gather of Ex for the explicit
        Ex + Ex^{baji} (eom_ccsd.py:377)."""
        self.no = no
        self.shard = shard
        self.nv = nv = T2.shape[0]
        # bk.narrow: the blocks keep the Fock matrix's momentum rule (a sector's products need it)
        rows_o, rows_v = bk.narrow(fock, 0, 0, no), bk.narrow(fock, 0, no, nv)
        self.static = {"foo": bk.narrow(rows_o, 1, 0, no), "fov": bk.narrow(rows_o, 1, no, nv),
                       "fvv": bk.narrow(rows_v, 1, no, nv), "T": T2}
        for key in V_KEYS_USED:
            self.static[key] = dV[key]
        # a hoisted intermediate may be as large as one o.v^3 integral block
        self.hoist_cap = hoist_cap if hoist_cap is not None else max(no * nv ** 3, no * no * nv * nv) * 1.01
        self.flops_per_vector = 0.0
        self.hoist_flops = 0.0
        self.programs = {"s1": self._compile(SIGMA1_TERMS), "s2p": self._compile(SIGMA2_P_TERMS),
                         "s2n": self._compile(SIGMA2_NP_TERMS)}

    # ---- planning ------------------------------------------------------
    def _compile(self, table):
        direct, twostep, operators = {}, {}, []
        for coef, spec, names in table:
            lhs, out = spec.split("->")
            subs, names = lhs.split(","), names.split()
            ext = {}
            for s, n in zip(subs, names):
                if n not in _U_CANON:
                    for ch, e in zip(s, self.static[n].shape):
                        ext[ch] = int(e)
            dyn = [i for i, n in enumerate(names) if n in _U_CANON]
            assert len(dyn) == 1, spec
            usub, uname = subs[dyn[0]], names[dyn[0]]
            for ch, e in zip(usub, (self.nv, self.no) if uname == "u1" else (self.nv, self.nv, self.no, self.no)):
                ext[ch] = e
            stat = [(subs[i], names[i]) for i in range(len(subs)) if i != dyn[0]]
            all_idx = set("".join(subs))
            if len(stat) == 1:
                self.flops_per_vector += 2.0 * _prod(ext, all_idx)
                if isinstance(self.static[stat[0][1]], bk.LinearOperator):
                    # the dressed V_abcd given as an operator (ccsd.DressedLadder): applied, not read
                    assert (stat[0][0], usub, out) == ("abcd", "cdij", "abij"), spec
                    operators.append((coef, self.static[stat[0][1]]))
                    continue
                self._add_direct(direct, coef, [stat[0]], usub, uname, out, ext)
                continue
            (s1, n1), (s2, n2) = stat
            options = []
            # (a) hoist S1.S2
            summed = {ch for ch in s1 if ch in s2 and ch not in usub and ch not in out}
            widx = (set(s1) | set(s2)) - summed
            if len(widx) <= 4 and _prod(ext, widx) <= self.hoist_cap:
                options.append((2.0 * _prod(ext, widx | set(usub) | set(out)), "hoist", None))
            # (b)/(c) X.u first, then Z
            for (xs, xn), (zs, zn) in (((s1, n1), (s2, n2)), ((s2, n2), (s1, n1))):
                sm = {ch for ch in xs if ch in usub and ch not in zs and ch not in out}
                yidx = (set(xs) | set(usub)) - sm
                if len(yidx) <= 4 and sm:
                    fl = 2.0 * _prod(ext, set(xs) | set(usub)) + 2.0 * _prod(ext, yidx | set(zs))
                    options.append((fl, "two", ((xs, xn), (zs, zn), yidx)))
            fl, kind, extra = min(options, key=lambda o: o[0])
            self.flops_per_vector += fl
            if kind == "hoist":
                self.hoist_flops += 2.0 * _prod(ext, set(s1) | set(s2))
                self._add_direct(direct, coef, stat, usub, uname, out, ext)
            else:
                (xs, xn), (zs, zn), yidx = extra
                ren = {}
                for pos, ch in enumerate(zs):
                    if ch not in out:
                        ren[ch] = _Z_CANON[pos]
                ysub = "".join(sorted(_rename("".join(yidx), ren)))
                key = (zn, _rename(zs, ren), ysub, out)
                twostep.setdefault(key, []).append((coef, _rename(xs, ren), xn, _rename(usub, ren), uname))
        prog = {"direct": [], "twostep": [], "operators": operators}
        for (wsub, usub, uname, out), items in direct.items():
            prog["direct"].append((wsub, usub, uname, out, self._materialise(wsub, items)))
        for (zn, zsub, ysub, out), items in twostep.items():
            prog["twostep"].append((self.static[zn], zsub, ysub, out, items))
        return prog

    def _add_direct(self, direct, coef, stat, usub, uname, out, ext):
        ren = {}
        for pos, ch in enumerate(usub):
            if ch not in out:
                ren[ch] = _U_CANON[uname][pos]
        if len(stat) == 1:
            widx = set(stat[0][0])
        else:
            (s1, _), (s2, _) = stat
            summed = {ch for ch in s1 if ch in s2 and ch not in usub and ch not in out}
            widx = (set(s1) | set(s2)) - summed
        wsub = "".join(sorted(_rename("".join(widx), ren)))
        key = (wsub, _rename(usub, ren), uname, out)
        direct.setdefault(key, []).append((coef, [(_rename(s, ren), n) for s, n in stat]))

    def _materialise(self, wsub, items):
        """(alpha, W): a zero-copy permuted view when the group is one plain operand, otherwise
        the coefficient-weighted sum of the group's operands / hoisted products.  In a sharded
        plan a W that carries the output index ``a`` is built for this rank's rows only (the
        hoisted products are the big replicated memory otherwise: up to o.v^3 each).  The first
        item is written, not accumulated, so that W carries the momentum rule its items derive."""
        rows = self._rows
        if len(items) == 1 and len(items[0][1]) == 1:
            coef, [(s, n)] = items[0]
            return coef, rows(wsub, bk.permute(self.static[n], [s.index(ch) for ch in wsub]))
        ext = {}
        for _, stat in items:
            for s, n in stat:
                for ch, e in zip(s, self.static[n].shape):
                    ext[ch] = int(e)
        if self.shard is not None and "a" in wsub:
            ext["a"] = self.shard.na
        W = bk.empty(*[ext[ch] for ch in wsub])
        beta = 0.0
        for coef, stat in items:
            if len(stat) == 1:
                s, n = stat[0]
                bk.axpby(coef, rows(wsub, bk.permute(self.static[n], [s.index(ch) for ch in wsub])), beta, W)
            else:
                (s1, n1), (s2, n2) = stat
                bk.contract_terms(wsub, [(coef, s1, rows(s1, self.static[n1]), s2, rows(s2, self.static[n2]))],
                                  out=W, beta=beta)
            beta = 1.0
        return 1.0, W

    # ---- execution -----------------------------------------------------
    def _rows(self, sub, t):
        """``t`` restricted to this rank's rows of the output index ``a`` (summed indices are
        renamed to e, f, m, n, w..z or keep k, l, c, d: ``a`` is always the sharded one)."""
        if self.shard is None or "a" not in sub:
            return t
        return self.shard.rows(t, sub.index("a"))

    def _run(self, prog, U, out_t):
        """out_t[r,...] += program applied to the stacked vectors U = {"u1": [r,v,o], "u2": [r,v,v,o,o]};
        with a shard, out_t holds the local rows of ``a`` only."""
        ct = bk.contract_terms
        rows = self._rows
        for wsub, usub, uname, out, (alpha, W) in prog["direct"]:      # W: local rows already
            ct("r" + out, [(alpha, wsub, W, "r" + usub, rows("r" + usub, U[uname]))], out=out_t, beta=1.0)
        for Z, zsub, ysub, out, items in prog["twostep"]:
            Y = None
            for coef, xsub, xn, usub, uname in items:
                term = [(coef, xsub, rows(xsub, self.static[xn]), "r" + usub, rows("r" + usub, U[uname]))]
                if Y is None:
                    Y = ct("r" + ysub, term)
                else:
                    ct("r" + ysub, term, out=Y, beta=1.0)
            ct("r" + out, [(1.0, "r" + ysub, Y, zsub, rows(zsub, Z))], out=out_t, beta=1.0)
        for coef, op in prog["operators"]:
            op.apply(U["u2"], out_t, coef, shard=self.shard)

    def apply(self, U1, U2, out=None):
        """sigma for a batch: U1 [r,v,o], U2 [r,v,v,o,o] device tensors (any strides along r,
        each vector contiguous) -> (S1, S2).  eom_ccsd.py:268-385 for every r at once.  Stacks
        with a momentum rule (``bk.stack`` of sector vectors) run every product on momentum groups
        and give S1, S2 with the same rules."""
        U = {"u1": U1, "u2": U2}
        r = U2.shape[0]
        if self.shard is not None:
            return self._apply_sharded(U, r, out)
        if out is None:
            S1, S2 = bk.zeros(*U1.shape, rule=bk.momentum_of(U1)), bk.empty(*U2.shape)
        else:
            S1, S2 = out
            bk.clear(S1, bk.momentum_of(U1))
        self._run(self.programs["s1"], U, S1)
        Ex = bk.zeros(*U2.shape, rule=bk.momentum_of(U2))
        self._run(self.programs["s2p"], U, Ex)
        bk.sym_baji_stack(Ex, S2)                                      # eom_ccsd.py:377
        del Ex
        self._run(self.programs["s2n"], U, S2)
        return S1, S2

    def _apply_sharded(self, U, r, out):
        """Row-block evaluation (see ``__init__``); returns / fills the FULL sigma vectors."""
        sh, no, nv = self.shard, self.no, self.nv

        def gather_rows(loc):                  # [r, na, ...] -> [r, nv, ...]
            return sh.gather(loc.transpose(0, 1).contiguous()).transpose(0, 1)

        S1l = bk.zeros(r, sh.na, no)
        self._run(self.programs["s1"], U, S1l)
        Exl = bk.zeros(r, sh.na, nv, no, no)
        self._run(self.programs["s2p"], U, Exl)
        Exf = gather_rows(Exl)                 # the (ba) block lives on another rank
        S2l = bk.empty(r, sh.na, nv, no, no)
        for k in range(r):                                             # eom_ccsd.py:377
            bk.axpby(1.0, Exl[k], 0.0, S2l[k])
            bk.axpby(1.0, sh.rows(Exf[k].permute(1, 0, 3, 2), 0), 1.0, S2l[k])
        del Exl, Exf
        self._run(self.programs["s2n"], U, S2l)
        S1f, S2f = gather_rows(S1l), gather_rows(S2l)
        if out is None:
            return S1f.contiguous(), S2f.contiguous()
        for k in range(r):
            bk.axpby(1.0, S1f[k], 0.0, out[0][k])
            bk.axpby(1.0, S2f[k], 0.0, out[1][k])
        return out

    def apply_packed(self, X):
        """Same for vectors packed as rows [singles | doubles] of X [r, v*o + v*v*o*o]."""
        no, nv = self.no, self.nv
        n1 = nv * no
        r = X.shape[0]
        Y = bk.empty(r, X.shape[1])
        self.apply(X[:, :n1].view(r, nv, no), X[:, n1:].view(r, nv, nv, no, no),
                   out=(Y[:, :n1].view(r, nv, no), Y[:, n1:].view(r, nv, nv, no, no)))
        return Y


# --------------------------------------------------------------------------
# diagonal of H-bar (FEAST preconditioner) -- eom_ccsd.py:169-266
# --------------------------------------------------------------------------
DIAG1_TERMS = [  # (coef, spec, target subscripts); operands (V_ijab, T2)       eom_ccsd.py:185-196
    (+4., "jiba,baji->ai", "ai"), (-2., "jkba,abjk->a", "a"), (-2., "jicb,bcji->i", "i"),
    (-2., "jiba,abji->ai", "ai"), (-2., "jiab,baji->ai", "ai"), (+1., "jkab,abjk->a", "a"),
    (+1., "jicb,bcji->i", "i"), (+1., "jiab,abji->ai", "ai"),
]
DIAG2_P_TERMS = [  # eom_ccsd.py:208-249, operands (V_ijab, T2)
    (+4., "kica,caki->ai", "ai"), (-2., "klca,cakl->a", "a"), (-2., "kicd,cdki->i", "i"),
    (-2., "kica,caki->ai", "ai"), (-2., "kica,acki->ai", "ai"), (-2., "kiac,caki->ai", "ai"),
    (-2., "kjab,abkj->abj", "abj"), (-2., "ijcb,cbij->ij", "ij"), (+1., "klca,ackl->a", "a"),
    (+1., "kidc,cdki->i", "i"), (+1., "kicb,acki->ai", None), (+1., "kiac,acki->ai", "ai"),
    (+1., "kiab,abkj->abij", "abij"), (+1., "kjac,caki->aij", "aij"), (+1., "kjac,ackj->aj", "aj"),
    (+1., "ijca,cbij->abij", "abij"),
]
DIAG2_NP_TERMS = [  # eom_ccsd.py:258-260
    (+1., "klab,abkl->ab", "ab"), (+1., "ijcd,cdij->ij", "ij"),
]


def diag_singles(no, fock, dV, T2):
    nv = T2.shape[0]
    d = bk.zeros(nv, no)
    foo, fvv = fock[:no, :no], fock[no:, no:]
    bk.add_broadcast(-1.0, torch.diagonal(foo), "i", d, "ai")
    bk.add_broadcast(+1.0, torch.diagonal(fvv), "a", d, "ai")
    bk.add_broadcast(+2.0, bk.diag_view(dV["iabj"], "iaai", "ai"), "ai", d, "ai")
    bk.add_broadcast(-1.0, bk.diag_view(dV["iajb"], "iaia", "ai"), "ai", d, "ai")
    for coef, spec, tgt in DIAG1_TERMS:
        bk.add_broadcast(coef, bk.bdot(spec, dV["ijab"], T2), tgt, d, "ai")
    return d


def diag_doubles(no, fock, dV, T2):
    nv = T2.shape[0]
    P = bk.zeros(nv, nv, no, no)
    foo, fvv = fock[:no, :no], fock[no:, no:]
    for coef, spec, tgt in DIAG2_P_TERMS:
        if tgt is None:
            # eom_ccsd.py:240 is written einsum("kicb, acki -> ai") with b summed on V only
            Vs = bk.contract_terms("kic", [(1.0, "kicb", dV["ijab"], "b", torch.ones(nv, dtype=bk.F64, device=T2.device))])
            bk.add_broadcast(coef, bk.bdot("kic,acki->ai", Vs, T2), "ai", P, "abij")
            continue
        bk.add_broadcast(coef, bk.bdot(spec, dV["ijab"], T2), tgt, P, "abij")
    x = bk.diag_view(dV["iabj"], "iaai", "ai")
    bk.add_broadcast(+2.0 - 1.0, x, "ai", P, "abij")                   # eom_ccsd.py:217,242
    bk.add_broadcast(-1.0, torch.diagonal(foo), "i", P, "abij")        # eom_ccsd.py:227
    bk.add_broadcast(+1.0, torch.diagonal(fvv), "a", P, "abij")
    y = bk.diag_view(dV["iajb"], "iaia", "ai")
    bk.add_broadcast(-1.0, y, "ai", P, "abij")                         # eom_ccsd.py:229
    bk.add_broadcast(-1.0, y, "ai", P, "abij")                         # eom_ccsd.py:231 ("bi" added at [a,i])
    D = bk.sym_baji(P)                                                 # eom_ccsd.py:254
    bk.add_broadcast(1.0, bk.diag_view(dV["klij"], "ijij", "ij"), "ij", D, "abij")
    for coef, spec, tgt in DIAG2_NP_TERMS:
        bk.add_broadcast(coef, bk.bdot(spec, dV["ijab"], T2), tgt, D, "abij")
    vabab = dV["abcd"].diag_abab() if isinstance(dV["abcd"], bk.LinearOperator) \
        else bk.diag_view(dV["abcd"], "abab", "ab")
    bk.add_broadcast(1.0, vabab, "ab", D, "abij")
    return D


# --------------------------------------------------------------------------
# block-vector helpers (HBM-bound kernels pmb_dots / pmb_lincomb)
# --------------------------------------------------------------------------
def pair_dot(a1, a2, b1, b2):
    """<a|b> over the (singles, doubles) pair, plain product (no conjugation)."""
    return float(bk.dots([a1], b1).item() + bk.dots([a2], b2).item())


def orthonormalise(u1s, u2s, start=0):
    """Modified Gram-Schmidt with one re-orthogonalisation pass on vectors ``start..`` against
    all earlier ones (the device stand-in for the dense Householder QR of eom_ccsd.py:512-541;
    the spanned subspace, hence every Ritz value, is the same)."""
    for n in range(start, len(u1s)):
        for _ in range(2):
            if n:
                c = (bk.dots(u1s[:n], u1s[n]) + bk.dots(u2s[:n], u2s[n])).cpu().numpy()
                u1s[n] = bk.lincomb([1.0] + list(-c), [u1s[n]] + u1s[:n])
                u2s[n] = bk.lincomb([1.0] + list(-c), [u2s[n]] + u2s[:n])
        nrm = np.sqrt(pair_dot(u1s[n], u2s[n], u1s[n], u2s[n]))
        u1s[n] = bk.lincomb([1.0 / nrm], [u1s[n]])
        u2s[n] = bk.lincomb([1.0 / nrm], [u2s[n]])
    return u1s, u2s


def _as_dict_dev(dict_t_V):
    return {k: bk.asdev(dict_t_V[k]) for k in V_KEYS_USED}


class EOM_CCSD:
    def __init__(self, no, n_excit=3, comm=None, parallel="rows", sector=None):
        """``comm`` (extension, ``pymes_b200.parallel.Comm``) with ``parallel="rows"``: the sigma
        product is evaluated in (ab) row blocks over the ranks of ``comm`` (operators too large
        for one GPU); with ``parallel="vectors"``: every rank holds the full operator and applies
        it to its share of each batch of new trial vectors, the results are summed over the ranks
        (no exchange inside sigma).  Everything else (trial vectors, the projected eigenproblem) is
        replicated and identical on every rank.

        ``sector`` (extension, ``model.ueg.excitation_sector``): :meth:`solve` finds the lowest
        states of ONE total momentum of a UEG reference.  H-bar built from momentum-conserving
        integrals never mixes sectors, so the Davidson space is kept inside the sector: the guesses
        are the sector's lowest singles, and every new trial vector is checked to lie in it (one
        pass per vector; a vector with weight outside raises) before sigma sees it, which then runs
        every product that involves it on momentum groups.  The dressed Fock matrix, T2 and the
        integral blocks are checked to conserve momentum when the sigma program is built
        (``ValueError`` if one does not: the sector would not be invariant).  Vectors keep the dense
        [v,o] / [v,v,o,o] layout.  Not available together with a sector: a ``comm`` of more than one
        rank and ``preconditioner = "diagonal"`` (both raise ``NotImplementedError``)."""
        if parallel not in ("rows", "vectors"):
            raise ValueError("parallel must be 'rows' or 'vectors'")
        if sector is not None and comm is not None and comm.size > 1:
            raise NotImplementedError("EOM-CCSD in a momentum sector runs on one device (no comm)")
        self.algo_name = "EOM-CCSD"
        # "scalar": the reference's correction vectors, r / (e_n - D_guess_n + 1e-5) with ONE number per
        # root (eom_ccsd.py:140-141).  "diagonal" (extension, not the reference's iterates): the usual
        # Davidson correction r / (e_n - diag(H-bar) + 1e-5) with the diagonal of get_diag_singles /
        # get_diag_doubles -- what converges the 54-electron systems.
        self.preconditioner = "scalar"
        self.comm = comm if parallel == "rows" else None
        self.vec_comm = comm if (parallel == "vectors" and comm is not None and comm.size > 1) else None
        self.max_rhs = 16                 # right-hand sides per batched sigma call (bounds the temporaries)
        self.no = no
        self.n_excit = n_excit
        self.u_singles = []
        self.u_doubles = []
        self.e_excit = np.zeros(n_excit)
        self.max_dim = n_excit * 4
        self.e_epsilon = 1.e-8
        self.max_iter = 500
        self._plan = None
        self._plan_key = None
        self.sector = sector

    def write_logging_info(self):
        return

    # ---- sigma ----------------------------------------------------------
    def invalidate(self):
        """Forget the compiled sigma program and the cached single-vector sigma (call after
        modifying the Fock matrix, an integral block or T2 IN PLACE: ``plan`` recognises its
        operands by identity, and for tensors by their in-place version counter)."""
        self._plan = self._plan_key = None
        self._last = None

    @staticmethod
    def _ident(x):
        return (id(x), getattr(x, "_version", None))

    def plan(self, t_fock_pq, dict_t_V, t_T_abij):
        """Compile (or fetch) the sigma program for these operands.  The hoisted H-bar
        intermediates are built from the operands' CURRENT contents; see :meth:`invalidate`."""
        key = (self._ident(t_fock_pq), id(dict_t_V), self._ident(t_T_abij))
        if self._plan is None or self._plan_key != key:
            T2 = bk.asdev(t_T_abij).contiguous()
            fock, dV = bk.asdev(t_fock_pq), _as_dict_dev(dict_t_V)
            shard = None
            if self.sector is not None:
                self._adopt_operands(t_fock_pq, fock, dV, T2)
            elif self.comm is not None and self.comm.size > 1:
                from ..parallel import Shard
                shard = Shard(self.comm, T2.shape[0])
            self._plan = SigmaPlan(self.no, fock, dV, T2, shard=shard)
            self._plan_key = key
            self._keep = (t_fock_pq, dict_t_V, t_T_abij)        # keep ids alive
        return self._plan

    def _adopt_operands(self, t_fock_pq, fock, dV, T2):
        """Tag the operands of a sector's sigma with their (total 0) momentum rules, after checking
        that every element a rule forbids is zero; ``ValueError`` names the first that breaks it."""
        sec = self.sector
        host = None if isinstance(t_fock_pq, torch.Tensor) else np.asarray(t_fock_pq)
        checks = [("the Fock matrix", bk.adopt_momentum(fock, sec.fock_rule(), host=host)),
                  ("T2", bk.adopt_momentum(T2, sec.rule("abij")))]
        for k in V_KEYS_USED:
            if isinstance(dV[k], bk.LinearOperator):
                checks.append(("V_" + k, dV[k].adopt_momentum(sec.rule)))
            else:
                checks.append(("V_" + k, bk.adopt_momentum(dV[k], sec.rule(k))))
        for what, ok in checks:
            if not ok:
                raise ValueError("%s does not conserve momentum: H-bar would mix the sector %r with others"
                                 % (what, sec))

    def sigma_batched(self, t_fock_pq, dict_t_V, U1, U2, t_T_abij):
        """(H-bar U)_singles, (H-bar U)_doubles for stacked vectors U1 [r,v,o], U2 [r,v,v,o,o]."""
        plan = self.plan(t_fock_pq, dict_t_V, t_T_abij)
        return plan.apply(bk.asdev(U1).contiguous(), bk.asdev(U2).contiguous())

    def update_singles(self, t_fock_pq, dict_t_V, t_u_ai, t_u_abij, t_T_abij):
        want_numpy = not isinstance(t_u_abij, torch.Tensor)
        S1, _ = self._single(0, t_fock_pq, dict_t_V, t_u_ai, t_u_abij, t_T_abij)
        return bk.tonumpy(S1) if want_numpy else S1

    def update_doubles(self, t_fock_pq, dict_t_V, t_u_ai, t_u_abij, t_T_abij):
        want_numpy = not isinstance(t_u_abij, torch.Tensor)
        _, S2 = self._single(1, t_fock_pq, dict_t_V, t_u_ai, t_u_abij, t_T_abij)
        return bk.tonumpy(S2) if want_numpy else S2

    def _single(self, half, t_fock_pq, dict_t_V, t_u_ai, t_u_abij, t_T_abij):
        """One vector; the (S1, S2) pair is kept so that the reference's update_singles +
        update_doubles call PAIR costs one sigma.  The kept pair serves each half once and only
        for the very same vector objects (tensors: same in-place version), so a vector that is
        modified in place between two pairs of calls is never answered from the cache."""
        key = (self._ident(t_u_ai), self._ident(t_u_abij))
        cache = getattr(self, "_last", None)
        if cache is not None and cache[0] == key and cache[1] is t_u_ai and cache[2] is t_u_abij \
                and half not in cache[4]:
            cache[4].add(half)
            return cache[3]
        u1 = bk.asdev(t_u_ai)
        u2 = bk.asdev(t_u_abij)
        if torch.is_complex(u1) or torch.is_complex(u2):
            raise TypeError("complex vectors: stack real and imaginary parts as two right-hand sides")
        S1, S2 = self.sigma_batched(t_fock_pq, dict_t_V, u1.contiguous()[None], u2.contiguous()[None], t_T_abij)
        res = (S1[0], S2[0])
        self._last = (key, t_u_ai, t_u_abij, res, {half})
        return res

    def sigma_list(self, plan, u1s, u2s):
        """sigma for lists of device vectors -> lists, in batches of at most ``max_rhs``.  In the
        "vectors" parallel mode every rank evaluates one contiguous share of the list with its
        own full operator and the shares are combined by an all-reduce over zero-filled slots."""
        n, no, nv = len(u1s), self.no, plan.nv
        vc = self.vec_comm
        lo, hi = 0, n
        if vc is not None:
            per = (n + vc.size - 1) // vc.size
            lo, hi = min(vc.rank * per, n), min((vc.rank + 1) * per, n)
        S1 = bk.zeros(n, nv, no) if vc is not None else bk.empty(n, nv, no)
        S2 = bk.zeros(n, nv, nv, no, no) if vc is not None else bk.empty(n, nv, nv, no, no)
        for b0 in range(lo, hi, self.max_rhs):
            b1 = min(b0 + self.max_rhs, hi)
            plan.apply(bk.stack(u1s[b0:b1]), bk.stack(u2s[b0:b1]), out=(S1[b0:b1], S2[b0:b1]))
        if vc is not None:
            vc.all_reduce_sum(S1)
            vc.all_reduce_sum(S2)
        return [S1[k] for k in range(n)], [S2[k] for k in range(n)]

    def get_diag_singles(self, t_fock_pq, dict_t_V, t_T_abij):
        want_numpy = not isinstance(t_T_abij, torch.Tensor)
        d = diag_singles(self.no, bk.asdev(t_fock_pq), _as_dict_dev(dict_t_V), bk.asdev(t_T_abij).contiguous())
        return bk.tonumpy(d) if want_numpy else d

    def get_diag_doubles(self, t_fock_pq, dict_t_V, t_T_abij):
        want_numpy = not isinstance(t_T_abij, torch.Tensor)
        d = diag_doubles(self.no, bk.asdev(t_fock_pq), _as_dict_dev(dict_t_V), bk.asdev(t_T_abij).contiguous())
        return bk.tonumpy(d) if want_numpy else d

    def QR(self, u_singles, u_doubles):
        """Orthonormalise the (singles, doubles) vectors; same span as eom_ccsd.py:512-541."""
        want_numpy = not isinstance(u_doubles[0], torch.Tensor)
        u1s = [bk.asdev(u).contiguous() for u in u_singles]
        u2s = [bk.asdev(u).contiguous() for u in u_doubles]
        u1s, u2s = orthonormalise(u1s, u2s)
        if want_numpy:
            return [bk.tonumpy(u) for u in u1s], [bk.tonumpy(u) for u in u2s]
        return u1s, u2s

    # ---- Davidson -------------------------------------------------------
    def solve(self, t_fock_dressed_pq, dict_t_V_dressed, t_T_abij):
        """Lowest ``n_excit`` right eigenvalues of H-bar by block Davidson, the algorithm of
        eom_ccsd.py:46-167 (unit-vector guesses on the smallest eps_a - eps_i, scalar
        preconditioner e_n - D_guess + 1e-5, collapse at 4 n_excit vectors).  Differences that do
        not change the iterates: sigma is evaluated only for vectors that are new (the reference
        recomputes all of them every sweep), in one batch; orthonormalisation is Gram-Schmidt."""
        print_title("EOM-CCSD Solver", )
        time_init = time.time()
        no, n_excit = self.no, self.n_excit
        fock = bk.asdev(t_fock_dressed_pq)
        T2 = bk.asdev(t_T_abij).contiguous()
        nv = T2.shape[0]
        fd = bk.tonumpy(fock).diagonal()
        D_ai = -(fd[:no][None, :] - fd[no:][:, None]).ravel()
        sec = self.sector
        if sec is None:
            lowest = np.argsort(D_ai)[:n_excit]
        else:
            if self.preconditioner != "scalar":
                raise NotImplementedError("EOM-CCSD in a momentum sector uses the scalar preconditioner")
            inside = sec.singles_mask().ravel()
            if not inside.any():
                raise ValueError("the sector %r holds no single excitation" % (sec,))
            if n_excit > inside.sum():
                raise ValueError("n_excit = %d exceeds the %d singles of the sector %r" % (n_excit, inside.sum(), sec))
            lowest = np.argsort(np.where(inside, D_ai, np.inf))[:n_excit]
            rule1, rule2 = sec.singles_rule(), sec.doubles_rule()
        plan = self.plan(t_fock_dressed_pq, dict_t_V_dressed, t_T_abij)

        print_logging_info("Initialising u tensors...", level=1)
        u1s = [bk.asdev(u).contiguous() for u in self.u_singles]
        u2s = [bk.asdev(u).contiguous() for u in self.u_doubles]
        for n in range(n_excit):
            A = np.zeros(nv * no)
            A[lowest[n]] = 1.
            u1s.append(bk.asdev(A.reshape(nv, no)))
            u2s.append(bk.zeros(nv, nv, no, no))
        w1s, w2s = [], []
        if self.preconditioner not in ("scalar", "diagonal"):
            raise ValueError("preconditioner must be 'scalar' or 'diagonal'")
        hdiag = None
        if self.preconditioner == "diagonal":
            dV = _as_dict_dev(dict_t_V_dressed)
            hdiag = (diag_singles(no, fock, dV, T2).reshape(-1), diag_doubles(no, fock, dV, T2).reshape(-1))
        B = np.zeros((0, 0))
        e = np.zeros(n_excit)
        e_imag = np.zeros(n_excit)
        diff_e_norm = np.inf
        for it in range(self.max_iter):
            t_it = time.time()
            m = len(u1s)
            n_done = len(w1s)
            u1s, u2s = orthonormalise(u1s, u2s, start=n_done)
            if sec is not None:
                for n in range(n_done, m):
                    if not (bk.adopt_momentum(u1s[n], rule1) and bk.adopt_momentum(u2s[n], rule2)):
                        raise RuntimeError("trial vector %d has weight outside the sector %r" % (n, sec))
            if n_done < m:
                S1, S2 = self.sigma_list(plan, u1s[n_done:], u2s[n_done:])
                w1s += S1
                w2s += S2
            Bn = np.zeros((m, m))
            Bn[:n_done, :n_done] = B
            for l in range(n_done, m):                                 # eom_ccsd.py:103-109
                col = (bk.dots(u1s, w1s[l]) + bk.dots(u2s, w2s[l])).cpu().numpy()
                Bn[:, l] = col
                row = (bk.dots(w1s[:n_done], u1s[l]) + bk.dots(w2s[:n_done], u2s[l])).cpu().numpy() \
                    if n_done else np.zeros(0)
                Bn[l, :n_done] = row
            B = Bn
            e_old = self.e_excit
            ev, v = np.linalg.eig(B)
            low = ev.argsort()[:n_excit]
            e_imag = np.imag(ev[low])
            e = np.real(ev[low])
            v = np.real(v[:, low])
            if m >= self.max_dim:                                      # collapse, eom_ccsd.py:122-133
                nu1 = [bk.lincomb(v[:, n], u1s) for n in range(n_excit)]
                nu2 = [bk.lincomb(v[:, n], u2s) for n in range(n_excit)]
                u1s, u2s, w1s, w2s, B = nu1, nu2, [], [], np.zeros((0, 0))
                self.e_excit = e_old
            else:                                                      # expand, eom_ccsd.py:134-147
                for n in range(n_excit):
                    if hdiag is None:
                        scale = 1.0 / (e[n] - D_ai[lowest[n]] + 1e-5)
                        cw = list(v[:, n] * scale)
                        cu = list(-e[n] * v[:, n] * scale)
                        u1s.append(bk.lincomb(cw + cu, w1s + u1s[:m]))
                        u2s.append(bk.lincomb(cw + cu, w2s + u2s[:m]))
                    else:                                          # residual / (e_n - diag + 1e-5), elementwise
                        cw, cu = list(v[:, n]), list(-e[n] * v[:, n])
                        for us, ws, hd in ((u1s, w1s, hdiag[0]), (u2s, w2s, hdiag[1])):
                            r = bk.lincomb(cw + cu, ws + us[:m])
                            y, _ = bk.cdiv_shifted(hd, complex(e[n]), 1e-5, r.reshape(-1), r.reshape(-1))
                            us.append(y.view(r.shape))
                diff_e_norm = np.linalg.norm(self.e_excit - e)
                self.e_excit = e
            if diff_e_norm < self.e_epsilon:
                print_logging_info("Iterative solver converged.", level=1)
                print_logging_info("Norm of energy difference = {:.12f}".format(diff_e_norm), level=2)
                for r in range(n_excit):
                    print_logging_info("Excited state {:d} energy = {:.12f}".format(r, e[r]), level=2)
                print_logging_info("Excited states energies imaginary part = ", e_imag, level=2)
                break
            print_logging_info("Iteration = ", it, level=1)
            print_logging_info("Norm of energy difference = ", diff_e_norm, level=2)
            for r in range(n_excit):
                print_logging_info("Excited state {:d} energy = {:.12f}".format(r, e[r]), level=2)
            print_logging_info("Excited states energies imaginary part = ", e_imag, level=2)
            print_logging_info("Took {:.3f} seconds ".format(time.time() - t_it), level=2)
        self.iterations = it + 1
        self.u_singles, self.u_doubles = u1s, u2s
        print_logging_info("EOM-CCSD finished in {:.3f} seconds".format(time.time() - time_init), level=1)
        print_logging_info("Converged excited states energies:", level=1)
        for r in range(n_excit):
            print_logging_info("Excited state {:d} energy = {:.12f}".format(r, e[r]), level=2)
        return self.e_excit
