"""CCD / DCD doubles solver on the B200 contraction engine.

Call surface of the reference ``pymes.solver.ccd.CCD`` (pymes/solver/ccd.py:10-262):
same constructor, ``solve`` / ``get_residual`` / ``get_energy`` signatures, the
same returned dict keys and the same log lines.  Inputs may be numpy arrays
(copied to the device once, results returned as numpy) or CUDA tensors.

The doubles residual (ccd.py:164-254) is evaluated as a short list of strided
DMMA contractions (``backend.contract_terms``) in which every index permutation
lives in the operand strides, plus three HBM-bound elementwise kernels.  Terms
that share an output layout are accumulated inside one launch:

    R   = V_abij + T.I + V_abcd.T                 hh + pp ladder   (one launch)
    R  += X1.T, Tt.Xai                            quadratic ring terms
    Ex  = Xac.T - Xki.T                           Fock-like terms
    Ex += -V_iajb.T + Tt.V_iabj - Xp.T + Xp.T'    four ring terms  (one launch)
    Ex += -V_iajb.T                               (permuted output, own launch)
    R  += Ex + Ex^{baji}                          no hermiticity assumed

No symmetrisation shortcut is taken anywhere: V_klij != V_ijkl and Ex != Ex^{baji}
for transcorrelated integrals (ccd.py:172,244-249).
"""
import time

import numpy as np
import torch

from .. import backend as bk
from ..log import print_logging_info
from ..mixer import diis
from . import drccd, mp2


class _Whole:
    """Trivial shard: one rank owns every row (the single-GPU case)."""
    lo, size = 0, 1

    def __init__(self, nv):
        self.na = nv

    def rows(self, t, dim=0):
        return t

    def gather(self, local):
        return local

    def all_reduce(self, x):
        return x


def _resolved(x):
    """A tensor, or the result of a collective still in flight (``parallel.Pending``)."""
    return x.wait_result() if hasattr(x, "wait_result") else x


def block2(t, r0, nr, c0, nc):
    """``t[r0:r0+nr, c0:c0+nc]`` as a view that keeps the momentum tag of ``t``."""
    return bk.narrow(bk.narrow(t, 0, r0, nr), 1, c0, nc)


def fock_rules(V_abij, no, nv):
    """Momentum rules of the Fock matrix (+,-), T1 [a,i] and T2 [a,b,i,j] over the labels of the
    tagged integral block ``V_abij``; None when the integrals carry no momentum tag."""
    k = bk.momentum_of(V_abij)
    if k is None:
        return None
    n = no + nv
    return {"fock": k.with_axes([(0, n, 1), (0, n, -1)]), "t1": k.with_axes([(no, nv, 1), (0, no, -1)]),
            "t2": k.with_axes([(no, nv, 1), (no, nv, 1), (0, no, -1), (0, no, -1)])}


def doubles_residual(no, fock, T2, V_klij, V_ijab, V_abij, V_iajb, V_iabj, V_abcd,
                     is_dcd=False, is_bruekner=False, pp_ladder=None, shard=None):
    """R_abij for device tensors (reference ccd.py:164-254).

    ``pp_ladder``: optional callable ``(T2, R) -> None`` adding V_abcd.T2 into R; used by
    CCSD (dressed ladder without forming the dressed V_abcd) and by sharded runs.

    ``shard`` (``pymes_b200.parallel.Shard``): this rank owns the rows a in [lo, lo+na) of
    every [a,b,i,j] quantity.  T2 and the o^2v^2-sized integral blocks are replicated; V_abij
    and V_abcd are the LOCAL row blocks; the returned R is the local row block.  The exchanges
    are an all-gather of the ring intermediate Xai (built sharded over its row index; started
    before the ladder and collected after it, so it travels while the ladder runs) and an
    all-to-all of the column blocks of Ex for the explicit Ex + Ex^{baji} permutation.
    ``V_iajb`` / ``V_iabj`` may be collectives still in flight (``parallel.Pending``): they are
    waited for at their first use, after the ladder.
    """
    nv = T2.shape[0]
    ccd = not is_dcd
    ct = bk.contract_terms
    sh = shard if shard is not None else _Whole(nv)
    T2a = sh.rows(T2, 0)            # T2[a in A, ., ., .]
    T2b = sh.rows(T2, 1)            # T2[., a in A, ., .]

    Tt = bk.tilde(T2)                                                # ccd.py:199
    Tta = sh.rows(Tt, 0)
    # Xai[c,b,k,j]: every rank builds its rows c, then all ranks need all of it   ccd.py:202
    Xai = ct("cbkj", [(1.0, "klcd", sh.rows(V_ijab, 2), "dblj", Tt)])
    if shard is not None:
        Xai = sh.gather_async(Xai)

    # I_klij = V_klij (+ V_ijab.T)                                   ccd.py:178-180
    # (sharded: each rank sums over its c in A, the o^4 partial sums are all-reduced)
    I = bk.copy(V_klij)
    if ccd:
        if shard is None:
            ct("klij", [(1.0, "klcd", V_ijab, "cdij", T2)], out=I, beta=1.0)
        else:
            bk.axpby(1.0, sh.all_reduce(ct("klij", [(1.0, "klcd", sh.rows(V_ijab, 2), "cdij", T2a)])), 1.0, I)

    # R = V_abij + I.T (hh ladder) + V_abcd.T (pp ladder)             ccd.py:185-187
    R = bk.copy(V_abij)
    ladder = [(1.0, "abkl", T2a, "klij", I)]
    if pp_ladder is None:
        ladder.append((1.0, "abcd", V_abcd, "cdij", T2))
    ct("abij", ladder, out=R, beta=1.0)
    if pp_ladder is not None:
        pp_ladder(T2, R)

    if ccd:                                                          # ccd.py:189-191
        X1 = ct("alcj", [(1.0, "klcd", V_ijab, "adkj", T2a)])
        ct("abij", [(1.0, "alcj", X1, "cbil", T2)], out=R, beta=1.0)
        del X1

    ct("abij", [(1.0, "acik", Tta, "cbkj", _resolved(Xai))], out=R, beta=1.0)   # ccd.py:204
    del Xai

    # Fock-like intermediates; the reference adds the same product twice for CCD
    # (ccd.py:213-221): X_ac = f_ab - c.Tt.V, X_ki = f_ij + c.Tt.V, c = 1/2 (DCD) or 1
    # Only the local rows a in A of X_ac are ever used; X_ki is summed over the local c in A
    # and all-reduced (o^2 numbers).
    if is_bruekner:
        # ccd.py:209-211 binds t_X_ac / t_X_ki to VIEWS of t_fock_pq, so the in-place updates of
        # ccd.py:218-221 modify the Fock matrix itself, sweep after sweep.  Reproduced: the
        # contractions below accumulate into the views of ``fock``.
        if shard is not None:
            raise NotImplementedError("is_bruekner is not available in sharded runs")
        Xac, Xki = fock[no:, no:], fock[:no, :no]
    else:
        Xac = bk.copy(sh.rows(block2(fock, no, nv, no, nv), 0))
        Xki = bk.copy(block2(fock, 0, no, 0, no))
    c = (1.0 if ccd else 0.5) if not is_bruekner else (0.5 if ccd else 0.0)
    if c != 0.0:
        ct("ac", [(-c, "adkl", Tta, "lkdc", V_ijab)], out=Xac, beta=1.0)
        if shard is None:
            ct("ki", [(+c, "cdil", Tt, "lkdc", V_ijab)], out=Xki, beta=1.0)
        else:
            bk.axpby(1.0, sh.all_reduce(ct("ki", [(+c, "cdil", Tta, "lkdc", sh.rows(V_ijab, 3))])), 1.0, Xki)

    V_iajb, V_iabj = _resolved(V_iajb), _resolved(V_iabj)
    Ex = ct("abij", [(1.0, "ac", Xac, "cbij", T2)])                  # ccd.py:231
    ct("abij", [(-1.0, "ki", Xki, "abkj", T2a)], out=Ex, beta=1.0)   # ccd.py:232
    ring = [(-1.0, "kaic", sh.rows(V_iajb, 1), "cbkj", T2),          # ccd.py:233
            (+1.0, "acik", Tta, "kbcj", V_iabj)]                     # ccd.py:235
    if ccd:                                                          # ccd.py:238-240
        Xp = ct("alci", [(1.0, "klcd", V_ijab, "daki", T2b)])
        # -Xp.T_cblj + Xp.T_bclj = Xp.(T^{ba} - T)_cblj and T^{ba} - T = T - Tt: one ring
        # contraction instead of two (one HBM pass builds the combined operand)
        ring.append((+1.0, "alci", Xp, "cblj", bk.lincomb([1.0, -1.0], [T2, Tt])))
    ct("abij", ring, out=Ex, beta=1.0)
    ct("abij", [(-1.0, "kbic", V_iajb, "ackj", T2a)], out=Ex, beta=1.0)   # ccd.py:234

    if shard is None:
        bk.sym_baji(Ex, R, accumulate=True)                          # ccd.py:249-252
    else:
        bk.axpby(1.0, Ex, 1.0, R)
        bk.axpby(1.0, sh.transposed_rows(Ex), 1.0, R)    # the (ba) blocks live on the other ranks
    return R


def _write_back(target, dev):
    """Copy a device tensor into the caller's array / tensor unless it already IS that tensor."""
    if isinstance(target, torch.Tensor):
        if target.data_ptr() != dev.data_ptr():
            target.copy_(dev)
    elif isinstance(target, np.ndarray) and target.flags.writeable:
        target[...] = bk.tonumpy(dev)


class CCD:
    def __init__(self, no, delta_e=1.e-8, is_dcd=False, is_diis=True, is_dr_ccd=False,
                 is_bruekner=False):
        self.is_dcd = is_dcd
        self.is_diis = is_diis
        self.is_dr_ccd = is_dr_ccd
        self.is_bruekner = is_bruekner
        self.no = no
        self.delta_e = delta_e
        self.max_iter = 50
        if self.is_diis:
            self.mixer = diis.DIIS(dim_space=6)

    # ------------------------------------------------------------------
    def get_residual(self, t_fock_pq, t_T_abij, t_V_klij, t_V_ijab, t_V_abij, t_V_iajb, t_V_iabj,
                     t_V_abcd):
        want_numpy = not isinstance(t_T_abij, torch.Tensor)
        fock = bk.asdev(t_fock_pq)
        R = doubles_residual(self.no, fock, bk.asdev(t_T_abij).contiguous(),
                             bk.asdev(t_V_klij), bk.asdev(t_V_ijab), bk.asdev(t_V_abij),
                             bk.asdev(t_V_iajb), bk.asdev(t_V_iabj), bk.asdev(t_V_abcd),
                             is_dcd=self.is_dcd, is_bruekner=self.is_bruekner)
        if self.is_bruekner:
            _write_back(t_fock_pq, fock)             # ccd.py:209-221 updates t_fock_pq in place
        return bk.tonumpy(R) if want_numpy else R

    def get_energy(self, t_T_abij, t_V_ijab):
        """(direct, exchange) contributions, ccd.py:256-262."""
        scal = bk.zeros(8)
        bk.energy_doubles(bk.asdev(t_T_abij).contiguous(), bk.asdev(t_V_ijab), scal)
        s = scal.cpu().numpy()
        return float(s[0]), float(s[1])

    # ------------------------------------------------------------------
    def solve(self, t_fock_pq, t_V_pqrs, level_shift=0., sp=0, amps=None, **kwargs):
        algo_name = "ccd.solve"
        t_start = time.time()
        no = self.no
        max_iter = kwargs.get("max_iter", self.max_iter)
        delta_e = kwargs.get("delta_e", self.delta_e)
        delta = 1.0
        want_numpy = not isinstance(t_V_pqrs, torch.Tensor)

        fock_host = bk.tonumpy(t_fock_pq)
        eps_i_host = fock_host.diagonal()[:no].copy()
        eps_a_host = fock_host.diagonal()[no:].copy()
        fock = bk.asdev(fock_host)
        eps_i, eps_a = bk.asdev(eps_i_host), bk.asdev(eps_a_host)
        V = bk.asdev(t_V_pqrs)
        V_iabj = V[:no, no:, no:, :no]
        V_aijb = V[no:, :no, :no, no:]
        V_ijab = V[:no, :no, no:, no:]
        V_klij = V[:no, :no, :no, :no]
        V_iajb = V[:no, no:, :no, no:]
        V_abij = V[no:, no:, :no, :no]
        V_abcd = V[no:, no:, no:, no:]

        print_logging_info(algo_name)
        print_logging_info("Using DCD: ", self.is_dcd, level=1)
        print_logging_info("Using dr-CCD: ", self.is_dr_ccd, level=1)
        print_logging_info("Solving doubles amplitude equation", level=1)
        print_logging_info("Using data type %s" % str(V.dtype).replace("torch.", ""), level=1)
        print_logging_info("Using DIIS mixer: ", self.is_diis, level=1)
        print_logging_info("Using Bruekner quasi-particle energy: ", self.is_bruekner, level=1)
        print_logging_info("Iteration = 0", level=1)
        e_mp2, T2 = mp2.solve_device(eps_i, eps_a, V_ijab, V_abij, level_shift)
        print("MP2 energy = ", e_mp2)
        amps_host = None
        if amps is not None:
            if isinstance(amps, torch.Tensor):
                T2 = bk.asdev(amps)          # aliased: updated in place like the reference
                if not T2.is_contiguous():   # the elementwise kernels index the amplitudes flat
                    raise ValueError("amps given as a tensor must be contiguous [nv,nv,no,no]")
            else:
                amps_host = amps
                T2 = bk.asdev(amps).contiguous()

        scal = bk.zeros(8)
        dE = abs(e_mp2)
        iteration = 0
        e_last = e_mp2
        e_ccd = e_dir = e_ex = 0.0
        while abs(dE) > delta_e and iteration <= max_iter:
            iteration += 1
            if self.is_dr_ccd:                                       # ccd.py:95-98
                R = drccd.residual_device(eps_i, eps_a, T2, V_abij, V_aijb, V_iabj, V_ijab)
            else:
                R = doubles_residual(no, fock, T2, V_klij, V_ijab, V_abij, V_iajb, V_iabj, V_abcd,
                                     is_dcd=self.is_dcd, is_bruekner=self.is_bruekner)
            if self.is_bruekner:
                if iteration == 1:
                    # t_epsilon_i / t_epsilon_a are VIEWS of the Fock diagonal in the reference
                    # (ccd.py:40-41) until the first rebinding at ccd.py:110: they see what
                    # get_residual has just done to the matrix
                    eps_i = torch.diagonal(fock)[:no].contiguous()
                    eps_a = torch.diagonal(fock)[no:].contiguous()
                eps_i, eps_a = self._bruekner_energies(eps_i, eps_a, T2, V_ijab)
            dT = bk.update_doubles(eps_i, eps_a, level_shift, delta, R, T2, scal[3:4],
                                   product_denominator=self.is_bruekner)         # ccd.py:118
            del R
            if amps_host is not None and (iteration == 1 or not self.is_diis):
                amps_host[...] = bk.tonumpy(T2)      # the reference mutates `amps` in place
            if self.is_diis:
                T2 = self.mixer.mix([dT], [T2])[0]
            bk.energy_doubles(T2, V_ijab, scal)
            s = scal.cpu().numpy()
            e_dir, e_ex = float(s[0]), float(s[1])
            e_ccd = e_dir + e_ex
            dE = e_ccd - e_last
            e_last = e_ccd
            t2_norm, res_norm = float(np.sqrt(s[2])), float(np.sqrt(s[3]))
            if iteration <= max_iter:
                print_logging_info("Iteration = ", iteration, level=1)
                print_logging_info("Correlation Energy = {:.12f}".format(e_ccd), level=2)
                print_logging_info("dE = {:.12e}".format(dE), level=2)
                print_logging_info("L1 Norm of T2 = {:.12f}".format(t2_norm), level=2)
                print_logging_info("Norm Residual = {:.12f}".format(res_norm), level=2)
            else:
                print_logging_info("A converged solution is not found!", level=1)

        print_logging_info("Direct contribution = {:.12f}".format(e_dir), level=1)
        print_logging_info("Exchange contribution = {:.12f}".format(e_ex), level=1)
        print_logging_info("CCD correlation energy = {:.12f}".format(e_ccd), level=1)
        print_logging_info("{:.3f} seconds spent on CCD".format(time.time() - t_start), level=1)
        self.iterations = iteration
        if self.is_bruekner:
            _write_back(t_fock_pq, fock)             # the reference leaves its caller's matrix modified
        if want_numpy:
            return {"ccd e": e_ccd, "t2 amp": bk.tonumpy(T2), "hole e": bk.tonumpy(eps_i),
                    "particle e": bk.tonumpy(eps_a), "dE": dE}
        return {"ccd e": e_ccd, "t2 amp": T2, "hole e": eps_i, "particle e": eps_a, "dE": dE}

    def _bruekner_energies(self, eps_i, eps_a, T2, V_ijab):
        """Amplitude-dependent quasi-particle energies, ccd.py:104-113.  i / a are batch indices
        (in both operands and the output): ``pmb_bdot``, not a matrix product."""
        Tt = bk.tilde(T2)
        di = bk.bdot("ilcd,cdil->i", V_ijab, Tt, alpha=0.5)
        da = bk.bdot("klad,adkl->a", V_ijab, Tt, alpha=-0.5)
        return eps_i + di, eps_a + da
