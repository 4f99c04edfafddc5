"""FEAST-EOM-CCSD: contour-integral eigensolver for the non-hermitian H-bar on the B200 engine.

Call surface of the reference ``pymes.solver.feast_eom_ccsd.FEAST_EOM_CCSD``
(pymes/solver/feast_eom_ccsd.py:17-181): ``FEAST_EOM_CCSD(no, e_c, e_r, n_trial, max_iter, tol)``,
attributes ``n_excit = 2, linear_solver, ls_max_iter = 20, u_singles, u_doubles, eigvals, eigvecs``,
``solve(fock_dressed, dictV_dressed, T2) -> eigvals`` and the module functions
``get_gauss_legendre_quadrature`` / ``normalize_amps``.  New attribute: ``n_nodes`` (the
reference hard-codes 8 quadrature points, feast:97).

The algorithm is the reference's: Gauss-Legendre nodes on the upper half circle
z_e = e_c + e_r exp(i theta_e), one linear solve (z_e - H-bar) Q_e = u_l per (node, trial
vector), Q_l = - sum_e w_e/2 Re(e_r exp(i theta_e) Q_e), Rayleigh-Ritz with the NON-orthogonal
Q (generalised eigenproblem H_proj c = lambda B c), trial space grown until n_trial.

What is different is how the linear systems are solved.  The reference runs scipy's
GCROT(m,k) once per system, i.e. 8 x n_trial sequential Krylov solvers, each calling the
62-term sigma for one complex vector.  Here ALL systems advance in lock-step through the same
GCROT(m,k) (``_solve_group``: inner flexible GMRES cycles of m + max(k - |CU|, 0) steps -- 40
in the first cycle -- with the same right preconditioner 1/(z - diag + 0.01), the same relative
tolerance 1e-4, the same recycling of (c, u) pairs with the oldest dropped beyond k = m = 20 and
the same outer limit ``ls_max_iter``): every Krylov step makes ONE batched sigma call whose
right-hand sides are the real and imaginary parts of the current vector of every unconverged
system (H-bar is real, so a complex vector is two real ones).  Systems that converge within the
first cycle reproduce scipy's iterate to rounding.
"""
import time

import numpy as np
import torch
from scipy.linalg import eig

from .. import backend as bk
from ..log import print_logging_info, print_title
from .eom_ccsd import EOM_CCSD


def get_gauss_legendre_quadrature(n):
    return np.polynomial.legendre.leggauss(n)


def normalize_amps(u_singles, u_doubles):
    """feast:626-631 for numpy arrays (in place) or device tensors (new tensors)."""
    if isinstance(u_singles, torch.Tensor):
        nrm = np.sqrt(bk.dots([u_singles], u_singles).item() + bk.dots([u_doubles], u_doubles).item())
        return bk.lincomb([1.0 / nrm], [u_singles]), bk.lincomb([1.0 / nrm], [u_doubles])
    nrm = np.sqrt(np.tensordot(np.conj(u_singles), u_singles, axes=2)
                  + np.tensordot(np.conj(u_doubles), u_doubles, axes=4))
    u_singles /= nrm
    u_doubles /= nrm
    return u_singles, u_doubles


class _CVec:
    """Complex vector as two flat real device tensors."""
    __slots__ = ("re", "im")

    def __init__(self, re, im):
        self.re, self.im = re, im


def _cdots_launch(vs, w):
    """Launch the dot products <v_k, w> = sum conj(v_k) w for a list of _CVec; returns the device
    results (no synchronisation) for :func:`_cdots_finish`."""
    flat = []
    for v in vs:
        flat += [v.re, v.im]
    parts = []
    for lo in range(0, len(flat), 16):
        chunk = flat[lo:lo + 16]
        parts.append((bk.dots(chunk, w.re), bk.dots(chunk, w.im)))
    return len(vs), parts


def _cdots_finish(pending):
    n, parts = pending
    out = np.zeros(n, dtype=complex)
    k0 = 0
    for a, b in parts:
        a, b = a.cpu().numpy(), b.cpu().numpy()
        for k in range(len(a) // 2):
            out[k0 + k] = (a[2 * k] + b[2 * k + 1]) + 1j * (b[2 * k] - a[2 * k + 1])
        k0 += len(a) // 2
    return out


def _cdots(vs, w):
    """<v_k, w> for a list of _CVec (numpy complex array)."""
    return _cdots_finish(_cdots_launch(vs, w))


def _norms(vecs):
    """2-norms of a list of _CVec with ONE host synchronisation."""
    if not vecs:
        return []
    sq = torch.stack([bk.dots([v.re], v.re)[0] + bk.dots([v.im], v.im)[0] for v in vecs])
    return list(np.sqrt(sq.cpu().numpy()))


def _caxpy(w, coefs, vs):
    """w + sum_k coefs[k] * vs[k] (complex coefficients) as a new _CVec."""
    cr, ci, tr, ti = [1.0], [1.0], [w.re], [w.im]
    for c, v in zip(coefs, vs):
        cr += [c.real, -c.imag]
        tr += [v.re, v.im]
        ci += [c.real, c.imag]
        ti += [v.im, v.re]
    return _CVec(bk.lincomb(cr, tr), bk.lincomb(ci, ti))


class FEAST_EOM_CCSD(EOM_CCSD):
    def __init__(self, no, e_c=0., e_r=1, n_trial=5, max_iter=20, tol=1e-12, **kwargs):
        """Extensions (keywords): ``comm`` (``pymes_b200.parallel.Comm``) and ``parallel``:
        ``"rows"`` -- every batched sigma is evaluated in (ab) row blocks over the ranks (for
        operators that do not fit one GPU); ``"systems"`` -- the (quadrature node x trial vector)
        linear systems of the contour are dealt out over the ranks, every rank applies the full
        (replicated, never-materialised-V_abcd) operator to its own systems and the only exchanges
        are the all-reduce of the filtered vectors Q and of H-bar Q (SURVEY 8e, second form).

        ``sector`` (``model.ueg.excitation_sector``): the states of ONE total momentum of a UEG
        reference.  The operators are checked and tagged as in ``EOM_CCSD(sector=...)`` (``ValueError``
        names one that breaks momentum conservation), and every vector the driver holds -- trial
        vectors, contour sums Q, H-bar Q and every GCROT vector -- is COMPACT: the ``n_sec`` allowed
        elements of the packed [singles | doubles] layout (``ExcitationSector.packed_index``).  Sigma
        scatters up to ``max_rhs`` of them into a persistent dense staging stack that carries the
        sector rules, runs ``SigmaPlan.apply`` on momentum groups and gathers the result (after
        checking that both outputs still carry the sector rules).  ``max_rhs`` defaults to 16 in a
        sector: the dense staging (U2, S2 and the Ex temporary of ``apply``, 3 x 16 doubles vectors)
        then stays under 37 GB at 389 plane waves (v = 362, o = 27).  The seeded start vectors are the
        reference's dense draws restricted to the sector; ``u_singles`` / ``u_doubles`` come back
        dense ([v,o] / [v,v,o,o], zero outside the sector, tagged with its rules) and are accepted as
        start vectors when they lie in the sector (``ValueError`` otherwise).  The K = 0 sector
        (doubles only) is allowed; an empty sector or one smaller than ``n_trial`` raises
        ``ValueError``.  ``parallel="systems"`` works in a sector; ``parallel="rows"`` with more than
        one rank raises ``NotImplementedError``."""
        self.parallel = kwargs.get("parallel", "rows")
        if self.parallel not in ("rows", "systems"):
            raise ValueError("parallel must be 'rows' or 'systems'")
        comm = kwargs.get("comm")
        sector = kwargs.get("sector")
        if sector is not None and self.parallel == "rows" and comm is not None and comm.size > 1:
            raise NotImplementedError("FEAST-EOM-CCSD in a momentum sector: row-sharded sigma is not available; "
                                      "use parallel='systems'")
        super().__init__(no, n_excit=2, comm=comm if self.parallel == "rows" else None, sector=sector)
        self.sys_comm = comm if (self.parallel == "systems" and comm is not None and comm.size > 1) else None
        self.e_c = e_c
        self.e_r = e_r
        self.n_trial = n_trial
        self.n_excit = 2
        self.max_iter = max_iter
        self.tol = tol
        self.linear_solver = "Jacobi"
        self.ls_max_iter = 20
        self.ls_tol = 1e-4           # gcrotmk(tol=1e-4), feast:346
        self.ls_restart = 20         # scipy's default m (inner steps per cycle once the recycle space is full)
        self.ls_recycle = None       # scipy's k: recycled (c, u) pairs kept; None = m, like gcrotmk(k=None)
        self.n_nodes = 8             # feast:97
        # real right-hand sides per batched sigma call (in a sector: per dense staging stack)
        self.max_rhs = 64 if sector is None else 16
        self.max_systems = None      # systems advanced together (None: all); bounds the Krylov memory
        self._layout = None          # sector mode: the compact layout and the dense staging stack
        self.u_singles = []
        self.u_doubles = []
        self.eigvals = np.array([self.e_c - self.e_r, self.e_c + self.e_r])
        self.eigvecs = None
        self.ls_matvecs = 0
        self.ls_residuals = []

    def dump_log(self):
        pass

    # ---- sector layout ----------------------------------------------------
    def sector_layout(self, nv):
        """Sector mode: the compact layout of the sector for ``nv`` virtuals, built once -- a dict with
        ``host`` (``packed_index``, numpy), ``idx`` (the same on the device), ``i1`` / ``i2`` (device
        offsets of the singles in [v,o] and of the doubles in [v,v,o,o]), ``n1`` (singles in the
        sector) and ``n`` (all elements).  ``ValueError`` for an empty sector or one smaller than
        ``n_trial``."""
        sec = self.sector
        if self._layout is None or self._layout["nv"] != nv:
            host = sec.packed_index()
            if len(host) == 0:
                raise ValueError("the sector %r holds no excitation" % (sec,))
            if len(host) < self.n_trial:
                raise ValueError("n_trial = %d exceeds the %d excitations of the sector %r"
                                 % (self.n_trial, len(host), sec))
            n1 = int(np.searchsorted(host, nv * self.no))
            dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(bk.device())
            self._layout = {"nv": nv, "host": host, "idx": dev(host), "i1": dev(host[:n1]),
                            "i2": dev(host[n1:] - nv * self.no), "n1": n1, "n": len(host), "staging": None}
        return self._layout

    def _staging(self, lay, r):
        """The first ``r`` rows of the dense staging stacks U1 [R,v,o] / U2 [R,v,v,o,o]: zeroed once and
        tagged with the stacked sector rules (scatters write only allowed elements, so they keep them)."""
        st = lay["staging"]
        if st is None or st[0].shape[0] < r:
            st = lay["staging"] = None                      # free the smaller stack before the larger one
            sec, nv, no = self.sector, lay["nv"], self.no
            st = lay["staging"] = [bk.zeros(r, *shape, rule=rule.with_axes([(0, r, 0)] + list(rule.axes)))
                                   for rule, shape in ((sec.singles_rule(), (nv, no)),
                                                       (sec.doubles_rule(), (nv, nv, no, no)))]
        return bk.narrow(st[0], 0, 0, r), bk.narrow(st[1], 0, 0, r)

    def _sigma_compact(self, plan, X):
        """H-bar on the compact sector vectors X [r, n_sec]: scatter into the staging stack, sigma on
        momentum groups, gather."""
        lay = self.sector_layout(plan.nv)
        n1, r = lay["n1"], X.shape[0]
        U1, U2 = self._staging(lay, r)
        if n1:
            bk.sector_scatter(X[:, :n1], lay["i1"], U1)
        bk.sector_scatter(X[:, n1:], lay["i2"], U2)
        k1, k2 = bk.momentum_of(U1), bk.momentum_of(U2)
        S1, S2 = plan.apply(U1, U2)
        if k1 is None or k2 is None or bk.momentum_of(S1) != k1 or bk.momentum_of(S2) != k2:
            raise RuntimeError("sigma in the sector %r lost the sector rule: gathering it would drop weight"
                               % (self.sector,))
        Y = bk.empty(r, lay["n"])
        if n1:
            bk.sector_gather(S1, lay["i1"], out=Y[:, :n1])
        bk.sector_gather(S2, lay["i2"], out=Y[:, n1:])
        return Y

    def _apply_block(self, plan, X):
        """H-bar on the rows of X: packed dense vectors, or compact ones in a sector."""
        return plan.apply_packed(X) if self.sector is None else self._sigma_compact(plan, X)

    # ---- batched linear solves -------------------------------------------
    def _sigma_c(self, plan, vecs):
        """H-bar applied to a list of _CVec through batched real sigma calls."""
        flat = []
        for v in vecs:
            flat += [v.re, v.im]
        out = []
        for lo in range(0, len(flat), self.max_rhs):
            Y = self._apply_block(plan, torch.stack(flat[lo:lo + self.max_rhs]))
            out += [Y[k] for k in range(Y.shape[0])]
        self.ls_matvecs += len(vecs)
        return [_CVec(out[2 * k], out[2 * k + 1]) for k in range(len(vecs))]

    def solve_shifted_systems(self, plan, diag, zs, rhs, hscale=1.0):
        """Solve (z_s - hscale * H-bar) x_s = rhs_s for every s (``rhs``: list of flat device
        vectors, real tensors or complex ``_CVec``; ``zs``: complex shifts; ``hscale``: a complex
        scalar, 1 for FEAST, i*dt for the real-time propagator of rt_eom_ccsd.py).
        The reference's GCROT(m,k) (``_solve_group``) advanced in lock-step over groups of at most
        ``max_systems`` systems (each system keeps up to ``ls_restart + ls_recycle + 1`` complex
        Krylov vectors and ``ls_recycle`` recycled pairs); returns the list of complex solutions
        (_CVec)."""
        group = self.max_systems or len(zs)
        out, res = [], []
        for lo in range(0, len(zs), group):
            x, r = self._solve_group(plan, diag, list(zs[lo:lo + group]), list(rhs[lo:lo + group]), hscale)
            out += x
            res += r
        self.ls_residuals = res
        return out

    def _solve_group(self, plan, diag, zs, rhs, hscale):
        """GCROT(m,k) as scipy runs it for the reference (``gcrotmk(A, b, x0=0, M=M, maxiter=ls_max_iter,
        tol=1e-4)``, feast:346; scipy/sparse/linalg/_isolve/_gcrotmk.py, m = 20, k = m, truncate =
        'oldest'), for every system of the group in lock-step.  Per outer iteration and system:

        * an inner flexible GMRES cycle of ``ml = m + max(k - len(CU), 0)`` steps at most (40 in the
          first cycle, when nothing has been recycled yet) on ``r / |r|`` with the right
          preconditioner, every new direction first projected off the recycled C vectors
          (coefficients B), stopped when the estimated residual drops below ``tol |b|``;
        * ``u = Z y - U (B y)``, ``c = V (H y)`` normalised to ``|c| = 1``, ``x += <c, r> u``,
          ``r -= <c, r> c`` (the residual is carried by this recurrence and recomputed from x only
          when it signals convergence, as scipy does), ``(c, u)`` appended to the recycle space,
          the oldest pair dropped beyond k.

        With an empty recycle space the first cycle is a plain right-preconditioned GMRES(40): a
        system that converges within it -- every system of the fixtures -- reproduces scipy's
        iterate to rounding (LiH: 7e-15 relative; FEAST eigenvalues of a seeded run: 3e-14 Eh)."""
        nsys = len(zs)
        hscale = complex(hscale)
        m_inner = self.ls_restart
        k_keep = m_inner if self.ls_recycle is None else int(self.ls_recycle)
        first = rhs[0].re if isinstance(rhs[0], _CVec) else rhs[0]
        zero = torch.zeros_like(first)
        rhs = [b if isinstance(b, _CVec) else _CVec(b, zero) for b in rhs]
        bnorm = _norms(rhs)
        x = [None] * nsys
        res = list(rhs)                                     # x0 = 0 -> r0 = b
        rnorm = list(bnorm)
        CU = [[] for _ in range(nsys)]                      # recycled (c, u) pairs per system
        active = [s for s in range(nsys) if bnorm[s] > 0]

        def apply_op(vecs_s, vecs):
            """(z_s - hscale H-bar) v for a list of systems / vectors."""
            HV = self._sigma_c(plan, vecs)
            out = []
            for s, v, hv in zip(vecs_s, vecs, HV):
                if hscale == 1.0:
                    out.append(_caxpy(_CVec(bk.lincomb([-1.0], [hv.re]), bk.lincomb([-1.0], [hv.im])), [zs[s]], [v]))
                else:
                    out.append(_caxpy(_CVec(zero, zero), [zs[s], -hscale], [v, hv]))
            return out

        for _outer in range(self.ls_max_iter):
            # scipy's loop head: a residual (from the recurrence) at the tolerance is recomputed from x
            # before it ends the solve
            check = [s for s in active if rnorm[s] <= self.ls_tol * bnorm[s] and x[s] is not None]
            if check:
                AX = apply_op(check, [x[s] for s in check])
                for s, ax in zip(check, AX):
                    res[s] = _caxpy(rhs[s], [-1.0 + 0j], [ax])
                del AX
                for s, rn in zip(check, _norms([res[s] for s in check])):
                    rnorm[s] = rn
            active = [s for s in active if rnorm[s] > self.ls_tol * bnorm[s]]
            if not active:
                break
            ml = {s: m_inner + max(k_keep - len(CU[s]), 0) for s in active}
            V = {s: [_CVec(bk.lincomb([1.0 / rnorm[s]], [res[s].re]), bk.lincomb([1.0 / rnorm[s]], [res[s].im]))]
                 for s in active}
            H = {s: np.zeros((ml[s] + 1, ml[s]), dtype=complex) for s in active}
            B = {s: np.zeros((len(CU[s]), ml[s]), dtype=complex) for s in active}
            y = {}
            running = list(active)
            for j in range(max(ml.values())):
                if not running:
                    break
                P = [_CVec(*bk.cdiv_shifted(diag, zs[s], 0.01, V[s][j].re, V[s][j].im)) for s in running]
                W = apply_op(running, P)
                del P
                # GCROT projection off the recycled C vectors, then Gram-Schmidt against V with one
                # refinement.  Every pass launches the dot products of ALL running systems, reads them
                # back together, then launches all the updates: the host waits for the device a fixed
                # number of times per Krylov step, not per system and dot.
                if any(CU[s] for s in running):
                    for _ in range(2):
                        pend = [_cdots_launch([c for c, _u in CU[s]], w) if CU[s] else None
                                for s, w in zip(running, W)]
                        for n, (s, pd) in enumerate(zip(running, pend)):
                            if pd is None:
                                continue
                            h = _cdots_finish(pd)
                            W[n] = _caxpy(W[n], list(-h), [c for c, _u in CU[s]])
                            B[s][:, j] += h
                for _ in range(2):
                    pend = [_cdots_launch(V[s], w) for s, w in zip(running, W)]
                    hs = [_cdots_finish(pd) for pd in pend]
                    for n, (s, h) in enumerate(zip(running, hs)):
                        W[n] = _caxpy(W[n], list(-h), V[s])
                        H[s][:j + 1, j] += h
                hns = _norms(W)
                nxt = []
                for s, w, hn in zip(running, W, hns):
                    H[s][j + 1, j] = hn
                    e1 = np.zeros(j + 2, dtype=complex)
                    e1[0] = rnorm[s]
                    ys, *_ = np.linalg.lstsq(H[s][:j + 2, :j + 1], e1, rcond=None)
                    y[s] = ys
                    est = np.linalg.norm(e1 - H[s][:j + 2, :j + 1] @ ys)
                    ok = hn > 1e-14 * rnorm[s]
                    if ok:                                  # v_{j+1}: needed for c = V (H y) as well
                        V[s].append(_CVec(bk.lincomb([1.0 / hn], [w.re]), bk.lincomb([1.0 / hn], [w.im])))
                    if est > self.ls_tol * bnorm[s] and ok and j + 1 < ml[s]:
                        nxt.append(s)
                del W
                running = nxt
            # outer update: u = M (V y) - U (B y), c = V (H y), normalised; x += <c,r> u, r -= <c,r> c
            cxs, uxs = [], []
            for s in active:
                k = len(y[s])
                vy = _caxpy(_CVec(zero, zero), list(y[s]), V[s][:k])
                ux = _CVec(*bk.cdiv_shifted(diag, zs[s], 0.01, vy.re, vy.im))
                if CU[s]:
                    ux = _caxpy(ux, list(-(B[s][:, :k] @ y[s])), [u for _c, u in CU[s]])
                hy = H[s][:k + 1, :k] @ y[s]
                nv_ = min(len(V[s]), k + 1)                 # after a breakdown v_{k} does not exist (its weight is ~0)
                cxs.append(_caxpy(_CVec(zero, zero), list(hy[:nv_]), V[s][:nv_]))
                uxs.append(ux)
            del V
            cn = _norms(cxs)
            upd = []
            for n, s in enumerate(active):
                if not (cn[n] > 0 and np.isfinite(cn[n])):
                    continue                                # scipy: "cannot update, so skip it"
                a_ = 1.0 / cn[n]
                cxs[n] = _CVec(bk.lincomb([a_], [cxs[n].re]), bk.lincomb([a_], [cxs[n].im]))
                uxs[n] = _CVec(bk.lincomb([a_], [uxs[n].re]), bk.lincomb([a_], [uxs[n].im]))
                upd.append((n, s))
            gam = [_cdots_launch([cxs[n]], res[s]) for n, s in upd]
            for (n, s), pd in zip(upd, gam):
                g_ = _cdots_finish(pd)[0]
                res[s] = _caxpy(res[s], [-g_], [cxs[n]])
                x[s] = _caxpy(x[s] if x[s] is not None else _CVec(zero, zero), [g_], [uxs[n]])
                while len(CU[s]) >= k_keep and CU[s]:
                    del CU[s][0]
                CU[s].append((cxs[n], uxs[n]))
            for (n, s), rn in zip(upd, _norms([res[s] for _n, s in upd])):
                rnorm[s] = rn
            del cxs, uxs
        return ([xs if xs is not None else _CVec(zero, zero) for xs in x],
                [rn / bn if bn > 0 else 0.0 for rn, bn in zip(rnorm, bnorm)])

    # ---- reference-shaped single solve (used by the parity tests) ---------
    def _gcrotmk(self, l, ze, diag_ai, diag_abij, t_fock_dressed_pq, dict_t_V_dressed, t_T_abij, **kwargs):
        """(Q_singles, Q_doubles) = (ze - H-bar)^-1 u_l as complex numpy arrays, feast:293-350."""
        if self.sector is not None:
            raise NotImplementedError("_gcrotmk takes dense vectors; in a sector use solve_shifted_systems")
        plan = self.plan(t_fock_dressed_pq, dict_t_V_dressed, t_T_abij)
        d1, d2 = bk.asdev(diag_ai), bk.asdev(diag_abij)
        diag = torch.cat([d1.reshape(-1), d2.reshape(-1)])
        b = torch.cat([bk.asdev(self.u_singles[l]).reshape(-1), bk.asdev(self.u_doubles[l]).reshape(-1)])
        q = self.solve_shifted_systems(plan, diag, [complex(ze)], [b])[0]
        qc = bk.tonumpy(q.re) + 1j * bk.tonumpy(q.im)
        n1 = d1.numel()
        return qc[:n1].reshape(tuple(d1.shape)), qc[n1:].reshape(tuple(d2.shape))

    # ---- FEAST -----------------------------------------------------------
    def _share(self, n):
        """Indices 0..n-1 dealt out round-robin over the ranks of the system-parallel mode."""
        if self.sys_comm is None:
            return list(range(n))
        return list(range(self.sys_comm.rank, n, self.sys_comm.size))

    def _sum_over_ranks(self, t):
        if self.sys_comm is not None:
            self.sys_comm.all_reduce_sum(t)
        return t

    def _start_vector(self, u_singles, u_doubles):
        """A user-supplied start vector as one flat device vector (compact in a sector, after checking
        that it lies in the sector: ``ValueError`` otherwise)."""
        u1, u2 = bk.asdev(u_singles).contiguous(), bk.asdev(u_doubles).contiguous()
        sec = self.sector
        if sec is None:
            return torch.cat([u1.reshape(-1), u2.reshape(-1)])
        if not (bk.adopt_momentum(u1, sec.singles_rule()) and bk.adopt_momentum(u2, sec.doubles_rule())):
            raise ValueError("a start vector has weight outside the sector %r" % (sec,))
        lay = self.sector_layout(u1.shape[0])
        out = bk.empty(1, lay["n"])
        if lay["n1"]:
            bk.sector_gather(u1.reshape(1, -1), lay["i1"], out=out[:, :lay["n1"]])
        bk.sector_gather(u2.reshape(1, -1), lay["i2"], out=out[:, lay["n1"]:])
        return out[0]

    def solve(self, t_fock_dressed_pq, dict_t_V_dressed, t_T_abij):
        print_title("FEAST-EOM-CCSD Solver")
        time_init = time.time()
        no = self.no
        plan = self.plan(t_fock_dressed_pq, dict_t_V_dressed, t_T_abij)
        nv = plan.nv
        n1 = nv * no
        d1 = self.get_diag_singles(t_fock_dressed_pq, dict_t_V_dressed, bk.asdev(t_T_abij))
        d2 = self.get_diag_doubles(t_fock_dressed_pq, dict_t_V_dressed, bk.asdev(t_T_abij))
        diag = torch.cat([d1.reshape(-1), d2.reshape(-1)])
        sec = self.sector
        if sec is not None:                                 # every vector below is compact
            lay = self.sector_layout(nv)
            diag = bk.sector_gather(diag[None], lay["idx"])[0]

        print_logging_info("Initialising u tensors...", level=1)
        U = [self._start_vector(a, b) for a, b in zip(self.u_singles, self.u_doubles)]
        for _ in range(self.n_excit):                       # same RNG call order as feast:89-91
            a = 0.5 - np.random.rand(nv, no)
            b = (0.5 - np.random.rand(nv, nv, no, no)) * 0.01
            u = np.concatenate([a.ravel(), b.ravel()])
            U.append(bk.asdev(u if sec is None else u[lay["host"]]))
        if self.sys_comm is not None:                       # one start for all ranks: rank 0's
            for u in U:
                if self.sys_comm.rank != 0:
                    u.zero_()
                self.sys_comm.all_reduce_sum(u)
        x, w = get_gauss_legendre_quadrature(self.n_nodes)
        theta = -np.pi / 2 * (x - 1)
        z = self.e_c + self.e_r * np.exp(1j * theta)
        self.timings = []

        e_norm_prev = 1e10
        for it in range(self.max_iter):
            t_it = time.time()
            nrm = np.sqrt(torch.stack([bk.dots([u], u)[0] for u in U]).cpu().numpy())
            U = [bk.lincomb([1.0 / n], [u]) for u, n in zip(U, nrm)]
            m = len(U)
            # all (node, trial vector) systems in lock-step batches                 feast:113-121
            # (system-parallel mode: this rank's share of them)
            mine = self._share(len(z) * m)
            zs = [z[g // m] for g in mine]
            rhs = [U[g % m] for g in mine]
            mv0 = self.ls_matvecs
            sol = self.solve_shifted_systems(plan, diag, zs, rhs)
            Q = [None] * m
            per_l = {}
            for g, s_ in zip(mine, sol):
                per_l.setdefault(g % m, []).append((g // m, s_))
            for l in range(m):
                coefs, vecs = [], []
                for e, s_ in per_l.get(l, []):
                    f = -w[e] / 2 * self.e_r * np.exp(1j * theta[e])
                    coefs += [f.real, -f.imag]              # Re(f * q) = f_r q_r - f_i q_i
                    vecs += [s_.re, s_.im]
                q = torch.zeros_like(U[0]) if not vecs else None
                for lo in range(0, len(vecs), 16):
                    q = bk.lincomb(coefs[lo:lo + 16], vecs[lo:lo + 16], out=q, beta=0.0 if q is None else 1.0)
                Q[l] = q
            del sol, per_l
            Qs = self._sum_over_ranks(torch.stack(Q))       # contour sum over every rank's nodes
            Q = [Qs[l] for l in range(m)]
            # H-bar Q, each rank its share of the columns                             feast:128-134
            Wq = torch.zeros_like(Qs)
            cols = self._share(m)
            for lo in range(0, len(cols), self.max_rhs):
                sel = cols[lo:lo + self.max_rhs]
                Wq[sel] = self._apply_block(plan, Qs[sel])
            self._sum_over_ranks(Wq)
            H_proj, B = np.zeros((m, m)), np.zeros((m, m))
            hb = [(bk.dots(Q, Wq[i]), bk.dots(Q, Q[i])) for i in range(m)]
            for i, (h_, b_) in enumerate(hb):               # one read-back after all launches
                H_proj[:, i] = h_.cpu().numpy()
                B[:, i] = b_.cpu().numpy()
            self.eigvals, self.eigvecs = eig(H_proj, B)     # feast:148
            C = np.real(self.eigvecs)
            if m < self.n_trial:                            # feast:151-159
                for l in range(len(self.eigvals)):
                    U.append(bk.lincomb(list(C[:, l]), Q))
            else:                                           # feast:160-164
                for l in range(len(self.eigvals)):
                    U[l] = bk.lincomb([1.0] + list(C[:, l]), [U[l]] + Q)
            del Q, Qs, Wq
            e_norm = np.linalg.norm(self.eigvals)
            self.timings.append({"iteration": it, "trial_vectors": m, "systems_this_rank": len(mine),
                                 "matvecs_this_rank": self.ls_matvecs - mv0,
                                 "max_rel_residual": max(self.ls_residuals) if self.ls_residuals else 0.0,
                                 "seconds": time.time() - t_it})
            if np.abs(e_norm - e_norm_prev) < self.tol:
                break
            print_logging_info(f"Iter = {it}, Eigenvalues: {self.eigvals}", level=1)
            print_logging_info(f"Norm of eigenvalues: {e_norm}, Difference: {np.abs(e_norm - e_norm_prev)}",
                               level=1)
            e_norm_prev = e_norm
        self.iterations = it + 1
        if sec is None:
            self.u_singles = [u[:n1].view(nv, no) for u in U]
            self.u_doubles = [u[n1:].view(nv, nv, no, no) for u in U]
        else:                                               # dense, zero outside the sector, tagged
            ns = lay["n1"]
            self.u_singles = [bk.sector_scatter(u[:ns], lay["i1"], bk.zeros(nv, no, rule=sec.singles_rule()))
                              for u in U]
            self.u_doubles = [bk.sector_scatter(u[ns:], lay["i2"],
                                                bk.zeros(nv, nv, no, no, rule=sec.doubles_rule())) for u in U]
        print_logging_info(f"FEAST-EOM-CCSD finished in {time.time() - time_init:.2f} seconds.", level=0)
        self.e_excit = self.eigvals
        return self.eigvals
