"""Real-time propagation of the EOM-CCSD linear ansatz by a Cauchy contour integral
(reference pymes/solver/rt_eom_ccsd.py:13-133, SURVEY 8(f).3).

One step maps a state Y = (u_singles, u_doubles) to

    Q = - sum_e  w_e/2 * e_r*dt*exp(i theta_e) * (Z_e - i*dt*H-bar)^-1 exp(Z_e) Y ,
    Z_e = (i*e_c + e_r*exp(i theta_e)) * dt ,   theta_e = -pi * x_e   (8 Gauss-Legendre nodes),

followed by ``normalize_amps`` (rt_eom_ccsd.py:92-124).  The eight shifted systems are the same
kind FEAST solves, with H-bar scaled by i*dt: they run together through the lock-step batched
GCROT(m,k) of ``FEAST_EOM_CCSD.solve_shifted_systems`` (one batched sigma call per Krylov step), with
the reference's diagonal preconditioner 1/(Z_e - diag + 0.01) (feast_eom_ccsd.py:341-342).

The reference class cannot run at HEAD (it calls the ctf-era ``.to_nparray()`` on numpy arrays,
rt_eom_ccsd.py:84-85, and never sets ``ls_max_iter``, which ``_gcrotmk`` reads); the golden
fixture tests/golden/rt_LiH.npz was produced by running it with those two points shimmed
(tests/golden/make_golden.py::sec_rt) -- no arithmetic touched."""
import time

import numpy as np
import torch

from .. import backend as bk
from ..log import print_logging_info, print_title
from .feast_eom_ccsd import FEAST_EOM_CCSD, _CVec, get_gauss_legendre_quadrature


class RT_EOM_CCSD(FEAST_EOM_CCSD):
    def __init__(self, no, e_c=0., e_r=1, dt=0.1, tol=1e-12, max_iter=100, **kwargs):
        if kwargs.get("sector") is not None:
            raise NotImplementedError("RT-EOM-CCSD in a momentum sector is not available")
        super().__init__(no, e_c=e_c, e_r=e_r, n_trial=1, max_iter=max_iter, tol=tol, **kwargs)
        self.dt = dt
        self.u_singles = None
        self.u_doubles = None

    def solve(self, t_fock_dressed_pq, dict_t_V_dressed, t_T_abij, dt=0.1, u_singles=None, u_doubles=None):
        """One propagation step; returns (Q_singles, Q_doubles) as complex numpy arrays (device
        complex tensors when the state came in as tensors), normalised like the reference."""
        print_title("RT-EOM-CCSD Solver")
        time_init = time.time()
        if u_doubles is None or u_singles is None:
            raise RuntimeError("No initial state specified!")
        want_numpy = not isinstance(u_doubles, torch.Tensor)
        no = self.no
        plan = self.plan(t_fock_dressed_pq, dict_t_V_dressed, t_T_abij)
        nv = plan.nv
        n1 = nv * no
        d1 = self.get_diag_singles(t_fock_dressed_pq, dict_t_V_dressed, bk.asdev(t_T_abij))
        d2 = self.get_diag_doubles(t_fock_dressed_pq, dict_t_V_dressed, bk.asdev(t_T_abij))
        diag = torch.cat([bk.asdev(d1).reshape(-1), bk.asdev(d2).reshape(-1)])

        def flat(part):
            s, d = (bk.tonumpy(u_singles), bk.tonumpy(u_doubles)) if want_numpy else (u_singles, u_doubles)
            if want_numpy:
                v = np.concatenate([np.asarray(part(s)).ravel(), np.asarray(part(d)).ravel()])
                return bk.asdev(np.ascontiguousarray(v, dtype=np.float64))
            return torch.cat([part(s).reshape(-1), part(d).reshape(-1)]).to(bk.F64).contiguous()

        is_complex = np.iscomplexobj(bk.tonumpy(u_singles)) if want_numpy else u_singles.is_complex()
        y_re = flat(lambda t: t.real if is_complex else t)
        y_im = flat(lambda t: t.imag) if is_complex else torch.zeros_like(y_re)
        self.u_singles, self.u_doubles = [u_singles], [u_doubles]

        x, w = get_gauss_legendre_quadrature(self.n_nodes)              # rt_eom_ccsd.py:92-95
        theta = -np.pi * x
        z = (self.e_c * 1j + self.e_r * np.exp(1j * theta)) * dt
        rhs = []
        for e in range(len(z)):                                         # exp(Z_e) * Y
            ph = np.exp(z[e])
            rhs.append(_CVec(bk.lincomb([ph.real, -ph.imag], [y_re, y_im]),
                             bk.lincomb([ph.imag, ph.real], [y_re, y_im])))
        sol = self.solve_shifted_systems(plan, diag, list(z), rhs, hscale=1j * dt)
        cr, ci, vr, vi = [], [], [], []
        for e in range(len(z)):                                         # rt_eom_ccsd.py:112-115
            f = -w[e] / 2 * self.e_r * dt * np.exp(1j * theta[e])
            cr += [f.real, -f.imag]
            vr += [sol[e].re, sol[e].im]
            ci += [f.imag, f.real]
            vi += [sol[e].re, sol[e].im]
        q_re, q_im = bk.lincomb(cr, vr), bk.lincomb(ci, vi)
        nrm = np.sqrt(bk.dots([q_re], q_re).item() + bk.dots([q_im], q_im).item())
        print_logging_info("Norm of new u vec before normalization = ", nrm * nrm)
        q_re, q_im = bk.lincomb([1.0 / nrm], [q_re]), bk.lincomb([1.0 / nrm], [q_im])
        print_logging_info(f"RT-EOM-CCSD finished in {time.time() - time_init:.2f} seconds.", level=0)
        if want_numpy:
            q = bk.tonumpy(q_re) + 1j * bk.tonumpy(q_im)
            Q1, Q2 = q[:n1].reshape(nv, no), q[n1:].reshape(nv, nv, no, no)
        else:
            q = torch.complex(q_re, q_im)
            Q1, Q2 = q[:n1].view(nv, no), q[n1:].view(nv, nv, no, no)
        self.u_singles, self.u_doubles = [Q1], [Q2]
        return Q1, Q2
