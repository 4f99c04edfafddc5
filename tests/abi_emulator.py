"""TEST INFRASTRUCTURE: a numpy emulation of the C ABI in include/pymes_b200.h.

It exists so that the *host logic* of pymes_b200 (einsum parsing, descriptor
building, dressing term tables, DIIS bookkeeping, solver drivers) can be checked
against the oracle in the GPU-less build container.  It is installed only by the
``cpu_abi`` fixture in tests/conftest.py (monkeypatching ``_lib.load`` and the
device helpers); the product package never imports it, has no CPU path of its
own, and raises if the CUDA library is missing.  The semantics implemented here
are exactly the ones documented in the header, descriptor field by field.
"""
import ctypes as C
import itertools

import numpy as np
import torch


def _window(ptr, n):
    """float64 view of n host doubles starting at raw address ptr."""
    return np.ctypeslib.as_array((C.c_double * n).from_address(ptr))


def _val(p):
    if p is None:
        return None
    return p.value if hasattr(p, "value") else int(p)


def _offsets(exts, strides):
    """Offsets of a composite index, first listed index fastest."""
    mult = [np.arange(e, dtype=np.int64) * s for e, s in zip(exts, strides)]
    out = np.zeros(1, dtype=np.int64)
    for m in mult[::-1]:
        out = (out[:, None] + m[None, :]).reshape(-1)
    return out


def _gather(ptr, offs):
    lo, hi = int(offs.min()), int(offs.max())
    win = _window(ptr + 8 * lo, hi - lo + 1)
    return win[offs - lo], win, lo


class FakeLib:
    """Drop-in for the ctypes library object."""

    def __init__(self):
        self.launches = 0

    # ---- info -------------------------------------------------------
    def pmb_version(self):
        return 100

    def pmb_launch_count(self):
        return self.launches

    def pmb_launch_count_reset(self):
        self.launches = 0

    def pmb_error_string(self, code):
        return b"emulated error %d" % code

    def pmb_reduce_workspace(self):
        return 8 * 64

    def pmb_contract_workspace(self, dref):
        return 0

    def pmb_contract_set_tuning(self, a, b):
        return None

    def pmb_contract_set_panel_bytes(self, n):
        return None

    # ---- contraction ------------------------------------------------
    def pmb_contract(self, dref, ws, ws_bytes, stream):
        d = dref._obj
        self.launches += 1
        m_ext = [d.m_ext[i] for i in range(d.nm)]
        n_ext = [d.n_ext[i] for i in range(d.nn)]
        M = int(np.prod(m_ext)) if m_ext else 1
        N = int(np.prod(n_ext)) if n_ext else 1
        acc = np.zeros((M, N))
        for ti in range(d.nterms):
            t = d.terms[ti]
            k_ext = [t.k_ext[i] for i in range(t.nk)]
            am = _offsets(m_ext, [t.a_mstr[i] for i in range(d.nm)])
            ak = _offsets(k_ext, [t.a_kstr[i] for i in range(t.nk)])
            bk_ = _offsets(k_ext, [t.b_kstr[i] for i in range(t.nk)])
            bn = _offsets(n_ext, [t.b_nstr[i] for i in range(d.nn)])
            if t.a_gen:
                A = self._generated(t.a_gen, m_ext, k_ext)
            else:
                A, _, _ = _gather(t.A, (am[:, None] + ak[None, :]).reshape(-1))
            B, _, _ = _gather(t.B, (bk_[:, None] + bn[None, :]).reshape(-1))
            acc += t.alpha * (A.reshape(M, -1) @ B.reshape(-1, N))
        cm = _offsets(m_ext, [d.c_mstr[i] for i in range(d.nm)])
        cn = _offsets(n_ext, [d.c_nstr[i] for i in range(d.nn)])
        offs = (cm[:, None] + cn[None, :]).reshape(-1)
        old, win, lo = _gather(d.C, offs)
        new = acc.reshape(-1) + (d.beta * old if d.beta != 0.0 else 0.0)
        win[offs - lo] = new
        return 0

    def pmb_cdiv_shifted(self, n, diag, zr, zi, shift, xr, xi, yr, yi, stream):
        self.launches += 1
        x = _window(_val(xr), n) + 1j * _window(_val(xi), n)
        y = x / (complex(zr, zi) - _window(_val(diag), n) + shift)
        _window(_val(yr), n)[:] = y.real
        _window(_val(yi), n)[:] = y.imag
        return 0

    def pmb_gemv(self, dref, stream):
        d = dref._obj
        self.launches += 1
        k_ext = [d.k_ext[i] for i in range(d.nk)]
        x_ext = [d.x_ext[i] for i in range(d.nx)]
        vk = _offsets(k_ext, [d.v_kstr[i] for i in range(d.nk)])
        bk_ = _offsets(k_ext, [d.b_kstr[i] for i in range(d.nk)])
        bx = _offsets(x_ext, [d.b_xstr[i] for i in range(d.nx)])
        ox = _offsets(x_ext, [d.o_xstr[i] for i in range(d.nx)])
        vec, _, _ = _gather(d.vec, vk)
        B, _, _ = _gather(d.B, (bk_[:, None] + bx[None, :]).reshape(-1))
        val = d.alpha * (vec @ B.reshape(len(vk), len(bx)))
        old, win, lo = _gather(d.out, ox)
        win[ox - lo] = val if d.beta == 0.0 else val + d.beta * old
        return 0

    def pmb_bdot(self, dref, stream):
        d = dref._obj
        self.launches += 1
        i_ext = [d.i_ext[i] for i in range(d.ni)]
        r_ext = [d.r_ext[i] for i in range(d.nr)]
        oi = _offsets(i_ext, [d.o_istr[i] for i in range(d.ni)])
        ai = _offsets(i_ext, [d.a_istr[i] for i in range(d.ni)])
        bi = _offsets(i_ext, [d.b_istr[i] for i in range(d.ni)])
        ar = _offsets(r_ext, [d.a_rstr[i] for i in range(d.nr)])
        br = _offsets(r_ext, [d.b_rstr[i] for i in range(d.nr)])
        A, _, _ = _gather(d.A, (ai[:, None] + ar[None, :]).reshape(-1))
        B, _, _ = _gather(d.B, (bi[:, None] + br[None, :]).reshape(-1))
        val = d.alpha * (A * B).reshape(len(oi), -1).sum(axis=1)
        old, win, lo = _gather(d.out, oi)
        win[oi - lo] = val if d.beta == 0.0 else val + d.beta * old
        return 0

    # ---- elementwise ------------------------------------------------
    def pmb_axpby4(self, ext, alpha, inp, in_str, beta, out, out_str, stream):
        self.launches += 1
        e = [ext[i] for i in range(4)]
        oi = _offsets(e[::-1], [in_str[i] for i in range(4)][::-1])
        oo = _offsets(e[::-1], [out_str[i] for i in range(4)][::-1])
        src, _, _ = _gather(_val(inp), oi)
        old, win, lo = _gather(_val(out), oo)
        # beta = 0: alpha x is stored as it is (a -0.0 stays -0.0) and the output is never read
        win[oo - lo] = alpha * src if beta == 0.0 else alpha * src + beta * old
        return 0

    @staticmethod
    def _denoms(no, nv, ei, ea, shift):
        ei, ea = _window(_val(ei), no), _window(_val(ea), nv)
        return (ei[None, None, :, None] + ei[None, None, None, :] - ea[:, None, None, None]
                - ea[None, :, None, None] + shift), ei, ea

    def pmb_mp2_amplitudes(self, no, nv, a_lo, na, ei, ea, shift, V, v_str, T2, stream):
        self.launches += 1
        D, _, _ = self._denoms(no, nv, ei, ea, shift)
        offs = _offsets([no, no, nv, na], [v_str[3], v_str[2], v_str[1], v_str[0]])
        v, _, _ = _gather(_val(V), offs)
        _window(_val(T2), na * nv * no * no)[:] = (v.reshape(na, nv, no, no) / D[a_lo:a_lo + na]).reshape(-1)
        return 0

    def pmb_update_doubles(self, no, nv, a_lo, na, ei, ea, shift, delta, denom_mode, R, dT, T2, scal, ws, wsb,
                           stream):
        self.launches += 2
        n = na * nv * no * no
        D, e_i, e_a = self._denoms(no, nv, ei, ea, shift)
        if denom_mode:
            # the product in the kernel's order: ((e_i e_j) (-e_a)) (-e_b)
            D = (((e_i[None, None, :, None] * e_i[None, None, None, :]) * -e_a[:, None, None, None])
                 * -e_a[None, :, None, None]) + shift
        d = _window(_val(R), n) * (1.0 / D[a_lo:a_lo + na]).reshape(-1)
        _window(_val(dT), n)[:] = d
        _window(_val(T2), n)[:] += delta * d
        _window(_val(scal), 1)[0] = np.sum(d * d)
        return 0

    def pmb_update_singles(self, no, nv, ei, ea, shift, delta, R1, dT1, T1, stream):
        self.launches += 1
        ei_, ea_ = _window(_val(ei), no), _window(_val(ea), nv)
        D = ei_[None, :] - ea_[:, None] + shift
        d = _window(_val(R1), nv * no) * (1.0 / D).reshape(-1)
        _window(_val(dT1), nv * no)[:] = d
        _window(_val(T1), nv * no)[:] += delta * d
        return 0

    def pmb_energy_doubles(self, no, nv, a_lo, na, T2, T1, V, v_str, mp2_form, scal, ws, wsb, stream):
        self.launches += 3
        n = na * nv * no * no
        t = _window(_val(T2), n).reshape(na, nv, no, no)
        tau = t
        if _val(T1):
            t1 = _window(_val(T1), nv * no).reshape(nv, no)
            tau = t + np.einsum("ai,bj->abij", t1[a_lo:a_lo + na], t1)
        offs = _offsets([nv, nv, no, no], [v_str[3], v_str[2], v_str[1], v_str[0]])
        v, _, _ = _gather(_val(V), offs)
        v = v.reshape(no, no, nv, nv)
        s = _window(_val(scal), 3)
        s[0] = 2.0 * np.einsum("abij,ijab->", tau, v[:, :, a_lo:a_lo + na, :])
        if mp2_form:
            s[1] = -np.einsum("abij,jiab->", tau, v[:, :, a_lo:a_lo + na, :])
        else:
            s[1] = -np.einsum("abij,ijba->", tau, v[:, :, :, a_lo:a_lo + na])
        s[2] = np.sum(t * t)
        return 0

    def pmb_tilde(self, no, nv, T2, Tt, swap_ij, stream):
        if no <= 0 or nv <= 0 or _val(T2) == _val(Tt):
            return -1                     # PMB_E_BADARG, as the library does
        self.launches += 1
        n = nv * nv * no * no
        t = _window(_val(T2), n).reshape(nv, nv, no, no)
        perm = (0, 1, 3, 2) if swap_ij else (1, 0, 2, 3)
        _window(_val(Tt), n)[:] = (2.0 * t - t.transpose(perm)).reshape(-1)
        return 0

    def pmb_sym_baji(self, no, nv, Ex, R, accumulate, stream):
        if no <= 0 or nv <= 0 or _val(Ex) == _val(R):
            return -1
        self.launches += 1
        n = nv * nv * no * no
        e = _window(_val(Ex), n).reshape(nv, nv, no, no)
        v = (e + e.transpose(1, 0, 3, 2)).reshape(-1)
        r = _window(_val(R), n)
        r[:] = r + v if accumulate else v
        return 0

    def pmb_dots(self, nvec, X, Y, n, out, ws, wsb, stream):
        if not 1 <= nvec <= 16 or n <= 0:
            return -1                     # PMB_E_BADARG, as the library does
        self.launches += 2
        y = _window(_val(Y), n)
        o = _window(_val(out), nvec)
        for k in range(nvec):
            o[k] = np.dot(_window(X[k], n), y)
        return 0

    def pmb_lincomb(self, nvec, c, X, n, beta, out, stream):
        if not 1 <= nvec <= 16 or n <= 0:
            return -1
        self.launches += 1
        o = _window(_val(out), n)
        acc = beta * o if beta != 0.0 else np.zeros(n)
        for k in range(nvec):
            acc = acc + c[k] * _window(X[k], n)
        o[:] = acc
        return 0

    # ---- UEG --------------------------------------------------------
    @staticmethod
    def _ueg(u):
        u = getattr(u, "_obj", u)          # byref(...) from the shim, or the struct itself
        nP = u.n_orb
        kvec = np.ctypeslib.as_array((C.c_int32 * (3 * nP)).from_address(u.kvec)).reshape(nP, 3)
        kp = _window(u.kp, 3 * nP).reshape(nP, 3)
        n = 2 * u.imax + 1
        imap = np.ctypeslib.as_array((C.c_int32 * n ** 3).from_address(u.index_map))
        tab = _window(u.u_table, u.u_table_len) if u.u_table else None
        return u, nP, kvec.astype(np.int64), kp, imap, tab

    @staticmethod
    def _u(tab, v):
        n2 = np.sum(np.asarray(v) ** 2, axis=-1)
        return np.where(n2 < len(tab), tab[np.minimum(n2, len(tab) - 1)], 0.0)

    def pmb_ueg_umat(self, u, box_len, cutoff, nq, qvec, out, stream):
        self.launches += 1
        u, nP, kvec, kp, imap, tab = self._ueg(u)
        q = np.ctypeslib.as_array((C.c_int32 * (3 * nq)).from_address(_val(qvec))).reshape(nq, 3)
        g = np.arange(-cutoff, cutoff + 1)
        kprime = np.array(list(itertools.product(g, g, g)), dtype=np.int64)
        k1 = 2 * np.pi * kprime / box_len
        o = _window(_val(out), nq)
        for n in range(nq):
            qf = 2 * np.pi * q[n].astype(float) / box_len
            k2 = qf - k1
            o[n] = np.sum(np.einsum("ni,ni->n", k1, k2) * self._u(tab, kprime)
                          * self._u(tab, q[n].astype(np.int64) - kprime)) / u.omega
        return 0

    def pmb_ueg_pair_tables(self, u, mode, umat_pr, W0, W1, stream):
        self.launches += 1
        u, nP, kvec, kp, imap, tab = self._ueg(u)
        um = _window(_val(umat_pr), nP * nP).reshape(nP, nP) if _val(umat_pr) else np.zeros((nP, nP))
        w0 = np.zeros((nP, nP))
        w1 = np.zeros((nP, nP))
        no = u.n_occ
        for p in range(nP):
            for r in range(nP):
                d = kp[r] - kp[p]
                di = kvec[r] - kvec[p]
                d2 = d.dot(d)
                nz = abs(d2) > 0
                ud = float(self._u(tab, di)) if tab is not None else 0.0

                def ex3(o):
                    v = kp[o] - kp[:no]
                    return np.sum(v.dot(d) * ud * self._u(tab, kvec[o] - kvec[:no])) / u.omega

                def pk(o):
                    b = kp[o] - kp[:no]
                    a = b - d
                    bi = kvec[o] - kvec[:no]
                    return np.sum(np.einsum("ni,ni->n", a, b) * self._u(tab, bi - di)
                                  * self._u(tab, bi)) / u.omega
                if mode == 0:
                    w0[p, r] = 4 * np.pi / d2 / u.omega if nz else 0.0
                elif mode == 1:
                    w0[p, r] = (-u.n_ele * d2 * ud ** 2 / u.omega) / u.omega if nz else 0.0
                elif mode == 2:
                    if nz:
                        w0[p, r] = (4 * np.pi / d2 + um[p, r] + d2 * ud) / u.omega
                        w1[p, r] = -ud / u.omega
                    else:
                        w0[p, r] = um[p, r] / u.omega
                elif mode == 3:
                    w0[p, r] = ((4 * np.pi / d2 + um[p, r] + d2 * ud) if nz else um[p, r]) / u.omega
                elif mode == 4:
                    if nz:
                        w0[p, r] = 4 * np.pi / d2 / u.omega
                        w1[p, r] = -ud / u.omega
                elif mode == 5:
                    if nz:
                        w0[p, r] = (-u.n_ele * d2 * ud ** 2 / u.omega + 2 * ex3(r) - 2 * ex3(p)
                                    + 2 * pk(r)) / u.omega
                    else:
                        w0[p, r] = 2 * pk(r) / u.omega
                elif mode == 6:
                    w0[p, r] = 2 * ex3(r) / u.omega if nz else 0.0
                elif mode == 7:
                    w0[p, r] = -2 * ex3(p) / u.omega if nz else 0.0
                elif mode == 8:
                    w0[p, r] = 2 * pk(r) / u.omega
        _window(_val(W0), nP * nP)[:] = w0.reshape(-1)
        if _val(W1):
            _window(_val(W1), nP * nP)[:] = w1.reshape(-1)
        return 0

    def pmb_blocked_contract(self, dref, stream):
        """Block-diagonal contraction, exactly as the header states it: per tile, the tile's rows
        meet the tile's entries; columns n = n1 * n0_ext + n0."""
        d = dref._obj
        self.launches += 1
        if d.n_tiles == 0:
            return 0
        ints = lambda ptr, n, ct: np.ctypeslib.as_array((ct * n).from_address(ptr))
        tiles = ints(d.tiles, 4 * d.n_tiles, C.c_int32).reshape(-1, 4)
        assert tiles[:, 1].min() >= 1 and tiles[:, 1].max() <= 64 and tiles[:, 3].min() >= 1
        n_rows = int((tiles[:, 0] + tiles[:, 1]).max())
        n_ent = int((tiles[:, 2] + tiles[:, 3]).max())
        a_moff, c_moff = ints(d.a_moff, n_rows, C.c_int64), ints(d.c_moff, n_rows, C.c_int64)
        a_koff, b_koff = ints(d.a_koff, n_ent, C.c_int64), ints(d.b_koff, n_ent, C.c_int64)
        n = np.arange(d.n0_ext * d.n1_ext, dtype=np.int64)
        bn = (n // d.n0_ext) * d.b_n1str + n % d.n0_ext
        cn = (n // d.n0_ext) * d.c_n1str + n % d.n0_ext
        seen = np.zeros(n_rows, dtype=bool)
        for m0, mn, k0, kn in tiles:
            assert not seen[m0:m0 + mn].any(), "a row belongs to two tiles"
            seen[m0:m0 + mn] = True
            A, _, _ = _gather(d.A, (a_moff[m0:m0 + mn, None] + a_koff[None, k0:k0 + kn]).reshape(-1))
            B, _, _ = _gather(d.B, (b_koff[k0:k0 + kn, None] + bn[None, :]).reshape(-1))
            offs = (c_moff[m0:m0 + mn, None] + cn[None, :]).reshape(-1)
            old, win, lo = _gather(d.C, offs)
            val = d.alpha * (A.reshape(mn, kn) @ B.reshape(kn, -1)).reshape(-1)
            win[offs - lo] = val + (d.beta * old if d.beta != 0.0 else 0.0)
        return 0

    def pmb_gather_expand(self, dref, stream):
        """out[x0,x1,x2,j] = beta*out + alpha * val[x] * D[idx[x], j], as the header states it."""
        d = dref._obj
        self.launches += 1
        ext = [d.ext[i] for i in range(4)]
        role = [d.role[i] for i in range(4)]
        assert sorted(role) == [0, 1, 2, 3]
        grids = np.meshgrid(*[np.arange(e, dtype=np.int64) for e in ext], indexing="ij")
        xoff = np.zeros(ext, dtype=np.int64)
        j = None
        for dim, r in enumerate(role):
            if r == 3:
                j = grids[dim]
            else:
                xoff += grids[dim] * d.x_str[r]
        n_tab = int(xoff.max()) + 1
        val = _window(d.val, n_tab)
        idx = np.ctypeslib.as_array((C.c_int32 * n_tab).from_address(d.idx))
        t = idx[xoff]
        doff = np.where(t >= 0, t, 0) * d.d_ystr + j * d.d_jstr
        Dv, _, _ = _gather(d.D, doff.reshape(-1))
        new = np.where(t.reshape(-1) >= 0, d.alpha * val[xoff].reshape(-1) * Dv, 0.0)
        out = _window(d.out, int(np.prod(ext)))
        out[:] = new + (d.beta * out if d.beta != 0.0 else 0.0)
        return 0

    def _generated(self, addr, m_ext, k_ext):
        """A[M,K] of a generated operand (pmb_ueg_operand_t): the block pmb_ueg_build_block
        would write, with its axes arranged as the M / K index groups (first listed fastest)."""
        from pymes_b200 import _lib
        g = _lib.UegOperand.from_address(addr)
        axes = [g.m_axis[i] for i in range(len(m_ext))] + [g.k_axis[i] for i in range(len(k_ext))]
        assert sorted(axes) == [0, 1, 2, 3]
        ext = [0] * 4
        for ax, e in zip(axes, list(m_ext) + list(k_ext)):
            ext[ax] = e
        lo = [g.lo[i] for i in range(4)]
        if g.nz:
            # compressed values: expand nz[p,q,r] to its dense position s*(p,q,r)
            u, nP, kvec, kp, imap, tab = self._ueg(g.ueg)
            nz = _window(g.nz, ext[0] * ext[1] * ext[2]).reshape(ext[:3])
            blk = np.zeros(ext)
            n = 2 * u.imax + 1
            for p in range(ext[0]):
                for q in range(ext[1]):
                    for r in range(ext[2]):
                        v = kvec[lo[1] + q] - (kvec[lo[2] + r] - kvec[lo[0] + p]) + u.imax
                        loc = n * n * v[0] + n * v[1] + v[2]
                        if 0 <= loc < n ** 3 and lo[3] <= imap[loc] < lo[3] + ext[3]:
                            blk[p, q, r, imap[loc] - lo[3]] = nz[p, q, r]
                        else:
                            assert nz[p, q, r] == 0.0
        else:
            blk = self._block(g.ueg, g.W0a, g.W1a, g.W0s, lo, ext)
        nm = len(m_ext)
        order = axes[:nm][::-1] + axes[nm:][::-1]           # slowest first, M group then K group
        M = int(np.prod(m_ext)) if m_ext else 1
        return np.ascontiguousarray(blk.transpose(order)).reshape(M, -1).reshape(-1)

    def pmb_synth_block(self, n_orb, seed, eps, table, lo, ext, out, stream):
        """csrc/synth_build.cu restated with numpy integer arithmetic (written independently of
        pymes_b200/util/synthetic.py so that the two check each other)."""
        self.launches += 1
        seed = int(seed.value if hasattr(seed, "value") else seed)
        n = np.uint64(n_orb)
        tab = _window(_val(table), 65536)
        idx = [np.arange(lo[d], lo[d] + ext[d], dtype=np.uint64) for d in range(4)]
        p, q, r, s = np.meshgrid(*idx, indexing="ij")
        m1, m2, gold = np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB), np.uint64(0x9E3779B97F4A7C15)

        def mix(x):
            x = (x ^ (x >> np.uint64(30))) * m1
            x = (x ^ (x >> np.uint64(27))) * m2
            return x ^ (x >> np.uint64(31))
        with np.errstate(over="ignore"):
            c = np.minimum(((p * n + q) * n + r) * n + s, ((q * n + p) * n + s) * n + r)
            h = mix(mix(c * gold + np.uint64(seed) * m1 + np.uint64(1)))
        vals = eps * tab[(h >> np.uint64(48)).astype(np.int64)]
        _window(_val(out), vals.size)[:] = vals.reshape(-1)
        return 0

    def pmb_ueg_build_nz(self, u, W0a, W1a, W0s, lo, ext, out, stream):
        self.launches += 1
        blk = self._block(u, W0a, W1a, W0s, [lo[i] for i in range(4)], [ext[i] for i in range(4)])
        # at most one non-zero per dense row: the row sum IS that element
        assert (np.count_nonzero(blk, axis=3) <= 1).all()
        _window(_val(out), blk[..., 0].size)[:] = blk.sum(axis=3).reshape(-1)
        return 0

    def pmb_ueg_build_block(self, u, W0a, W1a, W0s, lo, ext, out, stream):
        self.launches += 1
        blk = self._block(u, W0a, W1a, W0s, [lo[i] for i in range(4)], [ext[i] for i in range(4)])
        _window(_val(out), blk.size)[:] = blk.reshape(-1)
        return 0

    def _block(self, u, W0a, W1a, W0s, lo, ext):
        u, nP, kvec, kp, imap, tab = self._ueg(u)
        get = lambda p: _window(_val(p), nP * nP).reshape(nP, nP) if _val(p) else None
        W0a, W1a, W0s = get(W0a), get(W1a), get(W0s)
        blk = np.zeros(ext)
        n = 2 * u.imax + 1
        for p in range(lo[0], lo[0] + ext[0]):
            for q in range(lo[1], lo[1] + ext[1]):
                for r in range(lo[2], lo[2] + ext[2]):
                    v = kvec[q] - (kvec[r] - kvec[p]) + u.imax
                    loc = n * n * v[0] + n * v[1] + v[2]
                    if not 0 <= loc < n ** 3:
                        continue
                    s = imap[loc]
                    if s < 0 or s >= nP or not lo[3] <= s < lo[3] + ext[3]:
                        continue
                    w = 0.0
                    if W0a is not None:
                        w = W0a[p, r]
                    if W1a is not None and W1a[p, r] != 0.0:
                        w += W1a[p, r] * (kp[r] - kp[s]).dot(kp[r] - kp[p])
                    if W0s is not None:
                        w += 0.5 * (W0s[p, r] + W0s[q, s])
                    blk[p - lo[0], q - lo[1], r - lo[2], s - lo[3]] = w
        return blk


def install(monkeypatch):
    """Route pymes_b200 through the emulator with host tensors (tests only)."""
    from pymes_b200 import _lib, backend as bk
    fake = FakeLib()
    cpu = torch.device("cpu")
    monkeypatch.setattr(_lib, "load", lambda: fake)

    def check(rc, what=""):
        if rc != 0:
            raise RuntimeError("%s failed (%d)" % (what, rc))
    monkeypatch.setattr(_lib, "check", check)
    monkeypatch.setattr(bk, "require_cuda", lambda: None)
    monkeypatch.setattr(bk, "device", lambda: cpu)
    monkeypatch.setattr(bk, "_stream", lambda: None)
    monkeypatch.setattr(bk, "_device_key", lambda: "cpu-emulator")

    def asdev(x):
        if isinstance(x, (bk.GeneratedOperand, bk.LinearOperator)):
            return x
        if isinstance(x, torch.Tensor):
            return x.to(torch.float64)
        a = np.asarray(x, dtype=np.float64)
        return torch.from_numpy(np.ascontiguousarray(a))
    monkeypatch.setattr(bk, "asdev", asdev)
    bk._scratch.pop("cpu-emulator", None)
    return fake
