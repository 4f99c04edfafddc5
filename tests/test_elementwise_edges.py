"""Edges of the elementwise, reduction and matrix-vector kernels (csrc/cc_elementwise.cu).

Every entry point there picks one of several kernels by a size or stride test, and most kernels
walk their data with a grid-stride loop whose grid is capped.  Each case below sits on both sides
of those switches and past those caps.  The dispatch thresholds are read from the CUDA source, so
each case knows which kernel it must reach; on the device the profiler must see exactly that
kernel, and a guard checks that the cases name every kernel of the file.

The operands are small integers or dyadic rationals and the coefficients powers of two, so every
product and partial sum is exact in any order: results are compared bit for bit with numpy, and a
dropped, doubled or misplaced term moves an element by at least one unit.  Divisions are compared
bit for bit with the same operations in the same order.  Each kernel also gets one random-valued
case with an explicit bound of the form c n eps sum|term|.  Outputs that must not be read are
filled with NaN first; strided outputs sit inside a tensor of sentinels that must stay untouched.

Each case is a function of ``abi``: the CPU tests pass the numpy emulation of the C ABI
(tests/abi_emulator.py), the ``gpu`` tests pass None and run the same body on the kernels."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pymes_b200", "csrc")


def _read(name):
    with open(os.path.join(CSRC, name)) as fh:
        return fh.read()


SRC, COMMON = _read("cc_elementwise.cu"), _read("common.cuh")


def _const(text, pattern):
    """The integer (or product of integers) that ``pattern`` captures in ``text``."""
    m = re.search(pattern, text)
    assert m, "not found in the CUDA source: %s" % pattern
    return math.prod(int(f) for f in m.group(1).split("*"))


SM = _const(COMMON, r"constexpr int kSmCount = (\d+);")
REDUCE_CTAS = SM * _const(COMMON, r"constexpr int kReduceBlocks = (\d+) \* kSmCount;")
REDUCE_THREADS = _const(COMMON, r"constexpr int kReduceThreads = (\d+);")
ROW_MAX = _const(SRC, r"constexpr int kRowMax = (\d+);")                       # tilde: o^2 <= kRowMax
PAIR_BYTES = _const(SRC, r"if \(2 \* sizeof\(double\) \* no \* no <= ([\d *]+)\)")   # sym_baji row pair
T_EXT3 = _const(SRC, r"in_str\[3\] != 1 && ext\[3\] >= (\d+)\)")               # axpby4 transpose rule
T_EXTD = _const(SRC, r"in_str\[d\] == 1 && ext\[d\] >= (\d+)\)")
BDOT_WARP_R = _const(SRC, r"if \(k\.R >= (\d+)\)")
GEMV_KFAST_N0 = _const(SRC, r"bk0 < bx0 && k\.k_ext\[0\] >= (\d+)\)")
EW_COPY = _const(SRC, r"constexpr int kEwCopy = (\d+);")
EW_UNROLL = _const(SRC, r"constexpr int kEwUnroll = (\d+);")

# elements (or rows, tiles, outputs) one pass of each capped grid covers
COPY_PASS = 16 * SM * 256 * EW_COPY            # axpby4_kernel
MP2_PASS = 16 * SM * 256 * EW_UNROLL            # mp2_kernel
THREAD_PASS = 16 * SM * 256                     # lincomb, tilde, sym_baji, bdot_thread, cdiv
UPDATE_PASS = REDUCE_CTAS * REDUCE_THREADS * EW_UNROLL
REDUCE_PASS = REDUCE_CTAS * REDUCE_THREADS      # dots, energy_kernel
SINGLES_PASS = SM * 256
PAIR_PASS = 16 * SM                             # row pairs of tilde_pair / sym_baji_pair
TRANSPOSE_TILES = 32 * SM
BDOT_WARPS = 32 * SM * 8

HELPERS = {"finish_reduce_kernel", "scale3_kernel"}      # second stage of every reduction
KERNELS = set(re.findall(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s+)?(\w+)\s*\(", SRC)) - HELPERS
SENT = -12345.625
EPS = np.finfo(np.float64).eps


# --------------------------------------------------------------------------
# the dispatch conditions of the C entry points, restated
# --------------------------------------------------------------------------
def _axpby4_kernel(ext, si, so):
    dt = -1
    if so[3] == 1 and si[3] != 1 and ext[3] >= T_EXT3:
        for d in range(3):
            if si[d] == 1 and ext[d] >= T_EXTD:
                dt = d
    return "axpby4_transpose_kernel" if dt >= 0 else "axpby4_kernel"


def _tilde_kernel(no):
    return "tilde_pair_kernel" if no * no <= ROW_MAX else "tilde_kernel"


def _sym_baji_kernel(no):
    return "sym_baji_pair_kernel" if 16 * no * no <= PAIR_BYTES else "sym_baji_kernel"


def _energy_kernel(no, nv, v_str, mp2_form):
    if not mp2_form and tuple(v_str) == (no, 1, nv * no * no, no * no):
        return "energy_rows_kernel"
    return "energy_kernel" if mp2_form else "energy_tiled_kernel"


def _dots_kernels(nvec):
    return ["dots_kernel<%d>" % min(4, nvec - k) for k in range(0, nvec, 4)]


def _bdot_kernel(R):
    return "bdot_warp_kernel" if R >= BDOT_WARP_R else "bdot_thread_kernel"


def _gemv_kernel(k_ext, b_kstr, b_xstr):
    bk0 = abs(b_kstr[0])
    bx0 = abs(b_xstr[0]) if b_xstr else 1 << 62
    return "gemv_kfast_kernel" if bk0 < bx0 and k_ext[0] >= GEMV_KFAST_N0 else "gemv_xfast_kernel"


# --------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------
_NAMED = []         # the kernels the running case expected, in order


def _launch(abi, want, fn):
    """Run ``fn`` (one entry point).  On the device the profiler must record exactly the kernels
    ``want`` of this file (the reduction helpers aside)."""
    want = [want] if isinstance(want, str) else list(want)
    _NAMED.extend(want)
    if abi is not None:
        return fn()
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    got = []
    for e in prof.events():
        m = re.search(r"pmb::(\w+(?:<\d+>)?)\(", e.name)
        if m and m.group(1) not in HELPERS:
            got.append(m.group(1))
    assert sorted(got) == sorted(want), (got, want)
    return res


def _bk():
    from pymes_b200 import backend as bk
    return bk


def _lib():
    from pymes_b200 import _lib
    return _lib


def _n(x):
    return np.array(x.detach().cpu().numpy(), order="C")


def _dev(a):
    return torch.from_numpy(np.array(a, dtype=np.float64, order="C")).to(_bk().device())   # a copy


def _ints(rng, shape, hi=7):
    return rng.integers(-hi, hi + 1, shape).astype(np.float64)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    assert np.array_equal(_bits(got), _bits(want)), "%d elements differ" % np.count_nonzero(_bits(got) != _bits(want))


def _layout(a, order):
    """A device view of ``a`` whose memory order is ``order`` (logical axes, slowest first)."""
    base = _dev(np.ascontiguousarray(np.transpose(a, order)))
    return base.permute(*np.argsort(order).tolist())


def _sum_check(got, terms, c=2.0):
    """|got - sum(terms)| <= c n eps sum|terms|, the sum taken in long double."""
    t = np.asarray(terms, dtype=np.longdouble).reshape(-1)
    ref = float(t.sum())
    tol = c * max(t.size, 1) * EPS * float(np.abs(t).sum())
    assert abs(got - ref) <= tol, (got, ref, tol)


def _axpb(alpha, x, beta, old):
    """alpha x + beta old as the kernels form it: for beta = 0 they store alpha x unchanged (a
    -0.0 product stays -0.0) and never read the output."""
    return alpha * x if beta == 0.0 else alpha * x + beta * old


def _pow2(rng, shape, lo=-2, hi=2):
    return np.ldexp(1.0, rng.integers(lo, hi + 1, shape)) * rng.choice([-1.0, 1.0], shape)


def _padded(shape, pads, fill_inner):
    """(big, view, keep): a tensor of sentinels with ``pads[d] = (before, after)`` around ``shape``,
    the inner view filled with ``fill_inner``, and the mask of the sentinel positions."""
    big_shape = [n + a + b for n, (a, b) in zip(shape, pads)]
    host = np.full(big_shape, SENT)
    inner = tuple(slice(a, a + n) for n, (a, _b) in zip(shape, pads))
    host[inner] = fill_inner
    big = _dev(host)
    keep = np.ones(big_shape, dtype=bool)
    keep[inner] = False
    return big, big[inner], keep


def _strides(ext, order, pad=0):
    """Element strides of ``ext`` stored in ``order`` (dims slowest first), each row padded by ``pad``."""
    st, acc = [0] * len(ext), 1
    for k, d in enumerate(reversed(order)):
        st[d] = acc
        acc *= ext[d] + (pad if k == 0 else 0)
    return st


def _span(ext, st, off=0):
    return off + 1 + sum((e - 1) * abs(s) for e, s in zip(ext, st))


def _np_view(flat, off, ext, st):
    return np.lib.stride_tricks.as_strided(flat[off:], shape=tuple(ext), strides=tuple(8 * s for s in st))


# --------------------------------------------------------------------------
# pmb_axpby4
# --------------------------------------------------------------------------
def _axpby4(abi, rng, ext, si, so, alpha, beta, soff=0, ooff=0, real=False):
    """pmb_axpby4 through the C ABI on flat buffers: ``in`` at offset ``soff`` with strides ``si``,
    ``out`` at ``ooff`` with strides ``so``; every other element of ``out`` is a sentinel."""
    lib, bk = _lib(), _bk()
    x = rng.standard_normal(_span(ext, si, soff)) if real else _ints(rng, _span(ext, si, soff))
    old = np.full(_span(ext, so, ooff), SENT)
    ov = _np_view(old, ooff, ext, so)
    ov[...] = np.nan if beta == 0.0 else _ints(rng, ext)
    want = old.copy()
    wv = _np_view(want, ooff, ext, so)
    wv[...] = _axpb(alpha, _np_view(x, soff, ext, si), beta, ov)
    src, out = _dev(x), _dev(old)
    rc = _launch(abi, _axpby4_kernel(ext, si, so), lambda: lib.load().pmb_axpby4(
        lib.I64x4(*ext), alpha, C.c_void_p(src.data_ptr() + 8 * soff), lib.I64x4(*si), beta,
        C.c_void_p(out.data_ptr() + 8 * ooff), lib.I64x4(*so), bk._stream()))
    lib.check(rc, "pmb_axpby4")
    _same(_n(out), want)


def _case_axpby4_elements(abi):
    """The element-per-thread copy: 1-D copies of 1, 255, 1025 and more than one grid pass of
    elements over NaN (beta = 0); e2 e3 = 1 with a transposed source; beta = -0.5 into a padded
    view; random values; and stride-0 (broadcast) sources through add_broadcast."""
    bk = _bk()
    rng = np.random.default_rng(11)
    for n in (1, 255, 1025, COPY_PASS + 37):
        _axpby4(abi, rng, (1, 1, 1, n), (n, n, n, 1), (n, n, n, 1), -2.0, 0.0)
    _axpby4(abi, rng, (37, 29, 1, 1), (1, 37, 5, 7), (29, 1, 1, 1), 0.5, 0.0)
    ext = (6, 5, 9, 11)
    _axpby4(abi, rng, ext, _strides(ext, (0, 1, 2, 3)), [7 * 10 * 14, 10 * 14, 14, 1], 0.5, -0.5, ooff=213)
    _axpby4(abi, rng, ext, _strides(ext, (3, 1, 2, 0)), _strides(ext, (0, 1, 2, 3), pad=3), -1.0, 1.0, real=True)
    # add_broadcast: out[abij] += alpha src[ai] (element kernel) and src[jb] (transposed, stride-0 batch)
    for no, nv, sub, shape in ((5, 7, "ai", (7, 5)), (17, 19, "jb", (17, 19))):
        s = _ints(rng, shape)
        old = _ints(rng, (nv, nv, no, no))
        out = _dev(old)
        src = _dev(s)
        sstr = dict(zip(sub, src.stride()))
        si = [sstr.get(ch, 0) for ch in "abij"]
        _launch(abi, _axpby4_kernel(out.shape, si, out.stride()),
                lambda: bk.add_broadcast(0.5, src, sub, out, "abij"))
        pos = dict(zip("abij", np.indices(old.shape)))
        _same(_n(out), old + 0.5 * s[tuple(pos[ch] for ch in sub)])


def _case_axpby4_transpose(abi):
    """The tiled transpose: input unit-stride along dt in {0, 1, 2}, output along 3, extents 15
    (must take the element kernel), 16, 31, 32, 33 and 65; beta in {0 over NaN, 1, -0.5}; padded
    outputs among sentinels; a stride-0 batch axis; more tiles than the capped grid."""
    rng = np.random.default_rng(12)
    pairs = ((15, 33), (33, 15), (16, 16), (31, 32), (32, 31), (33, 65), (65, 33), (16, 65))
    coefs = ((1.0, 0.0), (-2.0, 1.0), (0.5, -0.5))
    k = 0
    for dt in (0, 1, 2):
        others = [d for d in range(3) if d != dt]
        for et, e3 in pairs:
            ext = [0] * 4
            ext[dt], ext[3] = et, e3
            ext[others[0]], ext[others[1]] = 3, 2
            si = _strides(ext, others + [3, dt])
            if k % 4 == 3:
                si[others[1]] = 0                                   # a stride-0 batch axis
            pad = k % 2
            so = _strides(ext, [others[1], dt, others[0], 3], pad=2 * pad)
            alpha, beta = coefs[k % 3]
            _axpby4(abi, rng, ext, si, so, alpha, beta, soff=3 * pad, ooff=5 * pad)
            k += 1
    _axpby4(abi, rng, (40, 33, 17, 31), _strides((40, 33, 17, 31), (1, 2, 3, 0)), _strides((40, 33, 17, 31), (0, 1, 2, 3)),
            0.5, 1.0, real=True)
    ext = (32, 80, 80, 32)
    assert 80 * 80 > TRANSPOSE_TILES
    _axpby4(abi, rng, ext, _strides(ext, (1, 2, 3, 0)), _strides(ext, (0, 1, 2, 3)), -1.0, 0.0)


# --------------------------------------------------------------------------
# pmb_mp2_amplitudes, pmb_update_doubles, pmb_update_singles
# --------------------------------------------------------------------------
def _eps(rng, no, nv, real=False):
    if real:
        return -1.0 - rng.random(no), 1.0 + rng.random(nv)
    return -rng.integers(4, 33, no) / 8.0, rng.integers(4, 33, nv) / 8.0


def _den(ei, ea, a_lo, na, mode):
    """The kernels' denominator, in their order of operations."""
    i, j = ei[None, None, :, None], ei[None, None, None, :]
    a, b = ea[a_lo:a_lo + na, None, None, None], ea[None, :, None, None]
    return ((i * j) * -a) * -b if mode else ((i + j) - a) - b


def _case_mp2(abi):
    """T2 = V / (e_i + e_j - e_a - e_b + shift) bit for bit: V_abij a permuted, narrowed view of one
    V_pqrs, row blocks, random values, and more elements than one grid pass."""
    bk = _bk()
    rng = np.random.default_rng(13)
    for no, nv, a_lo, na, shift, real, big in ((5, 9, 2, 4, 0.375, False, False), (5, 9, 0, 9, -0.25, True, False),
                                               (1, 1, 0, 1, 0.0, False, False), (20, 91, 13, 70, 0.125, True, True)):
        ei, ea = _eps(rng, no, nv, real)
        if big:
            assert na * nv * no * no > MP2_PASS
            V = rng.standard_normal((no, no, nv, nv))
            Vab = _dev(V).permute(2, 3, 0, 1)[a_lo:a_lo + na]                # V_abij[a,b,i,j] = V[i,j,a,b]
            v = V.transpose(2, 3, 0, 1)[a_lo:a_lo + na]
        else:
            n = no + nv
            P = rng.standard_normal((n,) * 4) if real else _ints(rng, (n,) * 4)
            Vab = _dev(P).permute(2, 3, 0, 1)[no + a_lo:no + a_lo + na, no:, :no, :no]
            v = P.transpose(2, 3, 0, 1)[no + a_lo:no + a_lo + na, no:, :no, :no]
        T2 = _launch(abi, "mp2_kernel",
                     lambda: bk.mp2_amplitudes(_dev(ei), _dev(ea), shift, Vab, rows=(a_lo, na)))
        _same(_n(T2), v / (_den(ei, ea, a_lo, na, 0) + shift))


def _update(abi, ei, ea, shift, delta, mode, R, T, a_lo):
    bk = _bk()
    na = R.shape[0]
    Td, scal = _dev(T), _dev(np.full(2, np.nan))
    dT = _launch(abi, "update_doubles_kernel", lambda: bk.update_doubles(
        _dev(ei), _dev(ea), shift, delta, _dev(R), Td, scal, rows=(a_lo, na), product_denominator=bool(mode)))
    return _n(dT), _n(Td), float(_n(scal)[0])


def _fma_den(ei, ea, a_lo, na, shift):
    """The product denominator with its last multiply and the shift fused (one rounding)."""
    from fractions import Fraction
    i, j = ei[None, None, :, None], ei[None, None, None, :]
    p3 = (i * j) * -ea[a_lo:a_lo + na, None, None, None]
    b = np.broadcast_to(-ea[None, :, None, None], p3.shape[:1] + (len(ea),) + p3.shape[2:])
    p3 = np.broadcast_to(p3, b.shape)
    return np.vectorize(lambda x, y: float(Fraction(x) * Fraction(y) + Fraction(shift)))(p3, b)


def _case_update_doubles(abi):
    """dT = R (1/(D + shift)), T2 += delta dT, scal[0] = sum dT^2 for both denominators, shifts 0
    and != 0, row blocks, n < 256 and more than one grid pass; bit for bit where the operations
    are exact, scal[0] exact where every dT^2 is."""
    rng = np.random.default_rng(14)
    shapes = ((6, 11, 3, 5), (2, 4, 1, 2), (1, 1, 0, 1), (32, 41, 5, 30))
    assert 30 * 41 * 32 * 32 > UPDATE_PASS and 2 * 4 * 2 * 2 < 256
    for k, (no, nv, a_lo, na) in enumerate(shapes):
        # the sum denominator, random R and T: dT and T2 bit for bit, scal[0] within the bound
        ei, ea = _eps(rng, no, nv)
        shift, delta = (0.0, 0.25)[k % 2], (0.5, -2.0)[k % 2]
        R, T = rng.standard_normal((2, na, nv, no, no))
        dT, T2, s = _update(abi, ei, ea, shift, delta, 0, R, T, a_lo)
        d = R * (1.0 / (_den(ei, ea, a_lo, na, 0) + shift))
        _same(dT, d)
        _same(T2, T + delta * d)
        _sum_check(s, d * d)
    # the sum denominator, R non-zero only where D + shift is a power of two: scal[0] exact
    no, nv, a_lo, na = 6, 11, 3, 5
    ei, ea = _eps(rng, no, nv)
    D = _den(ei, ea, a_lo, na, 0) + 0.125
    m, _e = np.frexp(np.abs(D))
    R = np.where(m == 0.5, _ints(rng, D.shape), 0.0)
    assert np.count_nonzero(R) > 20
    T = _ints(rng, R.shape)
    dT, T2, s = _update(abi, ei, ea, 0.125, -0.5, 0, R, T, a_lo)
    d = R * (1.0 / D)
    _same(dT, d)
    _same(T2, T - 0.5 * d)
    assert s == math.fsum((d * d).reshape(-1))
    # the product denominator on powers of two: every operation exact, scal[0] too
    for no, nv, a_lo, na in ((6, 11, 3, 5), (2, 3, 0, 3)):
        ei, ea = -np.abs(_pow2(rng, no, -1, 1)), np.abs(_pow2(rng, nv, -1, 1))
        R, T = _ints(rng, (na, nv, no, no)), _ints(rng, (na, nv, no, no))
        dT, T2, s = _update(abi, ei, ea, 0.0, 2.0, 1, R, T, a_lo)
        d = R * (1.0 / _den(ei, ea, a_lo, na, 1))
        _same(dT, d)
        _same(T2, T + 2.0 * d)
        assert s == math.fsum((d * d).reshape(-1))
    # the product denominator on random values with a shift: the kernel may fuse the last multiply
    # with the shift, so each element equals the separate or the fused form
    no, nv, a_lo, na = 4, 7, 2, 3
    ei, ea = _eps(rng, no, nv, real=True)
    R, T = rng.standard_normal((2, na, nv, no, no))
    dT, T2, s = _update(abi, ei, ea, 0.3, 0.5, 1, R, T, a_lo)
    plain = R * (1.0 / (_den(ei, ea, a_lo, na, 1) + 0.3))
    fused = R * (1.0 / _fma_den(ei, ea, a_lo, na, 0.3))
    ok = (_bits(dT) == _bits(plain)) | (_bits(dT) == _bits(fused))
    assert ok.all(), np.count_nonzero(~ok)
    _same(T2, T + 0.5 * dT)
    _sum_check(s, plain * plain)


def _case_update_singles(abi):
    """dT1 = R1 (1/(e_i - e_a + shift)), T1 += delta dT1 bit for bit, past one grid pass."""
    bk = _bk()
    rng = np.random.default_rng(15)
    assert 130 * 300 > SINGLES_PASS
    for no, nv, shift, real in ((1, 1, 0.0, False), (3, 7, 0.5, True), (130, 300, -0.25, True)):
        ei, ea = _eps(rng, no, nv, real)
        R1, T1 = (rng.standard_normal((2, nv, no)) if real else _ints(rng, (2, nv, no)))
        T1d = _dev(T1)
        dT1 = _launch(abi, "update_singles_kernel",
                      lambda: bk.update_singles(_dev(ei), _dev(ea), shift, 0.5, _dev(R1), T1d))
        d = R1 * (1.0 / ((ei[None, :] - ea[:, None]) + shift))
        _same(_n(dT1), d)
        _same(_n(T1d), T1 + 0.5 * d)


# --------------------------------------------------------------------------
# pmb_energy_doubles
# --------------------------------------------------------------------------
def _energy(abi, rng, no, nv, a_lo, na, form, with_t1, real=False):
    """scal[0:3] of one call against numpy: exact for integers, within the bound for random values."""
    bk = _bk()
    draw = (lambda s, hi=7: rng.standard_normal(s)) if real else (lambda s, hi=7: _ints(rng, s, hi))
    T = draw((na, nv, no, no))
    T1 = draw((nv, no), 3) if with_t1 else None
    V = draw((no, no, nv, nv))
    Vd = _layout(V, (2, 3, 0, 1)) if form == "rows" else _dev(V)
    mp2 = form == "mp2"
    name = _energy_kernel(no, nv, Vd.stride(), mp2)
    if not (no == 1 and nv == 1):
        assert name == {"rows": "energy_rows_kernel", "tiled": "energy_tiled_kernel", "mp2": "energy_kernel"}[form]
    scal = _dev(np.full(4, np.nan))
    _launch(abi, name, lambda: bk.energy_doubles(_dev(T), Vd, scal, T1=_dev(T1) if with_t1 else None,
                                                  mp2_form=mp2, rows=(a_lo, na)))
    got = _n(scal)
    tau = T + (np.einsum("ai,bj->abij", T1[a_lo:a_lo + na], T1) if with_t1 else 0.0)
    vd = V.transpose(2, 3, 0, 1)[a_lo:a_lo + na]                                   # V[i,j,a,b] as [a,b,i,j]
    vx = V.transpose(2, 3, 1, 0)[a_lo:a_lo + na] if mp2 else V.transpose(3, 2, 0, 1)[a_lo:a_lo + na]
    if real:
        _sum_check(got[0], 2.0 * tau * vd)
        _sum_check(got[1], -tau * vx)
        _sum_check(got[2], T * T)
    else:
        ti, vdi, vxi = tau.astype(np.int64), vd.astype(np.int64), vx.astype(np.int64)
        # the kernels scale the finished sums by 2 and -1 (an exchange sum of 0 becomes -0.0)
        _same(got[:3], [2.0 * float(np.sum(ti * vdi)), -1.0 * float(np.sum(ti * vxi)),
                        float(np.sum(T.astype(np.int64) ** 2))])
    assert np.isnan(got[3])


def _case_energy(abi):
    """Each of the rows / tiled / mp2_form kernels with T1 NULL and set, whole tensors and row
    blocks, o in {1, 5, 6} and v in {1, 31, 33} (ragged 32-wide tiles), one case past every
    grid cap, and random values."""
    rng = np.random.default_rng(16)
    shapes = ((1, 1, 0, 1), (5, 31, 0, 31), (6, 33, 4, 20), (1, 33, 32, 1), (6, 1, 0, 1), (5, 33, 1, 31))
    big = (6, 180, 0, 180)
    assert 180 * 180 * 36 > REDUCE_PASS and 180 * 180 > REDUCE_CTAS * REDUCE_THREADS // 32
    assert 180 * 6 * 2 > REDUCE_CTAS
    for form in ("rows", "tiled", "mp2"):
        for k, (no, nv, a_lo, na) in enumerate(shapes + (big,)):
            _energy(abi, rng, no, nv, a_lo, na, form, with_t1=bool(k % 2))
        _energy(abi, rng, 6, 33, 3, 17, form, with_t1=True, real=True)


# --------------------------------------------------------------------------
# pmb_tilde, pmb_sym_baji
# --------------------------------------------------------------------------
def _case_tilde(abi):
    """Tt = 2 T - T with (a,b) or (i,j) swapped, bit for bit, on both sides of kRowMax, v in
    {1, 2, 3}, one pass past the element grid, 4.5M row pairs (o = 1, v = 3000), and T2 == Tt."""
    bk, lib = _bk(), _lib()
    rng = np.random.default_rng(17)
    assert 63 * 63 <= ROW_MAX < 65 * 65 and 13 * 13 * 65 * 65 > THREAD_PASS
    cases = [(no, nv, sw) for no in (1, 63, 64, 65) for nv in (1, 2, 3) for sw in (0, 1)]
    cases += [(65, 13, 0), (65, 13, 1), (1, 3000, 0)]
    for no, nv, sw in cases:
        T = _ints(rng, (nv, nv, no, no))
        Tt = _launch(abi, _tilde_kernel(no), lambda: bk.tilde(_dev(T), swap_ij=bool(sw)))
        _same(_n(Tt), 2.0 * T - T.transpose((0, 1, 3, 2) if sw else (1, 0, 2, 3)))
    assert 3000 * 3001 // 2 > 1000 * PAIR_PASS
    T = _dev(_ints(rng, (2, 2, 3, 3)))
    assert lib.load().pmb_tilde(3, 2, bk._ptr(T), bk._ptr(T), 0, bk._stream()) == -1      # PMB_E_BADARG


def _case_sym_baji(abi):
    """R (+)= Ex + Ex^{baji} bit for bit at o = 55 (row pair in shared memory) and 56 (element
    kernel), accumulate 0 (over NaN) and 1, one pass past the element grid, 4.5M row pairs,
    and Ex == R."""
    bk, lib = _bk(), _lib()
    rng = np.random.default_rng(18)
    assert 16 * 55 * 55 <= PAIR_BYTES < 16 * 56 * 56 and 14 * 14 * 56 * 56 > THREAD_PASS
    cases = [(no, nv, acc) for no in (55, 56) for nv in (1, 3) for acc in (0, 1)] + [(56, 14, 1), (1, 3000, 1)]
    for no, nv, acc in cases:
        Ex = _ints(rng, (nv, nv, no, no))
        old = _ints(rng, Ex.shape) if acc else np.full(Ex.shape, np.nan)
        R = _dev(old)
        _launch(abi, _sym_baji_kernel(no), lambda: bk.sym_baji(_dev(Ex), R, accumulate=bool(acc)))
        v = Ex + Ex.transpose(1, 0, 3, 2)
        _same(_n(R), old + v if acc else v)
    E = _dev(_ints(rng, (2, 2, 3, 3)))
    assert lib.load().pmb_sym_baji(3, 2, bk._ptr(E), bk._ptr(E), 1, bk._stream()) == -1


# --------------------------------------------------------------------------
# pmb_dots, pmb_lincomb
# --------------------------------------------------------------------------
def _case_dots_lincomb(abi):
    """dots for 1..16 vectors (chunks of 4, 3, 2 and 1 per pass over Y), n in {1, 256, more
    than one reduction pass}, exact; random values within the bound; lincomb with power-of-two
    coefficients, beta = 0 over NaN; nvec = 17 and n = 0 are refused."""
    bk, lib = _bk(), _lib()
    rng = np.random.default_rng(19)
    big = REDUCE_PASS + 1001
    assert big > THREAD_PASS // 2
    for nvec, n in [(k, 256) for k in range(1, 17)] + [(3, 1), (7, big)]:
        X, y = _ints(rng, (nvec, n)), _ints(rng, n)
        xs = [_dev(x) for x in X]
        out = _dev(np.full(nvec, np.nan))
        _launch(abi, _dots_kernels(nvec), lambda: bk.dots(xs, _dev(y), out=out))
        _same(_n(out), (X.astype(np.int64) @ y.astype(np.int64)).astype(np.float64))
    X, y = rng.standard_normal((5, big)), rng.standard_normal(big)
    out = _launch(abi, _dots_kernels(5), lambda: bk.dots([_dev(x) for x in X], _dev(y)))
    for k in range(5):
        _sum_check(float(_n(out)[k]), X[k] * y)
    for nvec, n, beta in ((1, 256, 0.0), (2, 1, 0.5), (3, 256, 0.0), (5, 256, -1.0), (16, 256, 0.0),
                          (3, THREAD_PASS + 77, 0.0), (4, THREAD_PASS + 77, -0.5)):
        X, c = _ints(rng, (nvec, n)), _pow2(rng, nvec)
        old = _ints(rng, n) if beta != 0.0 else np.full(n, np.nan)
        out = _dev(old)
        _launch(abi, "lincomb_kernel", lambda: bk.lincomb(c, [_dev(x) for x in X], out=out, beta=beta))
        want = beta * old if beta != 0.0 else np.zeros(n)       # the kernel's order: one term at a time
        for k in range(nvec):
            want = want + c[k] * X[k]
        _same(_n(out), want)
    x = _dev(np.ones(4))
    ptrs = _bk()._ptr_array([x] * 17)
    res = _dev(np.zeros(17))
    ws = bk.scratch().reduce_ws()
    L = lib.load()
    assert L.pmb_dots(17, ptrs, bk._ptr(x), 4, bk._ptr(res), bk._ptr(ws), ws.numel() * 8, bk._stream()) == -1
    assert L.pmb_dots(1, ptrs, bk._ptr(x), 0, bk._ptr(res), bk._ptr(ws), ws.numel() * 8, bk._stream()) == -1
    c = (C.c_double * 17)(*([1.0] * 17))
    assert L.pmb_lincomb(17, c, ptrs, 4, 0.0, bk._ptr(res), bk._stream()) == -1
    assert L.pmb_lincomb(1, c, ptrs, 0, 0.0, bk._ptr(res), bk._stream()) == -1


# --------------------------------------------------------------------------
# pmb_bdot, pmb_gemv through the C ABI
# --------------------------------------------------------------------------
def _fill(arr, vals):
    for k, v in enumerate(vals):
        arr[k] = int(v)


def _out_buffer(rng, shape, beta, pad):
    """(tensor, view, old, keep): the output view (inside sentinels when ``pad``), NaN for beta = 0."""
    old = _ints(rng, shape) if beta != 0.0 else np.full(shape, np.nan)
    if pad:
        big, view, keep = _padded(shape, [(1, 2)] * len(shape), old)
        return big, view, old, keep
    t = _dev(old)
    return t, t, old, None


def _check_out(big, view, keep, want):
    _same(_n(view), want)
    if keep is not None:
        _same(_n(big)[keep], np.full(keep.sum(), SENT))


def _bdot(abi, rng, i_shape, r_shape, a_order, b_order, alpha=1.0, beta=0.0, pad=False):
    bk, lib = _bk(), _lib()
    ni, nr = len(i_shape), len(r_shape)
    A, B = _ints(rng, i_shape + r_shape), _ints(rng, i_shape + r_shape)
    Ad, Bd = _layout(A, a_order), _layout(B, b_order)
    big, view, old, keep = _out_buffer(rng, i_shape, beta, pad)
    d = lib.Bdot()
    d.A, d.B, d.out = Ad.data_ptr(), Bd.data_ptr(), view.data_ptr()
    d.ni, d.nr, d.alpha, d.beta = ni, nr, alpha, beta
    _fill(d.i_ext, i_shape)
    _fill(d.o_istr, view.stride())
    _fill(d.a_istr, Ad.stride()[:ni])
    _fill(d.b_istr, Bd.stride()[:ni])
    _fill(d.r_ext, r_shape)
    _fill(d.a_rstr, Ad.stride()[ni:])
    _fill(d.b_rstr, Bd.stride()[ni:])
    rc = _launch(abi, _bdot_kernel(math.prod(r_shape)), lambda: lib.load().pmb_bdot(C.byref(d), bk._stream()))
    lib.check(rc, "pmb_bdot")
    acc = (A.astype(np.int64) * B.astype(np.int64)).sum(axis=tuple(range(ni, ni + nr)))
    _check_out(big, view, keep, _axpb(alpha, acc.astype(np.float64), beta, old))


def _case_bdot(abi):
    """out[I] = beta out + alpha sum_R A B on both sides of the thread / warp switch (R = 63, 64,
    one or two summed axes), ni = 0 (a scalar), nr = 0 (an elementwise product), strided outputs
    among sentinels, and more outputs than the warp grid covers."""
    rng = np.random.default_rng(20)
    assert BDOT_WARP_R == 64
    _bdot(abi, rng, (5, 7), (63,), (1, 2, 0), (2, 0, 1), 1.0, 0.0)
    _bdot(abi, rng, (5, 7), (64,), (1, 2, 0), (2, 0, 1), 2.0, 1.0, pad=True)
    _bdot(abi, rng, (5, 7), (3, 21), (0, 1, 2, 3), (3, 2, 1, 0), -0.5, 0.0, pad=True)
    _bdot(abi, rng, (5, 7), (8, 8), (2, 3, 0, 1), (0, 1, 2, 3), 1.0, -0.5)
    _bdot(abi, rng, (), (64,), (0,), (0,), 1.0, 0.0)
    _bdot(abi, rng, (), (10,), (0,), (0,), 0.5, 1.0)
    _bdot(abi, rng, (6, 9), (), (1, 0), (0, 1), 1.0, 0.0, pad=True)
    assert 40000 > BDOT_WARPS
    _bdot(abi, rng, (40000,), (64,), (0, 1), (1, 0), 1.0, 0.0)


def _gemv(abi, rng, k_shape, x_shape, b_order, v_order, alpha=1.0, beta=0.0, pad=False, hankel=False):
    """out[X] = beta out + alpha sum_K vec[K] B[K,X]; ``hankel``: B[k,x] = b[k + x] (one K and one
    X axis with equal strides)."""
    bk, lib = _bk(), _lib()
    nk = len(k_shape)
    vec = _ints(rng, k_shape)
    if hankel:
        flat = _ints(rng, k_shape[0] + x_shape[0] - 1)
        B = flat[np.add.outer(np.arange(k_shape[0]), np.arange(x_shape[0]))]
        Bd = torch.as_strided(_dev(flat), (k_shape[0], x_shape[0]), (1, 1))
    else:
        B = _ints(rng, k_shape + x_shape)
        Bd = _layout(B, b_order)
    vd = _layout(vec, v_order)
    big, view, old, keep = _out_buffer(rng, x_shape, beta, pad)
    d = lib.Gemv()
    d.vec, d.B, d.out = vd.data_ptr(), Bd.data_ptr(), view.data_ptr()
    d.nk, d.nx, d.alpha, d.beta = nk, len(x_shape), alpha, beta
    _fill(d.k_ext, k_shape)
    _fill(d.v_kstr, vd.stride())
    _fill(d.b_kstr, Bd.stride()[:nk])
    _fill(d.x_ext, x_shape)
    _fill(d.b_xstr, Bd.stride()[nk:])
    _fill(d.o_xstr, view.stride())
    name = _gemv_kernel(k_shape, Bd.stride()[:nk], Bd.stride()[nk:])
    rc = _launch(abi, name, lambda: lib.load().pmb_gemv(C.byref(d), bk._stream()))
    lib.check(rc, "pmb_gemv")
    acc = np.tensordot(vec.astype(np.int64), B.astype(np.int64), axes=nk)
    _check_out(big, view, keep, _axpb(alpha, acc.astype(np.float64), beta, old))
    return name


def _case_gemv(abi):
    """Both sides of the k-fast switch (k_ext[0] = 15, 16), a stride tie between the first K and
    X axes, nx = 0, K with k1..k3 > 1, and k-fast first extents 127, 129 and 200 (the loop of 128
    and its 32-wide tail); beta in {0 over NaN, 1, -0.5}, outputs among sentinels."""
    rng = np.random.default_rng(21)
    assert GEMV_KFAST_N0 == 16
    names = [
        _gemv(abi, rng, (15,), (40,), (1, 0), (0,), 1.0, 0.0),
        _gemv(abi, rng, (16,), (40,), (1, 0), (0,), 2.0, 1.0, pad=True),
        _gemv(abi, rng, (16,), (40,), (0, 1), (0,), 1.0, -0.5),
        _gemv(abi, rng, (20,), (30,), None, (0,), 1.0, 0.0, hankel=True),
        _gemv(abi, rng, (200,), (), (0,), (0,), 1.0, 0.0),
        _gemv(abi, rng, (10,), (), (0,), (0,), -1.0, 1.0),
        _gemv(abi, rng, (20, 3, 2, 2), (7, 5), (5, 4, 3, 2, 1, 0), (3, 2, 1, 0), 0.5, 0.0, pad=True),
        _gemv(abi, rng, (20, 3, 2, 2), (7, 5), (3, 2, 1, 0, 5, 4), (0, 1, 2, 3), 1.0, 1.0),
    ]
    for n0 in (127, 129, 200):
        names.append(_gemv(abi, rng, (n0, 2), (9,), (1, 2, 0), (1, 0), 1.0, 0.0 if n0 != 129 else -0.5))
    assert names[:6] == ["gemv_xfast_kernel", "gemv_kfast_kernel", "gemv_xfast_kernel", "gemv_xfast_kernel",
                         "gemv_kfast_kernel", "gemv_xfast_kernel"]
    assert names[6:] == ["gemv_kfast_kernel", "gemv_xfast_kernel"] + ["gemv_kfast_kernel"] * 3


# --------------------------------------------------------------------------
# pmb_cdiv_shifted
# --------------------------------------------------------------------------
def _case_cdiv(abi):
    """(yr + i yi) = (xr + i xi) / (z - diag + shift) written over its input (yr, yi alias xr, xi):
    within a few ulps of the kernel's formula and of numpy's complex division."""
    bk, lib = _bk(), _lib()
    rng = np.random.default_rng(22)
    zr, zi, shift = 0.3, 0.7, -0.1
    for n in (1, 1000, THREAD_PASS + 5):
        diag, xr, xi = rng.standard_normal((3, n))
        dd, yr, yi = _dev(diag), _dev(xr), _dev(xi)
        rc = _launch(abi, "cdiv_shifted_kernel", lambda: lib.load().pmb_cdiv_shifted(
            n, bk._ptr(dd), zr, zi, shift, bk._ptr(yr), bk._ptr(yi), bk._ptr(yr), bk._ptr(yi), bk._stream()))
        lib.check(rc, "pmb_cdiv_shifted")
        gr, gi = _n(yr), _n(yi)
        dr = (zr - diag) + shift
        inv = 1.0 / (dr * dr + zi * zi)
        mr, mi = dr * inv, -zi * inv
        scale = np.abs(inv) * np.hypot(dr, zi)                                   # 1 / |z - diag + shift|
        tol = 4 * EPS * scale * (np.abs(xr) + np.abs(xi))
        assert np.all(np.abs(gr - (mr * xr - mi * xi)) <= tol)
        assert np.all(np.abs(gi - (mr * xi + mi * xr)) <= tol)
        y = (xr + 1j * xi) / (complex(zr, zi) - diag + shift)
        tol = 8 * EPS * scale * np.hypot(xr, xi)
        assert np.all(np.abs(gr - y.real) <= tol) and np.all(np.abs(gi - y.imag) <= tol)


# --------------------------------------------------------------------------
# argument checks of the backend wrappers
# --------------------------------------------------------------------------
def _case_wrapper_argument_checks(abi):
    """tilde, sym_baji and energy_doubles index T2, Ex, R and T1 flat: a strided or mis-shaped
    argument raises ValueError before any launch."""
    bk = _bk()
    rng = np.random.default_rng(23)
    nv, no = 4, 3
    T = _dev(_ints(rng, (nv, nv, no, no)))
    V = _dev(_ints(rng, (no, no, nv, nv)))
    T1 = _dev(_ints(rng, (nv, no)))
    even = bk.empty_even_pitch(nv, nv, no)                 # o^2 = 9: rows padded to 10
    assert not even.is_contiguous()
    before = bk.launch_count()
    bad_t2 = [T.transpose(2, 3), T.permute(1, 0, 2, 3), even, _dev(np.zeros((nv, nv + 1, no, no))),
              _dev(np.zeros((nv, nv, no, no + 1)))]
    for t in bad_t2:
        with pytest.raises(ValueError):
            bk.tilde(t)
        with pytest.raises(ValueError):
            bk.sym_baji(t, _dev(np.zeros((nv, nv, no, no))))
        with pytest.raises(ValueError):
            bk.sym_baji(T, t)
        with pytest.raises(ValueError):
            bk.energy_doubles(t, V, bk.zeros(4))
    with pytest.raises(ValueError):
        bk.sym_baji(T, _dev(np.zeros((nv, nv, no, no))).transpose(2, 3), accumulate=False)
    with pytest.raises(ValueError):
        bk.energy_doubles(T, V, bk.zeros(4), rows=(1, 2))              # a row block must be [na,v,o,o]
    with pytest.raises(ValueError):
        bk.energy_doubles(T[:, 1:3], V, bk.zeros(4), rows=(1, 2))
    for t1 in (T1.t().contiguous(), _dev(np.zeros((nv + 1, no))), _dev(np.zeros((no, nv))).t(),
               _dev(np.zeros((nv, 2 * no)))[:, ::2]):
        with pytest.raises(ValueError):
            bk.energy_doubles(T, V, bk.zeros(4), T1=t1)
    assert bk.launch_count() == before
    # the same calls with well-formed arguments go through
    bk.tilde(T)
    bk.sym_baji(T, _dev(np.zeros((nv, nv, no, no))))
    bk.energy_doubles(T[1:3].contiguous(), V, bk.zeros(4), T1=T1, rows=(1, 2))
    assert bk.launch_count() > before


CASES = {
    _case_axpby4_elements: {"axpby4_kernel", "axpby4_transpose_kernel"},
    _case_axpby4_transpose: {"axpby4_kernel", "axpby4_transpose_kernel"},
    _case_mp2: {"mp2_kernel"},
    _case_update_doubles: {"update_doubles_kernel"},
    _case_update_singles: {"update_singles_kernel"},
    _case_energy: {"energy_rows_kernel", "energy_tiled_kernel", "energy_kernel"},
    _case_tilde: {"tilde_pair_kernel", "tilde_kernel"},
    _case_sym_baji: {"sym_baji_pair_kernel", "sym_baji_kernel"},
    _case_dots_lincomb: {"dots_kernel<4>", "dots_kernel<3>", "dots_kernel<2>", "dots_kernel<1>", "lincomb_kernel"},
    _case_bdot: {"bdot_thread_kernel", "bdot_warp_kernel"},
    _case_gemv: {"gemv_xfast_kernel", "gemv_kfast_kernel"},
    _case_cdiv: {"cdiv_shifted_kernel"},
    _case_wrapper_argument_checks: set(),
}
IDS = [f.__name__[len("_case_"):] for f in CASES]


def _run(case, abi):
    del _NAMED[:]
    case(abi)
    assert set(_NAMED) == CASES[case]


@pytest.fixture
def abi(cpu_abi):
    return cpu_abi


@pytest.mark.parametrize("case", list(CASES), ids=IDS)
def test_on_the_emulated_abi(abi, case):
    _run(case, abi)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES), ids=IDS)
def test_on_the_device(case):
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    _run(case, None)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_axpby4_64bit_index_on_the_device():
    """A 1-D copy of 2^31 + 5 distinct values: e2 e3 >= 2^31, so axpby4_kernel splits its index
    with 64-bit arithmetic.  Needs about 34 GB of device memory."""
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    from pymes_b200 import _lib, backend as bk
    n = (1 << 31) + 5
    x = torch.arange(n, dtype=torch.float64, device="cuda")
    out = torch.full_like(x, float("nan"))
    ext, st = _lib.I64x4(1, 1, 1, n), _lib.I64x4(n, n, n, 1)
    rc = _launch(None, _axpby4_kernel((1, 1, 1, n), (n, n, n, 1), (n, n, n, 1)), lambda: _lib.load().pmb_axpby4(
        ext, -1.0, bk._ptr(x), st, 0.0, bk._ptr(out), st, bk._stream()))
    _lib.check(rc, "pmb_axpby4")
    assert torch.equal(out.neg_(), x)
    del x, out
    torch.cuda.empty_cache()


# --------------------------------------------------------------------------
# guards
# --------------------------------------------------------------------------
def test_every_kernel_has_a_case():
    """Every __global__ kernel of cc_elementwise.cu (the reduction helpers aside) is the expected
    kernel of some case: a kernel added without a case fails here."""
    named = {re.sub(r"<\d+>$", "", k) for ks in CASES.values() for k in ks}
    assert named == KERNELS
    assert KERNELS >= {"sym_baji_kernel", "tilde_kernel", "axpby4_transpose_kernel", "energy_kernel"}


def test_dispatch_thresholds_parse():
    """The thresholds read from the CUDA source have the values the shapes above straddle."""
    assert (ROW_MAX, PAIR_BYTES, T_EXT3, T_EXTD, BDOT_WARP_R, GEMV_KFAST_N0) == (4096, 48 * 1024, 16, 16, 64, 16)
    assert (COPY_PASS, REDUCE_PASS, SINGLES_PASS, PAIR_PASS, TRANSPOSE_TILES) == (2424832, 303104, 37888, 2368, 4736)
