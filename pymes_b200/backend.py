"""Device backend: the replacement for the reference's ``einsum`` seam.

The reference funnels every tensor operation through
``einsum = partial(np.einsum, optimize=True)`` (pymes/solver/ccsd.py:11 and the
other solver modules).  Here the same role is played by :func:`contract`, which
parses a two-operand einsum string into M / N / K index groups and hands a
stride-only description of the operands to the DMMA kernel behind
``pmb_contract`` -- index permutations are never materialised.

PyTorch is used for device memory and streams only.  Every arithmetic kernel is
in ``libpymes_b200.so``; there is no CPU path.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib

F64 = torch.float64


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("pymes_b200 needs a CUDA device (built for sm_100a / B200); "
                           "there is no CPU fallback")


def device():
    require_cuda()
    return torch.device("cuda", torch.cuda.current_device())


class GeneratedOperand:
    """An operand of :func:`contract_terms` that is never stored: the kernel's producer warps
    evaluate its tiles (``pmb_term_t.a_gen``).  Subclasses describe one source -- today the
    momentum-conserving UEG integrals (``model.ueg.VirtualBlock``).  It quacks like a tensor
    as far as the host-side index classification needs (shape / dim / C-order strides)."""

    shape = ()

    def dim(self):
        return len(self.shape)

    def stride(self):
        st, acc = [], 1
        for n in reversed(self.shape):
            st.append(acc)
            acc *= int(n)
        return tuple(reversed(st))

    def data_ptr(self):
        return 0

    def numel(self):
        n = 1
        for e in self.shape:
            n *= int(e)
        return n

    def gen_descriptor(self, sub, m_ord, k_ord):
        """ctypes ``pmb_ueg_operand_t`` for this operand indexed by ``sub`` with the M / K index
        groups ordered (fastest first) as ``m_ord`` / ``k_ord``."""
        raise NotImplementedError

    def momentum(self):
        """The operand's :class:`Momentum` selection rule, or None."""
        return None

    def blocked_lists(self):
        """Block-diagonal structure of the operand as the matrix [(axis 0, axis 1), (axis 2, axis 3)]
        for ``pmb_blocked_contract`` (see :func:`_blocked_term`), or None when the source has none."""
        return None


class LinearOperator:
    """Marker for objects that stand in for a tensor but are only ever APPLIED (e.g. the
    T1-dressed V_abcd of ``solver.ccsd.DressedLadder``).  ``asdev`` passes them through."""


def asdev(x):
    """numpy array / torch tensor -> float64 CUDA tensor (views keep their strides)."""
    if isinstance(x, (GeneratedOperand, LinearOperator)):
        return x
    if isinstance(x, torch.Tensor):
        if x.dtype != F64:
            x = x.to(F64)
        return x if x.is_cuda else x.to(device())
    a = np.asarray(x, dtype=np.float64)
    if not a.flags.c_contiguous:
        a = np.ascontiguousarray(a)
    return torch.from_numpy(a).to(device())


def tonumpy(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def empty(*shape):
    return torch.empty(shape, dtype=F64, device=device())


def zeros(*shape, rule=None):
    """Zeros; ``rule``: a momentum rule (:class:`Momentum`) to tag them with -- zeros satisfy any."""
    t = torch.zeros(shape, dtype=F64, device=device())
    if rule is not None:
        _set_momentum(t, rule)
    return t


def empty_stacked(shape_a, shape_b):
    """Two tensors of equal size carved out of ONE allocation, back to back (see ``stacked_rows``)."""
    na = int(np.prod(shape_a))
    if na != int(np.prod(shape_b)):
        raise ValueError("stacked tensors must have the same number of elements")
    buf = torch.empty(2 * na, dtype=F64, device=device())
    return buf[:na].view(*shape_a), buf[na:].view(*shape_b)


def empty_even_pitch(n0, n1, no):
    """An [n0, n1, no, no] amplitude-shaped tensor whose (i,j) rows start on 16-byte boundaries: the
    o^2 doubles of a row are followed by one pad double when o^2 is odd (o = 27: pitch 730).  The
    contraction kernel copies such an operand 16 bytes at a time (`b_vec2`, cc_contract.cu); the
    pad is zero and is never part of a result."""
    oo = no * no
    pitch = oo + (oo & 1)
    buf = torch.empty((n0, n1, pitch), dtype=F64, device=device())
    if pitch != oo:
        buf[:, :, oo:].zero_()
    return buf[:, :, :oo].view(n0, n1, no, no)


def stacked_rows(A, B, k_shape):
    """If the contiguous tensors A and B lie back to back in one allocation (``empty_stacked``) and
    both end in the index pattern ``k_shape`` (the contracted indices of a common contraction),
    return the VIEW [2, rows, *k_shape] over both -- one operand, so that two contractions with the
    same right-hand operand become one launch with twice the rows (two few-wave grids side by side
    become one grid without a second tail wave).  Otherwise None."""
    if not (isinstance(A, torch.Tensor) and isinstance(B, torch.Tensor)):
        return None
    if not (A.is_contiguous() and B.is_contiguous()) or A.numel() != B.numel() or A.numel() == 0:
        return None
    k = int(np.prod(k_shape))
    if tuple(A.shape[-len(k_shape):]) != tuple(k_shape) or tuple(B.shape[-len(k_shape):]) != tuple(k_shape):
        return None
    if A.untyped_storage().data_ptr() != B.untyped_storage().data_ptr() or \
            B.data_ptr() != A.data_ptr() + 8 * A.numel():
        return None
    rows = A.numel() // k
    strides, acc = [], 1
    for e in reversed(k_shape):
        strides.append(acc)
        acc *= int(e)
    return torch.as_strided(A, (2, rows) + tuple(int(e) for e in k_shape), (A.numel(), k) + tuple(reversed(strides)),
                            A.storage_offset())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _device_key():
    """Scratch buffers are per (device, stream): launches on different streams may overlap."""
    return (torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr())


class _Scratch:
    """Per-device scratch handed to the library (it never allocates itself)."""

    def __init__(self):
        self.reduce = None
        self.splitk = None

    def reduce_ws(self):
        if self.reduce is None:
            n = _lib.load().pmb_reduce_workspace()
            self.reduce = torch.empty(n // 8, dtype=F64, device=device())
        return self.reduce

    def splitk_ws(self, nbytes):
        if self.splitk is None or self.splitk.numel() * 8 < nbytes:
            self.splitk = torch.empty((nbytes + 7) // 8, dtype=F64, device=device())
        return self.splitk


_scratch = {}


def scratch():
    d = _device_key()
    if d not in _scratch:
        _scratch[d] = _Scratch()
    return _scratch[d]


def launch_count():
    return int(_lib.load().pmb_launch_count())


# --------------------------------------------------------------------------
# optional per-region device timing (CUDA events on the launching stream; used by
# bench.py for the roofline of the dominant kernel -- no synchronisation is added)
# --------------------------------------------------------------------------
_timing = {"on": False, "events": {}, "trace": None}


def enable_timing(flag=True):
    _timing["on"] = bool(flag)
    _timing["events"] = {}


def enable_trace(flag=True):
    """Record a (label, start, stop) event triple around EVERY contraction launch
    (tools/profile_sweep.py: which index patterns of a whole CCSD sweep cost what)."""
    _timing["trace"] = [] if flag else None


def trace_report():
    """[(label, flops, milliseconds)] in launch order (synchronises the device)."""
    torch.cuda.synchronize()
    return [(lab, fl, a.elapsed_time(b)) for lab, fl, a, b in (_timing["trace"] or [])]


class timed:
    """``with timed("pp_ladder"): ...`` records start/stop events when timing is enabled."""

    def __init__(self, tag):
        self.tag = tag

    def __enter__(self):
        if _timing["on"]:
            self.t0 = torch.cuda.Event(enable_timing=True)
            self.t1 = torch.cuda.Event(enable_timing=True)
            self.t0.record(torch.cuda.current_stream())
        return self

    def __exit__(self, *exc):
        if _timing["on"]:
            self.t1.record(torch.cuda.current_stream())
            _timing["events"].setdefault(self.tag, []).append((self.t0, self.t1))
        return False


def timing_report():
    """{tag: [milliseconds per recorded region]} (synchronises the device)."""
    torch.cuda.synchronize()
    return {tag: [a.elapsed_time(b) for a, b in ev] for tag, ev in _timing["events"].items()}


# --------------------------------------------------------------------------
# two independent launch sequences side by side
# --------------------------------------------------------------------------
_side_streams = {}


class side_by_side:
    """``with side_by_side() as side: main work; side(lambda: other work)`` -- runs ``other
    work`` on a second CUDA stream, ordered after everything already queued on the current
    stream, and joins it on exit.  For pairs of independent contractions whose grids are only
    a few waves long (W1 = V_iabc.tau, W2 = V_aibc.tau: 4.2 waves each): the second kernel's
    CTAs fill the SMs the first one's last partial wave leaves idle.  Every tensor the side
    work touches must be allocated beforehand (pass ``out=``): the caching allocator is
    per stream."""

    def __enter__(self):
        dev = _device_key()
        if dev not in _side_streams:
            _side_streams[dev] = torch.cuda.Stream() if torch.cuda.is_available() else None
        self.side = _side_streams[dev]
        self.main = torch.cuda.current_stream() if self.side is not None else None
        if self.side is not None:
            self.side.wait_stream(self.main)
        return self._run

    def _run(self, fn):
        if self.side is None:                 # host-logic tests without a device
            return fn()
        with torch.cuda.stream(self.side):
            return fn()

    def __exit__(self, *exc):
        if self.side is not None:
            self.main.wait_stream(self.side)
        return False


# --------------------------------------------------------------------------
# contraction front end
# --------------------------------------------------------------------------
def _parse(spec):
    lhs, out = spec.replace(" ", "").split("->")
    a, b = lhs.split(",")
    return a, b, out


def _fill(arr, vals):
    for i, v in enumerate(vals):
        arr[i] = int(v)


ALIGN_K_MIN_ELEMENTS = 1 << 16
SMALL_SIDE_TO_N = os.environ.get("PYMES_B200_SMALL_SIDE_TO_N", "1") == "1"


def _unit_index(sub, t):
    """The index along which ``t`` is unit-stride (extent > 1), or None."""
    for ch, n, st in zip(sub, t.shape, t.stride()):
        if st == 1 and n > 1:
            return ch
    return None


def _align_k(sa, A, sb, B):
    """Both operands stream their tiles along the contracted (K) indices in ONE common order.
    When each operand is unit-stride along a *different* contracted index (e.g.
    ``abjk,jkcb->ac``: T2 runs along k, V_ijab along b), any order leaves one of them gathering
    single 8-byte words out of 32-byte sectors, strides apart (measured: 3 TFLOP/s and 90 GB/s
    on o.v^3-sized operands).  The smaller operand is then re-laid out once -- its contracted
    indices in the other operand's order, innermost -- which costs one HBM-bound pass."""
    if isinstance(A, GeneratedOperand) or isinstance(B, GeneratedOperand):
        return sa, A, sb, B
    ks = set(sa) & set(sb)
    ua, ub = _unit_index(sa, A), _unit_index(sb, B)
    if ua is None or ub is None or ua == ub or ua not in ks or ub not in ks:
        return sa, A, sb, B
    if min(A.numel(), B.numel()) < ALIGN_K_MIN_ELEMENTS:
        return sa, A, sb, B                      # small enough to live in L2 either way
    if (B if B.numel() <= A.numel() else A).dim() > 4:
        return sa, A, sb, B                      # the copy kernel handles rank <= 4 (batched sigma: as is)

    def relaid(s_small, small, s_big, big):
        bstr = dict(zip(s_big, big.stride()))
        k_ord = sorted((ch for ch in s_small if ch in ks), key=lambda ch: -bstr[ch])
        new_sub = "".join(ch for ch in s_small if ch not in ks) + "".join(k_ord)
        return new_sub, copy(small.permute(*[s_small.index(ch) for ch in new_sub]))

    if B.numel() <= A.numel():
        sb, B = relaid(sb, B, sa, A)
    else:
        sa, A = relaid(sa, A, sb, B)
    return sa, A, sb, B


def describe_contraction(out_sub, terms, out=None, beta=0.0, conv=None, alloc=None):
    """Build the ``pmb_contract_t`` descriptor for ``contract_terms`` (pure host logic:
    index classification, operand swaps, group ordering, strides).  Returns
    ``(descriptor, out, operands)``; ``conv``/``alloc`` default to the device versions
    (the CPU tests substitute host tensors to check this logic without a GPU)."""
    conv = asdev if conv is None else conv
    alloc = empty if alloc is None else alloc
    if not 1 <= len(terms) <= _lib.MAX_TERMS:
        raise ValueError("1..%d terms per contraction" % _lib.MAX_TERMS)
    ext = {}
    norm = []
    for alpha, sa, A, sb, B in terms:
        A, B = conv(A), conv(B)
        if A.dim() != len(sa) or B.dim() != len(sb):
            raise ValueError("subscripts %s,%s do not match operand ranks" % (sa, sb))
        sa, A, sb, B = _align_k(sa, A, sb, B)
        for s, t in ((sa, A), (sb, B)):
            if len(set(s)) != len(s):
                raise ValueError("repeated index in %s is not supported" % s)
            for ch, n in zip(s, t.shape):
                if ext.setdefault(ch, int(n)) != int(n):
                    raise ValueError("extent mismatch for index %s" % ch)
        norm.append([float(alpha), sa, A, sb, B])
    if len(set(out_sub)) != len(out_sub):
        raise ValueError("repeated output index")
    # split of the output indices fixed by the first term
    m_set = frozenset(ch for ch in out_sub if ch in norm[0][1])
    n_set = frozenset(ch for ch in out_sub if ch in norm[0][3])
    if m_set & n_set or (m_set | n_set) != frozenset(out_sub):
        raise ValueError("batch / broadcast indices are not supported: %s" % out_sub)
    for t in norm:
        in_a = frozenset(ch for ch in out_sub if ch in t[1])
        if in_a == m_set and frozenset(ch for ch in out_sub if ch in t[3]) == n_set:
            continue
        if in_a == n_set and frozenset(ch for ch in out_sub if ch in t[3]) == m_set:
            t[1], t[2], t[3], t[4] = t[3], t[4], t[1], t[2]
            continue
        raise ValueError("terms split the output indices differently")
    for t in norm:
        ka = set(t[1]) - m_set
        kb = set(t[3]) - n_set
        if ka != kb:
            raise ValueError("indices %s appear in one operand only" % sorted(ka ^ kb))
        if len(ka) > _lib.MAX_DIMS:
            raise ValueError("too many contracted indices")
    shape = tuple(ext[ch] for ch in out_sub)
    if out is None:
        if beta != 0.0:
            raise ValueError("beta != 0 needs an output tensor")
        out = alloc(*shape)
    elif tuple(out.shape) != shape:
        raise ValueError("output shape %s != %s" % (tuple(out.shape), shape))
    cstr = dict(zip(out_sub, out.stride()))
    # keep the output's unit-stride index in the N group (coalesced epilogue)
    if out_sub and min(out_sub, key=lambda ch: (cstr[ch], -ext[ch])) in m_set and n_set:
        m_set, n_set = n_set, m_set
        for t in norm:
            t[1], t[2], t[3], t[4] = t[3], t[4], t[1], t[2]
    # When one side of the output is a single occupied index (27 wide: "ci,abcj->abij",
    # "cj,iacb->iajb") it goes to the N side: the 64x32 tile then wastes 5 of 32 columns instead of
    # 37 of 64 rows (measured at v = 362: 7.3 -> 4.2 ms and 7.0 -> 3.8 ms; PYMES_B200_SMALL_SIDE_TO_N=0
    # restores the old assignment for A/B runs).
    if SMALL_SIDE_TO_N and m_set and n_set:
        m_tot = int(np.prod([ext[ch] for ch in m_set]))
        n_tot = int(np.prod([ext[ch] for ch in n_set]))
        if m_tot <= 32 and n_tot >= 1024:
            m_set, n_set = n_set, m_set
            for t in norm:
                t[1], t[2], t[3], t[4] = t[3], t[4], t[1], t[2]
    # a generated operand can only be produced on the row (A) side of the kernel: that
    # outranks the epilogue preference above
    if any(isinstance(t[4], GeneratedOperand) for t in norm):
        if any(isinstance(t[2], GeneratedOperand) for t in norm):
            raise ValueError("generated operands on both sides of a contraction")
        m_set, n_set = n_set, m_set
        for t in norm:
            t[1], t[2], t[3], t[4] = t[3], t[4], t[1], t[2]
    if len(m_set) > _lib.MAX_DIMS or len(n_set) > _lib.MAX_DIMS:
        raise ValueError("too many indices in one group")
    a0 = dict(zip(norm[0][1], norm[0][2].stride()))
    m_ord = sorted(m_set, key=lambda ch: (a0[ch], ch))
    n_ord = sorted(n_set, key=lambda ch: (cstr[ch], ch))

    d = _lib.Contract()
    d.nm, d.nn, d.nterms = len(m_ord), len(n_ord), len(norm)
    _fill(d.m_ext, [ext[ch] for ch in m_ord])
    _fill(d.n_ext, [ext[ch] for ch in n_ord])
    _fill(d.c_mstr, [cstr[ch] for ch in m_ord])
    _fill(d.c_nstr, [cstr[ch] for ch in n_ord])
    d.C = out.data_ptr()
    d.beta = float(beta)
    for i, (alpha, sa, A, sb, B) in enumerate(norm):
        astr = dict(zip(sa, A.stride()))
        bstr = dict(zip(sb, B.stride()))
        ks = [ch for ch in sa if ch not in m_set]
        a_min = min(sa, key=lambda ch: astr[ch]) if sa else None
        b_min = min(sb, key=lambda ch: bstr[ch]) if sb else None
        if a_min in ks or b_min not in ks:
            k_ord = sorted(ks, key=lambda ch: (astr[ch], ch))
        else:
            k_ord = sorted(ks, key=lambda ch: (bstr[ch], ch))
        t = d.terms[i]
        t.A, t.B, t.nk, t.alpha = A.data_ptr(), B.data_ptr(), len(k_ord), alpha
        if isinstance(A, GeneratedOperand):
            gen = A.gen_descriptor(sa, m_ord, k_ord)
            keep = getattr(d, "_keep", [])
            keep.append(gen)
            d._keep = keep                      # the descriptor points into it
            t.a_gen = C.addressof(gen)
        _fill(t.k_ext, [ext[ch] for ch in k_ord])
        _fill(t.a_kstr, [astr[ch] for ch in k_ord])
        _fill(t.b_kstr, [bstr[ch] for ch in k_ord])
        _fill(t.a_mstr, [astr[ch] for ch in m_ord])
        _fill(t.b_nstr, [bstr[ch] for ch in n_ord])
    return d, out, norm


GEMV_MIN_ELEMENTS = 1 << 22
GEMV_MIN_OUTPUTS = 1 << 16           # one thread per output: needs that many to fill the GPU
GEMV_MIN_WARP_OUTPUTS = 1 << 11      # one warp per output


def _try_gemv(out_sub, terms, out, beta):
    """Matrix-vector contractions (one operand without any output index, the other o.v^3-sized:
    the T1 dressing of the Fock matrix and of the singles residual) go to ``pmb_gemv``, which
    streams the big operand once instead of feeding 1-row DMMA tiles.  Returns the result or
    None when the pattern does not apply."""
    if len(terms) != 1:
        return None
    alpha, sa, A, sb, B = terms[0]
    A, B = asdev(A), asdev(B)
    if isinstance(A, GeneratedOperand) or isinstance(B, GeneratedOperand):
        return None
    a_out = [ch for ch in sa if ch in out_sub]
    b_out = [ch for ch in sb if ch in out_sub]
    if bool(a_out) == bool(b_out):
        return None
    vsub, vec, bsub, big = (sa, A, sb, B) if not a_out else (sb, B, sa, A)
    if big.numel() < GEMV_MIN_ELEMENTS or vec.dim() != len(vsub) or big.dim() != len(bsub):
        return None
    if len(set(vsub)) != len(vsub) or len(set(bsub)) != len(bsub) or len(set(out_sub)) != len(out_sub):
        return None
    xs = [ch for ch in bsub if ch not in vsub]
    if set(vsub) - set(bsub) or set(xs) != set(out_sub) or not 1 <= len(vsub) <= 4 or len(xs) > 4:
        return None
    ext = dict(zip(bsub, big.shape))
    if any(ext[ch] != n for ch, n in zip(vsub, vec.shape)):
        raise ValueError("extent mismatch in %s,%s" % (sa, sb))
    # enough outputs to fill the GPU?  When the big operand is unit-stride along a summed index the
    # kernel gives a whole WARP to each output (lanes walk that index): a few thousand outputs are
    # enough ("jb,abij->ai": 13 176 outputs of 13 176-term sums over T2 ran at 0.3 TB/s as a split-K
    # tensor contraction).  Unit-stride along an output index means one THREAD per output.
    bs = dict(zip(bsub, big.stride()))
    k0 = min(vsub, key=lambda ch: (bs[ch], ch))
    warp_per_output = ext[k0] >= 16 and (not xs or bs[k0] < min(bs[ch] for ch in xs))
    n_out = big.numel() // max(vec.numel(), 1)
    if n_out < (GEMV_MIN_WARP_OUTPUTS if warp_per_output else GEMV_MIN_OUTPUTS):
        return None                      # few outputs, long sums: left to the split-K contraction
    shape = tuple(ext[ch] for ch in out_sub)
    if out is None:
        if beta != 0.0:
            raise ValueError("beta != 0 needs an output tensor")
        out = empty(*shape)
    elif tuple(out.shape) != shape:
        raise ValueError("output shape %s != %s" % (tuple(out.shape), shape))
    bstr, vstr, ostr = dict(zip(bsub, big.stride())), dict(zip(vsub, vec.stride())), dict(zip(out_sub, out.stride()))
    k_ord = sorted(vsub, key=lambda ch: (bstr[ch], ch))
    x_ord = sorted(xs, key=lambda ch: (bstr[ch], ch))
    d = _lib.Gemv()
    d.vec, d.B, d.out = vec.data_ptr(), big.data_ptr(), out.data_ptr()
    d.nk, d.nx, d.alpha, d.beta = len(k_ord), len(x_ord), float(alpha), float(beta)
    _fill(d.k_ext, [ext[ch] for ch in k_ord])
    _fill(d.v_kstr, [vstr[ch] for ch in k_ord])
    _fill(d.b_kstr, [bstr[ch] for ch in k_ord])
    _fill(d.x_ext, [ext[ch] for ch in x_ord])
    _fill(d.b_xstr, [bstr[ch] for ch in x_ord])
    _fill(d.o_xstr, [ostr[ch] for ch in x_ord])
    trace = _timing["trace"]
    if trace is not None:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(torch.cuda.current_stream())
    rc = _lib.load().pmb_gemv(C.byref(d), _stream())
    if trace is not None:
        t1.record(torch.cuda.current_stream())
        trace.append(("%s,%s->%s [gemv]" % (sa, sb, out_sub), 2.0 * big.numel(), t0, t1))
    _lib.check(rc, "pmb_gemv")
    return out


# Momentum-blocked evaluation of contractions whose row operand is a generated (momentum-
# conserving) integral block: on by default, PYMES_B200_BLOCKED=0 or set_blocked(False) sends them
# through the dense generated-operand path of pmb_contract instead (A/B runs, bench --ladder dense).
_BLOCKED = [os.environ.get("PYMES_B200_BLOCKED", "1") != "0"]


def set_blocked(flag):
    old = _BLOCKED[0]
    _BLOCKED[0] = bool(flag)
    return old


def blocked_enabled():
    return _BLOCKED[0]


def blocked_companion(t):
    """The never-materialised twin of a STORED integral block (``UEG.eval_2b_blocks`` attaches one
    to V_iabc / V_aibc: their compressed values are 1/v of the block), for the contractions that
    can run momentum-blocked; None when there is none, the blocked path is switched off, or the
    block was edited in place since (its twin holds the old values)."""
    return getattr(t, "_pmb_blocked", None) if _BLOCKED[0] and block_rule(t) is not None else None


def _column_groups(n_sub, ext, bstr, cstr):
    """Split the column indices into (n0, n1): n0 the innermost indices that are dense and
    unit-stride in BOTH B and C, n1 the rest flattened into one index.  Returns
    ``(n0_ext, n1_ext, b_n1str, c_n1str)`` or None when the layouts do not allow it."""
    idx = [ch for ch in n_sub if ext[ch] > 1]
    if not idx:
        return 1, 1, 0, 0
    order = sorted(idx, key=lambda ch: (cstr[ch], ch))
    if sorted(idx, key=lambda ch: (bstr[ch], ch)) != order:
        return None
    if bstr[order[0]] != 1 or cstr[order[0]] != 1:
        return None
    n0, i = ext[order[0]], 1
    while i < len(order) and bstr[order[i]] == n0 and cstr[order[i]] == n0:
        n0 *= ext[order[i]]
        i += 1
    if i == len(order):
        return n0, 1, 0, 0
    b1, c1, n1 = bstr[order[i]], cstr[order[i]], ext[order[i]]
    i += 1
    while i < len(order) and bstr[order[i]] == b1 * n1 and cstr[order[i]] == c1 * n1:
        n1 *= ext[order[i]]
        i += 1
    if i != len(order):
        return None
    return n0, n1, b1, c1


# --------------------------------------------------------------------------
# momentum tags: which elements of a tensor can be non-zero
# --------------------------------------------------------------------------
class Momentum:
    """Selection rule of a tensor: ``x[i_0, i_1, ..]`` can be non-zero only where
    ``sum_d sign_d * lin[lo_d + i_d] == total``, ``lin`` the linearised momentum of every orbital
    (``model.ueg.momentum_groups``) and one ``(lo, ext, sign)`` per axis.  A stored UEG integral block
    has signs (+,+,-,-) and total 0; an excitation vector of one total-momentum sector
    (``model.ueg.excitation_sector``) has total l(K).  Contractions, linear combinations and index
    swaps of tensors with such rules have one as well (:func:`contract_terms` derives it), and a
    tensor from outside gets one only by :func:`adopt_momentum`, which checks it.  A sign 0 leaves
    its axis unconstrained.  Kept in a normal form (first non-zero sign positive, the total flipped
    with the signs): rules equal up to an overall sign compare equal."""

    __slots__ = ("lin", "lin_key", "axes", "total")

    def __init__(self, lin, axes, lin_key=None, total=0):
        axes = tuple((int(lo), int(n), int(sg)) for lo, n, sg in axes)
        total = int(total)
        first = next((sg for _lo, _n, sg in axes if sg), 1)
        if first < 0:
            axes = tuple((lo, n, -sg) for lo, n, sg in axes)
            total = -total
        self.lin = lin
        self.lin_key = lin_key if lin_key is not None else (lin.tobytes() if lin is not None else None)
        self.axes = axes
        self.total = total

    def __eq__(self, other):
        return isinstance(other, Momentum) and self.axes == other.axes and self.total == other.total \
            and self.lin_key == other.lin_key

    def __hash__(self):
        return hash((self.axes, self.total, self.lin_key))

    def with_axes(self, axes):
        return Momentum(self.lin, axes, self.lin_key, self.total)

    def with_total(self, total):
        return Momentum(self.lin, self.axes, self.lin_key, total)

    def narrow(self, dim, lo, n):
        axes = list(self.axes)
        a_lo, _a_n, sg = axes[dim]
        axes[dim] = (a_lo + int(lo), int(n), sg)
        return self.with_axes(axes)

    def permute(self, dims):
        return self.with_axes([self.axes[d] for d in dims])

    def signed(self, d):
        """Signed momentum labels ``sign * lin[lo:lo+ext]`` of axis ``d`` (int64), without the total."""
        lo, n, sg = self.axes[d]
        if sg == 0:
            return np.zeros(n, dtype=np.int64)
        return sg * np.asarray(self.lin[lo:lo + n], dtype=np.int64)

    def labels(self, d):
        """Labels of axis ``d`` such that an allowed element's labels sum to 0: the signed labels,
        with the total subtracted from those of axis 0 (what ``pmb_momentum_residue`` checks)."""
        lab = self.signed(d)
        return lab - self.total if d == 0 and self.total else lab


def _set_momentum(t, key, block=False):
    """Tag ``t`` with the rule ``key`` (None: untagged); ``block`` marks a stored integral block
    (:func:`tag_block`).  One version stamp serves both: an in-place edit ends the two."""
    t._pmb_mom = (key, t._version, block) if key is not None else None


def momentum_of(x):
    """The live :class:`Momentum` tag of ``x`` (None when there is none, or when the tensor was
    edited in place after it was tagged: the tag records the tensor's version counter)."""
    if isinstance(x, GeneratedOperand):
        return x.momentum()
    if not isinstance(x, torch.Tensor):
        return None
    tag = getattr(x, "_pmb_mom", None)
    if tag is not None and tag[1] == x._version:
        return tag[0]
    # a view of a tensor whose rule is live (written through a sibling view since it was made)
    link = getattr(x, "_pmb_parent", None)
    if link is not None:
        pk = momentum_of(link[0])
        if pk is not None:
            return pk.narrow(*link[1:])
    return None


def ones(n):
    """A vector of ones; it satisfies the rule without constraint (sign 0)."""
    t = torch.ones(n, dtype=F64, device=device())
    _set_momentum(t, Momentum(None, [(0, n, 0)]))
    return t


def adopt_momentum(t, key, host=None):
    """Tag ``t`` (a tensor that enters from outside) with the rule ``key`` if and only if every
    element the rule forbids is exactly zero (``pmb_momentum_residue``: one pass over the tensor).
    ``host``: the same values as a numpy array the caller holds anyway (e.g. the Fock matrix); they
    are checked there instead.  Returns True when it was tagged.  A stored integral block adopted
    under its own rule stays one (:func:`block_rule`)."""
    if key is None or not isinstance(t, torch.Tensor) or t.dim() != len(key.axes) or not 1 <= t.dim() <= 4:
        return False
    block = block_rule(t) == key
    if any(int(n) != a[1] for n, a in zip(t.shape, key.axes)):
        raise ValueError("momentum rule %s does not fit a tensor of shape %s" % (key.axes, tuple(t.shape)))
    if host is not None:
        host = np.asarray(host)
        if host.shape != tuple(t.shape):
            raise ValueError("host copy of shape %s for a tensor of shape %s" % (host.shape, tuple(t.shape)))
        total = np.zeros((), dtype=np.int64)
        for d in range(t.dim()):
            total = np.add.outer(total, key.labels(d))
        ok = not np.any(host[total != 0] != 0)           # NaN != 0: not adopted
        _set_momentum(t, key if ok else None, ok and block)
        return ok
    if t.numel() == 0:
        # no element can break the rule (and pmb_momentum_residue takes no extent of 0)
        _set_momentum(t, key, block)
        return True
    labels = torch.from_numpy(np.concatenate([key.labels(d) for d in range(t.dim())])).to(device())
    res = zeros(1)
    _lib.check(_lib.load().pmb_momentum_residue(t.dim(), _lib.I64x4(*_pad4r(t.shape, 1)),
                                                 _lib.I64x4(*_pad4r(t.stride(), 0)), _ptr(t), _ptr(labels),
                                                 _ptr(res), _stream()), "pmb_momentum_residue")
    ok = float(res.item()) == 0.0
    _set_momentum(t, key if ok else None, ok and block)
    return ok


def drop_momentum(t):
    """Remove the momentum tag of ``t`` (always safe: the tensor then takes the dense paths)."""
    if isinstance(t, torch.Tensor):
        _set_momentum(t, None)


def _pad4r(vals, fill):
    vals = [int(v) for v in vals]
    return vals + [fill] * (4 - len(vals))


def _chain(out):
    """``[(parent, dim, lo, n, parent's live tag)]`` up the :func:`narrow` chain of ``out``, read
    BEFORE a write into it."""
    links, t = [], out
    while True:
        link = getattr(t, "_pmb_parent", None)
        if link is None:
            return links
        p, dim, lo, n = link
        links.append((p, dim, lo, n, momentum_of(p)))
        t = p


def _written(out, key, chain):
    """A backend kernel has written ``out``: its storage changed behind torch's back, so the version
    counter it shares with its base and every other view is bumped (their tags die), then ``out``
    gets ``key``.  A :func:`narrow` parent whose rule, restricted to the view, is ``key`` keeps its
    tag: the write stayed inside its selection rule."""
    torch.autograd.graph.increment_version(out)
    _set_momentum(out, key)
    child = key
    for p, dim, lo, n, pk in chain:
        if child is None or pk is None or pk.narrow(dim, lo, n) != child:
            break
        _set_momentum(p, pk)
        child = pk


def _term_keys(out_sub, sa, ka, sb, kb):
    """The rules the product ``einsum(sa, sb -> out_sub)`` of operands with rules ``ka`` / ``kb``
    satisfies: with one sign sigma for the whole term, every summed axis must cancel
    (``sign_a + sigma * sign_b == 0`` over the same orbitals); the output axes then carry the signs
    of A and sigma times those of B, and the total ``total_A + sigma * total_B``.  Both sigmas when
    nothing constrains it (outer products)."""
    if ka.lin_key is not None and kb.lin_key is not None and ka.lin_key != kb.lin_key:
        return set()
    lin, lin_key = (ka.lin, ka.lin_key) if ka.lin_key is not None else (kb.lin, kb.lin_key)
    xa, xb = dict(zip(sa, ka.axes)), dict(zip(sb, kb.axes))
    sigmas = {1, -1}
    for ch in sa:
        if ch not in sb:
            if ch not in out_sub:
                return set()
            continue
        if ch in out_sub:
            return set()
        (la, na, ga), (lb, nb, gb) = xa[ch], xb[ch]
        if ga == 0 and gb == 0:
            continue
        if (la, na) != (lb, nb) or abs(ga) != abs(gb):
            return set()
        sigmas &= {-1 if ga == gb else 1}
    if any(ch not in sa and ch not in out_sub for ch in sb) or any(ch not in xa and ch not in xb for ch in out_sub):
        return set()
    return {Momentum(lin, [xa[ch] if ch in xa else (xb[ch][0], xb[ch][1], sg * xb[ch][2]) for ch in out_sub],
                     lin_key, ka.total + sg * kb.total) for sg in sigmas}


def _derive(out_sub, terms, old, accumulate):
    """The rule of ``out = beta*out + sum of terms``: one that every term satisfies (and, when the
    output accumulates, the one it already has); None when there is none."""
    if accumulate and old is None:
        return None
    cands = None
    for _alpha, sa, A, sb, B in terms:
        ka, kb = momentum_of(A), momentum_of(B)
        if ka is None or kb is None or len(ka.axes) != len(sa) or len(kb.axes) != len(sb):
            return None
        c = _term_keys(out_sub, sa, ka, sb, kb)
        cands = c if cands is None else cands & c
        if not cands:
            return None
    if old is not None:
        return old if old in cands else None
    return min(cands, key=lambda k: k.axes)


def tag_block(t, rule):
    """Mark ``t`` as a stored integral block whose elements obey ``rule`` (``UEG.eval_2b_blocks``):
    products of such a block with an untagged operand run on its momentum groups
    (``pmb_blocked_contract``, ``pmb_gather_expand``).  Returns the tensor."""
    _set_momentum(t, rule, block=True)
    return t


def block_rule(t):
    """The live rule of a stored integral block (:func:`tag_block`); None for any other tensor and
    after an in-place edit.  :func:`narrow` and :func:`copy` keep the mark, every backend write and
    :func:`permute` end it: amplitudes, intermediates and permuted views take the paths their rules
    alone select."""
    tag = getattr(t, "_pmb_mom", None) if isinstance(t, torch.Tensor) else None
    if tag is None or tag[1] != t._version or not tag[2]:
        return None
    return tag[0]


def narrow(t, dim, lo, n):
    """``t.narrow(dim, lo, n)`` that keeps the tags of ``t``, restricted to the view."""
    out = t.narrow(dim, lo, n)
    k = momentum_of(t)
    if k is not None:
        _set_momentum(out, k.narrow(dim, lo, n), block_rule(t) is not None)
    out._pmb_parent = (t, int(dim), int(lo), int(n))
    return out


def permute(t, dims):
    """``t.permute(dims)`` that keeps the momentum tag of ``t``."""
    out = t.permute(*dims)
    k = momentum_of(t)
    if k is not None:
        _set_momentum(out, k.permute(dims))
    return out


def _structured(x):
    """Does ``x`` carry a block-diagonal momentum structure ``pmb_blocked_contract`` can use?"""
    if isinstance(x, GeneratedOperand):
        return x.blocked_lists() is not None
    return block_rule(x) is not None


def _blocked_term(out_sub, term):
    """``(alpha, sa, S, sb, D, m_axes, k_axes)`` if this term can go to ``pmb_blocked_contract``:
    S a momentum-structured 4-index operand (a generated block with block lists, or a stored
    integral block, :func:`block_rule`) with two of its indices in the output (``m_axes``, rows) and two
    contracted with D (``k_axes``, entries); every other index of D an output index.  A generated
    operand only in its native split (p,q | r,s).  Else None."""
    if not _BLOCKED[0]:
        return None
    alpha, sa, A, sb, B = term
    if isinstance(A, LinearOperator) or isinstance(B, LinearOperator):
        return None
    if not _structured(A):
        if not _structured(B):
            return None
        sa, A, sb, B = sb, B, sa, A
    if isinstance(B, GeneratedOperand):
        return None
    B = asdev(B)
    if len(sa) != 4 or len(set(sa)) != 4 or len(set(sb)) != len(sb) or len(set(out_sub)) != len(out_sub):
        return None
    if B.dim() != len(sb) or A.dim() != 4:
        return None
    m_axes = tuple(i for i, ch in enumerate(sa) if ch in out_sub)
    k_axes = tuple(i for i, ch in enumerate(sa) if ch not in out_sub)
    if len(m_axes) != 2 or any(sa[i] in sb for i in m_axes) or any(sa[i] not in sb for i in k_axes):
        return None
    n_sub = [ch for ch in sb if ch not in sa]
    if not n_sub or any(ch not in out_sub for ch in n_sub) or len(n_sub) + 2 != len(out_sub):
        return None
    if isinstance(A, GeneratedOperand) and (m_axes, k_axes) != ((0, 1), (2, 3)):
        return None
    return float(alpha), sa, A, sb, B, m_axes, k_axes


def _run_blocked(out_sub, term, out, beta):
    """One term through ``pmb_blocked_contract``; returns False when the operand layouts rule it
    out (the caller then uses the dense path)."""
    alpha, sa, A, sb, B, m_axes, k_axes = term
    ext = dict(zip(sb, (int(n) for n in B.shape)))
    if any(int(A.shape[i]) != ext[sa[i]] for i in k_axes):
        raise ValueError("extent mismatch in %s,%s" % (sa, sb))
    bstr, cstr = dict(zip(sb, B.stride())), dict(zip(out_sub, out.stride()))
    cols = _column_groups([ch for ch in sb if ch not in sa], ext, bstr, cstr)
    if cols is None:
        return False
    n0, n1, b1, c1 = cols
    dev = device()
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    if isinstance(A, GeneratedOperand):
        L = A.blocked_lists()
        values, a_moff, a_koff = L["values"], L["a_moff"], L["a_koff"]
    else:
        L = block_lists(block_rule(A), m_axes, k_axes)
        astr = A.stride()
        akey = ("a", astr[m_axes[0]], astr[m_axes[1]], astr[k_axes[0]], astr[k_axes[1]])
        aoffs = L["offsets"].get(akey)
        if aoffs is None:
            aoffs = (up(L["row_i0"] * akey[1] + L["row_i1"] * akey[2]), up(L["ent_j0"] * akey[3] + L["ent_j1"] * akey[4]))
            L["offsets"][akey] = aoffs
        values, (a_moff, a_koff) = A, aoffs
    key = (cstr[sa[m_axes[0]]], cstr[sa[m_axes[1]]], bstr[sa[k_axes[0]]], bstr[sa[k_axes[1]]])
    offs = L["offsets"].get(key)
    if offs is None:
        offs = (up(L["row_i0"] * key[0] + L["row_i1"] * key[1]), up(L["ent_j0"] * key[2] + L["ent_j1"] * key[3]))
        L["offsets"][key] = offs
    if beta != 1.0 and not L["rows_covered"]:
        # rows outside every group are part of the result: zero, or scaled by beta
        if beta == 0.0:
            out.zero_()
        else:
            axpby(beta, out, 0.0, out)
        beta = 1.0
    d = _lib.Blocked()
    d.A, d.B, d.C = values.data_ptr(), B.data_ptr(), out.data_ptr()
    d.a_moff, d.a_koff = a_moff.data_ptr(), a_koff.data_ptr()
    d.c_moff, d.b_koff = offs[0].data_ptr(), offs[1].data_ptr()
    d.tiles, d.n_tiles = L["tiles"].data_ptr(), int(L["n_tiles"])
    d.n0_ext, d.n1_ext, d.b_n1str, d.c_n1str = n0, n1, b1, c1
    d.alpha, d.beta = alpha, float(beta)
    trace = _timing["trace"]
    if trace is not None:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(torch.cuda.current_stream())
    rc = _lib.load().pmb_blocked_contract(C.byref(d), _stream())
    if trace is not None:
        t1.record(torch.cuda.current_stream())
        trace.append(("%s,%s->%s [momentum-blocked]" % (sa, sb, out_sub), 2.0 * L["nnz"] * n0 * n1, t0, t1))
    _lib.check(rc, "pmb_blocked_contract")
    return True


# T1 dressing products of a stored UEG block with ONE summed index ("abid,dj->abij", ...): gathers
# over the partner tables instead of a pass over the o.v^3 block (pmb_gather_expand).
_GATHER = [os.environ.get("PYMES_B200_T1_GATHER", "1") != "0"]


def set_gather(flag):
    old = _GATHER[0]
    _GATHER[0] = bool(flag)
    return old


def partner_tables(S, y_axis):
    """For a contiguous stored integral block ``S`` and one of its axes ``y_axis``: ``idx[x0,x1,x2]``
    = the local index along that axis of the ONE orbital whose label completes the other three to
    the block's rule (:func:`block_rule`), or -1, and ``val[x0,x1,x2] = S[x0,x1,x2 | idx]`` (0 where
    there is none) -- what ``pmb_gather_expand`` reads instead of the block.  (x0,x1,x2) are the
    other three axes in S's own order.  Device tensors, cached on the tensor that owns S's storage
    (they go with the block, and a row block narrowed again every sweep finds them) until the
    storage is next written."""
    rule = block_rule(S)
    if rule is None or not S.is_contiguous():
        raise ValueError("partner tables need a contiguous stored integral block")
    owner = S if S._base is None else S._base
    cache = getattr(owner, "_pmb_partner", None)
    if cache is None or cache[0] != S._version:
        cache = owner._pmb_partner = (S._version, {})
    key = (rule, int(y_axis), S.data_ptr())
    tab = cache[1].get(key)
    if tab is None:
        others = [ax for ax in range(4) if ax != y_axis]
        l0, l1, l2 = (rule.labels(ax) for ax in others)
        want = -(l0[:, None, None] + l1[None, :, None] + l2[None, None, :]).reshape(-1)
        ly = rule.labels(y_axis)
        order = np.argsort(ly)
        pos = np.minimum(np.searchsorted(ly[order], want), len(ly) - 1)
        hit = ly[order][pos] == want
        idx = np.where(hit, order[pos], -1).astype(np.int32)
        # flat position in S of (x0,x1,x2 | idx)
        grid = np.meshgrid(*[np.arange(S.shape[ax], dtype=np.int64) for ax in others], indexing="ij")
        flat = sum(g * S.stride(ax) for g, ax in zip(grid, others)).reshape(-1)
        flat = flat + np.maximum(idx, 0).astype(np.int64) * S.stride(y_axis)
        idx_d = torch.from_numpy(idx).to(device())
        val = torch.index_select(S.reshape(-1), 0, torch.from_numpy(flat).to(device()))
        val = torch.where(idx_d >= 0, val, torch.zeros_like(val))
        tab = cache[1][key] = dict(idx=idx_d, val=val, ext=tuple(int(S.shape[ax]) for ax in others),
                                   n_hit=int(hit.sum()))
    return tab


def _try_gather(out_sub, terms, out, beta):
    """``out[x0,x1,x2,j] = beta*out + alpha * sum_y S[x0,x1,x2|y] D[y,j]`` for a stored, tagged UEG
    integral block S (three of its indices in the output, one summed) and a two-index D (T1): one
    candidate y per (x0,x1,x2), so the product is an HBM-bound pass over the output
    (``pmb_gather_expand``).  Returns the result or None when the pattern / layouts do not apply."""
    if not (_BLOCKED[0] and _GATHER[0]) or len(terms) != 1 or len(out_sub) != 4 or len(set(out_sub)) != 4:
        return None
    alpha, sa, A, sb, B = terms[0]
    if block_rule(A) is None:
        sa, A, sb, B = sb, B, sa, A
    if block_rule(A) is None or isinstance(B, (GeneratedOperand, LinearOperator)) or len(sa) != 4 or len(sb) != 2:
        return None
    if len(set(sa)) != 4 or len(set(sb)) != 2 or not A.is_contiguous():
        return None
    B = asdev(B)
    if B.dim() != 2 or block_rule(B) is not None:
        return None
    ys = [ch for ch in sa if ch in sb]
    if len(ys) != 1 or ys[0] in out_sub:
        return None
    y = ys[0]
    j = sb[1 - sb.index(y)]
    xs = [ch for ch in sa if ch != y]
    if j in sa or set(xs) | {j} != set(out_sub):
        return None
    ext = dict(zip(sa, (int(n) for n in A.shape)))
    if int(B.shape[sb.index(y)]) != ext[y]:
        raise ValueError("extent mismatch in %s,%s" % (sa, sb))
    ext[j] = int(B.shape[sb.index(j)])
    shape = tuple(ext[ch] for ch in out_sub)
    if out is None:
        if beta != 0.0:
            raise ValueError("beta != 0 needs an output tensor")
        out = empty(*shape)
    elif tuple(out.shape) != shape:
        raise ValueError("output shape %s != %s" % (tuple(out.shape), shape))
    elif not out.is_contiguous():
        return None
    elif out.device != device():
        raise RuntimeError("pymes_b200: output tensor lives on %s, the kernels write to %s "
                           "(there is no CPU fallback)" % (out.device, device()))
    tab = partner_tables(A, sa.index(y))
    d = _lib.Gather()
    d.val, d.idx, d.D, d.out = tab["val"].data_ptr(), tab["idx"].data_ptr(), B.data_ptr(), out.data_ptr()
    xe = tab["ext"]
    for k, ch in enumerate(out_sub):
        d.ext[k] = ext[ch]
        d.role[k] = 3 if ch == j else xs.index(ch)
    d.x_str[0], d.x_str[1], d.x_str[2] = xe[1] * xe[2], xe[2], 1
    d.d_ystr, d.d_jstr = B.stride(sb.index(y)), B.stride(sb.index(j))
    d.alpha, d.beta = float(alpha), float(beta)
    trace = _timing["trace"]
    if trace is not None:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(torch.cuda.current_stream())
    rc = _lib.load().pmb_gather_expand(C.byref(d), _stream())
    if trace is not None:
        t1.record(torch.cuda.current_stream())
        trace.append(("%s,%s->%s [momentum-gather]" % (sa, sb, out_sub), 2.0 * out.numel(), t0, t1))
    _lib.check(rc, "pmb_gather_expand")
    return out


def _group_term(out_sub, term):
    """``(alpha, sa, A, sb, B, sigma)`` if this term can go to ``pmb_group_contract``: both operands
    stored tensors of rank 1-4 with a live momentum rule that the term conserves (``_term_keys``).
    Every index of A is an output index (a row) or summed with B (an entry), every other index of B
    is an output index (a column), and there is at least one output index.  A summed axis with a
    non-zero sign on both operands fixes the sign sigma; a term whose summed axes all have sign 0
    (a trace with :func:`ones`) is left to the other paths.  Without summed axes (an outer
    product) only group 0 exists and sigma = 1.  Else None."""
    if not _BLOCKED[0]:
        return None
    alpha, sa, A, sb, B = term
    if not (isinstance(A, torch.Tensor) and isinstance(B, torch.Tensor)) or not out_sub:
        return None
    if not (1 <= len(sa) <= 4 and 1 <= len(sb) <= 4) or A.dim() != len(sa) or B.dim() != len(sb):
        return None
    if len(set(sa)) != len(sa) or len(set(sb)) != len(sb) or len(set(out_sub)) != len(out_sub):
        return None
    ka, kb = momentum_of(A), momentum_of(B)
    if ka is None or kb is None or len(ka.axes) != len(sa) or len(kb.axes) != len(sb):
        return None
    if not _term_keys(out_sub, sa, ka, sb, kb):
        return None
    ents = [ch for ch in sa if ch in sb]
    signs = [(ka.axes[sa.index(ch)][2], kb.axes[sb.index(ch)][2]) for ch in ents]
    signs = [(ga, gb) for ga, gb in signs if ga != 0 and gb != 0]
    if ents and not signs:
        return None
    ga, gb = signs[0] if signs else (1, -1)
    return float(alpha), sa, A, sb, B, (-1 if ga == gb else 1)


_GROUP_CACHE = {}
GROUP_TILE = 32          # rows / columns per tile of pmb_group_contract (its GT)


def _side_keys(k, axes, sign, shift=0):
    """The distinct labels of one side (``sign`` times the sum of its axes' signed labels, plus
    ``shift``), grown one axis at a time so that the labels of a long side (o.v^2 members) are
    never all formed."""
    keys = np.zeros(1, dtype=np.int64)
    for d in axes:
        keys = np.unique(np.add.outer(keys, np.unique(k.signed(d))))
    return sign * keys + shift


def _side_members(k, axes, sign, shift, common):
    """Flat positions (C order over ``axes``) of the side's members whose label is in ``common``,
    stably sorted by label, with each group's first index and count in that list."""
    lab = np.full(1, shift, dtype=np.int64)
    for d in axes:
        lab = np.add.outer(lab, sign * k.signed(d)).reshape(-1)
    pos = np.flatnonzero(np.isin(lab, common))
    pos = pos[np.argsort(lab[pos], kind="stable")]
    _keys, first, cnt = np.unique(lab[pos], return_index=True, return_counts=True)
    return pos, first, cnt


def block_groups(rule, m_axes, k_axes):
    """The 4-index tensor with momentum rule ``rule`` as the matrix [rows = axes ``m_axes``, entries =
    axes ``k_axes``] is block diagonal: a row and an entry can meet only where their labels cancel.
    Returns ``(row_pos, ent_pos, g_row0, g_rows, g_ent0, g_ents)``: the flat positions (C order over
    the side's axes) of the rows / entries of the groups present on both sides, sorted by group
    (index order inside a group), and each group's first position and length in the two lists."""
    sides = ((rule, m_axes, 1, -rule.total), (rule, k_axes, -1, 0))
    common = np.intersect1d(_side_keys(*sides[0]), _side_keys(*sides[1]))
    (r_pos, r_first, r_cnt), (e_pos, e_first, e_cnt) = (_side_members(*s_, common) for s_ in sides)
    return r_pos, e_pos, r_first, r_cnt, e_first, e_cnt


def blocked_tiles(g_first, g_cnt, g_e0, g_en, tile_rows=64):
    """Row tiles of ``pmb_blocked_contract``: every group's rows in equal pieces of whole 8-row
    fragments, at most ``tile_rows`` each; {first row, rows, first entry, entries} per tile,
    long groups first."""
    pieces = -(-g_cnt // tile_rows)
    size = -(-g_cnt // np.maximum(pieces, 1))
    size = np.minimum(-(-size // 8) * 8, tile_rows)
    pieces = -(-g_cnt // np.maximum(size, 1))
    grp = np.repeat(np.arange(len(g_cnt)), pieces)
    within = np.arange(len(grp)) - np.repeat(np.cumsum(pieces) - pieces, pieces)
    t_m0 = g_first[grp] + within * size[grp]
    t_mn = np.minimum(size[grp], g_cnt[grp] - within * size[grp])
    tiles = np.stack([t_m0, t_mn, g_e0[grp], g_en[grp]], axis=1).astype(np.int32)
    return np.ascontiguousarray(tiles[np.argsort(-tiles[:, 3], kind="stable")])


_LIST_CACHE = {}


def block_lists(rule, m_axes=(0, 1), k_axes=(2, 3)):
    """Lists of ``pmb_blocked_contract`` for a 4-index tensor with momentum rule ``rule`` split as
    :func:`block_groups`: the index pairs of the rows / entries (numpy int64, sorted by group), the
    device tile table and a cache for the offset tables derived from them.  Cached by value (a
    sharded sweep narrows the same blocks every iteration)."""
    key = (rule, tuple(m_axes), tuple(k_axes), str(device()))
    L = _LIST_CACHE.get(key)
    if L is None:
        r_pos, e_pos, g_first, g_cnt, g_e0, g_en = block_groups(rule, m_axes, k_axes)
        ext = [n for _lo, n, _sg in rule.axes]
        tiles = blocked_tiles(g_first, g_cnt, g_e0, g_en)
        L = _LIST_CACHE[key] = dict(
            row_i0=r_pos // ext[m_axes[1]], row_i1=r_pos % ext[m_axes[1]],
            ent_j0=e_pos // ext[k_axes[1]], ent_j1=e_pos % ext[k_axes[1]],
            tiles=torch.from_numpy(tiles).to(device()), n_tiles=len(tiles),
            nnz=int((g_cnt * g_en).sum()), n_groups=len(g_cnt), offsets={},
            # every row meets at least one entry: a fresh output needs no clearing
            rows_covered=int(g_cnt.sum()) == ext[m_axes[0]] * ext[m_axes[1]])
    return L


def _side_offsets(pos, ext, *strides):
    """Element offsets of flat positions ``pos`` over extents ``ext``, one array per stride set."""
    idx = np.unravel_index(pos, ext) if ext else ()
    offs = []
    for st in strides:
        o = np.zeros(len(pos), dtype=np.int64)
        for i, s_ in zip(idx, st):
            o += i.astype(np.int64) * int(s_)
        offs.append(o)
    return offs


def _group_plan(out_sub, g, out):
    """Device lists and tiles of one group term, cached by value: the three sides' momentum labels
    and the strides of A, B and C (intermediates are new tensors every sweep and hit the cache).
    A side without axes (rows of a matrix-vector product, entries of an outer product) has one
    member, label 0 and offset 0.  Only members of groups common to all three sides are listed;
    when there is none, the plan has no tile and nothing is uploaded."""
    _alpha, sa, A, sb, B, sigma = g
    ka, kb = momentum_of(A), momentum_of(B)
    rows = [d for d, ch in enumerate(sa) if ch in out_sub]
    ents = [d for d, ch in enumerate(sa) if ch not in out_sub]
    cols = [d for d, ch in enumerate(sb) if ch in out_sub]
    b_ents = [sb.index(sa[d]) for d in ents]
    cstr = dict(zip(out_sub, out.stride()))
    key = (ka.lin_key, kb.lin_key, tuple(ka.axes[d] for d in rows + ents), tuple(kb.axes[d] for d in cols), sigma,
           ka.total, kb.total,
           tuple(A.stride(d) for d in rows + ents), tuple(B.stride(d) for d in b_ents + cols),
           tuple(cstr[sa[d]] for d in rows), tuple(cstr[sb[d]] for d in cols), str(out.device))
    plan = _GROUP_CACHE.get(key)
    if plan is not None:
        return plan
    # group label g = R - t_A = -E_A = sigma (t_B - C_B): R, E_A the signed row / entry sums of A,
    # C_B the column sum of B, t_A / t_B the totals (A: R + E_A = t_A; B: -sigma E_A + C_B = t_B)
    sides = ((ka, rows, 1, -ka.total), (ka, ents, -1, 0), (kb, cols, -sigma, sigma * kb.total))
    common = np.intersect1d(_side_keys(*sides[0]), _side_keys(*sides[2]))
    if len(common):
        common = np.intersect1d(common, _side_keys(*sides[1]))
    if not len(common):
        plan = dict(tiles=torch.zeros((0, 6), dtype=torch.int32), n_tiles=0, flops=0.0)
        _GROUP_CACHE[key] = plan
        return plan
    (r_pos, r_first, r_cnt), (e_pos, e_first, e_cnt), (c_pos, c_first, c_cnt) = (
        _side_members(*s_, common) for s_ in sides)
    tiles = []
    for r0, rn, e0, en, c0, cn in zip(r_first, r_cnt, e_first, e_cnt, c_first, c_cnt):
        for rt in range(0, int(rn), GROUP_TILE):
            for ct_ in range(0, int(cn), GROUP_TILE):
                tiles.append((r0 + rt, min(GROUP_TILE, rn - rt), e0, en, c0 + ct_, min(GROUP_TILE, cn - ct_)))
    tiles = np.asarray(tiles, dtype=np.int32).reshape(-1, 6)
    dev = out.device
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(dev)
    a_row, c_row = _side_offsets(r_pos, [A.shape[d] for d in rows], [A.stride(d) for d in rows],
                                 [cstr[sa[d]] for d in rows])
    a_ent, b_ent = _side_offsets(e_pos, [A.shape[d] for d in ents], [A.stride(d) for d in ents],
                                 [B.stride(d) for d in b_ents])
    b_col, c_col = _side_offsets(c_pos, [B.shape[d] for d in cols], [B.stride(d) for d in cols],
                                 [cstr[sb[d]] for d in cols])
    plan = dict(
        a_row=up(a_row), a_ent=up(a_ent), b_ent=up(b_ent), b_col=up(b_col), c_row=up(c_row), c_col=up(c_col),
        tiles=torch.from_numpy(np.ascontiguousarray(tiles)).to(dev), n_tiles=len(tiles),
        flops=2.0 * float((r_cnt * e_cnt * c_cnt).sum()))
    _GROUP_CACHE[key] = plan
    return plan


def _run_group(out_sub, g, out, beta):
    """One term through ``pmb_group_contract``.  Elements outside every group get no product: they
    are cleared (beta = 0) or scaled (beta != 1) here, before the kernel accumulates."""
    alpha, sa, A, sb, B, _sigma = g
    plan = _group_plan(out_sub, g, out)
    if beta == 0.0:
        out.zero_()
    elif beta != 1.0:
        axpby(beta, out, 0.0, out)
    d = _lib.Group()
    if not plan["n_tiles"]:
        # no group is common to the three sides: the product is zero and nothing is launched
        # (pmb_group_contract returns before it reads a table)
        _lib.check(_lib.load().pmb_group_contract(C.byref(d), _stream()), "pmb_group_contract")
        return
    d.A, d.B, d.C = A.data_ptr(), B.data_ptr(), out.data_ptr()
    d.a_row, d.a_ent, d.b_ent = plan["a_row"].data_ptr(), plan["a_ent"].data_ptr(), plan["b_ent"].data_ptr()
    d.b_col, d.c_row, d.c_col = plan["b_col"].data_ptr(), plan["c_row"].data_ptr(), plan["c_col"].data_ptr()
    d.tiles, d.n_tiles, d.alpha = plan["tiles"].data_ptr(), int(plan["n_tiles"]), alpha
    trace = _timing["trace"]
    if trace is not None:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(torch.cuda.current_stream())
    rc = _lib.load().pmb_group_contract(C.byref(d), _stream())
    if trace is not None:
        t1.record(torch.cuda.current_stream())
        trace.append(("%s,%s->%s [momentum-blocked]" % (sa, sb, out_sub), plan["flops"], t0, t1))
    _lib.check(rc, "pmb_group_contract")


def _batched_group_term(out_sub, term):
    """``(alpha, sa, A, sb, B, g, n_batch, a_bstr, b_bstr)`` if this term is a group product
    (:func:`_group_term`) repeated over a batch axis: the output's leading index ``r`` is held by A
    and / or B on an axis of sign 0 (stacked right-hand sides, :func:`stack`), and the product of
    one slice qualifies.  ``g`` is that slice's group term (views of right-hand side 0, tagged with
    the rules less the batch axis); a stride of 0 marks the operand without ``r``.  Else None."""
    if not _BLOCKED[0]:
        return None
    alpha, sa, A, sb, B = term
    if not (isinstance(A, torch.Tensor) and isinstance(B, torch.Tensor)) or len(out_sub) < 2:
        return None
    r = out_sub[0]
    if r not in sa and r not in sb:
        return None
    sliced, n_batch = [], None
    for s_, T in ((sa, A), (sb, B)):
        k = momentum_of(T)
        if k is None or len(k.axes) != T.dim() or T.dim() != len(s_):
            return None
        if r not in s_:
            sliced.append((s_, T, 0))
            continue
        d = s_.index(r)
        if k.axes[d][2] != 0 or int(T.shape[d]) < 1 or (n_batch is not None and n_batch != int(T.shape[d])):
            return None
        n_batch = int(T.shape[d])
        v = T.select(d, 0)
        _set_momentum(v, k.with_axes(k.axes[:d] + k.axes[d + 1:]))
        sliced.append((s_.replace(r, ""), v, int(T.stride(d))))
    (sa1, A1, a_bstr), (sb1, B1, b_bstr) = sliced
    g = _group_term(out_sub[1:], (alpha, sa1, A1, sb1, B1))
    if g is None:
        return None
    return float(alpha), sa, A, sb, B, g, n_batch, a_bstr, b_bstr


def _run_group_batched(out_sub, t, out, beta):
    """One term of :func:`_batched_group_term` through ``pmb_group_contract_batched``: the group
    plan of one right-hand side serves all of them (planned once per geometry, whatever the batch
    size).  Elements outside every group are cleared (beta = 0) or scaled (beta != 1) here."""
    _alpha, sa, _A, sb, _B, g, n_batch, a_bstr, b_bstr = t
    c_bstr = int(out.stride(0))
    plan = _group_plan(out_sub[1:], g, out.select(0, 0))
    if beta == 0.0:
        out.zero_()
    elif beta != 1.0:
        for k in range(out.shape[0]):
            axpby(beta, out[k], 0.0, out[k])
    d = _lib.GroupBatched()
    d.n_batch, d.a_bstr, d.b_bstr, d.c_bstr = n_batch, a_bstr, b_bstr, c_bstr
    if not plan["n_tiles"]:
        _lib.check(_lib.load().pmb_group_contract_batched(C.byref(d), _stream()), "pmb_group_contract_batched")
        return
    alpha, _sa1, A1, _sb1, B1, _sigma = g
    p = d.g
    p.A, p.B, p.C = A1.data_ptr(), B1.data_ptr(), out.data_ptr()
    p.a_row, p.a_ent, p.b_ent = plan["a_row"].data_ptr(), plan["a_ent"].data_ptr(), plan["b_ent"].data_ptr()
    p.b_col, p.c_row, p.c_col = plan["b_col"].data_ptr(), plan["c_row"].data_ptr(), plan["c_col"].data_ptr()
    p.tiles, p.n_tiles, p.alpha = plan["tiles"].data_ptr(), int(plan["n_tiles"]), alpha
    trace = _timing["trace"]
    if trace is not None:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(torch.cuda.current_stream())
    rc = _lib.load().pmb_group_contract_batched(C.byref(d), _stream())
    if trace is not None:
        t1.record(torch.cuda.current_stream())
        trace.append(("%s,%s->%s [momentum-blocked x%d]" % (sa, sb, out_sub, n_batch), plan["flops"] * n_batch,
                      t0, t1))
    _lib.check(rc, "pmb_group_contract_batched")


def _try_blocked(out_sub, terms, out, beta):
    """Terms with momentum structure are evaluated on their diagonal blocks only: both operands
    with a live momentum rule by ``pmb_group_contract`` (``_group_term``; repeated over stacked
    right-hand sides by ``pmb_group_contract_batched``, ``_batched_group_term``), a
    stored or generated integral block times a dense operand by ``pmb_blocked_contract``
    (``_blocked_term``).  The other terms of the same call (e.g. the hole-hole ladder next to the
    particle-particle one, ccd.py:185-187) keep the dense kernel.  Returns the result, or None when
    no term qualifies."""
    picked = []
    for i, t in enumerate(terms):
        bt = _batched_group_term(out_sub, t)
        if bt is not None:
            picked.append((i, "batched", bt))
            continue
        g = _group_term(out_sub, t)
        if g is not None:
            picked.append((i, "group", g))
            continue
        b = _blocked_term(out_sub, t)
        if b is not None:
            picked.append((i, "blocked", b))
    if not picked:
        return None
    _alpha, sa, A, sb, B = picked[0][2][:5]
    ext = dict(zip(sb, (int(n) for n in B.shape)))
    ext.update(zip(sa, (int(n) for n in A.shape)))
    shape = tuple(ext[ch] for ch in out_sub)
    if out is None:
        if beta != 0.0:
            raise ValueError("beta != 0 needs an output tensor")
        out = empty(*shape)
    elif tuple(out.shape) != shape:
        raise ValueError("output shape %s != %s" % (tuple(out.shape), shape))
    elif out.device != device():
        raise RuntimeError("pymes_b200: output tensor lives on %s, the kernels write to %s "
                           "(there is no CPU fallback)" % (out.device, device()))
    done = set()
    rest = [t for i, t in enumerate(terms) if i not in {j for j, _k, _t in picked}]
    if rest:
        contract_terms(out_sub, rest, out=out, beta=beta)
        beta = 1.0
    for i, kind, t in picked:
        if kind == "batched":
            _run_group_batched(out_sub, t, out, beta)
        elif kind == "group":
            _run_group(out_sub, t, out, beta)
        elif not _run_blocked(out_sub, t, out, beta):
            continue
        done.add(i)
        beta = 1.0
    left = [terms[i] for i, _k, _t in picked if i not in done]
    if left:
        old = set_blocked(False)
        try:
            contract_terms(out_sub, left, out=out, beta=beta)
        finally:
            set_blocked(old)
    return out


def contract_terms(out_sub, terms, out=None, beta=0.0):
    """out[out_sub] = beta*out + sum_t alpha_t * einsum(subA_t, subB_t -> out_sub).

    ``terms`` is a list of ``(alpha, subA, A, subB, B)``.  All terms must split the
    output indices between their two operands in the same way (operands are
    swapped automatically when needed); contracted indices may differ per term.
    One kernel launch accumulates every term in registers.

    The result carries the momentum rule every term derives from its operands' rules (and, when
    ``beta != 0``, the one ``out`` already had); otherwise none.
    """
    accumulate = out is not None and beta != 0.0
    chain = _chain(out) if out is not None else []
    key = _derive(out_sub, terms, momentum_of(out) if accumulate else None, accumulate)
    out = _contract_terms(out_sub, terms, out, beta)
    _written(out, key, chain)
    return out


def _contract_terms(out_sub, terms, out, beta):
    lib = _lib.load()
    if out is not None and out.device != device():
        raise RuntimeError("pymes_b200: output tensor lives on %s, the kernels write to %s "
                           "(there is no CPU fallback)" % (out.device, device()))
    # a term whose operands both carry a live rule runs on its momentum groups, however cheap the
    # matrix-vector or gather kernel would be: the group plan skips every product the rules make zero
    if any(_group_term(out_sub, t) is not None or _batched_group_term(out_sub, t) is not None for t in terms):
        return _try_blocked(out_sub, terms, out, beta)
    res = _try_gemv(out_sub, terms, out, beta)
    if res is not None:
        return res
    res = _try_gather(out_sub, terms, out, beta)
    if res is not None:
        return res
    res = _try_blocked(out_sub, terms, out, beta)
    if res is not None:
        return res
    d, out, _operands = describe_contraction(out_sub, terms, out, beta)
    need = lib.pmb_contract_workspace(C.byref(d))
    ws = scratch().splitk_ws(need) if need else None
    trace = _timing["trace"]
    if trace is not None:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(torch.cuda.current_stream())
    rc = lib.pmb_contract(C.byref(d), _ptr(ws) if ws is not None else None, need, _stream())
    if trace is not None:
        t1.record(torch.cuda.current_stream())
        flops = 0.0
        for _a, sa, A, sb, B in _operands:
            n = 2.0
            for ch, e in {**dict(zip(sa, A.shape)), **dict(zip(sb, B.shape))}.items():
                n *= e
            flops += n
        label = " + ".join("%s,%s" % (t[1], t[3]) for t in _operands) + "->" + out_sub
        trace.append((label + (" [split-K]" if need else ""), flops, t0, t1))
    _lib.check(rc, "pmb_contract")
    return out


def contract(spec, A, B, out=None, alpha=1.0, beta=0.0):
    """Two-operand einsum on the DMMA engine: out = beta*out + alpha*einsum(spec, A, B)."""
    sa, sb, so = _parse(spec)
    return contract_terms(so, [(alpha, sa, asdev(A), sb, asdev(B))], out=out, beta=beta)


# --------------------------------------------------------------------------
# elementwise / reduction wrappers
# --------------------------------------------------------------------------
def _pad4(vals, fill):
    vals = list(vals)
    return [fill] * (4 - len(vals)) + vals


def axpby(alpha, src, beta=0.0, out=None):
    """out = alpha*src + beta*out for tensors of rank <= 4; ``src`` may be any view."""
    lib = _lib.load()
    src = asdev(src)
    if src.dim() > 4:
        raise ValueError("rank <= 4 only")
    if out is None:
        if beta != 0.0:
            raise ValueError("beta != 0 needs an output tensor")
        out = empty(*src.shape)
    if tuple(out.shape) != tuple(src.shape):
        raise ValueError("shape mismatch")
    key, chain = momentum_of(src), _chain(out)
    if beta != 0.0 and momentum_of(out) != key:
        key = None
    ext = _lib.I64x4(*_pad4(src.shape, 1))
    si = _lib.I64x4(*_pad4(src.stride(), 0))
    so = _lib.I64x4(*_pad4(out.stride(), 0))
    _lib.check(lib.pmb_axpby4(ext, float(alpha), _ptr(src), si, float(beta), _ptr(out), so, _stream()),
               "pmb_axpby4")
    _written(out, key, chain)
    return out


def copy(src):
    """A copy keeps the tags of its source (a copy of a stored integral block IS the block)."""
    out = axpby(1.0, src)
    rule = block_rule(src)
    if rule is not None:
        tag_block(out, rule)
    return out


def mp2_amplitudes(eps_i, eps_a, shift, V_abij, rows=None):
    """T2 = V_abij / D.  ``rows=(a_lo, na)``: V_abij is the local row block [na,nv,no,no]."""
    lib = _lib.load()
    no, nv = eps_i.numel(), eps_a.numel()
    a_lo, na = rows if rows is not None else (0, nv)
    T2 = empty(na, nv, no, no)
    _lib.check(lib.pmb_mp2_amplitudes(no, nv, a_lo, na, _ptr(eps_i), _ptr(eps_a), float(shift), _ptr(V_abij),
                                      _lib.I64x4(*V_abij.stride()), _ptr(T2), _stream()),
               "pmb_mp2_amplitudes")
    _written(T2, momentum_of(V_abij), [])        # the denominators are diagonal: same rule
    return T2


def update_doubles(eps_i, eps_a, shift, delta, R, T2, scal, rows=None, product_denominator=False):
    """dT = R/D, T2 += delta*dT (in place); scal[0] = |dT|^2.  Returns dT.
    ``rows=(a_lo, na)``: R and T2 are local row blocks [na,nv,no,no].
    ``product_denominator``: D = e_i e_j e_a e_b + shift (the reference's Brueckner branch,
    ccd.py:118) instead of e_i + e_j - e_a - e_b + shift."""
    if not T2.is_contiguous() or not R.is_contiguous():
        raise ValueError("update_doubles needs contiguous R and T2 (they are indexed flat)")
    lib = _lib.load()
    no, nv = eps_i.numel(), eps_a.numel()
    a_lo, na = rows if rows is not None else (0, nv)
    dT = torch.empty_like(T2)
    kR, kT, chain = momentum_of(R), momentum_of(T2), _chain(T2)
    ws = scratch().reduce_ws()
    _lib.check(lib.pmb_update_doubles(no, nv, a_lo, na, _ptr(eps_i), _ptr(eps_a), float(shift), float(delta),
                                      int(bool(product_denominator)), _ptr(R), _ptr(dT), _ptr(T2), _ptr(scal),
                                      _ptr(ws), ws.numel() * 8,
                                      _stream()), "pmb_update_doubles")
    _written(dT, kR, [])
    _written(T2, kT if kT == kR else None, chain)
    return dT


def update_singles(eps_i, eps_a, shift, delta, R1, T1):
    lib = _lib.load()
    no, nv = eps_i.numel(), eps_a.numel()
    dT1 = torch.empty_like(T1)
    kR, kT, chain = momentum_of(R1), momentum_of(T1), _chain(T1)
    _lib.check(lib.pmb_update_singles(no, nv, _ptr(eps_i), _ptr(eps_a), float(shift), float(delta), _ptr(R1),
                                      _ptr(dT1), _ptr(T1), _stream()), "pmb_update_singles")
    _written(dT1, kR, [])
    _written(T1, kT if kT == kR else None, chain)
    return dT1


def _flat(what, t, shape):
    """Raise unless ``t`` is a contiguous tensor of ``shape``: the kernels index it flat."""
    if tuple(t.shape) != tuple(shape) or not t.is_contiguous():
        raise ValueError("%s must be a contiguous tensor of shape %s (got shape %s, strides %s)"
                         % (what, tuple(shape), tuple(t.shape), tuple(t.stride())))


def energy_doubles(T2, V_ijab, scal, T1=None, mp2_form=False, rows=None):
    """scal[0:3] = (E_direct, E_exchange, |T2|^2) on the device (partial sums over the local
    row block when ``rows=(a_lo, na)``; V_ijab and T1 are always the full tensors)."""
    lib = _lib.load()
    nv, no = T2.shape[1], T2.shape[2]
    a_lo, na = rows if rows is not None else (0, nv)
    _flat("energy_doubles: T2", T2, (na, nv, no, no))
    if T1 is not None:
        _flat("energy_doubles: T1", T1, (nv, no))
    ws = scratch().reduce_ws()
    _lib.check(lib.pmb_energy_doubles(no, nv, a_lo, na, _ptr(T2), _ptr(T1) if T1 is not None else None,
                                      _ptr(V_ijab), _lib.I64x4(*V_ijab.stride()), int(mp2_form), _ptr(scal),
                                      _ptr(ws), ws.numel() * 8, _stream()), "pmb_energy_doubles")
    return scal


def tilde(T2, swap_ij=False):
    lib = _lib.load()
    nv, no = T2.shape[0], T2.shape[2]
    _flat("tilde: T2", T2, (nv, nv, no, no))
    Tt = torch.empty_like(T2)
    k = momentum_of(T2)
    _lib.check(lib.pmb_tilde(no, nv, _ptr(T2), _ptr(Tt), int(swap_ij), _stream()), "pmb_tilde")
    # 2 T - T with two indices swapped: the rule survives when the swap leaves it unchanged
    _written(Tt, k if k is not None and k.permute((0, 1, 3, 2) if swap_ij else (1, 0, 2, 3)) == k else None, [])
    return Tt


def sym_baji(Ex, R=None, accumulate=True):
    """R (+)= Ex + Ex^{baji}."""
    lib = _lib.load()
    nv, no = Ex.shape[0], Ex.shape[2]
    _flat("sym_baji: Ex", Ex, (nv, nv, no, no))
    if R is None:
        R, accumulate = torch.empty_like(Ex), False
    _flat("sym_baji: R", R, (nv, nv, no, no))
    k, chain = momentum_of(Ex), _chain(R)
    if k is not None and (k.permute((1, 0, 3, 2)) != k or (accumulate and momentum_of(R) != k)):
        k = None
    _lib.check(lib.pmb_sym_baji(no, nv, _ptr(Ex), _ptr(R), int(accumulate), _stream()), "pmb_sym_baji")
    _written(R, k, chain)
    return R


def sym_baji_stack(Ex, R):
    """R[k] = Ex[k] + Ex[k]^{baji} for every k of the stacks Ex, R [r,v,v,o,o] (``sym_baji`` per
    right-hand side); R keeps the rule of Ex when the swap leaves it unchanged."""
    k, chain = momentum_of(Ex), _chain(R)
    if k is not None and k.permute((0, 2, 1, 4, 3)) != k:
        k = None
    for i in range(Ex.shape[0]):
        sym_baji(Ex[i], R[i], accumulate=False)
    _written(R, k, chain)
    return R


def stack(tensors):
    """``torch.stack`` along a new leading axis; the result keeps the rule the inputs share (the new
    axis, a batch of right-hand sides, gets sign 0), none when they do not all carry the same one."""
    keys = {momentum_of(t) for t in tensors}
    out = torch.stack(list(tensors))
    key = keys.pop() if len(keys) == 1 else None
    _set_momentum(out, key.with_axes([(0, len(tensors), 0)] + list(key.axes)) if key is not None else None)
    return out


def clear(t, rule=None):
    """Zero ``t`` in place and tag it with ``rule`` (zeros satisfy any rule); returns ``t``."""
    t.zero_()
    _set_momentum(t, rule)
    return t


def _ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def dots(xs, y, out=None):
    """out[k] = <xs[k], y> (plain products, no conjugation) for contiguous tensors."""
    lib = _lib.load()
    for t in list(xs) + [y]:
        if not t.is_contiguous():
            raise ValueError("dots needs contiguous tensors")
    if out is None:
        out = empty(len(xs))
    ws = scratch().reduce_ws()
    for lo in range(0, len(xs), 16):                 # the C entry point takes up to 16 vectors per call
        chunk = list(xs[lo:lo + 16])
        _lib.check(lib.pmb_dots(len(chunk), _ptr_array(chunk), _ptr(y), y.numel(), _ptr(out[lo:lo + len(chunk)]),
                                _ptr(ws), ws.numel() * 8, _stream()), "pmb_dots")
    return out


def lincomb(coefs, xs, out=None, beta=0.0):
    """out = beta*out + sum_k coefs[k]*xs[k] for contiguous tensors of one shape."""
    lib = _lib.load()
    for t in xs:
        if not t.is_contiguous():
            raise ValueError("lincomb needs contiguous tensors")
    if out is None:
        out = torch.empty_like(xs[0])
    keys = {momentum_of(t) for t in xs} | ({momentum_of(out)} if beta != 0.0 else set())
    key, chain = (keys.pop() if len(keys) == 1 else None), _chain(out)
    done = 0
    while done < len(xs):
        chunk = xs[done:done + 16]
        c = (C.c_double * len(chunk))(*[float(v) for v in coefs[done:done + 16]])
        _lib.check(lib.pmb_lincomb(len(chunk), c, _ptr_array(chunk), out.numel(),
                                   float(beta) if done == 0 else 1.0, _ptr(out), _stream()), "pmb_lincomb")
        done += len(chunk)
    _written(out, key, chain)
    return out


def bdot(spec, A, B, out=None, alpha=1.0, beta=0.0):
    """out[I] = beta*out + alpha * sum_R A[I,R]*B[I,R] for einsum strings in which some index is
    shared by both operands AND the output (e.g. "kica,caki->ai"), which no GEMM expresses.
    Indices of one operand only must appear in the output.  HBM-bound ``pmb_bdot``."""
    lib = _lib.load()
    sa, sb, so = _parse(spec)
    A, B = asdev(A), asdev(B)
    ext = {}
    for sub, t in ((sa, A), (sb, B)):
        if len(set(sub)) != len(sub) or t.dim() != len(sub):
            raise ValueError("bad subscripts %s" % sub)
        for ch, n in zip(sub, t.shape):
            if ext.setdefault(ch, int(n)) != int(n):
                raise ValueError("extent mismatch for %s" % ch)
    red = [ch for ch in sa if ch in sb and ch not in so]
    if (set(sa) | set(sb)) - set(red) != set(so) or len(set(so)) != len(so):
        raise ValueError("every non-summed index must appear in the output: %s" % spec)
    if len(so) > 4 or len(red) > 4:
        raise ValueError("at most 4 output and 4 summed indices")
    shape = tuple(ext[ch] for ch in so)
    if out is None:
        if beta != 0.0:
            raise ValueError("beta != 0 needs an output tensor")
        out = empty(*shape)
    elif tuple(out.shape) != shape:
        raise ValueError("output shape mismatch")
    astr, bstr, ostr = dict(zip(sa, A.stride())), dict(zip(sb, B.stride())), dict(zip(so, out.stride()))
    iord = sorted(so, key=lambda ch: (ostr[ch], ch))            # fastest output index first
    rord = sorted(red, key=lambda ch: (astr[ch], ch))
    d = _lib.Bdot()
    d.A, d.B, d.out = A.data_ptr(), B.data_ptr(), out.data_ptr()
    d.ni, d.nr, d.alpha, d.beta = len(iord), len(rord), float(alpha), float(beta)
    _fill(d.i_ext, [ext[ch] for ch in iord])
    _fill(d.o_istr, [ostr[ch] for ch in iord])
    _fill(d.a_istr, [astr.get(ch, 0) for ch in iord])
    _fill(d.b_istr, [bstr.get(ch, 0) for ch in iord])
    _fill(d.r_ext, [ext[ch] for ch in rord])
    _fill(d.a_rstr, [astr[ch] for ch in rord])
    _fill(d.b_rstr, [bstr[ch] for ch in rord])
    chain = _chain(out)
    _lib.check(lib.pmb_bdot(C.byref(d), _stream()), "pmb_bdot")
    _written(out, None, chain)
    return out


def cdiv_shifted(diag, z, shift, xr, xi):
    """(yr, yi) = (xr + i xi) / (z - diag + shift), elementwise, for flat contiguous tensors."""
    lib = _lib.load()
    yr, yi = torch.empty_like(xr), torch.empty_like(xi)
    _lib.check(lib.pmb_cdiv_shifted(diag.numel(), _ptr(diag), float(np.real(z)), float(np.imag(z)), float(shift),
                                    _ptr(xr), _ptr(xi), _ptr(yr), _ptr(yi), _stream()), "pmb_cdiv_shifted")
    return yr, yi


def _sector_index(idx, row):
    """Host copy of a sector index list ``idx`` (1-D contiguous int64 device tensor), checked once per
    version of ``idx``: strictly increasing offsets inside a row of ``row`` elements."""
    if not (isinstance(idx, torch.Tensor) and idx.dtype == torch.int64 and idx.dim() == 1 and idx.is_contiguous()):
        raise ValueError("a sector index is a 1-D contiguous int64 tensor")
    tag = getattr(idx, "_pmb_index", None)
    if tag is None or tag[0] != idx._version:
        h = idx.cpu().numpy()
        if len(h) and (h[0] < 0 or np.any(np.diff(h) <= 0)):
            raise ValueError("a sector index must be strictly increasing and non-negative")
        tag = (idx._version, h, {})
        idx._pmb_index = tag
    h = tag[1]
    if len(h) and h[-1] >= row:
        raise ValueError("sector index %d is outside a row of %d elements" % (h[-1], row))
    return tag


def _sector_rows(t, batched, what):
    """(n_batch, batch stride, row length) of a stack [r, ...] (``batched``) or one vector whose rows
    are contiguous."""
    if batched and (t.dim() < 2 or t.shape[0] < 1):
        raise ValueError("%s: a stack [r, ...] of r >= 1 vectors" % what)
    first = t[0] if batched else t
    if not first.is_contiguous():
        raise ValueError("%s: rows of a sector stack must be contiguous" % what)
    return (t.shape[0] if batched else 1), (int(t.stride(0)) if batched else 0), first.numel()


def sector_gather(x_packed_stack, idx, out=None):
    """out[b, k] = x[b].flatten()[idx[k]]: the allowed elements of one momentum sector taken out of a
    stack of dense vectors [r, ...] (each vector contiguous; ``pmb_sector_gather``).  ``out``: an
    [r, len(idx)] tensor with contiguous rows (any row stride, e.g. columns of a wider compact stack),
    allocated when None.  The result carries no rule."""
    x = x_packed_stack
    nb, xb, row = _sector_rows(x, True, "sector_gather")
    _sector_index(idx, row)
    n = idx.numel()
    if out is None:
        out = empty(nb, n)
    if tuple(out.shape) != (nb, n) or out.stride(1) != 1:
        raise ValueError("sector_gather: out must be [%d, %d] with contiguous rows" % (nb, n))
    chain = _chain(out)
    if n:
        _lib.check(_lib.load().pmb_sector_gather(nb, n, _ptr(idx), _ptr(x), xb, _ptr(out), out.stride(0),
                                                 _stream()), "pmb_sector_gather")
    _written(out, None, chain)
    return out


def _index_fits(tag, key, shape):
    """Whether every offset of a sector index lies where ``key`` allows a non-zero in a tensor of
    ``shape`` (host check on the index alone, cached with it)."""
    memo = tag[2]
    if (key, shape) not in memo:
        pos = np.unravel_index(tag[1], shape) if len(tag[1]) else [np.zeros(0, dtype=np.int64)] * len(shape)
        tot = sum(key.labels(d)[p] for d, p in enumerate(pos))
        memo[(key, shape)] = bool(np.all(tot == 0))
    return memo[(key, shape)]


def sector_scatter(compact, idx, out):
    """out[b].flatten()[idx[k]] = compact[b, k] (``pmb_sector_scatter``); every other element of
    ``out`` is left as it is.  ``compact`` [r, len(idx)] (or one vector [len(idx)]), ``out`` [r, ...]
    (or one tensor), rows contiguous.  When ``out`` carried a live momentum rule before the write (a
    ``zeros(..., rule=...)`` buffer) and every offset of ``idx`` is allowed by it, the write keeps
    ``out`` inside the rule and ``out`` is re-stamped with it; otherwise ``out`` is left untagged."""
    batched = compact.dim() == 2
    if compact.dim() not in (1, 2) or compact.stride(-1) != 1:
        raise ValueError("sector_scatter: compact must be [r, n] or [n] with contiguous rows")
    nb, ob, row = _sector_rows(out, batched, "sector_scatter")
    tag = _sector_index(idx, row)
    n = idx.numel()
    if tuple(compact.shape) != ((nb, n) if batched else (n,)):
        raise ValueError("sector_scatter: compact of shape %s for %d vectors of %d elements"
                         % (tuple(compact.shape), nb, n))
    key, chain = momentum_of(out), _chain(out)
    if key is not None:
        shape = tuple(int(e) for e in out.shape)
        if batched:                          # a stack: its batch axis must be unconstrained
            key_row = key.with_axes(key.axes[1:]) if key.axes[0][2] == 0 else None
            shape = shape[1:]
        else:
            key_row = key
        if key_row is None or not _index_fits(tag, key_row, shape):
            key = None
    if n:
        _lib.check(_lib.load().pmb_sector_scatter(nb, n, _ptr(idx), _ptr(compact),
                                                  int(compact.stride(0)) if batched else 0, _ptr(out), ob,
                                                  _stream()), "pmb_sector_scatter")
    _written(out, key, chain)
    return out


def diag_view(t, sub, out_sub):
    """Strided VIEW of a tensor with repeated subscripts, e.g. diag_view(V, "iaai", "ai")[a,i] =
    V[i,a,a,i] (the einsum("iaai->ai") of eom_ccsd.py:182); no data is moved."""
    strides, sizes = {}, {}
    for ch, st, n in zip(sub, t.stride(), t.shape):
        strides[ch] = strides.get(ch, 0) + st
        if sizes.setdefault(ch, n) != n:
            raise ValueError("repeated index %s with different extents" % ch)
    if set(out_sub) != set(sub):
        raise ValueError("diag_view keeps every index: %s -> %s" % (sub, out_sub))
    view = torch.as_strided(t, [sizes[ch] for ch in out_sub], [strides[ch] for ch in out_sub],
                            t.storage_offset())
    k = momentum_of(t)
    if k is not None:
        # a repeated index carries the sum of its axes' signs (the axes must cover the same orbitals)
        axes = {}
        for ch, (lo, n, sg) in zip(sub, k.axes):
            lo0, n0, sg0 = axes.get(ch, (lo, n, 0))
            if (lo0, n0) != (lo, n):
                return view
            axes[ch] = (lo, n, sg0 + sg)
        _set_momentum(view, k.with_axes([axes[ch] for ch in out_sub]))
    return view


def add_broadcast(alpha, src, src_sub, out, out_sub):
    """out[out_sub] += alpha * src[src_sub] with src broadcast over the indices it lacks
    (numpy's ``x[:, None, :, None]`` adds of eom_ccsd.py:206-262)."""
    lib = _lib.load()
    src = asdev(src)
    sstr = dict(zip(src_sub, src.stride()))
    ext = _lib.I64x4(*_pad4(out.shape, 1))
    si = _lib.I64x4(*_pad4([sstr.get(ch, 0) for ch in out_sub], 0))
    so = _lib.I64x4(*_pad4(out.stride(), 0))
    chain = _chain(out)
    _lib.check(lib.pmb_axpby4(ext, float(alpha), _ptr(src), si, 1.0, _ptr(out), so, _stream()), "pmb_axpby4")
    _written(out, None, chain)
    return out


# --------------------------------------------------------------------------
# N-operand einsum (pairwise evaluation on the DMMA engine)
# --------------------------------------------------------------------------
def _pair_result(sa, sb, shared):
    """Subscripts of contract(sa, sb): keep the bigger operand's order and put the
    other operand's surviving indices where the first contracted index was."""
    keep_b = [ch for ch in sb if ch not in shared]
    out, placed = [], False
    for ch in sa:
        if ch in shared:
            if not placed:
                out += keep_b
                placed = True
        else:
            out.append(ch)
    if not placed:
        out += keep_b
    return "".join(out)


def einsum(spec, *ops, out=None, alpha=1.0, beta=0.0):
    """out = beta*out + alpha * einsum(spec, *ops) for the class of expressions the
    coupled-cluster equations use: every index appears exactly twice (in two
    operands, or in one operand and the output).  Products of more than two
    operands are evaluated pairwise, smallest intermediate first -- the device
    counterpart of the reference's ``einsum(..., optimize=True)``."""
    lhs, so = spec.replace(" ", "").split("->")
    subs = lhs.split(",")
    if len(subs) != len(ops):
        raise ValueError("operand count does not match %s" % spec)
    items = [[s, asdev(t)] for s, t in zip(subs, ops)]
    count = {}
    for s in subs + [so]:
        for ch in s:
            count[ch] = count.get(ch, 0) + 1
    if any(v != 2 for v in count.values()):
        raise ValueError("every index must appear exactly twice: %s" % spec)
    ext = {}
    for s, t in items:
        for ch, n in zip(s, t.shape):
            ext[ch] = int(n)
    if len(items) == 1:
        s, t = items[0]
        src = permute(t, [s.index(ch) for ch in so])
        return axpby(alpha, src, beta, out)
    while len(items) > 2:
        best = None
        for i in range(len(items)):
            for j in range(i + 1, len(items)):
                shared = set(items[i][0]) & set(items[j][0])
                if not shared:
                    continue
                size = 1
                for ch in (set(items[i][0]) | set(items[j][0])) - shared:
                    size *= ext[ch]
                if best is None or size < best[0]:
                    best = (size, i, j, shared)
        if best is None:
            raise ValueError("disconnected product in %s" % spec)
        _, i, j, shared = best
        (sa, ta), (sb, tb) = items[i], items[j]
        if tb.numel() > ta.numel():
            sa, ta, sb, tb = sb, tb, sa, ta
        res = _pair_result(sa, sb, shared)
        tmp = contract_terms(res, [(1.0, sa, ta, sb, tb)])
        items = [it for n, it in enumerate(items) if n not in (i, j)] + [[res, tmp]]
    (sa, ta), (sb, tb) = items
    return contract_terms(so, [(alpha, sa, ta, sb, tb)], out=out, beta=beta)
