"""Edges of the tensor contraction engine (csrc/cc_contract.cu, ``pmb_contract``).

The host side of ``pmb_contract`` picks one of twelve kernel instantiations and a launch plan:
the tile configuration (``choose_cfg``), split-K (``split_for``), k windows (``panel_ktiles``),
the cut of a sparse last wave (``tail_plan``), the banded tile order, 16-byte copies of B
(``b_vec2``) and, for a generated UEG operand, one of three producer paths (walker, scanner and
the global-map fallback).  The plan is restated below with its constants read from the CUDA
source, so every call knows which kernels it must launch; on the device the profiler must
record exactly that list and the launch counter must move by its length.  A guard checks that
the cases reach every instantiation of the launch switch.

The operands are integers in [-7, 7] and the coefficients powers of two, so every partial sum
is an exact integer and any summation order gives the same bits: results are compared bit for
bit with numpy, and a dropped, doubled or misplaced k-tile, row or column moves an element by
at least one.  Outputs with beta = 0 are NaN before the call (any read of C shows); strided
outputs sit among sentinels that must come back unchanged; operands sit in NaN-filled buffers,
so NaN in pitch padding or in the gaps of strided views must not reach a stored element.  One
random-valued case per kernel family is checked against a long-double sum with an explicit
bound.

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


SRC, COMMON = _read("cc_contract.cu"), _read("common.cuh")


def _const(text, pattern):
    m = re.search(pattern, text)
    assert m, "not found in the CUDA source: %s" % pattern
    return int(m.group(1))


def _body(name):
    """Body of the host function ``name`` (up to its closing brace in column 0)."""
    m = re.search(r"\n[^\n]*\b%s\([^)]*\)\s*\{(.*?)\n\}\n" % name, SRC, re.S)
    assert m, "function %s not found" % name
    return m.group(1)


SM = _const(COMMON, r"constexpr int kSmCount = (\d+);")
BK = _const(SRC, r"constexpr int BK = (\d+);")
CFG = [(int(a), int(b), int(c), float(e)) for a, b, c, e in
       re.findall(r"\{(\d+), (\d+), (\d+), ([\d.]+)\}", re.search(r"kCfg\[\] = \{(.*?)\};", SRC, re.S).group(1))]
NUM_CFG = _const(SRC, r"constexpr int kNumCfg = (\d+);")
RASTER_BAND = _const(SRC, r"constexpr int kRasterBand = (\d+);")
PANEL_DEFAULT = _const(SRC, r"kPanelDefault = (\d+)LL << 20") << 20
PANEL_DEFAULT_WS = _const(SRC, r"kPanelDefaultWs = (\d+);")
MAX_SMEM = _const(SRC, r"constexpr size_t kMaxSmemOptin = (\d+);")
WS_KRING = _const(SRC, r"constexpr int kWsKRing = (\d+);")
COEF_SPREAD = _const(SRC, r"constexpr int kCoefSpread = (\d+);")
_SPLIT = _body("split_for")
SPLIT_MIN_KT = _const(_SPLIT, r"kt < (\d+)\) return 1")
SPLIT_KT_DIV = _const(_SPLIT, r"n > kt / (\d+)\)")
SPLIT_MAX = _const(_SPLIT, r"if \(n > (\d+)\) n = ")
_TAIL = _body("tail_plan")
TAIL_MIN_KT = _const(_TAIL, r"p\.total_ktiles < (\d+)\)")
TAIL_KT_DIV = _const(_TAIL, r"p\.total_ktiles / (\d+);")
TAIL_REST_DIV = _const(_TAIL, r"rest > kSmCount / (\d+) ")
_CHOOSE = _body("choose_cfg")
assert "kt >= %d" % TAIL_MIN_KT in _CHOOSE and "kt / %d" % TAIL_KT_DIV in _CHOOSE
assert "rest <= slots / %d" % TAIL_REST_DIV in _CHOOSE and "cost < best_cost * 0.999" in _CHOOSE


def _switch():
    """cfg -> kernel template arguments of the launch switch in pmb_contract (default: the rest)."""
    body = re.search(r"switch \(cfg\) \{(.*?)\n        \}", SRC, re.S).group(1)
    cases = {int(c): (kind, args) for c, kind, args in
             re.findall(r"case (\d+): rc = (launch_cfg|launch_ws)<([\d, ]+)>", body)}
    kind, args = re.search(r"default: rc = (launch_cfg|launch_ws)<([\d, ]+)>", body).groups()
    return {c: cases.get(c, (kind, args)) for c in range(NUM_CFG)}


SWITCH = _switch()
WS_STAGES = {c: int(args.split(",")[-1]) for c, (kind, args) in SWITCH.items() if kind == "launch_ws"}
# the tail launch names the warp-specialised instantiations itself
assert "cfg == 5 ? launch_ws<%s>(p, g1, s) : launch_ws<%s>(p, g1, s)" % (SWITCH[5][1], SWITCH[6][1]) in SRC


def _kernel(cfg, il):
    kind, args = SWITCH[cfg]
    if kind == "launch_ws":
        return "contract_ws_kernel<%s>" % args
    return "contract_kernel<%s, %s>" % (args, "true" if il else "false")


ALL_KERNELS = ({_kernel(c, il) for c in range(NUM_CFG) for il in (False, True) if SWITCH[c][0] == "launch_cfg"}
               | {_kernel(c, False) for c in range(NUM_CFG) if SWITCH[c][0] == "launch_ws"}
               | {"splitk_reduce_kernel", "tail_reduce_kernel"})
SENT = -12345.625
EPS = np.finfo(np.float64).eps
NAN = float("nan")

# --------------------------------------------------------------------------
# the launch plan, restated
# --------------------------------------------------------------------------
_TUNE = {"cfg": -1, "split": 0, "panel": PANEL_DEFAULT, "panel_ws": PANEL_DEFAULT_WS}


def _bits_of(name):
    c = _TUNE["cfg"]
    return c >= 0 and bool(c & {"no_walk": 16, "no_mraster": 32, "no_tail": 64, "no_vec2": 128,
                                "no_band": 256}[name])


def _force():
    return _TUNE["cfg"] & 15 if _TUNE["cfg"] >= 0 else _TUNE["cfg"]


def _cdiv(a, b):
    return -(-a // b)


def split_for(tiles, slots, kt):
    if tiles >= slots or kt < SPLIT_MIN_KT:
        return 1
    return max(1, min(slots // tiles, kt // SPLIT_KT_DIV, SPLIT_MAX))


def choose_cfg(M, N, kt):
    best, best_cost, nsplit = 0, 1e300, 1
    force = _force()
    for c in range(NUM_CFG):
        if force >= 0 and (force & 7) < NUM_CFG and c != (force & 7):
            continue
        bm, bn, threads, eff = CFG[c]
        tiles = _cdiv(M, bm) * _cdiv(N, bn)
        per_sm = 3 if threads == 128 else 1
        slots = SM * per_sm
        split = split_for(tiles, slots, kt)
        waves = float(_cdiv(tiles * split, slots))
        if c >= 5 and split == 1 and not _bits_of("no_tail") and kt >= TAIL_MIN_KT:
            rest = tiles % slots
            if tiles > slots and 0 < rest <= slots // TAIL_REST_DIV:
                ts = min(slots // rest, kt // TAIL_KT_DIV)
                if ts >= 2:
                    waves = float(tiles // slots) + 1.0 / ts
        cost = waves * per_sm * bm * bn / (eff * split)
        if cost < best_cost * 0.999:
            best, best_cost, nsplit = c, cost, split
    return best, nsplit


def panel_ktiles(cfg, nsplit, M, N, kt):
    budget = _TUNE["panel_ws"] if cfg >= 5 else _TUNE["panel"]
    if nsplit > 1 or budget <= 0:
        return kt
    small = float(min(M, N))
    if small * kt * BK * 8.0 <= budget:
        return kt
    w = max(int(budget / (small * BK * 8.0)), 64)
    return _cdiv(kt, _cdiv(kt, w))


def tail_plan(cfg, nsplit, M, N, kt, tiles):
    if cfg < 5 or _bits_of("no_tail") or nsplit != 1 or panel_ktiles(cfg, nsplit, M, N, kt) < kt:
        return None
    full = (tiles // SM) * SM
    rest = tiles - full
    if full == 0 or rest == 0 or rest > SM // TAIL_REST_DIV or kt < TAIL_MIN_KT:
        return None
    split = min(SM // rest, kt // TAIL_KT_DIV)
    return (full, rest, split) if split >= 2 else None


def ws_smem_bytes(stages, nterms):
    return 128 + 8 * stages * BK * (2 * 128 + 8) + 8 * (WS_KRING * 2 * BK + (nterms + 1) * 256)


def coef_runs(alphas):
    """[first, last) term ranges of the coefficient runs pmb_contract issues one after another."""
    first, lo, hi = [0], None, None
    for i, a in enumerate(alphas):
        if a == 0.0 or not math.isfinite(a):
            continue
        e = math.frexp(a)[1] - 1
        if lo is None:
            lo = hi = e
        elif max(e, hi) - min(e, lo) > COEF_SPREAD:
            first.append(i)
            lo = hi = e
        else:
            lo, hi = min(lo, e), max(hi, e)
    return list(zip(first, first[1:] + [len(alphas)]))


class Plan:
    """Expected kernels (launch order) and workspace of one pmb_contract call."""

    def __init__(self, M, N, terms, gen=None):
        """``terms``: (alpha, K, generated?) per term; ``gen``: the Gen of the generated one."""
        self.kernels, self.ws, self.runs = [], 0, []
        for lo, hi in coef_runs([t[0] for t in terms]):
            run = self._run(M, N, terms[lo:hi], gen)
            self.runs.append(run)
            self.kernels += run["kernels"]
            self.ws = max(self.ws, run["ws"])

    @staticmethod
    def _run(M, N, terms, g):
        kept = [t for t in terms if t[0] != 0.0]
        kept = kept or [terms[-1]]
        gen = any(t[2] for t in kept)
        kt = sum(_cdiv(t[1], BK) for t in kept)
        cfg, nsplit = choose_cfg(M, N, kt)
        if gen and cfg < 5:
            cfg, nsplit = 5, split_for(_cdiv(M, 128) * _cdiv(N, 128), SM, kt)
        bm, bn = CFG[cfg][:2]
        tm, tn = _cdiv(M, bm), _cdiv(N, bn)
        if _TUNE["split"] > 0:
            nsplit = _TUNE["split"]
        nsplit = max(1, min(nsplit, kt))
        nsplit = _cdiv(kt, _cdiv(kt, nsplit))
        r = dict(cfg=cfg, nsplit=nsplit, kt=kt, tiles=(tm, tn), nterms=len(kept),
                 band=cfg >= 5 and not gen and not _bits_of("no_band") and tm > RASTER_BAND and tn > RASTER_BAND)
        if gen:
            # launch_ws: index map, plane-wave vectors and lin[] in shared memory if they fit next to
            # the ring; the walker needs them there and K = (s fastest, r)
            n_orb = g.model.n_orb
            extra = 24 * n_orb + 4 * ((2 * g.model.imax + 1) ** 3 + 1 + n_orb)
            r["map_smem"] = ws_smem_bytes(WS_STAGES[cfg], len(kept)) + extra <= MAX_SMEM
            r["walk"] = r["map_smem"] and tuple(g.k_ord) == (3, 2) and not _bits_of("no_walk")
        il = (cfg == 0) != (_force() >= 0 and bool(_force() & 8))
        name = _kernel(cfg, il)
        tail = tail_plan(cfg, nsplit, M, N, kt, tm * tn)
        r["tail"] = tail
        if tail:
            r["kernels"] = [name, name, "tail_reduce_kernel"]
            r["ws"] = 8 * tail[1] * tail[2] * 128 * 128
            r["windows"] = 1
        else:
            w = panel_ktiles(cfg, nsplit, M, N, kt)
            r["windows"] = _cdiv(kt, w)
            r["kernels"] = [name] * r["windows"] + (["splitk_reduce_kernel"] if nsplit > 1 else [])
            r["ws"] = 8 * nsplit * M * N if nsplit > 1 else 0
        return r


def kfast(nk, kstr, kext, nx, xstr):
    if nk == 0:
        return False
    ks = abs(kstr[0])
    if nx == 0:
        return True
    xs = abs(xstr[0])
    if ks == 1 and kext[0] > 1:
        return xs != 1
    return ks < xs


def b_vec2(ptr, k_ext, b_kstr, n_ext, b_nstr):
    if _bits_of("no_vec2") or not n_ext or not k_ext or kfast(len(k_ext), b_kstr, k_ext, len(n_ext), b_nstr):
        return False
    if ptr % 16:
        return False
    dense = 1
    for e, s in zip(n_ext, b_nstr):
        if s != dense:
            return False
        dense *= e
    return all(s % 2 == 0 for s in b_kstr)


# --------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------
_NAMED = []          # the kernels the running case expected


def _bk():
    from pymes_b200 import backend as bk
    return bk


def _lib():
    from pymes_b200 import _lib
    return _lib


def _tune(cfg, split=0):
    _TUNE["cfg"], _TUNE["split"] = cfg, split
    _lib().load().pmb_contract_set_tuning(cfg, split)


def _panel(nbytes):
    _TUNE["panel"] = PANEL_DEFAULT if nbytes < 0 else nbytes
    _TUNE["panel_ws"] = PANEL_DEFAULT_WS if nbytes < 0 else nbytes
    _lib().load().pmb_contract_set_panel_bytes(nbytes)


def _launch(abi, want, fn):
    """Run ``fn``.  On the device the profiler must record exactly the kernels ``want`` of this
    library, and the launch counter must move by their number."""
    _NAMED.extend(want)
    if abi is not None:
        return fn()
    from torch.profiler import ProfilerActivity, profile
    bk = _bk()
    torch.cuda.synchronize()
    before = bk.launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    got = []
    for e in prof.events():
        m = re.search(r"pmb::(\w+(?:<[^()]*>)?)\(", e.name)
        if m:
            got.append(m.group(1).replace(" ", ""))
    assert sorted(got) == sorted(k.replace(" ", "") for k in want), (got, want)
    assert bk.launch_count() - before == len(want)
    return res


def _ints(rng, shape, hi=7):
    return rng.integers(-hi, hi + 1, shape).astype(np.float64)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(got, want):
    """Bit for bit, except the sign of an exact zero (alpha * (+0) keeps alpha's sign in the
    kernels' epilogue, numpy's sum of terms starts from +0)."""
    assert got.shape == want.shape
    got, want = got + 0.0, want + 0.0
    diff = _bits(got) != _bits(want)
    assert not diff.any(), "%d of %d elements differ, first at %s: %r vs %r" % (
        diff.sum(), diff.size, np.argwhere(diff)[0], got[tuple(np.argwhere(diff)[0])],
        want[tuple(np.argwhere(diff)[0])])


def _order(kind, na, nb):
    """Memory order (axes slowest first) of an operand with ``na`` leading and ``nb`` trailing
    axes: ``"a"`` makes the first leading axis unit-stride, ``"b"`` the first trailing one."""
    lead, trail = list(range(na))[::-1], list(range(na, na + nb))[::-1]
    return trail + lead if kind == "a" else lead + trail


class Op:
    """A tensor of logical shape ``val.shape`` placed in a flat buffer of ``fill`` (NaN for
    operands, sentinels for outputs): memory order ``order`` (axes slowest first), ``pad``
    elements of pitch padding after the innermost axis, strides times ``gap`` (NaN between the
    elements), ``off`` elements in, and negative strides along the axes ``neg``."""

    def __init__(self, abi, val, order, pad=0, gap=1, off=0, neg=(), fill=NAN):
        self.val = np.asarray(val, dtype=np.float64)
        ext = self.val.shape
        st, acc = [0] * len(ext), 1
        for k, d in enumerate(reversed(order)):
            st[d] = acc
            acc *= ext[d] + (pad if k == 0 else 0)
        st = [s * gap for s in st]
        base = off
        for d in neg:
            base += (ext[d] - 1) * st[d]
            st[d] = -st[d]
        span = off + 1 + sum((e - 1) * abs(s) for e, s in zip(ext, st)) + 2 + pad
        flat = np.full(span, fill)
        self._view(flat, base, st)[...] = self.val
        self.st, self.base, self.ext = st, base, ext
        t = torch.from_numpy(flat)
        self.t = t.clone() if abi is not None else t.to(_bk().device())
        self.ptr = self.t.data_ptr() + 8 * base
        self.flat0 = flat

    def _view(self, flat, base, st):
        return np.lib.stride_tricks.as_strided(flat[base:], shape=self.val.shape, strides=tuple(8 * s for s in st))

    def mat(self, nrow):
        rows = int(np.prod(self.val.shape[:nrow]))
        return self.val.reshape(rows, -1, order="F")

    def expect(self, new):
        """The buffer after its view is overwritten by ``new`` (same shape as val)."""
        flat = self.flat0.copy()
        self._view(flat, self.base, self.st)[...] = new
        return flat

    def now(self):
        return self.t.detach().cpu().numpy()


class Gen:
    """A generated A operand: a VirtualBlock of ``model`` whose compressed values are replaced by
    the integers ``nz`` at the partner positions (NaN elsewhere on the device; the emulator asserts
    zeros there), or with ``nz = None`` and the pair tables ``tables`` (the kernel evaluates the
    integral formula).  ``m_ord`` / ``k_ord``: the block's axes (0-3 = p, q, r, s) in the M / K
    groups, first listed fastest."""

    def __init__(self, abi, model, lo, ext, m_ord, k_ord, rng=None, tables=None, dense=None):
        from pymes_b200.model import ueg
        bk = _bk()
        self.model, self.lo, self.ext, self.m_ord, self.k_ord = model, tuple(lo), tuple(ext), m_ord, k_ord
        if tables is None:
            tables = (bk.zeros(model.n_orb, model.n_orb), None, None)
        self.virt = ueg.VirtualBlock(model, lo, ext, *tables, compressed=False)
        s, ok = self.partners()
        if rng is not None:
            nz = np.where(ok, _ints(rng, ext[:3]), 0.0)
            blk = np.zeros(ext)
            P, Q, R = np.nonzero(ok)
            blk[P, Q, R, s[ok] - lo[3]] = nz[ok]
            self.virt.nz = torch.from_numpy(np.where(ok, nz, NAN if abi is None else 0.0)).to(bk.device())
            self.blk = blk
        else:
            self.blk = dense
        self.desc = self.virt.gen_descriptor("pqrs", ["pqrs"[a] for a in m_ord], ["pqrs"[a] for a in k_ord])

    def partners(self):
        """s*(p, q, r) of the block's rows, and whether it lies in the block (the kernel's test:
        flattened bounds check on the index map, then the s range)."""
        m, lo, ext = self.model, self.lo, self.ext
        k = m.k_int().astype(np.int64)
        n = 2 * m.imax + 1
        P, Q, R = np.meshgrid(*[np.arange(lo[d], lo[d] + ext[d]) for d in range(3)], indexing="ij")
        v = k[Q] - (k[R] - k[P]) + m.imax
        loc = n * n * v[..., 0] + n * v[..., 1] + v[..., 2]
        inside = (loc >= 0) & (loc < n ** 3)
        s = np.where(inside, m.basis_indices_map[np.clip(loc, 0, n ** 3 - 1)], -1)
        return s, inside & (s >= lo[3]) & (s < lo[3] + ext[3])

    def mat(self):
        axes = list(self.m_ord) + list(self.k_ord)
        M = int(np.prod([self.ext[a] for a in self.m_ord]))
        return np.transpose(self.blk, axes).reshape(M, -1, order="F")


def _gemm(abi, rng, m_ext, n_ext, terms, beta=0.0, c_kind="b", c_pad=0, c_neg=(), c_gap=1, real=False,
          check=None):
    """One pmb_contract call.  ``terms``: dicts with alpha, k_ext and the layouts of A and B
    (a_kind / b_kind "a" or "b" for the unit-stride group, a_pad, a_gap, a_off, a_neg, the same for
    b, b_zero for an all-zero B) or gen = a Gen.  Checks bits (or the bound with ``real``), the
    workspace, the kernels, the sentinels; returns the plan."""
    lib, bk = _lib(), _bk()
    nm, nn = len(m_ext), len(n_ext)
    draw = (lambda shape: rng.standard_normal(shape)) if real else (lambda shape: _ints(rng, shape))
    M, N = int(np.prod(m_ext)), int(np.prod(n_ext))
    d = lib.Contract()
    d.nm, d.nn, d.nterms = nm, nn, len(terms)
    for i in range(nm):
        d.m_ext[i] = m_ext[i]
    for i in range(nn):
        d.n_ext[i] = n_ext[i]
    ref = np.zeros((M, N), dtype=np.longdouble if real else np.float64)
    mag = np.zeros((M, N))
    keep, spec = [], []
    for i, t in enumerate(terms):
        k_ext = list(t["k_ext"])
        nk = len(k_ext)
        T = d.terms[i]
        T.nk, T.alpha = nk, t["alpha"]
        for j in range(nk):
            T.k_ext[j] = k_ext[j]
        if "gen" in t:
            g = t["gen"]
            T.A, T.a_gen = None, C.addressof(g.desc)
            A = g.mat()
            keep.append(g)
        else:
            a = Op(abi, draw(list(m_ext) + k_ext), t.get("a_order") or _order(t.get("a_kind", "b"), nm, nk),
                   t.get("a_pad", 0), t.get("a_gap", 1), t.get("a_off", 0), t.get("a_neg", ()))
            T.A = a.ptr
            for j in range(nm):
                T.a_mstr[j] = a.st[j]
            for j in range(nk):
                T.a_kstr[j] = a.st[nm + j]
            A = a.mat(nm)
            keep.append(a)
        bval = np.zeros(k_ext + list(n_ext)) if t.get("b_zero") else draw(k_ext + list(n_ext))
        b = Op(abi, bval, t.get("b_order") or _order(t.get("b_kind", "b"), nk, nn), t.get("b_pad", 0),
               t.get("b_gap", 1), t.get("b_off", 0), t.get("b_neg", ()))
        T.B = b.ptr
        for j in range(nk):
            T.b_kstr[j] = b.st[j]
        for j in range(nn):
            T.b_nstr[j] = b.st[nk + j]
        keep.append(b)
        t["vec2"] = b_vec2(b.ptr, k_ext, b.st[:nk], list(n_ext), b.st[nk:])
        Bm = b.mat(nk)
        if real:
            ref += np.longdouble(t["alpha"]) * (A.astype(np.longdouble) @ Bm.astype(np.longdouble))
            mag += abs(t["alpha"]) * (np.abs(A) @ np.abs(Bm))
        elif t["alpha"] != 0.0:
            ref = ref + t["alpha"] * (A @ Bm)
        spec.append((t["alpha"], int(np.prod(k_ext)), "gen" in t))
    old = np.full(list(m_ext) + list(n_ext), NAN) if beta == 0.0 else _ints(rng, list(m_ext) + list(n_ext))
    c = Op(abi, old, _order(c_kind, nm, nn), c_pad, c_gap, 3, c_neg, fill=SENT)
    d.C, d.beta = c.ptr, beta
    for j in range(nm):
        d.c_mstr[j] = c.st[j]
    for j in range(nn):
        d.c_nstr[j] = c.st[nm + j]
    g = next((t["gen"] for t in terms if "gen" in t), None)
    plan = Plan(M, N, spec, g)
    if check is not None:
        check(plan)
    need = lib.load().pmb_contract_workspace(C.byref(d))
    ws = torch.empty(max(need, 8) // 8, dtype=torch.float64, device=bk.device())
    if abi is None:
        assert need == plan.ws, (need, plan.ws)
        if need:
            before = bk.launch_count()
            assert lib.load().pmb_contract(C.byref(d), bk._ptr(ws), need - 1, bk._stream()) == -2
            assert bk.launch_count() == before
    rc = _launch(abi, plan.kernels, lambda: lib.load().pmb_contract(C.byref(d), bk._ptr(ws), need, bk._stream()))
    assert rc == 0, rc
    got = c.now()
    if real:
        fin = ref + (np.longdouble(beta) * c.mat(nm) if beta != 0.0 else 0)
        new = c._view(got, c.base, c.st)
        gm = new.reshape(M, N, order="F")
        tol = 2.0 * max(sum(s[1] for s in spec), 1) * EPS * (mag + abs(beta) * np.abs(c.mat(nm)))
        assert (np.abs(gm - fin.astype(np.float64)) <= tol).all()
        outside = np.ones(got.size, dtype=bool)
        outside[c._view(np.arange(got.size, dtype=np.int64), c.base, c.st).reshape(-1)] = False
        _same(got[outside], c.flat0[outside])
    else:
        want = ref + (beta * c.mat(nm) if beta != 0.0 else 0.0)
        _same(got, c.expect(want.reshape(c.val.shape, order="F")))
    del keep
    return plan


def _t(alpha, k_ext, **kw):
    return dict(alpha=alpha, k_ext=k_ext, **kw)


# --------------------------------------------------------------------------
# cases
# --------------------------------------------------------------------------
def _case_tile_configs(abi):
    """Forced configurations 0-6, each with and without +8, at M, N of 1, BM/BN +- 1 and 2 BM + 1
    and K of 1, 15, 16, 17 and 33; outer products (nk = 0), a scalar side (nm or nn = 0); the
    heuristic with its choice predicted; one random-valued case per kernel family."""
    rng = np.random.default_rng(21)
    for cfg in range(NUM_CFG):
        bm, bn = CFG[cfg][:2]
        shapes = [(1, 1, 1), (bm - 1, bn + 1, 15), (bm + 1, bn - 1, 16), (2 * bm + 1, 1, 17),
                  (1, 2 * bn + 1, 33), (bm, bn, 33)]
        for flip in (0, 8):
            _tune(cfg + flip, 0)
            for i, (M, N, K) in enumerate(shapes):
                p = _gemm(abi, rng, [M], [N], [_t((1.0, -2.0, 0.5)[i % 3], [K], a_kind="ab"[i % 2],
                                                 b_kind="ab"[(i // 2) % 2])], beta=(0.0, 1.0, -0.5)[(i + flip) % 3])
                assert p.runs[0]["cfg"] == cfg
        _tune(cfg, 0)
        _gemm(abi, rng, [bm + 3], [bn - 5], [_t(2.0, [])], beta=0.0)                        # outer product
        _gemm(abi, rng, [], [bn + 7], [_t(-1.0, [37], a_kind="b")], beta=1.0)             # one row
        _gemm(abi, rng, [bm + 9], [], [_t(0.5, [37], b_kind="a")], beta=0.0)              # one column
        _gemm(abi, rng, [5, 7], [3, 11], [_t(1.0, [4, 5])], beta=4.0)
    _tune(-1, 0)
    for M, N, K in ((3, 4, 5), (300, 200, 40), (1000, 700, 50), (2000, 1500, 24), (77, 4000, 16), (64, 64, 3000)):
        _gemm(abi, rng, [M], [N], [_t(1.0, [K])], beta=0.0)
    _tune(2, 1)
    _gemm(abi, rng, [150], [130], [_t(1.0, [1000])], beta=-0.5, real=True)
    _tune(5, 1)
    _gemm(abi, rng, [150], [130], [_t(1.0, [1000])], beta=-0.5, real=True)


def _case_ragged_ws_widths(abi):
    """cfg 5 and 6: both ends of each per-warp column width class of the last column tile (N mod
    128 in 1-16, 17-32, 33-64, 65-96, 97-128) and every active warp-row count of the last row tile
    (M mod 128 in 1, 32, 33, 64, 65, 96, 97, 128)."""
    rng = np.random.default_rng(22)
    nr = (1, 16, 17, 32, 33, 64, 65, 96, 97, 128)
    mr = (1, 32, 33, 64, 65, 96, 97, 128)
    for cfg in (5, 6):
        _tune(cfg, 1)
        for i, r in enumerate(nr):
            _gemm(abi, rng, [128 + mr[(i + cfg) % len(mr)]], [128 + r], [_t(-1.0, [40], a_kind="ab"[i % 2])],
                  beta=(0.0, 2.0)[i % 2])


def _case_multi_term(abi):
    """2-8 terms with K not a multiple of 16 and negative power-of-two alphas; an alpha = 0 term
    first, in the middle, last, and all of them; forced splits whose boundaries fall inside a
    term and on a term boundary."""
    rng = np.random.default_rng(23)
    Ks = [17, 33, 5, 49, 1, 70, 23, 15]
    for cfg in (2, 5):
        _tune(cfg, 1)
        for nt in range(2, 9):
            terms = [_t((-1.0) ** i * 2.0 ** (i % 5 - 2), [Ks[i]], a_kind="ab"[i % 2]) for i in range(nt)]
            p = _gemm(abi, rng, [70], [130], terms, beta=(0.0, 1.0)[nt % 2])
            assert p.runs[0]["nterms"] == nt and len(p.runs) == 1
        for zeros in ((0,), (1,), (2,), (0, 1, 2)):
            terms = [_t(0.0 if i in zeros else -2.0 ** i, [Ks[i + 1]]) for i in range(3)]
            p = _gemm(abi, rng, [70], [45], terms, beta=0.0)
            assert p.runs[0]["nterms"] == (1 if len(zeros) == 3 else 2)
        for split in (2, 3, 8):
            # k-tiles per term (3, 3, 2): split 3 cuts on the term boundaries, 2 inside term 1, 8 everywhere
            _tune(cfg, split)
            _gemm(abi, rng, [70], [45], [_t(0.5, [33]), _t(-4.0, [40], b_kind="a"), _t(0.25, [20])], beta=-0.5)


def _case_split_k(abi):
    """Forced splits 2, 3, 7, exactly kt and more than kt (clamped); a heuristic split; beta 0 over
    NaN, 1, -0.5 and 4; the workspace is exact (one byte less is refused without a launch)."""
    rng = np.random.default_rng(24)
    for cfg in (2, 0, 5):
        for i, split in enumerate((2, 3, 7, 41, 50)):
            _tune(cfg, split)
            p = _gemm(abi, rng, [70], [45], [_t(1.0, [16 * 40 + 3], a_kind="ab"[i % 2])],
                      beta=(0.0, 1.0, -0.5, 4.0)[i % 4])
            assert p.runs[0]["nsplit"] == min(split, 41) and p.ws == 8 * min(split, 41) * 70 * 45
    _tune(-1, 0)
    for beta in (0.0, 4.0):
        p = _gemm(abi, rng, [64], [64], [_t(1.0, [5000])], beta=beta)
        assert p.runs[0]["nsplit"] > 1


def _case_k_windows(abi):
    """set_panel_bytes(1) on cfg 0-4 and on cfg 5: the windows the mirror predicts, with edges that
    do not align with the term edge; windows are off when split-K is on."""
    rng = np.random.default_rng(25)
    _panel(1)
    for cfg in range(6):
        _tune(cfg, 1)
        p = _gemm(abi, rng, [70], [50], [_t(1.0, [1000]), _t(-0.5, [1407], a_kind="a")], beta=(0.0, 1.0)[cfg % 2])
        assert p.runs[0]["windows"] == 3
        _tune(cfg, 0)
        p = _gemm(abi, rng, [40], [40], [_t(1.0, [2407])], beta=0.0)
        assert p.runs[0]["nsplit"] > 1 and p.runs[0]["windows"] == 1


def _case_tail_and_band(abi):
    """The tail cut at 148 + 1 and 148 + 74 tiles (cut) and 2 x 148 + 75 and < 148 (not cut), kt 63
    vs 64, a split clamped by kt / 16; the banded order with a ragged last band and at tiles_m or
    tiles_n = 12 (off) vs 13 (on); +64 and +256; C stored transposed; band and tail together."""
    rng = np.random.default_rng(26)
    _tune(5, 0)
    p = _gemm(abi, rng, [149 * 128 - 3], [7], [_t(1.0, [1030])], beta=0.0)
    assert p.runs[0]["tail"] == (148, 1, 4)                           # 148 / 1 clamped by kt / 16 = 4
    p = _gemm(abi, rng, [37 * 128 - 5], [6 * 128 - 9], [_t(-1.0, [1030])], beta=1.0, c_kind="a")
    assert p.runs[0]["tail"] == (148, 74, 2)
    p = _gemm(abi, rng, [37 * 128 - 5], [6 * 128 - 9], [_t(1.0, [1009])], beta=0.0)
    assert p.runs[0]["kt"] == 64 and p.runs[0]["tail"]
    p = _gemm(abi, rng, [37 * 128 - 5], [6 * 128 - 9], [_t(1.0, [1008])], beta=0.0)
    assert p.runs[0]["kt"] == 63 and not p.runs[0]["tail"]
    p = _gemm(abi, rng, [7 * 128], [53 * 128 - 1], [_t(0.5, [1030], a_kind="a")], beta=0.0)
    assert p.runs[0]["tiles"] == (7, 53) and not p.runs[0]["tail"]
    p = _gemm(abi, rng, [10 * 128], [10 * 128 - 1], [_t(1.0, [1030])], beta=0.0)
    assert not p.runs[0]["tail"]
    _tune(5 + 64, 0)
    p = _gemm(abi, rng, [37 * 128 - 5], [6 * 128 - 9], [_t(1.0, [1030])], beta=-0.5)
    assert not p.runs[0]["tail"]
    # band order
    for cfg in (5, 6, 5 + 256):
        _tune(cfg, 0)
        for tm, tn in ((13, 13), (12, 13), (13, 12), (25, 14)):
            p = _gemm(abi, rng, [tm * 128 - 7], [tn * 128 - 3], [_t(1.0, [40])], beta=(0.0, 1.0)[tm % 2],
                      c_kind="ab"[tn % 2])
            assert p.runs[0]["band"] == (cfg < 256 and tm > 12 and tn > 12)
    _tune(5, 0)
    p = _gemm(abi, rng, [13 * 128 - 7], [13 * 128 - 3], [_t(1.0, [1030])], beta=1.0, c_kind="a")
    assert p.runs[0]["band"] and p.runs[0]["tail"] == (148, 21, 4)


def _case_copy_mappings(abi):
    """16-byte copies of B: eligible, then ineligible by a misaligned base, an odd k stride, a
    non-dense N group and nk = 0; +128 gives the same bits.  Operands unit-stride along k, along
    m / n, or along neither; negative strides on A, B and C."""
    rng = np.random.default_rng(27)
    for cfg in (5, 6, 0):
        _tune(cfg, 1)
        for N, pad, off, want in ((64, 0, 0, True), (37, 1, 0, True), (37, 1, 1, False), (37, 0, 0, False)):
            for no_vec2 in (0, 128):
                _tune(cfg + no_vec2, 1)
                terms = [_t(1.0, [40], b_kind="b", b_pad=pad, b_off=off)]
                _gemm(abi, rng, [150], [N], terms, beta=0.0)
                assert terms[0]["vec2"] == (want and not no_vec2)
        _tune(cfg, 1)
        terms = [_t(1.0, [24], b_order=[0, 2, 1], b_pad=1)]                 # N group (5, 7), gap in n1
        _gemm(abi, rng, [130], [5, 7], terms, beta=1.0)
        assert not terms[0]["vec2"]
        terms = [_t(1.0, [24], b_gap=2)]
        _gemm(abi, rng, [130], [33], terms, beta=1.0)
        assert not terms[0]["vec2"]
        terms = [_t(-1.0, [], b_kind="b")]
        _gemm(abi, rng, [130], [64], terms, beta=0.0)
        assert not terms[0]["vec2"]
        for ak in ("a", "b"):
            for bk_ in ("a", "b"):
                _gemm(abi, rng, [131], [67], [_t(2.0, [35], a_kind=ak, b_kind=bk_)], beta=0.0)
        _gemm(abi, rng, [131], [67], [_t(2.0, [35], a_gap=2, b_gap=3, a_pad=1)], beta=-0.5, c_gap=2)
        _gemm(abi, rng, [131], [67], [_t(1.0, [35], a_neg=(0, 1), b_neg=(1,))], beta=1.0, c_neg=(0,))
        _gemm(abi, rng, [5, 27], [3, 23], [_t(1.0, [7, 3], a_kind="a", a_neg=(1, 2), b_neg=(0, 3))], beta=0.0,
              c_neg=(1, 2), c_kind="a")


def _ueg_model(cutoff):
    from pymes_b200.model import ueg
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(cutoff)
    return m


def _case_generated(abi):
    """A generated A operand with integer compressed values: the walker (K = (s, r)) and the
    scanner (+16, the other K order, s in the M group); ext_s of 1, 5, 15, 16, 17 and 70; row blocks
    with lo != 0 and a ragged last row tile; split-K starting inside the generated term; the
    generated term after and before a stored one; k windows; a tail launch and +32."""
    bk = _bk()
    was = bk.set_blocked(False)
    try:
        rng = np.random.default_rng(28)
        m = _ueg_model(9.0)
        nP = m.n_orb
        assert nP == 117

        def gen(lo, ext, m_ord=(0, 1), k_ord=(3, 2)):
            return Gen(abi, m, lo, ext, m_ord, k_ord, rng=rng)

        for i, (ext_s, lo_s) in enumerate(((1, 50), (5, 7), (15, 20), (16, 0), (17, 33), (70, 40))):
            _tune(5 + 64, 0)
            g = gen((3, 10, 0, lo_s), (10, 15, nP, ext_s), m_ord=((0, 1), (1, 0))[i % 2])
            p = _gemm(abi, rng, [10, 15] if i % 2 == 0 else [15, 10], [37], [_t(1.0, [ext_s, nP], gen=g)],
                      beta=(0.0, 1.0)[i % 2])
            assert p.runs[0]["map_smem"] and p.runs[0]["walk"]
            _tune(5 + 64 + 16, 0)                                          # the scanner on the same operand
            p = _gemm(abi, rng, [10, 15] if i % 2 == 0 else [15, 10], [37], [_t(-2.0, [ext_s, nP], gen=g)], beta=0.0)
            assert p.runs[0]["map_smem"] and not p.runs[0]["walk"]
        _tune(6 + 64, 0)
        g = gen((3, 10, 0, 30), (10, 15, nP, 17))
        _gemm(abi, rng, [10, 15], [37], [_t(1.0, [17, nP], gen=g)], beta=0.0)
        _tune(5 + 64, 0)
        g = gen((3, 10, 5, 30), (10, 15, 100, 17), k_ord=(2, 3))               # K = (r, s): scanner
        p = _gemm(abi, rng, [10, 15], [37], [_t(1.0, [100, 17], gen=g)], beta=0.0)
        assert not p.runs[0]["walk"]
        g = gen((0, 0, 40, 50), (20, 30, 10, 15), m_ord=(2, 3), k_ord=(0, 1))  # s in the M group
        p = _gemm(abi, rng, [10, 15], [37], [_t(1.0, [20, 30], gen=g)], beta=0.0)
        assert not p.runs[0]["walk"]
        # split-K inside the generated term, after a stored term; the generated term first
        g = gen((3, 10, 0, 40), (10, 15, nP, 70))
        for split in (3, 7):
            _tune(5 + 64, split)
            _gemm(abi, rng, [10, 15], [37], [_t(0.5, [40]), _t(1.0, [70, nP], gen=g)], beta=0.0)
        _tune(5 + 64, 1)
        _gemm(abi, rng, [10, 15], [37], [_t(1.0, [70, nP], gen=g), _t(-1.0, [40], a_kind="a")], beta=1.0)
        _gemm(abi, rng, [10, 15], [37], [_t(2.0, [24]), _t(1.0, [70, nP], gen=g), _t(-1.0, [40])], beta=0.0)
        # k windows
        _panel(1)
        try:
            p = _gemm(abi, rng, [10, 15], [37], [_t(1.0, [70, nP], gen=g)], beta=0.0)
            assert p.runs[0]["windows"] == 8
        finally:
            _panel(-1)
        # m-fastest tail launch (37 x 6 = 148 + 74 tiles), then +32
        _tune(5, 0)
        g = gen((0, 0, 0, 60), (40, nP, nP, 17))
        p = _gemm(abi, rng, [40, nP], [6 * 128 - 9], [_t(1.0, [17, nP], gen=g)], beta=0.0)
        assert p.runs[0]["tail"] == (148, 74, 2)
        _tune(5 + 32 + 64, 2)
        _gemm(abi, rng, [10, 15], [37], [_t(1.0, [17, nP], gen=gen((3, 10, 0, 30), (10, 15, nP, 17)))], beta=1.0)
    finally:
        bk.set_blocked(was)


def _case_generated_fallback(abi):
    """The global-map producer: the 14-electron model (57 plane waves) with imax raised to 14 and 27,
    so the index map does not fit in shared memory next to the ring.  Integer values (walker and
    scanner K orders), and the formula (nz = NULL) bit for bit against the same kernel on the block
    pmb_ueg_build_block writes, and within the bound of a long-double product."""
    bk = _bk()
    was = bk.set_blocked(False)
    try:
        rng = np.random.default_rng(29)
        m = _ueg_model(5.0)
        nP = m.n_orb
        assert nP == 57
        for imax in (14, 27):
            m.imax = imax
            m.init_basis_indices_map()
            m._dev = None
            for cfg in (5 + 64, 6 + 64):
                _tune(cfg, 1)
                for k_ord in ((3, 2), (2, 3)):
                    g = Gen(abi, m, (2, 0, 0, 0), (6, 25, nP, nP), (0, 1), k_ord, rng=rng)
                    p = _gemm(abi, rng, [6, 25], [37], [_t(1.0, [nP, nP], gen=g)], beta=0.0)
                    assert p.runs[0]["map_smem"] is False and not p.runs[0]["walk"]
            W = [bk.asdev(rng.standard_normal((nP, nP))) for _ in range(3)]
            raw = Gen(abi, m, (2, 0, 0, 0), (6, 25, nP, nP), (0, 1), (3, 2), tables=W)
            dense = raw.virt.materialise()
            raw.blk = dense.cpu().numpy()
            assert np.count_nonzero(raw.blk) > 0
            _tune(5 + 64, 1)
            Bv = rng.standard_normal((nP, nP, 37))
            outs = []
            for A in (raw, dense):
                out = bk.empty(6, 25, 37).fill_(NAN)
                d = _lib().Contract()
                d.nm, d.nn, d.nterms, d.C, d.beta = 2, 1, 1, out.data_ptr(), 0.0
                d.m_ext[0], d.m_ext[1], d.n_ext[0], d.c_mstr[0], d.c_mstr[1], d.c_nstr[0] = 6, 25, 37, 25 * 37, 37, 1
                T = d.terms[0]
                T.nk, T.alpha, T.k_ext[0], T.k_ext[1] = 2, 1.0, nP, nP
                B = bk.asdev(Bv)                                        # [s, r, n] -> K = (s, r): strides nP*37, 37
                T.B, T.b_kstr[0], T.b_kstr[1], T.b_nstr[0] = B.data_ptr(), nP * 37, 37, 1
                if A is raw:
                    T.A, T.a_gen = None, C.addressof(raw.desc)
                    plan = Plan(150, 37, [(1.0, nP * nP, True)], raw)
                    assert plan.runs[0]["map_smem"] is False
                else:
                    T.A = A.data_ptr()                                  # [p, q, r, s]
                    T.a_mstr[0], T.a_mstr[1], T.a_kstr[0], T.a_kstr[1] = 25 * nP * nP, nP * nP, 1, nP
                    plan = Plan(150, 37, [(1.0, nP * nP, False)])
                rc = _launch(abi, plan.kernels, lambda: _lib().load().pmb_contract(C.byref(d), None, 0, bk._stream()))
                assert rc == 0
                outs.append(out.cpu().numpy())
            _same(outs[0], outs[1])
            Am = raw.blk.reshape(150, -1)                                  # rows (p, q), K = (r, s) s fastest
            Bm = np.transpose(Bv, (1, 0, 2)).reshape(-1, 37)
            ref = Am.astype(np.longdouble) @ Bm.astype(np.longdouble)
            tol = 2.0 * nP * nP * EPS * (np.abs(Am) @ np.abs(Bm))
            assert (np.abs(outs[0].reshape(150, 37) - ref.astype(np.float64)) <= tol).all()
    finally:
        bk.set_blocked(was)


def _case_argument_errors(abi):
    """Malformed descriptors return an error and launch nothing: 0 or 9 terms, nm = 5, a zero
    extent, M >= 2^31 and null pointers give -1; two generated terms, imax = 28 and n_orb = 2048
    give -3; a repeated or missing axis and lo + ext > n_orb give -1.  (Device only: the emulated
    ABI does not validate.)"""
    lib, bk = _lib(), _bk()
    buf = bk.zeros(64)
    m = _ueg_model(2.0)
    nP = m.n_orb
    g = Gen(abi, m, (0, 0, 0, 0), (nP, nP, nP, nP), (0, 1), (3, 2), rng=np.random.default_rng(1))

    def good():
        d = lib.Contract()
        d.nm, d.nn, d.nterms, d.C = 1, 1, 1, buf.data_ptr()
        d.m_ext[0] = d.n_ext[0] = 4
        d.c_mstr[0], d.c_nstr[0] = 4, 1
        T = d.terms[0]
        T.A, T.B, T.nk, T.alpha, T.k_ext[0] = buf.data_ptr(), buf.data_ptr(), 1, 1.0, 4
        T.a_mstr[0] = T.a_kstr[0] = 1
        T.b_kstr[0] = T.b_nstr[0] = 1
        return d

    def gen_term(d, i, desc):
        d.nm = 2
        d.m_ext[0] = d.m_ext[1] = nP
        T = d.terms[i]
        T.A, T.B, T.a_gen, T.nk, T.alpha = None, buf.data_ptr(), C.addressof(desc), 2, 1.0
        T.k_ext[0] = T.k_ext[1] = nP
        T.b_kstr[0] = T.b_kstr[1] = 0
        return d

    def copy_desc(mod):
        desc = _lib().UegOperand.from_buffer_copy(g.desc)
        mod(desc)
        keep.append(desc)
        return desc

    keep = []
    bad = []
    for mod, rc in ((lambda d: setattr(d, "nterms", 0), -1), (lambda d: setattr(d, "nterms", 9), -1),
                    (lambda d: setattr(d, "nm", 5), -1), (lambda d: d.n_ext.__setitem__(0, 0), -1),
                    (lambda d: (setattr(d, "nm", 2), d.m_ext.__setitem__(0, 1 << 16), d.m_ext.__setitem__(1, 1 << 15)), -1),
                    (lambda d: setattr(d, "C", None), -1), (lambda d: setattr(d.terms[0], "B", None), -1),
                    (lambda d: setattr(d.terms[0], "A", None), -1),
                    (lambda d: setattr(d.terms[0], "nk", 5), -1)):
        d = good()
        mod(d)
        bad.append((d, rc))
    d = gen_term(good(), 0, g.desc)
    d.nterms = 2
    gen_term(d, 1, g.desc)
    bad.append((d, -3))
    for field, value, rc in (("imax", 28, -3), ("n_orb", 2048, -3)):
        bad.append((gen_term(good(), 0, copy_desc(lambda x: setattr(x.ueg, field, value))), rc))
    bad.append((gen_term(good(), 0, copy_desc(lambda x: x.k_axis.__setitem__(0, 0))), -1))     # p twice
    d = gen_term(good(), 0, g.desc)
    d.terms[0].nk = 1                                                                          # r missing
    bad.append((d, -1))
    bad.append((gen_term(good(), 0, copy_desc(lambda x: x.k_axis.__setitem__(1, -1))), -1))    # no axis
    bad.append((gen_term(good(), 0, copy_desc(lambda x: x.lo.__setitem__(3, 1))), -1))         # s past n_orb
    if abi is not None:
        return
    before = bk.launch_count()
    for d, rc in bad:
        assert lib.load().pmb_contract(C.byref(d), None, 0, bk._stream()) == rc
        assert lib.load().pmb_contract_workspace(C.byref(d)) == 0
    torch.cuda.synchronize()
    assert bk.launch_count() == before
    d = good()                                          # and the well-formed one goes through
    assert lib.load().pmb_contract(C.byref(d), None, 0, bk._stream()) == 0
    assert bk.launch_count() == before + 1


def _case_coefficient_range(abi):
    """Alphas 2^600 and 2^-600, and 2^-600 with 2^500 over a zero B: the result equals
    a0 (A0 B0) + a1 (A1 B1) bit for bit, with no inf or NaN.  The terms go in two coefficient
    runs, each with its own plan."""
    rng = np.random.default_rng(30)
    for cfg, split in ((-1, 0), (2, 0), (5, 0), (2, 3), (5, 3)):
        _tune(cfg, split)
        for a0, a1, zero in ((2.0 ** 600, 2.0 ** -600, False), (2.0 ** -600, 2.0 ** 500, True),
                             (-(2.0 ** 30), 2.0 ** -8, False)):
            p = _gemm(abi, rng, [40], [70], [_t(a0, [20]), _t(a1, [37], b_zero=zero, a_kind="a")], beta=0.0)
            assert len(p.runs) == (1 if a1 == 2.0 ** -8 else 2)
        p = _gemm(abi, rng, [40], [70], [_t(2.0 ** 600, [20]), _t(0.0, [5]), _t(2.0 ** 560, [9]),
                                         _t(2.0 ** -600, [37]), _t(1.0, [3])], beta=0.0)
        assert [r["nterms"] for r in p.runs] == [2, 1, 1]


CASES = {
    _case_tile_configs: ALL_KERNELS - {"tail_reduce_kernel"},
    _case_ragged_ws_widths: {_kernel(5, False), _kernel(6, False)},
    _case_multi_term: {_kernel(2, False), _kernel(5, False), "splitk_reduce_kernel"},
    _case_split_k: None,
    _case_k_windows: None,
    _case_tail_and_band: {_kernel(5, False), _kernel(6, False), "tail_reduce_kernel"},
    _case_copy_mappings: {_kernel(5, False), _kernel(6, False), _kernel(0, True)},
    _case_generated: {_kernel(5, False), _kernel(6, False), "splitk_reduce_kernel", "tail_reduce_kernel"},
    _case_generated_fallback: {_kernel(5, False), _kernel(6, False)},
    _case_argument_errors: set(),
    _case_coefficient_range: None,
}
IDS = [f.__name__[len("_case_"):] for f in CASES]


def _run(case, abi):
    del _NAMED[:]
    try:
        case(abi)
    finally:
        _tune(-1, 0)
        _panel(-1)
    if CASES[case] is not None:
        assert set(_NAMED) == CASES[case], (set(_NAMED) ^ CASES[case])
    else:
        assert _NAMED


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
def test_contract_64bit_offsets_on_the_device():
    """A, B and C as strided views whose element offsets pass 2^31 (rows 2^28 elements apart in one
    buffer of 2^31 + 2^10 doubles): the offset tables, the tile gathers, the split-K and the
    epilogue index with 64-bit arithmetic.  Needs about 17.2 GB of device memory."""
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    from pymes_b200 import _lib as lib, backend as bk
    S, M, N, K = 1 << 28, 9, 9, 40
    rng = np.random.default_rng(31)
    A, B, old = _ints(rng, (M, K)), _ints(rng, (K, N)), _ints(rng, (M, N))
    buf = torch.full(((1 << 31) + (1 << 10),), NAN, dtype=torch.float64, device="cuda")
    rows = torch.arange(M, device="cuda") * S
    cols = torch.arange(N, device="cuda") * S
    # A[m, k] at m S + k, B[k, n] at n S + 100 + k, C[m, n] at m S + 200 + n
    buf[(rows[:, None] + torch.arange(K, device="cuda")[None, :]).reshape(-1)] = torch.from_numpy(A).cuda().reshape(-1)
    buf[(cols[None, :] + 100 + torch.arange(K, device="cuda")[:, None]).reshape(-1)] = \
        torch.from_numpy(B).cuda().reshape(-1)
    c_idx = (rows[:, None] + 200 + torch.arange(N, device="cuda")[None, :]).reshape(-1)
    assert int(c_idx.max()) > (1 << 31)
    d = lib.Contract()
    d.nm, d.nn, d.nterms, d.C, d.beta = 1, 1, 1, buf.data_ptr() + 8 * 200, 1.0
    d.m_ext[0], d.n_ext[0], d.c_mstr[0], d.c_nstr[0] = M, N, S, 1
    T = d.terms[0]
    T.A, T.B, T.nk, T.alpha, T.k_ext[0] = buf.data_ptr(), buf.data_ptr() + 8 * 100, 1, 1.0, K
    T.a_mstr[0], T.a_kstr[0], T.b_kstr[0], T.b_nstr[0] = S, 1, 1, S
    want = old.copy()
    try:
        for cfg, split in ((-1, 0), (2, 0), (5, 0), (2, 3)):
            _tune(cfg, split)
            buf[c_idx] = torch.from_numpy(old).cuda().reshape(-1)
            plan = Plan(M, N, [(1.0, K, False)])
            need = lib.load().pmb_contract_workspace(C.byref(d))
            ws = torch.empty(max(need, 8) // 8, dtype=torch.float64, device="cuda")
            rc = _launch(None, plan.kernels, lambda: lib.load().pmb_contract(C.byref(d), bk._ptr(ws), need, bk._stream()))
            assert rc == 0
            _same(buf[c_idx].cpu().numpy().reshape(M, N), want + A @ B)
        assert torch.isnan(buf[(1 << 31) + 300:]).all()
    finally:
        _tune(-1, 0)
        del buf
        torch.cuda.empty_cache()


# --------------------------------------------------------------------------
# guards
# --------------------------------------------------------------------------
def test_every_instantiation_has_a_case():
    """The cases name every kernel instantiation of the pmb_contract launch switch and both
    second-stage kernels: a configuration added without a case fails here."""
    named = set().union(*[k for k in CASES.values() if k])
    assert named == ALL_KERNELS
    assert len(ALL_KERNELS) == 2 * 5 + 2 + 2


def test_plan_constants_parse():
    """The constants read from the CUDA source have the values the shapes above straddle."""
    assert CFG == [(128, 128, 256, 1.0), (128, 64, 256, 0.9), (64, 64, 128, 1.0), (64, 32, 128, 0.8),
                   (128, 64, 128, 0.9), (128, 128, 384, 1.3), (128, 128, 384, 1.0)]
    assert (NUM_CFG, RASTER_BAND, PANEL_DEFAULT, PANEL_DEFAULT_WS) == (7, 12, 40 << 20, 0)
    assert (SPLIT_MIN_KT, SPLIT_KT_DIV, SPLIT_MAX) == (8, 4, 192)
    assert (TAIL_MIN_KT, TAIL_KT_DIV, TAIL_REST_DIV) == (64, 16, 2)
    assert (MAX_SMEM, WS_KRING, SM, BK, COEF_SPREAD) == (232448, 16, 148, 16, 64)
    assert WS_STAGES == {5: 4, 6: 6}
    # the fallback cases: imax 14 is the first that pushes the 4-stage kernel's map out of shared memory
    extra = lambda imax: 24 * 57 + 4 * ((2 * imax + 1) ** 3 + 1 + 57)
    assert ws_smem_bytes(4, 1) + extra(13) <= MAX_SMEM < ws_smem_bytes(4, 1) + extra(14)


def test_coefficient_runs():
    """The run rule: ordinary coefficients are one run, zero and non-finite ones join any run."""
    assert coef_runs([1.0, -0.5, 2.0 ** 30, 2.0 ** -30]) == [(0, 4)]
    assert coef_runs([2.0 ** 600, 2.0 ** -600]) == [(0, 1), (1, 2)]
    assert coef_runs([0.0, 2.0 ** 64, 0.0, 1.0, 2.0 ** -1]) == [(0, 4), (4, 5)]
    assert coef_runs([0.0, 0.0]) == [(0, 2)]
