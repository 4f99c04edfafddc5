"""Group products of any index split (pmb_group_contract beyond 2 | 2 | 2).

A term whose operands both carry a live momentum rule runs on its momentum groups whatever its
split: r row indices from A, e summed indices, c column indices from B (``backend._group_term``).
A side without indices has one member of label 0.  In the UEG every orbital has its own momentum,
so a two-index tensor with a rule is diagonal, and a rule that pairs a virtual with an occupied
index (T1) allows no element: such products have no common group, and nothing is launched.

Each case is a function of ``abi``: the CPU tests pass the numpy emulation of the C ABI
(tests/momentum_emulator.py), the ``gpu`` tests pass None and run the same body on the kernels.
The operands are integers in +-[1, 7], so every sum is exact in any order and results are compared
bit for bit with an int64 numpy einsum."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _kernel_consts():
    """(GK, GE) as csrc/cc_blocked.cu defines them for group_kernel."""
    with open(os.path.join(ROOT, "pymes_b200", "csrc", "cc_blocked.cu")) as fh:
        m = re.search(r"constexpr int GT = \d+, GK = (\d+), GNT = \d+, GE = (\d+);", fh.read())
    return int(m.group(1)), int(m.group(2))


GK, GE = _kernel_consts()

# one product of each new split r | e | c that the CCSD sweep runs, as (spec, r, e, c)
SPLITS = [("ac,cbij->abij", 1, 1, 3), ("abkj,ki->abij", 3, 1, 1), ("adkl,lkdc->ac", 1, 3, 1),
          ("ak,ki->ai", 1, 1, 1), ("abij,jb->ai", 2, 2, 0), ("jb,abij->ai", 0, 2, 2), ("ai,bj->abij", 2, 0, 2),
          ("ajbc,ijbc->ai", 1, 3, 1), ("kc,ci->ki", 1, 1, 1)]


@pytest.fixture
def abi(cpu_abi):
    from tests import momentum_emulator
    return momentum_emulator.extend(cpu_abi)


def _n(x):
    return np.ascontiguousarray(x.detach().cpu().numpy())


def _t(a):
    from pymes_b200 import backend as bk
    return torch.from_numpy(np.array(a, dtype=np.float64, order="C")).to(bk.device())


def _ints(rng, shape):
    return rng.integers(1, 8, shape) * rng.choice([-1, 1], shape)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


class _Calls:
    """Counts calls of C entry points and backend helpers until the ``with`` block ends."""

    def __init__(self, names=("pmb_group_contract", "pmb_gemv", "pmb_gather_expand", "pmb_contract")):
        from pymes_b200 import _lib
        self._mp = pytest.MonkeyPatch()
        self.n = dict.fromkeys(names, 0)
        lib = _lib.load()
        for name in names:
            def counted(*a, _fn=getattr(lib, name), _name=name):
                self.n[_name] += 1
                return _fn(*a)
            self._mp.setattr(lib, name, counted)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self._mp.undo()


class _Labels:
    """Momentum labels for one product: each index its own range of ``lin``, labels drawn from a
    few keys (so groups of several members meet), and a random sign folded into them, so both
    signs sigma of the summed axes occur.  A allows sum(rows) == sum(entries), B sum(entries) ==
    sum(columns); ``pad[ch] = n`` adds n orbitals in front of index ``ch`` for a parent tensor that
    the operand is a narrow of."""

    def __init__(self, spec, rng, ext=None, keys=4, pad=None):
        sa, rest = spec.split(",")
        sb, so = rest.split("->")
        self.sa, self.sb, self.so = sa, sb, so
        ext = ext or {}
        pad = pad or {}
        lin, at, self.lo, self.flip, self.ext, self.pad = [], 0, {}, {}, {}, pad
        for ch in sorted(set(sa + sb)):
            n = ext.get(ch, 5)
            lab = rng.integers(0, keys, n + pad.get(ch, 0))
            self.flip[ch] = int(rng.choice([-1, 1]))
            self.lo[ch], self.ext[ch] = at + pad.get(ch, 0), n
            lin.append(self.flip[ch] * lab)
            at += len(lab)
        self.lin = np.concatenate(lin).astype(np.int64)

    def rule(self, which, padded=False):
        from pymes_b200 import backend as bk
        sub, other = (self.sa, self.sb) if which == "a" else (self.sb, self.sa)
        # A: rows +, entries -;  B: entries +, columns -
        base = {ch: (1 if ch not in other else -1) if which == "a" else (1 if ch in other else -1) for ch in sub}
        p = (lambda ch: self.pad.get(ch, 0)) if padded else (lambda ch: 0)
        return bk.Momentum(self.lin, [(self.lo[ch] - p(ch), self.ext[ch] + p(ch), base[ch] * self.flip[ch])
                                      for ch in sub])

    def dense(self, which, rng, padded=False):
        rule = self.rule(which, padded)
        tot = np.zeros((), dtype=np.int64)
        for d in range(len(rule.axes)):
            tot = np.add.outer(tot, rule.labels(d))
        return np.where(tot == 0, _ints(rng, tot.shape), 0)


def _operands(spec, rng, **kw):
    from pymes_b200 import backend as bk
    lab = _Labels(spec, rng, **kw)
    Ai, Bi = lab.dense("a", rng), lab.dense("b", rng)
    A, B = _t(Ai), _t(Bi)
    assert bk.adopt_momentum(A, lab.rule("a")) and bk.adopt_momentum(B, lab.rule("b"))
    return lab, Ai, Bi, A, B


def _want(spec, Ai, Bi, old, beta):
    acc = np.einsum(spec, Ai.astype(np.int64), Bi.astype(np.int64)).astype(np.float64)
    return acc if beta == 0.0 else beta * old + acc


# --------------------------------------------------------------------------
# cases
# --------------------------------------------------------------------------
def _case_every_new_split(abi):
    """Each split of the sweep takes the group path and matches numpy bit for bit for beta = 0
    (output filled with NaN), 0.5 and 1, with both signs sigma."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(1)
    for spec, r, e, c in SPLITS:
        sigmas = set()
        for seed in range(16):
            lab, Ai, Bi, A, B = _operands(spec, np.random.default_rng(100 * seed + len(spec)))
            g = bk._group_term(lab.so, (1.0, lab.sa, A, lab.sb, B))
            assert g is not None, spec
            sigmas.add(g[5])
            rows, ents = [ch for ch in lab.sa if ch in lab.so], [ch for ch in lab.sa if ch not in lab.so]
            assert (len(rows), len(ents), len([ch for ch in lab.sb if ch in lab.so])) == (r, e, c)
            shape = np.einsum(spec, Ai, Bi).shape
            for beta in (0.0, 0.5, 1.0):
                old = _ints(rng, shape).astype(np.float64)
                out = _t(np.full(shape, np.nan) if beta == 0.0 else old)
                with _Calls() as calls:
                    bk.contract(spec, A, B, out=out, beta=beta)
                assert calls.n["pmb_group_contract"] == 1 and calls.n["pmb_contract"] == 0, spec
                assert calls.n["pmb_gemv"] == calls.n["pmb_gather_expand"] == 0, spec
                assert np.array_equal(_bits(_n(out)), _bits(_want(spec, Ai, Bi, old, beta))), (spec, beta)
            if seed >= 1 and (e == 0 or len(sigmas) == 2):
                break
        assert e == 0 or sigmas == {1, -1}, (spec, sigmas)


def _case_strided_and_narrowed_operands(abi):
    """A permuted A, a B narrowed from a larger tagged parent and an output that is a permuted
    view inside a tensor of sentinels."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(2)
    for spec in ("ac,cbij->abij", "adkl,lkdc->ac", "abkj,ki->abij", "jb,abij->ai"):
        lab = _Labels(spec, rng, pad={ch: 3 for ch in spec.split(",")[1].split("->")[0]})
        Ai = lab.dense("a", rng)
        Bp = lab.dense("b", rng, padded=True)
        At = _t(np.ascontiguousarray(Ai.transpose(tuple(range(Ai.ndim))[::-1])))
        assert bk.adopt_momentum(At, lab.rule("a").permute(tuple(range(Ai.ndim))[::-1]))
        A = bk.permute(At, tuple(range(Ai.ndim))[::-1])
        B = _t(Bp)
        assert bk.adopt_momentum(B, lab.rule("b", padded=True))
        for d in range(Bp.ndim):
            B = bk.narrow(B, d, 3, lab.ext[lab.sb[d]])
        Bi = _n(B)
        assert bk.momentum_of(A) is not None and bk.momentum_of(B) is not None
        shape = np.einsum(spec, Ai, Bi).shape
        for beta in (0.0, 0.5):
            old = _ints(rng, shape).astype(np.float64)
            big = np.full(shape[::-1] + (2,), 7.25)
            big[..., 0] = (np.full(shape, np.nan) if beta == 0.0 else old).T
            host = _t(big)
            out = host[..., 0].permute(*range(len(shape) - 1, -1, -1))
            with _Calls() as calls:
                bk.contract(spec, A, B, out=out, beta=beta)
            assert calls.n["pmb_group_contract"] == 1 and calls.n["pmb_contract"] == 0, spec
            assert np.array_equal(_bits(_n(out)), _bits(_want(spec, Ai, Bi, old, beta))), (spec, beta)
            assert np.all(_n(host)[..., 1] == 7.25)


def _case_empty_plans(abi):
    """Rules that never meet on all three sides (a T1-like operand pairs disjoint label sets): no
    tile, no upload, no launch, and the output gets only the beta treatment."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(3)
    for spec in ("ajbc,ijbc->ai", "bl,alij->abij", "ai,bj->abij", "kibc,ck->ib", "jb,abij->ai"):
        lab = _Labels(spec, rng)
        # move every label of index "a" or "b" (virtual) away from the occupied ones
        virt = [ch for ch in "abcd" if ch in lab.lo]
        for ch in virt:
            lo = lab.lo[ch]
            lab.lin[lo:lo + lab.ext[ch]] = lab.flip[ch] * (100 + np.arange(lab.ext[ch]) * 17 + 1000 * (ch == "c"))
        Ai, Bi = lab.dense("a", rng), lab.dense("b", rng)
        A, B = _t(Ai), _t(Bi)
        assert bk.adopt_momentum(A, lab.rule("a")) and bk.adopt_momentum(B, lab.rule("b"))
        assert not np.einsum(spec, Ai, Bi).any()
        shape = np.einsum(spec, Ai, Bi).shape
        g = bk._group_term(lab.so, (1.0, lab.sa, A, lab.sb, B))
        assert g is not None, spec
        for beta in (0.0, -0.5, 1.0):
            old = _ints(rng, shape).astype(np.float64)
            out = _t(np.full(shape, np.nan) if beta == 0.0 else old)
            launches = bk.launch_count()
            uploads = []
            orig_to = torch.Tensor.to

            def to(self, *a, **k):
                if self.dtype != torch.float64:          # an offset list or a tile table
                    uploads.append(tuple(self.shape))
                return orig_to(self, *a, **k)
            mp = pytest.MonkeyPatch()
            mp.setattr(torch.Tensor, "to", to)
            try:
                with _Calls() as calls:
                    bk.contract(spec, A, B, out=out, beta=beta)
            finally:
                mp.undo()
            assert calls.n["pmb_contract"] == calls.n["pmb_gemv"] == calls.n["pmb_gather_expand"] == 0, spec
            plan = bk._group_plan(lab.so, g, out)
            assert plan["n_tiles"] == 0 and len(plan["tiles"]) == 0 and "a_ent" not in plan
            assert uploads == [], (spec, uploads)
            if abi is None:
                # the beta treatment is the only launch: none for beta = 1, a clear or a scale else
                assert bk.launch_count() - launches <= (0 if beta == 1.0 else 1), spec
            want = np.zeros(shape) if beta == 0.0 else beta * old
            assert np.array_equal(_bits(_n(out)), _bits(want)), (spec, beta)


def _case_untagged_operands_keep_their_route(abi):
    """An untagged operand keeps today's route: the matrix-vector kernel for ``kibc,ck->ib`` and
    ``jb,abij->ai``, no group product.  The size thresholds of the matrix-vector path are lowered
    so that these small operands take it."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(4)
    mp = pytest.MonkeyPatch()
    for name in ("GEMV_MIN_ELEMENTS", "GEMV_MIN_WARP_OUTPUTS", "GEMV_MIN_OUTPUTS"):
        mp.setattr(bk, name, 1)
    try:
        _untagged_routes(bk, rng)
    finally:
        mp.undo()


def _untagged_routes(bk, rng):
    for spec in ("kibc,ck->ib", "jb,abij->ai"):
        lab, Ai, Bi, A, B = _operands(spec, rng, ext={"a": 6, "b": 7, "c": 8, "i": 3, "j": 3, "k": 3})
        untagged = _t(_n(B))
        with _Calls() as calls:
            out = bk.contract(spec, A, untagged)
        assert calls.n["pmb_gemv"] == 1 and calls.n["pmb_group_contract"] == 0, spec
        assert np.array_equal(_bits(_n(out)), _bits(_want(spec, Ai, Bi, None, 0.0)))
        with _Calls() as calls:
            bk.contract(spec, A, B)
        assert calls.n["pmb_gemv"] == 0 and calls.n["pmb_group_contract"] == 1, spec
        prev = bk.set_blocked(False)
        try:
            with _Calls() as calls:
                bk.contract(spec, A, B)
            assert calls.n["pmb_gemv"] == 1 and calls.n["pmb_group_contract"] == 0, spec
        finally:
            bk.set_blocked(prev)


# (rows, columns) per tile: rn*cn in {1, 2, 32} as asked, GE and GE + 1 at the switch of the form
TILE_SHAPES = [(1, 1), (1, 2), (2, 1), (2, 2), (1, 5), (4, 8)]
ENTRIES = [1, 32, 33, 1000, 9000]


def _case_entry_split_form(abi):
    """Hand-built tables: one tile per (rows, entries, columns), entries 1 .. 9000, so the kernel
    takes both the slab form and the entry-split form (rn*cn <= GE, en > GK).  Rows and columns of C
    are scattered, A and B have padded pitches."""
    from pymes_b200 import _lib, backend as bk
    rng = np.random.default_rng(5)
    shapes = [(rn, en, cn) for rn, cn in TILE_SHAPES for en in ENTRIES]
    assert any(rn * cn <= GE and en > GK for rn, en, cn in shapes)
    assert any(rn * cn > GE and en > GK for rn, en, cn in shapes)
    n_r, n_e, n_c = (sum(s[i] for s in shapes) for i in range(3))
    pa, pb = n_e + 3, n_c + 5
    A, B = _ints(rng, (n_r, pa)), _ints(rng, (n_e, pb))
    prow, pcol = rng.permutation(n_r), rng.permutation(n_c)
    Cwant = np.full((n_r, n_c), 0.5)
    tiles, r0, e0, c0 = [], 0, 0, 0
    a_ent, b_col = np.zeros(n_e, dtype=np.int64), np.zeros(n_c, dtype=np.int64)
    for rn, en, cn in shapes:
        tiles.append((r0, rn, e0, en, c0, cn))
        a_ent[e0:e0 + en] = np.arange(e0, e0 + en)
        b_col[c0:c0 + cn] = np.arange(c0, c0 + cn)
        acc = A[r0:r0 + rn, e0:e0 + en].astype(np.int64) @ B[e0:e0 + en, c0:c0 + cn].astype(np.int64)
        Cwant[np.ix_(prow[r0:r0 + rn], pcol[c0:c0 + cn])] += acc
        r0, e0, c0 = r0 + rn, e0 + en, c0 + cn
    dev = bk.device()
    up = lambda a, dt=np.int64: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
    Ad, Bd = _t(A), _t(B)
    Cd = _t(np.full((n_r, n_c), 0.5))
    lists = dict(a_row=up(np.arange(n_r) * pa), a_ent=up(a_ent), b_ent=up(np.arange(n_e) * pb), b_col=up(b_col),
                 c_row=up(prow * n_c), c_col=up(pcol), tiles=up(tiles, np.int32))
    d = _lib.Group()
    d.A, d.B, d.C = Ad.data_ptr(), Bd.data_ptr(), Cd.data_ptr()
    for k, v in lists.items():
        setattr(d, k, v.data_ptr())
    d.n_tiles, d.alpha = len(tiles), 1.0
    _lib.check(_lib.load().pmb_group_contract(C.byref(d), bk._stream()), "pmb_group_contract")
    assert np.array_equal(_bits(_n(Cd)), _bits(Cwant))


CASES = [_case_every_new_split, _case_strided_and_narrowed_operands, _case_empty_plans,
         _case_untagged_operands_keep_their_route, _case_entry_split_form]
IDS = [f.__name__[len("_case_"):] for f in CASES]


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_on_the_emulated_abi(abi, case):
    case(abi)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_on_the_device(case):
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    case(None)


# --------------------------------------------------------------------------
# the CCSD sweep: which products of two tagged operands still take another route
# --------------------------------------------------------------------------
def _ueg(n_ele, no, cutoff, k_cutoff, rs=0.5):
    from pymes_b200.model import ueg
    m = ueg.UEG(n_ele, no, no, rs)
    m.init_single_basis(cutoff)
    m.gamma, m.k_cutoff = None, k_cutoff
    return m, no, [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)]


def _fock(m, no):
    eps = np.asarray(m.kinetic(), dtype=np.float64).copy()
    eps[:no] -= 1.0
    return np.diag(eps)


def _other_route_reason(bk, out_sub, term):
    """Why a term of two tagged operands may leave the group path: a scalar result or summed axes
    that carry no sign (a trace with ``ones``).  None for any other term."""
    _alpha, sa, A, sb, B = term
    if not out_sub:
        return "scalar"
    ka, kb = bk.momentum_of(A), bk.momentum_of(B)
    ents = [ch for ch in sa if ch in sb]
    if ents and all(ka.axes[sa.index(ch)][2] == 0 and kb.axes[sb.index(ch)][2] == 0 for ch in ents):
        return "sign-0 trace"
    return None


def _sweep_guard(m, no, parts, n_sweeps, monkeypatch):
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd
    other, checked = [], []

    def tagged(t):
        return isinstance(t[2], torch.Tensor) and isinstance(t[4], torch.Tensor) and \
            bk.momentum_of(t[2]) is not None and bk.momentum_of(t[4]) is not None

    def watch(fn, route):
        def wrapped(out_sub, terms, out, beta):
            res = fn(out_sub, terms, out, beta)
            if res is not None:
                for t in terms:
                    if tagged(t):
                        other.append((route, "%s,%s->%s" % (t[1], t[3], out_sub),
                                      _other_route_reason(bk, out_sub, t)))
            return res
        return wrapped
    describe = bk.describe_contraction

    def described(out_sub, terms, *a, **k):
        for t in terms:
            if tagged(t):
                other.append(("dense", "%s,%s->%s" % (t[1], t[3], out_sub), _other_route_reason(bk, out_sub, t)))
        return describe(out_sub, terms, *a, **k)
    run = bk._run_group

    def shadow(out_sub, g, out, beta):
        alpha, sa, A, sb, B, _sigma = g
        old = out.clone()
        run(out_sub, g, out, beta)
        want = alpha * torch.einsum("%s,%s->%s" % (sa, sb, out_sub), A, B)
        if beta != 0.0:
            want += beta * old
        err = (out - want).abs().max().item()
        assert err <= 1e-13 * max(want.abs().max().item(), 1e-300), (sa, sb, out_sub, err)
        checked.append("%s,%s->%s" % (sa, sb, out_sub))
    monkeypatch.setattr(bk, "_try_gemv", watch(bk._try_gemv, "gemv"))
    monkeypatch.setattr(bk, "_try_gather", watch(bk._try_gather, "gather"))
    monkeypatch.setattr(bk, "describe_contraction", described)
    monkeypatch.setattr(bk, "_run_group", shadow)

    def sweeps():
        cc = ccsd.CCSD(no)
        cc.setup(_fock(m, no), m.eval_2b_blocks(no, list(KEYS), parts))
        return [cc.sweep()[:3] for _ in range(n_sweeps)]
    e = sweeps()
    assert all(why is not None for _route, _spec, why in other), sorted({(r, s) for r, s, w in other if w is None})
    specs = set(checked)
    for spec in ("ajbc,bcij->ai", "ac,cbij->abij", "ki,abkj->abij", "adkl,lkdc->ac", "cdil,lkdc->ki",
                 "bl,alij->abij", "ai,bj->abij", "jb,abij->ai", "kibc,ck->ib", "abid,dj->abij", "kaic,cbkj->abij"):
        assert spec in specs, (spec, sorted(specs))
    prev = bk.set_blocked(False)
    try:
        n0 = len(checked)
        e_dense = sweeps()
        assert len(checked) == n0
    finally:
        bk.set_blocked(prev)
    np.testing.assert_allclose(np.array(e), np.array(e_dense), rtol=0, atol=1e-12)


def test_sweep_products_of_tagged_operands_take_the_group_path(abi, monkeypatch):
    """TC-UEG 14e: every product of two tagged operands runs on its groups (scalars and sign-0
    traces aside), every group result matches torch.einsum, and the energies match the dense path."""
    m, no, parts = _ueg(14, 7, 2.0, 1.0)
    _sweep_guard(m, no, parts, 2, monkeypatch)


@pytest.mark.gpu
def test_sweep_products_of_tagged_operands_take_the_group_path_54e(monkeypatch):
    """The same at the bench's 54 electrons with a smaller basis (cutoff 7.0)."""
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    import bench
    m, no, _parts = _ueg(54, 27, 7.0, bench.K_CUTOFF, bench.RS)
    _sweep_guard(m, no, bench.tc_parts(m), 2, monkeypatch)
