"""Edges of pmb_group_contract (the product of two momentum-tagged tensors on their common groups)
and of pmb_momentum_residue (the check behind ``adopt_momentum``).

The kernel cuts every group into tiles of at most GT rows x GT columns, one CTA each, and walks the
group's entries in slabs of GK (csrc/cc_blocked.cu).  The momentum labels here are made by hand, so
each group's row, entry and column counts sit exactly on those edges.  The operands are integers
in +-[1, 7], so the FP64 products and sums are exact in any order and the result is compared bit
for bit with an int64 numpy einsum: a dropped, doubled or misplaced term moves an element by at
least 1.

Each case is a function of ``abi``: the CPU tests pass the numpy emulation of the C ABI
(tests/momentum_emulator.py), the ``gpu`` tests pass None and run the same body on the kernels."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _kernel_tiles():
    """(GT, GK) as csrc/cc_blocked.cu defines them for group_kernel."""
    with open(os.path.join(ROOT, "pymes_b200", "csrc", "cc_blocked.cu")) as fh:
        m = re.search(r"constexpr int GT = (\d+), GK = (\d+)", fh.read())
    return int(m.group(1)), int(m.group(2))


GT, GK = _kernel_tiles()
SEC = 1000          # label step of a side's second index: far above every group key

# key -> (rows, entries, columns) of the group; 0 = the group is missing from that side
EDGE = {1: (1, 1, 1), 2: (31, 32, 33), 3: (32, 33, 31), 4: (33, 64, 65), 5: (64, 65, 32),
        6: (65, 31, 64), 7: (2, 100, 3),
        8: (3, 0, 0), 9: (2, 3, 0), 10: (0, 2, 5), 11: (0, 0, 4), 12: (4, 0, 4)}
SMALL = {1: (33, 40, 34), 2: (3, 1, 65), 3: (2, 3, 0), 4: (4, 0, 5)}
DISJOINT = {1: (3, 4, 0), 2: (0, 5, 6), 3: (7, 0, 8)}        # no group on all three sides

# every 2 | 2 | 2 split of the doubles residual that reaches the group path (ccd.doubles_residual)
SPLITS = ["kaic,cbkj->abij", "kbic,ackj->abij", "acik,kbcj->abij", "acik,cbkj->abij", "alcj,cbil->abij",
          "alci,cblj->abij", "cbkj,kaic->abij", "abkl,klij->abij", "klcd,dblj->cbkj", "klcd,adkj->alcj",
          "klcd,daki->alci", "klcd,cdij->klij", "abcd,cdij->abij"]


@pytest.fixture
def abi(cpu_abi):
    """The emulated C ABI with pmb_group_contract and pmb_momentum_residue."""
    from tests import momentum_emulator
    return momentum_emulator.extend(cpu_abi)


def _n(x):
    return np.ascontiguousarray(x.detach().cpu().numpy())


def _t(a):
    from pymes_b200 import backend as bk
    return torch.from_numpy(np.array(a, dtype=np.float64, order="C")).to(bk.device())   # a copy, also on the host


def _ints(rng, shape):
    return rng.integers(1, 8, shape) * rng.choice([-1, 1], shape)


def _tag(a, rule):
    from pymes_b200 import backend as bk
    t = _t(a)
    assert bk.adopt_momentum(t, rule)
    return t


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


class _Probe:
    """Records (sigma, tiles) of every group plan the backend builds or reuses and counts the calls
    of pmb_group_contract and pmb_momentum_residue, until the ``with`` block ends."""

    def __init__(self):
        from pymes_b200 import _lib, backend as bk
        self._mp = pytest.MonkeyPatch()
        self.plans, self.calls = [], {"pmb_group_contract": 0, "pmb_momentum_residue": 0}
        orig = bk._group_plan

        def plan(out_sub, g, out):
            p = orig(out_sub, g, out)
            self.plans.append((g[5], p["tiles"].cpu().numpy().reshape(-1, 6).copy()))
            return p
        self._mp.setattr(bk, "_group_plan", plan)
        lib = _lib.load()
        for name in self.calls:
            def counted(*a, _fn=getattr(lib, name), _name=name):
                self.calls[_name] += 1
                return _fn(*a)
            self._mp.setattr(lib, name, counted)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self._mp.undo()


def _extents(tiles):
    return sorted((int(t[1]), int(t[3]), int(t[5])) for t in tiles)


def _col_split(tiles):
    """Does some group have a column tile that starts past its first column?"""
    first = {}
    for r0, _rn, e0, _en, c0, _cn in tiles:
        first.setdefault((int(r0), int(e0)), set()).add(int(c0))
    return any(len(c) > 1 for c in first.values())


class _Design:
    """Momentum labels for one 2 | 2 | 2 product ``spec``: rows from A, summed entries, columns
    from B.  On each side the first index carries the group keys, ``counts[key][side]`` orbitals of
    each in a shuffled order, and the second index the labels 0, SEC, 2 SEC, .. (``sec[side]`` of
    them), so the group key + s SEC of a side holds exactly ``counts[key][side]`` pairs.  A allows
    rows and entries of one key, B entries and columns of one key.  Each index gets its own range of
    ``lin`` and a random sign folded into its labels, so the rules mix their signs and both signs
    sigma of the summed axes occur.  ``pad[ch] = (before, after)`` adds orbitals around index
    ``ch`` for a parent tensor that the design is a narrow of."""

    def __init__(self, spec, counts, rng, sec=(2, 1, 2), pad=None):
        sa, rest = spec.split(",")
        sb, so = rest.split("->")
        self.spec, self.sa, self.sb, self.so = spec, sa, sb, so
        self.sides = ([ch for ch in sa if ch in so], [ch for ch in sa if ch not in so],
                      [ch for ch in sb if ch in so])
        self.counts, self.sec = counts, sec
        keys = sorted(counts)
        self.lab = {}
        for s, (first, second) in enumerate(self.sides):
            self.lab[first] = rng.permutation(np.repeat(keys, [counts[k][s] for k in keys]))
            self.lab[second] = SEC * np.arange(sec[s])
        self.base = {"a": {ch: 1 if ch in self.sides[0] else -1 for ch in sa},
                     "b": {ch: 1 if ch in self.sides[1] else -1 for ch in sb}}
        pad = pad or {}
        lin, at, self.lo, self.parent, self.flip = [], 0, {}, {}, {}
        for ch in sorted(self.lab):
            before, after = pad.get(ch, (0, 0))
            full = np.concatenate([rng.choice(keys, before), self.lab[ch], rng.choice(keys, after)])
            self.flip[ch] = int(rng.choice([-1, 1]))
            self.lo[ch], self.parent[ch] = at + before, (at, len(full))
            lin.append(self.flip[ch] * full)
            at += len(full)
        self.lin = np.concatenate(lin).astype(np.int64)

    def rule(self, which, padded=()):
        from pymes_b200 import backend as bk
        sub = self.sa if which == "a" else self.sb
        axes = [self.parent[ch] + (self.base[which][ch] * self.flip[ch],) if ch in padded else
                (self.lo[ch], len(self.lab[ch]), self.base[which][ch] * self.flip[ch]) for ch in sub]
        return bk.Momentum(self.lin, axes)

    def dense(self, which, rng, padded=(), real=False):
        """Integers in +-[1, 7] (standard normal values with ``real``) where the rule allows them."""
        rule = self.rule(which, padded)
        tot = np.zeros((), dtype=np.int64)
        for d in range(len(rule.axes)):
            tot = np.add.outer(tot, rule.labels(d))
        vals = rng.standard_normal(tot.shape) if real else _ints(rng, tot.shape)
        return np.where(tot == 0, vals, 0)

    def tiles(self):
        """(rows, entries, columns) of every tile the host plan must cut, sorted."""
        want = []
        for r, e, c in self.counts.values():
            if r and e and c:
                for rt in range(0, r, GT):
                    for ct in range(0, c, GT):
                        want += [(min(GT, r - rt), e, min(GT, c - ct))] * min(self.sec)
        return sorted(want)

    def inside(self):
        """Output elements in a group that has rows, entries and columns (the others get no term)."""
        def key(chs):
            k = np.zeros((1,) * len(self.so), dtype=np.int64)
            for ch in chs:
                shape = [1] * len(self.so)
                shape[self.so.index(ch)] = -1
                k = k + self.lab[ch].reshape(shape)
            return k
        rows, ents, cols = self.sides
        rk = key(rows)
        return (rk == key(cols)) & np.isin(rk, np.add.outer(self.lab[ents[0]], self.lab[ents[1]]))


def _want(acc, old, alpha, beta):
    return (beta * old if beta != 0.0 else np.zeros(old.shape)) + alpha * acc.astype(np.float64)


def _check(got, acc, old, alpha, beta, inside):
    """``got == beta * old + alpha * acc`` bit for bit, except where alpha * acc rounds (alpha not an
    integer): the kernel fuses it with the old value into one FMA, numpy rounds the product first,
    so there the two may differ by an ulp of the result plus half an ulp of the product (a missing
    or extra term moves the element by at least 0.7)."""
    got, want = _n(got), _want(acc, old, alpha, beta)
    if alpha == 1.0:
        assert np.array_equal(_bits(got), _bits(want))
        return
    assert np.array_equal(_bits(got[~inside]), _bits(want[~inside]))
    tol = np.spacing(np.abs(want[inside])) + np.spacing(np.abs(alpha * acc[inside].astype(np.float64)))
    assert np.all(np.abs(got[inside] - want[inside]) <= tol)


# --------------------------------------------------------------------------
# 1. synthetic momentum labels, exact references
# --------------------------------------------------------------------------
def _case_every_split_at_the_tile_edges(abi):
    """Each split of the doubles residual on groups of 1, 31, 32, 33, 64, 65 rows and columns and
    1 .. 100 entries, groups missing from one or two sides, alpha in {1, -0.7} and beta in
    {0 (NaN before), 0.5, 1, -1}: bit for bit against int64 numpy, and the host plan cuts exactly
    the tiles the counts imply."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(1)
    combos = [(a, b) for b in (0.0, 0.5, 1.0, -1.0) for a in (1.0, -0.7)]
    sigmas, tiles_seen = set(), []
    with _Probe() as probe:
        for i, spec in enumerate(SPLITS):
            alpha, beta = combos[i % len(combos)]
            d = _Design(spec, EDGE, rng)
            Ai, Bi = d.dense("a", rng), d.dense("b", rng)
            A, B = _tag(Ai, d.rule("a")), _tag(Bi, d.rule("b"))
            acc = np.einsum(spec, Ai, Bi)
            old = _ints(rng, acc.shape).astype(np.float64)
            out = _t(np.full(acc.shape, np.nan) if beta == 0.0 else old)
            n0 = probe.calls["pmb_group_contract"]
            bk.contract(spec, A, B, out=out, alpha=alpha, beta=beta)
            assert probe.calls["pmb_group_contract"] == n0 + 1, spec
            sigma, tiles = probe.plans[-1]
            assert _extents(tiles) == d.tiles(), spec
            _check(out, acc, old, alpha, beta, d.inside())
            sigmas.add(sigma)
            tiles_seen.append(tiles)
    every = np.concatenate(tiles_seen)
    assert sigmas == {1, -1}
    assert every[:, 1].max() == GT and every[:, 5].max() == GT and every[:, 3].max() >= 3 * GK + 1
    assert {1, GK + 1, 2 * GK + 1}.issubset(set(every[:, 3].tolist()))
    assert all(_col_split(t) for t in tiles_seen)


def _case_strided_operands_and_output(abi):
    """A permuted operand, a permuted and narrowed one, and outputs that are a contiguous tensor or
    a permuted, narrowed view of a larger tensor of sentinels; the same spec back to back on both
    outputs and on two narrows at different offsets (each must get its own plan)."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(2)
    spec = "kaic,cbkj->abij"
    d = _Design(spec, SMALL, rng, sec=(2, 2, 2), pad={"b": (3, 2), "k": (1, 4)})
    Ai = d.dense("a", rng)
    pa = (2, 0, 3, 1)
    A = bk.permute(_tag(Ai.transpose(pa), d.rule("a").permute(pa)), np.argsort(pa).tolist())
    Bp = d.dense("b", rng, padded=("b", "k"))
    pb = (1, 3, 0, 2)
    Bs = bk.permute(_tag(Bp.transpose(pb), d.rule("b", padded=("b", "k")).permute(pb)), np.argsort(pb).tolist())
    nb, nk = len(d.lab["b"]), len(d.lab["k"])

    def narrowed(b_lo):
        view = bk.narrow(bk.narrow(Bs, d.sb.index("b"), b_lo, nb), d.sb.index("k"), 1, nk)
        ref = Bp[:, b_lo:b_lo + nb, 1:1 + nk, :]
        return view, ref
    B, Bi = narrowed(3)
    assert A.stride(-1) != 1 and B.stride(-1) != 1
    assert bk.momentum_of(B) == d.rule("b")
    acc = np.einsum(spec, Ai, Bi)
    old = _ints(rng, acc.shape).astype(np.float64)
    sentinel = -12345.625
    pads, po = [(1, 2), (0, 3), (2, 1), (0, 0)], (3, 1, 0, 2)
    big_shape = [n + a + b for n, (a, b) in zip(acc.shape, pads)]
    big = torch.full([big_shape[p] for p in po], sentinel, dtype=torch.float64, device=bk.device())
    big = big.permute(*np.argsort(po).tolist())
    inner = tuple(slice(a, a + n) for n, (a, _b) in zip(acc.shape, pads))
    view = big[inner]
    keep = np.ones(big_shape, dtype=bool)
    keep[inner] = False
    with _Probe() as probe:
        out = _t(old)
        bk.contract(spec, A, B, out=out, beta=0.5)
        _check(out, acc, old, 1.0, 0.5, d.inside())
        view.copy_(_t(old))
        bk.contract(spec, A, B, out=view, alpha=-0.7, beta=-1.0)
        _check(view, acc, old, -0.7, -1.0, d.inside())
        assert np.array_equal(_bits(_n(big)[keep]), _bits(np.full(keep.sum(), sentinel)))
        assert [_extents(t) for _s, t in probe.plans] == [d.tiles()] * 2
        assert _col_split(probe.plans[-1][1])
        # a narrow at another offset: another rule, the same strides
        B2, Bi2 = narrowed(5)
        view.fill_(float("nan"))
        bk.contract(spec, A, B2, out=view, beta=0.0)
        assert np.array_equal(_bits(_n(view)), _bits(np.einsum(spec, Ai, Bi2).astype(np.float64)))
        assert np.array_equal(_bits(_n(big)[keep]), _bits(np.full(keep.sum(), sentinel)))
        assert probe.calls["pmb_group_contract"] == 3


def _case_group_term_next_to_a_dense_term(abi):
    """contract_terms with a group term and a dense term (untagged operands) and beta not in {0, 1}:
    the dense term runs first with beta, the group term then accumulates."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(3)
    spec = "acik,kbcj->abij"
    sa, rest = spec.split(",")
    sb, so = rest.split("->")
    d = _Design(spec, SMALL, rng)
    Ai, Bi = d.dense("a", rng), d.dense("b", rng)
    A, B = _tag(Ai, d.rule("a")), _tag(Bi, d.rule("b"))
    Di, Ei = _ints(rng, Ai.shape), _ints(rng, Bi.shape)
    D, E = _t(Di), _t(Ei)
    acc = np.einsum(spec, Ai, Bi) + np.einsum(spec, Di, Ei)
    with _Probe() as probe:
        for k, beta in enumerate((0.5, -1.0)):
            terms = [(1.0, sa, A, sb, B), (1.0, sa, D, sb, E)]
            old = _ints(rng, acc.shape).astype(np.float64)
            out = _t(old)
            bk.contract_terms(so, terms[::-1] if k else terms, out=out, beta=beta)
            assert probe.calls["pmb_group_contract"] == k + 1
            assert np.array_equal(_bits(_n(out)), _bits(_want(acc, old, 1.0, beta)))
            assert bk.momentum_of(out) is None


def _case_no_common_group(abi):
    """Non-zero operands whose groups never meet on all three sides: no tile, and the output is
    beta * old (cleared for beta = 0)."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(4)
    spec = "abkl,klij->abij"
    d = _Design(spec, DISJOINT, rng, sec=(1, 1, 1))
    Ai, Bi = d.dense("a", rng), d.dense("b", rng)
    assert np.count_nonzero(Ai) and np.count_nonzero(Bi) and not np.einsum(spec, Ai, Bi).any()
    A, B = _tag(Ai, d.rule("a")), _tag(Bi, d.rule("b"))
    with _Probe() as probe:
        for beta in (0.0, -1.0):
            old = _ints(rng, (Ai.shape[0], Ai.shape[1], Bi.shape[2], Bi.shape[3])).astype(np.float64)
            out = _t(np.full(old.shape, np.nan) if beta == 0.0 else old)
            bk.contract(spec, A, B, out=out, alpha=-0.7, beta=beta)
            assert np.array_equal(_bits(_n(out)), _bits(_want(np.zeros(old.shape), old, -0.7, beta)))
        assert probe.calls["pmb_group_contract"] == 2
        assert [len(t) for _s, t in probe.plans] == [0, 0]


def _case_real_values(abi):
    """Standard normal values on the edge groups: numpy float64 and the dense path agree to 1e-13."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(5)
    for spec in ("kaic,cbkj->abij", "abkl,klij->abij"):
        d = _Design(spec, EDGE, rng)
        Ai, Bi = d.dense("a", rng, real=True), d.dense("b", rng, real=True)
        A, B = _tag(Ai, d.rule("a")), _tag(Bi, d.rule("b"))
        ref = np.einsum(spec, Ai, Bi)
        old = rng.standard_normal(ref.shape)
        with _Probe() as probe:
            got = bk.contract(spec, A, B, out=_t(old), alpha=-0.7, beta=0.5)
            assert probe.calls["pmb_group_contract"] == 1
            prev = bk.set_blocked(False)
            try:
                dense = bk.contract(spec, A, B, out=_t(old), alpha=-0.7, beta=0.5)
            finally:
                bk.set_blocked(prev)
            assert probe.calls["pmb_group_contract"] == 1
        want = 0.5 * old - 0.7 * ref
        assert _rel(_n(got), want) < 1e-13, spec
        assert _rel(_n(got), _n(dense)) < 1e-13, spec


# --------------------------------------------------------------------------
# 2. the kernel through the C ABI, without the host plan
# --------------------------------------------------------------------------
def _case_c_abi_tiles(abi):
    """Hand-built tables: tiles of 1, GK, GK + 1 and 1000 entries with 1, GT - 1 and GT rows and
    columns, rows and columns of C scattered through permutations, B with a padded pitch.  The
    touched elements of C are exact, the untouched ones bit-identical."""
    from pymes_b200 import _lib, backend as bk
    rng = np.random.default_rng(6)
    shapes = [(rn, en, cn) for en in (1, GK, GK + 1, 1000)
              for rn, cn in ((1, GT), (GT - 1, 1), (GT, GT - 1), (GT, GT), (1, 1))]
    n_rows, n_ent, n_cols = (sum(s[i] for s in shapes) for i in range(3))
    e_max, pitch_b, pitch_c = max(s[1] for s in shapes), GT + 3, n_cols + 2
    A = _ints(rng, (n_rows, e_max))                         # A[row, entry of its group]
    B = _ints(rng, (n_ent, pitch_b))                        # B[entry, column of its group]
    Cm = _ints(rng, (n_rows, pitch_c)).astype(np.float64)
    prow, pcol = rng.permutation(n_rows), rng.permutation(n_cols)
    alpha, want = -1.5, Cm.copy()
    tiles, a_ent, b_col = [], np.zeros(n_ent, dtype=np.int64), np.zeros(n_cols, dtype=np.int64)
    r0 = e0 = c0 = 0
    for rn, en, cn in shapes:
        tiles.append((r0, rn, e0, en, c0, cn))
        a_ent[e0:e0 + en] = np.arange(en)
        b_col[c0:c0 + cn] = np.arange(cn)
        acc = A[r0:r0 + rn, :en] @ B[e0:e0 + en, :cn]
        rows, cols = prow[r0:r0 + rn], pcol[c0:c0 + cn]
        want[np.ix_(rows, cols)] = Cm[np.ix_(rows, cols)] + alpha * acc
        r0, e0, c0 = r0 + rn, e0 + en, c0 + cn
    lib = _lib.load()
    dev = bk.device()
    up = lambda a, dt=np.int64: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
    Ad, Bd, Cd = up(A, np.float64), up(B, np.float64), up(Cm, np.float64)
    tabs = dict(a_row=up(np.arange(n_rows) * e_max), a_ent=up(a_ent), b_ent=up(np.arange(n_ent) * pitch_b),
                b_col=up(b_col), c_row=up(prow * pitch_c), c_col=up(pcol), tiles=up(tiles, np.int32))
    d = _lib.Group()
    d.A, d.B, d.C = Ad.data_ptr(), Bd.data_ptr(), Cd.data_ptr()
    for name, t in tabs.items():
        setattr(d, name, t.data_ptr())
    d.n_tiles, d.alpha = len(tiles), alpha
    _lib.check(lib.pmb_group_contract(C.byref(d), bk._stream()), "pmb_group_contract")
    assert np.array_equal(_bits(_n(Cd)), _bits(want))
    d.n_tiles = 0
    _lib.check(lib.pmb_group_contract(C.byref(d), bk._stream()), "pmb_group_contract")
    assert np.array_equal(_bits(_n(Cd)), _bits(want))


# --------------------------------------------------------------------------
# 3. pmb_momentum_residue by value
# --------------------------------------------------------------------------
def _residue(t, rule):
    """pmb_momentum_residue of ``t`` under ``rule``, called directly."""
    from pymes_b200 import _lib, backend as bk
    keys = torch.from_numpy(np.concatenate([rule.labels(d) for d in range(t.dim())])).to(bk.device())
    res = bk.zeros(1)
    _lib.check(_lib.load().pmb_momentum_residue(t.dim(), _lib.I64x4(*bk._pad4r(t.shape, 1)),
                                                _lib.I64x4(*bk._pad4r(t.stride(), 0)), bk._ptr(t),
                                                bk._ptr(keys), bk._ptr(res), bk._stream()),
               "pmb_momentum_residue")
    return float(res.item())


def _forbidden(rule, shape):
    tot = np.zeros((), dtype=np.int64)
    for d in range(len(shape)):
        tot = np.add.outer(tot, rule.labels(d))
    return tot != 0


def _max_forbidden(x, rule):
    bad = np.abs(x[_forbidden(rule, x.shape)])
    return float(bad.max()) if bad.size else 0.0


def _same(got, want):
    return (np.isnan(got) and np.isnan(want)) or _bits(np.array([got]))[0] == _bits(np.array([want]))[0]


def _rule(rng, ext, signs=None, spread=2):
    """A rule over ``ext`` with random labels in [-spread, spread] on each axis."""
    from pymes_b200 import backend as bk
    signs = signs or [1] * len(ext)
    lin = rng.integers(-spread, spread + 1, sum(ext))
    los = np.cumsum([0] + list(ext))[:-1]
    return bk.Momentum(lin, [(int(lo), n, sg) for lo, n, sg in zip(los, ext, signs)])


def _adopt_both(t, rule):
    """adopt_momentum on the device and with ``host=``: the same decision."""
    from pymes_b200 import backend as bk
    dev = bk.adopt_momentum(t, rule)
    host = bk.adopt_momentum(t.clone(), rule, host=_n(t))
    assert dev == host
    return dev


def _case_residue_by_value(abi):
    """The returned maximum equals numpy's max |x| over the forbidden positions bit for bit: ranks
    1-4, permuted and narrowed views, axes with sign 0, 1.3M elements with the only forbidden
    value first or last, and the values 5e-324, Inf, NaN and -0.0."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(7)
    cases = []
    for ext in ((11,), (6, 9), (4, 5, 7), (3, 4, 5, 6)):
        rule = _rule(rng, ext)
        x = rng.standard_normal(ext)
        cases += [(_t(x), rule), (_t(np.where(_forbidden(rule, ext), 0.0, x)), rule)]
    # views: permuted, narrowed, both; the rule follows the view
    base_rule = _rule(rng, (6, 5, 4, 7))
    base = _t(rng.standard_normal((6, 5, 4, 7)))
    cases += [(base.permute(3, 1, 0, 2), base_rule.permute((3, 1, 0, 2))),
              (base.narrow(1, 2, 3), base_rule.narrow(1, 2, 3)),
              (base.permute(2, 3, 0, 1).narrow(3, 1, 3).narrow(0, 1, 2),
               base_rule.permute((2, 3, 0, 1)).narrow(3, 1, 3).narrow(0, 1, 2))]
    # sign 0: that axis does not count
    ext = (5, 4, 6)
    zero_rule = _rule(rng, ext, signs=[1, 0, -1])
    x = rng.standard_normal(ext)
    cases += [(_t(x), zero_rule), (_t(np.where(_forbidden(zero_rule, ext), 0.0, x)), zero_rule)]
    for t, rule in cases:
        want = _max_forbidden(_n(t), rule)
        assert _same(_residue(t, rule), want)
        assert _adopt_both(t, rule) == (want == 0.0)
    # larger than several grid-stride passes of the kernel (8 CTAs per SM x 256 threads)
    ext = (24, 24, 48, 48)
    lin = rng.integers(-3, 4, sum(ext))
    los = np.cumsum((0,) + ext)
    lin[los[:-1]] = lin[los[1:] - 1] = 1              # the first and the last element are forbidden
    big_rule = bk.Momentum(lin, [(int(lo), n, 1) for lo, n in zip(los, ext)])
    bad = _forbidden(big_rule, ext)
    assert bad.flat[0] and bad.flat[-1] and bad.size >= 1_300_000
    x = rng.standard_normal(ext)
    assert _same(_residue(_t(x), big_rule), _max_forbidden(x, big_rule))
    clean = np.where(bad, 0.0, x)
    for pos in (0, bad.size - 1):
        y = clean.copy()
        y.flat[pos] = -3.5
        assert _residue(_t(y), big_rule) == 3.5
    # special values at one forbidden position; -0.0 is a zero and is accepted
    ext = (3, 4, 5, 6)
    rule = _rule(rng, ext)
    bad = _forbidden(rule, ext)
    clean = np.where(bad, 0.0, rng.standard_normal(ext))
    pos = int(np.flatnonzero(bad)[len(np.flatnonzero(bad)) // 2])
    for v, want in ((5e-324, 5e-324), (float("inf"), float("inf")), (-float("inf"), float("inf")),
                    (float("nan"), float("nan")), (-0.0, 0.0)):
        y = clean.copy()
        y.flat[pos] = v
        t = _t(y)
        assert _same(_residue(t, rule), want), v
        assert _adopt_both(t, rule) == (want == 0.0), v
        assert (bk.momentum_of(t) == rule) == (want == 0.0), v


def _case_empty_tensor_is_adopted(abi):
    """An extent of 0: every rule holds, the tensor is tagged without a launch."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(8)
    with _Probe() as probe:
        for ext in ((3, 0), (2, 0, 3, 4), (0,)):
            rule = _rule(rng, ext)
            t = torch.zeros(ext, dtype=torch.float64, device=bk.device())
            assert bk.adopt_momentum(t, rule) and bk.momentum_of(t) == rule
            assert bk.adopt_momentum(t.clone(), rule, host=np.zeros(ext))
        assert probe.calls["pmb_momentum_residue"] == 0


CASES = [_case_every_split_at_the_tile_edges, _case_strided_operands_and_output,
         _case_group_term_next_to_a_dense_term, _case_no_common_group, _case_real_values, _case_c_abi_tiles,
         _case_residue_by_value, _case_empty_tensor_is_adopted]
IDS = [f.__name__[len("_case_"):] for f in CASES]


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_on_the_emulated_abi(abi, case):
    case(abi)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_on_the_device(case):
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    case(None)
    torch.cuda.synchronize()


# --------------------------------------------------------------------------
# 4. a CCSD sweep at o = 33, product by product
# --------------------------------------------------------------------------
@pytest.mark.gpu
def test_ccsd_at_o33_checks_every_group_product(monkeypatch):
    """TC-UEG 66 electrons / 81 plane waves (o = 33, v = 48): its (k,l) and (i,j) groups hold 33
    pairs, so the hh ladder takes a second entry slab and a second column tile.  Two CCSD sweeps;
    every pmb_group_contract result is compared with torch.einsum of the same operands, and the
    energies with the dense path."""
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    import bench
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd
    n_ele, no = 66, 33
    m = ueg.UEG(n_ele, no, no, bench.RS)
    m.init_single_basis(6.0)
    m.k_cutoff, m.gamma = bench.K_CUTOFF, None
    assert (m.n_orb, m.n_orb - no) == (81, 48)
    fock = bench.build_fock(m, no)
    seen = []
    run = bk._run_group

    def shadow(out_sub, g, out, beta):
        alpha, sa, A, sb, B, _sigma = g
        old = out.clone()
        run(out_sub, g, out, beta)
        spec = "%s,%s->%s" % (sa, sb, out_sub)
        want = alpha * torch.einsum(spec, A, B)
        if beta != 0.0:
            want += beta * old
        assert _rel(_n(out), _n(want)) < 1e-13, spec
        seen.append((spec, bk._group_plan(out_sub, g, out)["tiles"].cpu().numpy().reshape(-1, 6)))

    def sweeps():
        cc = ccsd.CCSD(no)
        cc.setup(fock, m.eval_2b_blocks(no, list(KEYS), bench.tc_parts(m)))
        return [cc.sweep()[:3] for _ in range(2)]
    monkeypatch.setattr(bk, "_run_group", shadow)
    e = sweeps()
    specs = {s for s, _t in seen}
    assert {"kaic,cbkj->abij", "kbic,ackj->abij", "acik,kbcj->abij", "acik,cbkj->abij", "alcj,cbil->abij",
            "alci,cblj->abij", "abkl,klij->abij"} <= specs, specs
    assert any((t[:, 3] > GK).any() for _s, t in seen)
    assert any(_col_split(t) for _s, t in seen)
    prev = bk.set_blocked(False)
    try:
        n0 = len(seen)
        e_dense = sweeps()
        assert len(seen) == n0
    finally:
        bk.set_blocked(prev)
    np.testing.assert_allclose(np.array(e), np.array(e_dense), rtol=0, atol=1e-12)


# --------------------------------------------------------------------------
# 5. guards
# --------------------------------------------------------------------------
def test_host_tile_is_the_kernel_tile():
    """group_kernel does not check rn <= GT: a larger host tile would drop rows silently."""
    from pymes_b200 import backend as bk
    assert bk.GROUP_TILE == GT
