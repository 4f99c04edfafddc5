"""FEAST-EOM-CCSD in one total-momentum sector of the UEG: the compact <-> dense copies
pmb_sector_gather / pmb_sector_scatter, ExcitationSector.packed_index, and the sector mode of
solver.feast_eom_ccsd (compact Krylov vectors, sigma on momentum groups), against numpy, the dense
solver and the oracle H-bar of the sector."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def abi(cpu_abi):
    """The emulated C ABI with the momentum, batched group and sector copy entry points."""
    from tests import feast_sector_emulator
    return feast_sector_emulator.extend(cpu_abi)


def _n(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def _ueg14():
    from pymes_b200.model import ueg
    m = ueg.UEG(14, 7, 7, 0.5)
    m.init_single_basis(2.0)
    m.gamma, m.k_cutoff = None, 1.0
    return m, 7, m.n_orb - 7, [("only_non_hermi_2b", m.trunc), ("effect_2b", m.trunc)]


def _masks(sec):
    lin, no = sec.lin, sec.no
    lo, lv = lin[:no], lin[no:]
    m1 = (lv[:, None] - lo[None, :]) == sec.label
    m2 = (lv[:, None, None, None] + lv[None, :, None, None] - lo[None, None, :, None] - lo[None, None, None, :]) \
        == sec.label
    return m1, m2


def _sectors():
    """K = (-1,0,0) (68 elements), the 8th sector with >= 2 singles (39) and K = 0 (204, doubles only)."""
    from pymes_b200.model import ueg
    m, no, nv, _parts = _ueg14()
    eight = [e["sector"] for e in ueg.excitation_sectors(m, no) if e["n_singles"] >= 2][7]
    return {"K-1": ueg.excitation_sector(m, no, (-1, 0, 0)), "8th": eight, "K0": ueg.excitation_sector(m, no, (0, 0, 0))}


_SYSTEM = {}


def _system():
    """_ueg14 after two CCSD sweeps on the active backend: host copies of the dressed Fock matrix,
    the dressed blocks and T2."""
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.solver import ccsd, eom_ccsd
    m, no, nv, parts = _ueg14()
    key = str(bk.device())
    if key not in _SYSTEM:
        eps = np.asarray(m.kinetic(), dtype=np.float64).copy()
        eps[:no] -= 1.0
        fock = np.diag(eps)
        dV = m.eval_2b_blocks(no, list(KEYS), parts)
        cc = ccsd.CCSD(no)
        cc.setup(fock, dV)
        for _ in range(2):
            cc.sweep()
        T1, T2 = cc._st["T1"], cc._st["T2"]
        ft = cc.get_T1_dressed_fock(bk.asdev(fock), T1, dV)
        dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
        _SYSTEM[key] = (_n(ft).copy(), {k: _n(dVd[k]).copy() for k in eom_ccsd.V_KEYS_USED}, _n(T2).copy())
    f, dVh, T2h = _SYSTEM[key]
    return m, no, nv, f, dVh, T2h


def _operands(f, dVh, T2h):
    """Fresh device tensors (untagged) of the host operands."""
    from pymes_b200 import backend as bk
    return bk.asdev(_t(f)), {k: bk.asdev(_t(v)) for k, v in dVh.items()}, bk.asdev(_t(T2h))


def _count(lib, name):
    calls = {"n": 0}
    orig = getattr(lib, name)

    def wrapped(*a):
        calls["n"] += 1
        return orig(*a)
    setattr(lib, name, wrapped)
    return calls


def _feast(sec, **kw):
    from pymes_b200.solver import feast_eom_ccsd
    return feast_eom_ccsd.FEAST_EOM_CCSD(7, sector=sec, **kw)


def _oracle_hbar(sec, no, f, dVh, T2h):
    """The oracle H-bar on the sector basis (packed_index order), built column by column."""
    from oracle import cc_oracle as oc
    m1, m2 = _masks(sec)
    i1, i2 = np.flatnonzero(m1), np.flatnonzero(m2)
    n1 = len(i1)
    H = np.zeros((n1 + len(i2), n1 + len(i2)))
    for c in range(H.shape[0]):
        u1, u2 = np.zeros(m1.size), np.zeros(m2.size)
        if c < n1:
            u1[i1[c]] = 1.0
        else:
            u2[i2[c - n1]] = 1.0
        u1, u2 = u1.reshape(m1.shape), u2.reshape(m2.shape)
        s1 = oc.eom_sigma_singles(no, f, dVh, u1, u2, T2h)
        s2 = oc.eom_sigma_doubles(no, f, dVh, u1, u2, T2h)
        H[:n1, c], H[n1:, c] = s1.reshape(-1)[i1], s2.reshape(-1)[i2]
    return H


# --------------------------------------------------------------------------
# bodies shared by the emulated and the device tests
# --------------------------------------------------------------------------
def _compact_sigma_body(lib):
    """scatter -> sector plan.apply -> gather on compact vectors == the gathered sector sigma of the
    same vectors; no pmb_contract launch."""
    from pymes_b200 import backend as bk
    m, no, nv, f, dVh, T2h = _system()
    for name in ("K-1", "K0"):
        sec = _sectors()[name]
        fe = _feast(sec)
        plan = fe.plan(*_operands(f, dVh, T2h))
        lay = fe.sector_layout(nv)
        rng = np.random.default_rng(11)
        X = rng.standard_normal((3, lay["n"]))
        dense = np.zeros((3, nv * no + nv * nv * no * no))
        dense[:, lay["host"]] = X
        n1 = nv * no
        U1 = [bk.asdev(_t(d[:n1].reshape(nv, no))) for d in dense]
        U2 = [bk.asdev(_t(d[n1:].reshape(nv, nv, no, no))) for d in dense]
        for a, b in zip(U1, U2):
            assert bk.adopt_momentum(a, sec.singles_rule()) and bk.adopt_momentum(b, sec.doubles_rule())
        S1, S2 = plan.apply(bk.stack(U1), bk.stack(U2))
        want = np.concatenate([_n(S1).reshape(3, -1), _n(S2).reshape(3, -1)], axis=1)
        calls = _count(lib, "pmb_contract") if lib is not None else None
        n0 = bk.launch_count()
        Y = fe._sigma_compact(plan, bk.asdev(_t(X)))
        assert bk.launch_count() > n0
        if calls is not None:
            assert calls["n"] == 0
        assert _rel(_n(Y), want[:, lay["host"]]) < 1e-13, name
        # sigma keeps a sector vector in the sector: what the gather drops is exactly zero
        outside = np.ones(want.shape[1], dtype=bool)
        outside[lay["host"]] = False
        assert not want[:, outside].any()


def _shifted_body():
    """One shifted system in the sector == the dense solve of the scattered right-hand side."""
    from pymes_b200 import backend as bk
    m, no, nv, f, dVh, T2h = _system()
    sec = _sectors()["K-1"]
    fs, fd = _feast(sec), _feast(None)
    ops_s, ops_d = _operands(f, dVh, T2h), _operands(f, dVh, T2h)
    ps, pd = fs.plan(*ops_s), fd.plan(*ops_d)
    lay = fs.sector_layout(nv)
    d = torch.cat([fd.get_diag_singles(*ops_d).reshape(-1), fd.get_diag_doubles(*ops_d).reshape(-1)])
    rng = np.random.default_rng(12)
    b = rng.standard_normal(lay["n"])
    bd = np.zeros(d.numel())
    bd[lay["host"]] = b
    z = complex(np.mean(np.diag(f)[no:]) + 0.3j)
    xs = fs.solve_shifted_systems(ps, bk.sector_gather(d[None], lay["idx"])[0], [z], [bk.asdev(_t(b))])[0]
    xd = fd.solve_shifted_systems(pd, d, [z], [bk.asdev(_t(bd))])[0]
    assert fs.ls_residuals[0] < fs.ls_tol and fd.ls_residuals[0] < fd.ls_tol
    cs, cd = _n(xs.re) + 1j * _n(xs.im), _n(xd.re) + 1j * _n(xd.im)
    assert _rel(cs, cd[lay["host"]]) < 1e-12
    outside = np.ones(cd.size, dtype=bool)
    outside[lay["host"]] = False
    assert np.abs(cd[outside]).max() < 1e-13 * np.abs(cd).max()


def _roots_body(name):
    """A contour around one isolated eigenvalue of the oracle sector H-bar: every Ritz value inside
    is an oracle eigenvalue to 1e-8, and the targeted one is found."""
    m, no, nv, f, dVh, T2h = _system()
    sec = _sectors()[name]
    ev = np.linalg.eigvals(_oracle_hbar(sec, no, f, dVh, T2h))
    real = np.sort(ev[np.abs(ev.imag) < 1e-10].real)
    gaps = np.minimum(np.diff(real, prepend=-np.inf), np.diff(real, append=np.inf))
    mid = real[len(real) // 3:]                            # away from the doubles-like bottom of the spectrum
    target = mid[np.argmax(gaps[len(real) // 3:])]
    gap = np.abs(ev[np.abs(ev - target) > 1e-9] - target).min()
    e_r = 0.4 * gap
    np.random.seed(3)
    fe = _feast(sec, e_c=float(target), e_r=float(e_r), n_trial=2, max_iter=12, tol=1e-12)
    fe.ls_tol = 1e-12
    ritz = np.asarray(fe.solve(*_operands(f, dVh, T2h)))
    inside = ritz[np.abs(ritz - target) < e_r]
    assert len(inside) >= 1, (target, ritz)
    for r in inside:
        assert np.abs(ev - r).min() < 1e-8, (r, target)
    assert np.abs(inside - target).min() < 1e-8


# --------------------------------------------------------------------------
# emulated ABI
# --------------------------------------------------------------------------
@pytest.mark.parametrize("nb", [1, 3])
def test_sector_copies_match_numpy_indexing(abi, nb):
    """Gather and scatter through the backend against numpy indexing, with batch strides wider than
    a row; the scatter leaves every other element as it was."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(1)
    row, pitch = 300, 317
    host = np.sort(rng.choice(row, 97, replace=False)).astype(np.int64)
    idx = torch.from_numpy(host)
    buf = rng.standard_normal((nb, pitch))
    x = _t(buf)[:, :row]
    got = bk.sector_gather(x, idx)
    assert np.array_equal(_n(got), buf[:, host])
    wide = torch.zeros(nb, 120, dtype=torch.float64)
    bk.sector_gather(x, idx, out=wide[:, 5:102])
    assert np.array_equal(_n(wide[:, 5:102]), buf[:, host]) and not _n(wide[:, :5]).any()
    dst0 = rng.standard_normal((nb, pitch))
    dst = _t(dst0)
    src = rng.standard_normal((nb, 130))
    bk.sector_scatter(_t(src)[:, :97], idx, dst[:, :row])
    want = dst0.copy()
    want[:, host] = src[:, :97]
    assert np.array_equal(_n(dst), want)
    one = _t(dst0[0, :row])
    bk.sector_scatter(_t(src[0, :97]), idx, one)
    assert np.array_equal(_n(one)[host], src[0, :97])


def test_sector_copies_reject_bad_arguments(abi):
    from pymes_b200 import backend as bk
    idx = torch.tensor([1, 4, 6], dtype=torch.int64)
    src, dst = _t(np.ones(8)), _t(np.zeros(8))
    p = lambda t: t.data_ptr()
    for fn in (abi.pmb_sector_gather, abi.pmb_sector_scatter):
        assert fn(0, 3, p(idx), p(src), 8, p(dst), 8, None) == -1
        assert fn(1, 0, p(idx), p(src), 8, p(dst), 8, None) == -1
        assert fn(1, 3, None, p(src), 8, p(dst), 8, None) == -1
        assert fn(1, 3, p(idx), None, 8, p(dst), 8, None) == -1
        assert fn(1, 3, p(idx), p(src), 8, None, 8, None) == -1
        assert fn(1, 3, p(idx), p(src), 8, p(dst), 8, None) == 0
    with pytest.raises(ValueError, match="increasing"):
        bk.sector_gather(src[None], torch.tensor([3, 3], dtype=torch.int64))
    with pytest.raises(ValueError, match="outside a row"):
        bk.sector_gather(src[None], torch.tensor([2, 8], dtype=torch.int64))
    with pytest.raises(ValueError, match="int64"):
        bk.sector_gather(src[None], torch.tensor([2, 5], dtype=torch.int32))


def test_sector_scatter_restamps_only_a_rule_it_keeps(abi):
    from pymes_b200 import backend as bk
    m, no, nv, _parts = _ueg14()
    sec = _sectors()["K-1"]
    m1, m2 = _masks(sec)
    k2 = sec.doubles_rule()
    idx = torch.from_numpy(np.flatnonzero(m2).astype(np.int64))
    vals = _t(np.arange(1.0, idx.numel() + 1))
    out = bk.zeros(nv, nv, no, no, rule=k2)
    bk.sector_scatter(vals, idx, out)
    assert bk.momentum_of(out) == k2 and np.array_equal(_n(out)[m2], _n(vals))
    stacked = k2.with_axes([(0, 2, 0)] + list(k2.axes))
    outs = bk.zeros(2, nv, nv, no, no, rule=stacked)
    bk.sector_scatter(torch.stack([vals, -vals]), idx, outs)
    assert bk.momentum_of(outs) == stacked
    plain = bk.zeros(nv, nv, no, no)
    bk.sector_scatter(vals, idx, plain)
    assert bk.momentum_of(plain) is None
    # an index with one element outside the rule: the write breaks it, so no tag
    bad = torch.from_numpy(np.sort(np.r_[np.flatnonzero(m2)[1:], np.flatnonzero(~m2)[0]]).astype(np.int64))
    out = bk.zeros(nv, nv, no, no, rule=k2)
    bk.sector_scatter(vals, bad, out)
    assert bk.momentum_of(out) is None


def test_packed_index_is_the_sector_mask():
    from pymes_b200.model import ueg
    m, no, nv, _parts = _ueg14()
    secs = ueg.excitation_sectors(m, no)
    for e in secs[:5] + [secs[-1]]:
        sec = e["sector"]
        m1, m2 = _masks(sec)
        want = np.concatenate([np.flatnonzero(m1), nv * no + np.flatnonzero(m2)])
        got = sec.packed_index()
        assert got.dtype == np.int64 and np.array_equal(got, want)
        assert len(got) == e["n_singles"] + e["n_doubles"]
        assert sec.packed_index() is got                   # cached
    sizes = {k: len(s.packed_index()) for k, s in _sectors().items()}
    assert sizes == {"K-1": 68, "8th": 39, "K0": 204}
    assert ueg.excitation_sector(m, no, (0, 0, 0)).packed_index().min() >= nv * no


def test_compact_sigma_equals_gathered_sector_sigma(abi):
    _compact_sigma_body(abi)


def test_shifted_system_in_sector_equals_dense_solve(abi):
    _shifted_body()


@pytest.mark.slow
@pytest.mark.parametrize("name", ["K-1", "K0"])
def test_sector_feast_roots_match_oracle_hbar(abi, name):
    _roots_body(name)


@pytest.mark.slow
def test_seeded_start_and_returned_vectors(abi, monkeypatch):
    from pymes_b200 import backend as bk
    m, no, nv, f, dVh, T2h = _system()
    sec = _sectors()["K-1"]
    lay_host = sec.packed_index()
    np.random.seed(7)
    want = []
    for _ in range(2):
        a = 0.5 - np.random.rand(nv, no)
        b = (0.5 - np.random.rand(nv, nv, no, no)) * 0.01
        u = np.concatenate([a.ravel(), b.ravel()])[lay_host]
        want.append(u / np.linalg.norm(u))
    fe = _feast(sec, e_c=0.5, e_r=0.2, n_trial=2, max_iter=1)
    seen = []

    class Stop(Exception):
        pass

    def record(plan, diag, zs, rhs, hscale=1.0):
        seen.extend(_n(r) for r in rhs[:2])
        raise Stop
    monkeypatch.setattr(fe, "solve_shifted_systems", record)
    np.random.seed(7)
    with pytest.raises(Stop):
        fe.solve(*_operands(f, dVh, T2h))
    for s, w in zip(seen, want):
        assert _rel(s, w) < 1e-14
    # one iteration; the vectors come back dense, zero outside the sector, tagged, and are taken back
    fe = _feast(sec, e_c=0.5, e_r=0.2, n_trial=2, max_iter=1)
    np.random.seed(7)
    fe.solve(*_operands(f, dVh, T2h))
    m1, m2 = _masks(sec)
    for u1, u2 in zip(fe.u_singles, fe.u_doubles):
        assert tuple(u1.shape) == (nv, no) and tuple(u2.shape) == (nv, nv, no, no)
        assert not _n(u1)[~m1].any() and not _n(u2)[~m2].any() and _n(u2)[m2].any()
        assert bk.momentum_of(u1) == sec.singles_rule() and bk.momentum_of(u2) == sec.doubles_rule()
    again = _feast(sec, e_c=0.5, e_r=0.2, n_trial=4, max_iter=1)
    again.u_singles, again.u_doubles = fe.u_singles, fe.u_doubles
    again.solve(*_operands(f, dVh, T2h))


def test_sector_feast_rejects_what_it_cannot_solve(abi):
    from pymes_b200.model import ueg
    from pymes_b200.solver import rt_eom_ccsd
    m, no, nv, f, dVh, T2h = _system()
    sec = _sectors()["K-1"]
    rng = np.random.default_rng(6)
    ft, dV, T2 = _operands(f, dVh, T2h)
    with pytest.raises(ValueError, match="Fock"):
        _feast(sec).solve(f + 1e-6 * rng.standard_normal(f.shape), dV, T2)
    with pytest.raises(ValueError, match="T2"):
        _feast(sec).solve(ft, dV, _t(T2h + 1e-6 * rng.standard_normal(T2h.shape)))
    m1, m2 = _masks(sec)
    fe = _feast(sec)
    u2 = np.where(m2, 1.0, 0.0)
    u2[np.argwhere(~m2)[0][0], np.argwhere(~m2)[0][1], np.argwhere(~m2)[0][2], np.argwhere(~m2)[0][3]] = 1e-3
    fe.u_singles, fe.u_doubles = [np.where(m1, 1.0, 0.0)], [u2]
    with pytest.raises(ValueError, match="outside the sector"):
        fe.solve(*_operands(f, dVh, T2h))
    with pytest.raises(ValueError, match="no excitation"):
        _feast(ueg.excitation_sector(m, no, (40, 0, 0))).solve(*_operands(f, dVh, T2h))
    small = _sectors()["8th"]
    with pytest.raises(ValueError, match="exceeds"):
        _feast(small, n_trial=40).solve(*_operands(f, dVh, T2h))

    class TwoRanks:
        size, rank = 2, 0
    with pytest.raises(NotImplementedError):
        _feast(sec, comm=TwoRanks(), parallel="rows")
    with pytest.raises(NotImplementedError):
        rt_eom_ccsd.RT_EOM_CCSD(no, sector=sec)


def _systems_run(f, dVh, T2h, comm=None):
    from pymes_b200.model import ueg
    m, no, nv, _parts = _ueg14()
    sec = ueg.excitation_sector(m, no, (-1, 0, 0))
    np.random.seed(5)
    fe = _feast(sec, e_c=float(np.mean(np.diag(f)[no:])), e_r=0.5, n_trial=4, max_iter=2, comm=comm,
                parallel="systems")
    fe.n_nodes = 4
    return np.sort_complex(np.asarray(fe.solve(*_operands(f, dVh, T2h)))), fe


def _systems_worker(rank, world, port, ops, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from tests import abi_emulator, feast_sector_emulator

        class _Patch:
            def setattr(self, obj, name, val):
                setattr(obj, name, val)
        feast_sector_emulator.extend(abi_emulator.install(_Patch()))
        from pymes_b200 import log, parallel
        log.set_quiet(True)
        if rank == 1:
            np.random.seed(12345)   # the start vectors must come from rank 0 alone
        ev, fe = _systems_run(*ops, comm=parallel.Comm())
        assert fe.sys_comm is not None
        q.put((rank, ev, [t["systems_this_rank"] for t in fe.timings]))
    finally:
        dist.destroy_process_group()


@pytest.mark.slow
def test_sector_feast_two_ranks_systems(abi):
    """parallel="systems" over two gloo ranks in a sector == the single-rank Ritz values."""
    import torch.multiprocessing as mp
    m, no, nv, f, dVh, T2h = _system()
    ev1, fe1 = _systems_run(f, dVh, T2h)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 30700 + (os.getpid() % 90)
    procs = [ctx.Process(target=_systems_worker, args=(r, 2, port, (f, dVh, T2h), q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=900) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, ev, nsys in res:
        np.testing.assert_allclose(ev, ev1, rtol=0, atol=1e-12)
        assert nsys == [t["systems_this_rank"] // 2 for t in fe1.timings]


# --------------------------------------------------------------------------
# on the B200
# --------------------------------------------------------------------------
@pytest.mark.gpu
def test_sector_copy_kernels_bit_exact_on_device():
    """pmb_sector_gather / pmb_sector_scatter against torch indexing, bit for bit: n_idx at and
    around one 256-thread block and a sector-sized list, batches up to 64, batch strides wider
    than a row."""
    from pymes_b200 import backend as bk
    rng = np.random.default_rng(21)
    for n_idx in (1, 255, 256, 257, 155120):
        row = max(2 * n_idx, 1000) + 3
        host = np.sort(rng.choice(row, n_idx, replace=False)).astype(np.int64)
        idx = torch.from_numpy(host).cuda()
        for nb in (1, 3, 64):
            if n_idx == 155120 and nb == 64:
                nb = 17
            pitch = row + 5
            buf = torch.from_numpy(rng.standard_normal((nb, pitch))).cuda()
            x = buf[:, :row]
            got = bk.sector_gather(x, idx)
            assert torch.equal(got, x[:, idx]), (n_idx, nb)
            dst = torch.from_numpy(rng.standard_normal((nb, pitch))).cuda()
            want = dst.clone()
            src = torch.from_numpy(rng.standard_normal((nb, n_idx + 7))).cuda()
            want[:, idx] = src[:, :n_idx]
            bk.sector_scatter(src[:, :n_idx], idx, dst[:, :row])
            assert torch.equal(dst, want), (n_idx, nb)
    bk.sector_gather(torch.zeros(64, 4, dtype=torch.float64, device="cuda"), torch.tensor([0, 3]).cuda())
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_compact_sigma_on_device():
    _compact_sigma_body(None)


@pytest.mark.gpu
def test_shifted_system_in_sector_on_device():
    _shifted_body()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["K-1", "K0"])
def test_sector_feast_roots_on_device(name):
    _roots_body(name)


@pytest.mark.gpu
def test_sector_shifted_solve_at_o27_equals_dense():
    """At the benchmark's o = 27 (TC-UEG 54e / 65 plane waves, 3 CCSD sweeps, K = (1,0,0)): one
    shifted solve on compact vectors equals the dense solve of the scattered right-hand side to
    1e-10 relative."""
    import bench
    from pymes_b200 import backend as bk
    from pymes_b200.integral.partition import KEYS
    from pymes_b200.model import ueg
    from pymes_b200.solver import ccsd, eom_ccsd, feast_eom_ccsd
    no = bench.N_ELE // 2
    m = ueg.UEG(bench.N_ELE, no, no, bench.RS)
    m.init_single_basis(6.0)
    m.k_cutoff, m.gamma = bench.K_CUTOFF, None
    fock = bk.asdev(bench.build_fock(m, no))
    dV = m.eval_2b_blocks(no, list(KEYS), bench.tc_parts(m))
    cc = ccsd.CCSD(no)
    cc.setup(fock, dV)
    for _ in range(3):
        cc.sweep()
    T1, T2 = cc._st["T1"], cc._st["T2"]
    ft = cc.get_T1_dressed_fock(fock, T1, dV)
    dVd = cc.get_T1_dressed_V(T1, dV, {k: None for k in eom_ccsd.V_KEYS_USED})
    f, dVh, T2h = _n(ft), {k: _n(dVd[k]) for k in eom_ccsd.V_KEYS_USED}, _n(T2)
    nv = T2h.shape[0]
    sec = ueg.excitation_sector(m, no, (1, 0, 0))
    fs, fd = feast_eom_ccsd.FEAST_EOM_CCSD(no, sector=sec), feast_eom_ccsd.FEAST_EOM_CCSD(no)
    ops_s, ops_d = _operands(f, dVh, T2h), _operands(f, dVh, T2h)
    ps, pd = fs.plan(*ops_s), fd.plan(*ops_d)
    lay = fs.sector_layout(nv)
    d = torch.cat([fd.get_diag_singles(*ops_d).reshape(-1), fd.get_diag_doubles(*ops_d).reshape(-1)])
    rng = np.random.default_rng(13)
    b = rng.standard_normal(lay["n"])
    bd = np.zeros(d.numel())
    bd[lay["host"]] = b
    z = complex(np.mean(np.diag(f)[no:]) + 0.3j)
    xs = fs.solve_shifted_systems(ps, bk.sector_gather(d[None], lay["idx"])[0], [z], [bk.asdev(_t(b))])[0]
    xd = fd.solve_shifted_systems(pd, d, [z], [bk.asdev(_t(bd))])[0]
    cs, cd = _n(xs.re) + 1j * _n(xs.im), _n(xd.re) + 1j * _n(xd.im)
    assert _rel(cs, cd[lay["host"]]) < 1e-10
