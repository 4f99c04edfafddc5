"""TEST INFRASTRUCTURE: numpy twins of pmb_group_contract and pmb_momentum_residue
(include/pymes_b200.h), added to the emulated library of tests/abi_emulator.py by ``extend``."""
import ctypes as C

import numpy as np

from tests.abi_emulator import _gather, _offsets, _val, _window


def pmb_group_contract(fake, dref, stream):
    """Per tile, C[c_row[r] + c_col[n]] += alpha * sum_k A[a_row[r] + a_ent[k]] B[b_ent[k] + b_col[n]]."""
    d = dref._obj
    fake.launches += 1
    if d.n_tiles == 0:
        return 0
    ints = lambda ptr, n, ct: np.ctypeslib.as_array((ct * n).from_address(ptr))
    tiles = ints(d.tiles, 6 * d.n_tiles, C.c_int32).reshape(-1, 6)
    assert tiles[:, [1, 3, 5]].min() >= 1 and max(tiles[:, 1].max(), tiles[:, 5].max()) <= 32
    n_r = int((tiles[:, 0] + tiles[:, 1]).max())
    n_e = int((tiles[:, 2] + tiles[:, 3]).max())
    n_c = int((tiles[:, 4] + tiles[:, 5]).max())
    a_row, c_row = ints(d.a_row, n_r, C.c_int64), ints(d.c_row, n_r, C.c_int64)
    a_ent, b_ent = ints(d.a_ent, n_e, C.c_int64), ints(d.b_ent, n_e, C.c_int64)
    b_col, c_col = ints(d.b_col, n_c, C.c_int64), ints(d.c_col, n_c, C.c_int64)
    seen = set()
    for r0, rn, e0, en, c0, cn in tiles:
        A, _, _ = _gather(d.A, (a_row[r0:r0 + rn, None] + a_ent[None, e0:e0 + en]).reshape(-1))
        B, _, _ = _gather(d.B, (b_ent[e0:e0 + en, None] + b_col[None, c0:c0 + cn]).reshape(-1))
        offs = (c_row[r0:r0 + rn, None] + c_col[None, c0:c0 + cn]).reshape(-1)
        assert not seen & set(offs.tolist()), "an element belongs to two tiles"
        seen |= set(offs.tolist())
        old, win, lo = _gather(d.C, offs)
        win[offs - lo] = old + d.alpha * (A.reshape(rn, en) @ B.reshape(en, cn)).reshape(-1)
    return 0


def pmb_momentum_residue(fake, ndim, ext, strides, x, keys, out, stream):
    """out[0] = max |x| over the elements whose per-axis labels do not sum to zero."""
    fake.launches += 1
    ext = [int(ext[i]) for i in range(ndim)]
    offs = _offsets(ext[::-1], [int(strides[i]) for i in range(ndim)][::-1])
    vals, _, _ = _gather(_val(x), offs)
    lab = np.ctypeslib.as_array((C.c_int64 * sum(ext)).from_address(_val(keys)))
    tot, start = np.zeros(1, dtype=np.int64), 0
    for e in ext:
        tot = (tot[:, None] + lab[start:start + e][None, :]).reshape(-1)
        start += e
    bad = np.abs(vals[tot != 0])
    _window(_val(out), 1)[0] = bad.max() if bad.size else 0.0
    return 0


def extend(fake):
    """Give an emulated library (``abi_emulator.FakeLib``) the two entry points; returns it."""
    fake.pmb_group_contract = lambda *a: pmb_group_contract(fake, *a)
    fake.pmb_momentum_residue = lambda *a: pmb_momentum_residue(fake, *a)
    return fake
