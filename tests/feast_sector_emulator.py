"""TEST INFRASTRUCTURE: numpy twins of pmb_sector_gather and pmb_sector_scatter
(include/pymes_b200.h), added together with the entry points of tests/sector_emulator.py by ``extend``."""
import ctypes as C

import numpy as np

from tests import sector_emulator
from tests.abi_emulator import _gather, _val


def _args(n_batch, n_idx, idx, src, dst):
    if n_batch < 1 or n_idx < 1 or not _val(idx) or not _val(src) or not _val(dst):
        return None                                 # PMB_E_BADARG, as the library does
    return np.ctypeslib.as_array((C.c_int64 * n_idx).from_address(_val(idx))).copy()


def pmb_sector_gather(fake, n_batch, n_idx, idx, src, src_bstr, dst, dst_bstr, stream):
    """dst[b*dst_bstr + k] = src[b*src_bstr + idx[k]]."""
    k = _args(n_batch, n_idx, idx, src, dst)
    if k is None:
        return -1
    fake.launches += 1
    for b in range(n_batch):
        vals, _, _ = _gather(_val(src) + 8 * b * src_bstr, k)
        _, win, lo = _gather(_val(dst) + 8 * b * dst_bstr, np.arange(n_idx, dtype=np.int64))
        win[:] = vals
    return 0


def pmb_sector_scatter(fake, n_batch, n_idx, idx, src, src_bstr, dst, dst_bstr, stream):
    """dst[b*dst_bstr + idx[k]] = src[b*src_bstr + k]; every other element of dst is kept."""
    k = _args(n_batch, n_idx, idx, src, dst)
    if k is None:
        return -1
    fake.launches += 1
    for b in range(n_batch):
        vals, _, _ = _gather(_val(src) + 8 * b * src_bstr, np.arange(n_idx, dtype=np.int64))
        _, win, lo = _gather(_val(dst) + 8 * b * dst_bstr, k)
        win[k - lo] = vals
    return 0


def extend(fake):
    """Give an emulated library (``abi_emulator.FakeLib``) the momentum and batched group entry points
    and the two sector copies; returns it."""
    sector_emulator.extend(fake)
    fake.pmb_sector_gather = lambda *a: pmb_sector_gather(fake, *a)
    fake.pmb_sector_scatter = lambda *a: pmb_sector_scatter(fake, *a)
    return fake
