"""TEST INFRASTRUCTURE: numpy twin of pmb_group_contract_batched (include/pymes_b200.h), added
together with the entry points of tests/momentum_emulator.py by ``extend``."""
from tests import momentum_emulator


class _Slice:
    """A pmb_group_t of one right-hand side, shaped like the ``byref`` the emulator reads."""

    def __init__(self, g):
        self._obj = g


def pmb_group_contract_batched(fake, dref, stream):
    """Right-hand side b: pmb_group_contract with A + b a_bstr, B + b b_bstr, C + b c_bstr."""
    d = dref._obj
    if d.n_batch < 1 or d.g.n_tiles < 0 or (d.c_bstr == 0 and d.n_batch > 1):
        return -1                                   # PMB_E_BADARG, as the library does
    if d.g.n_tiles == 0:
        fake.launches += 1
        return 0
    for b in range(d.n_batch):
        one = type(d.g).from_buffer_copy(d.g)
        one.A, one.B, one.C = d.g.A + 8 * b * d.a_bstr, d.g.B + 8 * b * d.b_bstr, d.g.C + 8 * b * d.c_bstr
        momentum_emulator.pmb_group_contract(fake, _Slice(one), stream)
    fake.launches -= d.n_batch - 1                  # one launch for the whole batch
    return 0


def extend(fake):
    """Give an emulated library (``abi_emulator.FakeLib``) the momentum entry points and the batched
    group product; returns it."""
    momentum_emulator.extend(fake)
    fake.pmb_group_contract_batched = lambda *a: pmb_group_contract_batched(fake, *a)
    return fake
