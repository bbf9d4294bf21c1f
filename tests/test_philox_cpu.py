"""The numpy Philox4x32-10 reference (tests/philox_ref.py) against the Random123 known-answer vectors."""
import numpy as np

from philox_ref import draws, keep_mask, philox4x32


def _kat(ctr, key):
    return [int(x) for x in philox4x32(*ctr, *key)]


def test_philox_known_answers():
    assert _kat([0, 0, 0, 0], [0, 0]) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert _kat([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert _kat([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]) == \
        [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_philox_vectorised_matches_scalar_and_carries():
    """The vectorised counter walk equals one call per counter, including the carry from ctr_lo into ctr_hi."""
    seed, base, sid = 0x0123456789ABCDEF, (1 << 32) - 3, 7
    got = draws(26, seed, base, sid)
    want = []
    for i in range(7):
        c = base + i
        want += [int(x) for x in philox4x32(c & 0xFFFFFFFF, c >> 32, sid, 0, seed & 0xFFFFFFFF, seed >> 32)]
    assert got.tolist() == want[:26]
    m = keep_mask(26, 0.5, seed, base, sid)
    assert m.tolist() == [int(((w >> 8) * 2.0 ** -24) < 0.5) for w in want[:26]]
    assert np.all(keep_mask(100, 1.0, 1, 0, 0) == 1) and np.all(keep_mask(100, 0.0, 1, 0, 0) == 0)
