"""The host Philox4x32-10 of the oracle (oracle/philox.py) against the published Random123 known-answer vectors.

The device streams (csrc/philox.cuh) are checked against this oracle; these vectors tie the oracle itself to the
published algorithm, so that a drift of both sides together cannot pass unnoticed."""
import numpy as np
import pytest

from oracle.philox import philox4x32

M = 0xFFFFFFFF

#: (counter c0..c3, key k0, k1) -> output x0..x3, Philox4x32-10 (Random123 kat_vectors)
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((M, M, M, M), (M, M), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


@pytest.mark.parametrize("ctr, key, want", KAT)
def test_philox4x32_10_matches_random123_known_answers(ctr, key, want):
    got = philox4x32(*ctr, *key)
    assert [int(x) for x in got] == list(want)
    # the same counter as one element of an array, the way the oracle draws whole path ranges
    arr = [np.array([0, c, 0], dtype=np.uint64) for c in ctr]
    assert [int(x[1]) for x in philox4x32(*arr, *key)] == list(want)
