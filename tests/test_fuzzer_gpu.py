"""The fuzz loop of the reference's tests/fuzzer.c on the drop-in entry points, on a GPU.

LZ4_compress_default, LZ4_compress_fast and LZ4_decompress_safe of lz4_b200/liblz4_b200.so run the seeded
cycles of tests/ref_answers.py: per cycle, compressed data must decode to the input, truncated / overlong
capacities and inputs must fail exactly where the contract says, nothing may be written past a capacity
(tests/fuzzer.c:479-727), and every return value and output must equal what the reference's own
lib/lz4.c returned for the same cycle (tests/golden/ref_answers.json).
"""
import pytest

import ref_answers as ra
from oracle.pyoracle import _Codec


class DropIn(_Codec):
    """the oracle's compress / decompress surface (guard bytes past every capacity) over the drop-in C functions;
    acceleration 1 goes through LZ4_compress_default"""

    def __init__(self, lib):
        self._bound = lib.LZ4_compressBound
        self._compress = lambda s, d, n, cap, acc: (lib.LZ4_compress_default(s, d, n, cap) if acc == 1
                                                    else lib.LZ4_compress_fast(s, d, n, cap, acc))
        self._decompress = lib.LZ4_decompress_safe


@pytest.mark.gpu
@pytest.mark.parametrize("seed", ra.FUZZ_SEEDS)
def test_reference_fuzzer_on_the_drop_in_entry_points(seed, oracle):
    from lz4_b200 import _lib
    got = ra.fuzz_records(oracle, DropIn(_lib.load()), seed)
    want = ra.load()["fuzz"][str(seed)]
    assert len(got) == len(want)
    for cycle, (g, w) in enumerate(zip(got, want)):
        n, _, rets, _ = g
        assert rets[0] > 0 and rets[1] > 0 and rets[2] == 0, (cycle, g)          # compress; one byte too little room
        assert rets[3] == n and rets[4] == n and rets[5] < 0, (cycle, g)         # capacity exact, +1, -1
        assert g == w, (cycle, g, w)
