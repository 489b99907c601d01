"""lz4_b200.lz4bench (SURVEY.md section 8 f-2): the `lz4 -b` harness.

CPU part: the codec-agnostic harness is driven by an oracle-backed codec (test infrastructure) and
its block split / level rule / sizes / ratio / result lines are compared with what the REFERENCE TOOL
`lz4 -b# -i0` (programs/*.c) printed for the same files (tests/golden/ref_answers.json).
GPU part: the same comparison for the product codec (GpuCodec).
"""
import os
import re
import time

import numpy as np
import pytest

import ref_answers as ra
from lz4_b200 import lz4bench
from oracle.pyoracle import Oracle


class OracleCodec(lz4bench.Codec):
    """bench.c's serial per-block loops, on the CPU oracle (checker only)."""

    def __init__(self, corrupt_at=None):
        self.codec = Oracle()
        self.corrupt_at = corrupt_at

    def setup(self, src, blocks, acceleration):
        self.src = bytes(src)
        self.blocks = blocks
        self.accel = acceleration
        self.comp = [b""] * len(blocks)
        self.csz = [0] * len(blocks)
        self.res = [b""] * len(blocks)
        self.rsz = [0] * len(blocks)

    def compress_passes(self, n):
        t0 = time.perf_counter_ns()
        for _ in range(n):
            for i, (off, sz) in enumerate(self.blocks):
                self.csz[i], self.comp[i] = self.codec.compress(self.src[off:off + sz], self.accel)
        return time.perf_counter_ns() - t0

    def compressed_sizes(self):
        return list(self.csz)

    def decompress_passes(self, n):
        t0 = time.perf_counter_ns()
        for _ in range(n):
            for i, (_, sz) in enumerate(self.blocks):
                r, o = self.codec.decompress(self.comp[i], sz)
                self.rsz[i], self.res[i] = r, bytes(o)
        return time.perf_counter_ns() - t0

    def decoded_sizes(self):
        return list(self.rsz)

    def verify(self):
        out = bytearray(b"".join(self.res))
        if self.corrupt_at is not None:
            out[self.corrupt_at] ^= 0x40
        a, b = np.frombuffer(self.src, dtype=np.uint8), np.frombuffer(bytes(out), dtype=np.uint8)
        if len(a) != len(b):
            return min(len(a), len(b))
        d = np.nonzero(a != b)[0]
        return int(d[0]) if len(d) else -1


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    return ra.write_bench_files(Oracle(), tmp_path_factory.mktemp("benchfiles"))


def ref_bench(args, paths):
    """What the reference tool printed for `lz4 <args> <files>`: (srcSize, cSize, ratio text)."""
    src, csz, ratio = ra.load()["lz4_bench"][ra.bench_key(args, paths)]
    return src, csz, ratio


def test_split_blocks_never_straddle_files():
    assert lz4bench.split_blocks([10, 0, 25, 8], 10) == [(0, 10), (10, 10), (20, 10), (30, 5), (35, 8)]
    assert lz4bench.split_blocks([], 64) == []
    assert lz4bench.split_blocks([65536], 65536) == [(0, 65536)]
    assert lz4bench.split_blocks([65537], 65536) == [(0, 65536), (65536, 1)]


def test_level_and_block_flags():
    assert [lz4bench.level_to_acceleration(l) for l in (1, 0, -1, -3, -64)] == [1, 1, 2, 4, 65]   # bench.c:229
    for hc in (2, 3, 9, 12):                                                                 # lz4hc.h:47
        with pytest.raises(ValueError):
            lz4bench.level_to_acceleration(hc)
    assert [lz4bench.block_size_from_flag(v) for v in (4, 5, 6, 7, 32, 65536)] == [65536, 262144, 1 << 20, 4 << 20, 32, 65536]
    with pytest.raises(ValueError):
        lz4bench.block_size_from_flag(8)


def test_fastest_pass_rule_and_loop_sizing():
    """bench.c:480-492: the speed comes from the fastest pass; loops are re-sized to ~1 s of work."""
    per_pass = iter([400_000_000, 250_000_000, 300_000_000, 260_000_000, 500_000_000, 500_000_000, 500_000_000])
    calls = []

    def run(n):
        calls.append(n)
        return next(per_pass) * n

    fastest, passes, total = lz4bench._timed_loop(run, 3, first_loops=1)
    assert fastest == 250_000_000
    assert calls[0] == 1 and calls[1] == 1_000_000_000 // 400_000_000 + 1 and calls[2] == 1_000_000_000 // 250_000_000 + 1
    assert total > 3_000_000_000 and passes == sum(calls)
    # -i0: exactly one pass
    calls.clear()
    fastest, passes, _ = lz4bench._timed_loop(lambda n: calls.append(n) or 7 * n, 0, first_loops=50)
    assert calls == [1] and passes == 1 and fastest == 7


@pytest.mark.parametrize("level_flag,level,block_flag,block", [
    ("-b1", 1, "-B4", 65536), ("-b1", 1, None, 0), ("-b0", 0, "-B5", 262144), ("-b1", 1, "-B1000", 1000),
])
def test_harness_matches_reference_tool(files, level_flag, level, block_flag, block):
    for subset in (files[:1], files):
        src = b"".join(open(p, "rb").read() for p in subset)
        sizes = [os.path.getsize(p) for p in subset]
        name = os.path.basename(subset[0]) if len(subset) == 1 else " %u files" % len(subset)
        res = lz4bench.bench_mem(OracleCodec(), src, sizes, name, level, block, nb_seconds=0)
        rsrc, rcsz, rratio = ref_bench([level_flag, "-i0"] + ([block_flag] if block_flag else []), subset)
        assert res.error == 0
        assert (res.src_size, res.c_size) == (rsrc, rcsz)
        assert "%5.3f" % res.ratio == rratio
        line = res.line()
        assert re.match(r"^ ?%d#.{17} :\s*%d ->\s*%d \(%s\),\s*[\d.]+ MB/s,\s*[\d.]+ MB/s$" % (level, rsrc, rcsz, rratio), line), line
        assert res.quiet_line().startswith("-%-3i%11i (%s)" % (level, rcsz, rratio))


def test_fast_levels_match_reference_tool(files):
    src = open(files[0], "rb").read()
    for fast in (1, 3, 9):
        res = lz4bench.bench_mem(OracleCodec(), src, [len(src)], "p50.bin", -fast, 65536, nb_seconds=0)
        assert (res.src_size, res.c_size) == ref_bench(["--fast=%d" % fast, "-b", "-i0", "-B4"], files[:1])[:2]


def test_verify_reports_corruption(files, capsys):
    src = open(files[0], "rb").read()
    res = lz4bench.bench_mem(OracleCodec(corrupt_at=70000), src, [len(src)], "p50.bin", 1, 65536, nb_seconds=0)
    assert res.error == 1
    err = capsys.readouterr().err
    assert "Invalid Checksum" in err and "Decoding error at pos 70000 (block 1, sub 0, pos 4464)" in err


def test_cli_refuses_hc_and_needs_files():
    with pytest.raises(SystemExit):
        lz4bench.main([])
    with pytest.raises(ValueError):
        lz4bench.level_to_acceleration(9)


@pytest.mark.gpu
def test_gpu_codec_matches_reference_tool(files):
    codec = lz4bench.GpuCodec()
    for subset, level, level_args, block_flag, block in ((files[:1], 1, ["-b1"], "-B4", 65536),
                                                         (files, 1, ["-b1"], "-B4", 65536),
                                                         (files, -3, ["--fast=3", "-b"], "-B4", 65536),
                                                         (files[:2], 1, ["-b1"], None, 0)):
        src = b"".join(open(p, "rb").read() for p in subset)
        sizes = [os.path.getsize(p) for p in subset]
        res = lz4bench.bench_mem(codec, src, sizes, "x", level, block, nb_seconds=0)
        assert res.error == 0
        assert (res.src_size, res.c_size) == ref_bench(level_args + ["-i0"] + ([block_flag] if block_flag else []), subset)[:2]
        assert res.c_ns > 0 and res.d_ns > 0
