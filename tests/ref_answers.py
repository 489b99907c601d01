"""Seeded cases whose answers were recorded from the compiled reference into tests/golden/ref_answers.json.

Every function below derives its cases from fixed seeds and returns one JSON-able record per case.
tests/golden/make_golden.py runs them on the reference (oracle/_ref/libref_lz4.so and the reference
`lz4` tool); the tests run them on the oracle or on the GPU entry points and compare the records, so
the comparison with the reference holds on machines that have none of its sources.

`gen` is anything with the oracle's `datagen`; `codec` anything with the oracle's `compress` /
`decompress` surface (oracle.pyoracle._Codec: both check that nothing is written past a capacity).
"""
import hashlib
import json
import os
import struct

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_answers.json")


def load():
    with open(GOLDEN) as f:
        return json.load(f)


def _digest(h):
    return h.hexdigest()[:16]


def _feed(h, ret, out=b""):
    h.update(struct.pack("<i", int(ret)))
    h.update(bytes(out))


# ---- generator and block codec (tests/test_oracle_vs_ref.py) -----------------------------------------------

DATAGEN_CASES = [(65536, 0.5, 0), (1 << 20, 0.9, 3), (100000, 0.0, 7), (300000, 1.0, 2), (1, 0.5, 0), (777777, 0.25, 99)]


def datagen_records(gen):
    return [hashlib.sha256(gen.datagen(n, p, s).tobytes()).hexdigest() for (n, p, s) in DATAGEN_CASES]


def compress_records(gen, codec):
    """Per trial: compress (full capacity, then six smaller ones) and decode the result at six capacities.
    Record: [n, proba, accel, returns, digest of the returns and of every successful output]."""
    rng = np.random.default_rng(1)
    sizes = [0, 1, 5, 12, 13, 14, 20, 64, 100, 1000, 4096, 65535, 65536, 65546, 65547, 65548, 70000, 200000, 1 << 20]
    recs = []
    for trial in range(250):
        n = int(rng.choice(sizes))
        p = float(rng.choice([0.0, 0.1, 0.5, 0.9, 1.0]))
        d = gen.datagen(n, p, trial)
        acc = int(rng.choice([1, 1, 1, 2, 8, 32, 1000, 65537, -3]))
        h = hashlib.sha256()
        r, c = codec.compress(d, acc)
        rets = [r]
        _feed(h, r, c)
        for cap in [r, r - 1, r - 7, max(r // 2, 0), 1, 0]:
            a = codec.compress(d, acc, cap)
            rets.append(a[0])
            _feed(h, a[0], a[1] if a[0] > 0 else b"")
        for cap in [n, n + 1, n + 100, n - 1, n - 10, n // 2]:
            if cap < 0:
                continue
            a = codec.decompress(c, cap)
            rets.append(a[0])
            _feed(h, a[0], a[1] if a[0] >= 0 else b"")
        recs.append([n, p, acc, rets, _digest(h)])
    return recs


def noisy_records(gen, codec):
    """tests/fuzzer.c:588-622 idea: corrupted blocks decoded at three capacities.
    Record per trial: [returns, digest of the compressed block, the returns and every successful output]."""
    rng = np.random.default_rng(2)
    recs = []
    for trial in range(1500):
        n = int(rng.choice([20, 64, 100, 300, 1000, 5000, 70000]))
        d = gen.datagen(n, float(rng.choice([0.1, 0.5, 0.9])), 1000 + trial)
        _, br = codec.compress(d, int(rng.choice([1, 4])))
        h = hashlib.sha256(br)
        b = bytearray(br)
        for _ in range(int(rng.integers(1, 6))):
            mode = rng.integers(0, 4)
            pos = int(rng.integers(0, len(b)))
            if mode == 0:
                b[pos] = int(rng.integers(0, 256))
            elif mode == 1:
                b[pos] = int(rng.choice([0, 0xFF, 0xF0, 0x0F, 0x10, 0x1F]))
            elif mode == 2:
                del b[pos:pos + int(rng.integers(1, 4))]
            else:
                b[pos:pos] = bytes(rng.integers(0, 256, int(rng.integers(1, 4)), dtype=np.uint8))
        if not b:
            recs.append([[], _digest(h)])
            continue
        rets = []
        for cap in [n, n + int(rng.integers(0, 80)), max(n - int(rng.integers(0, 80)), 0)]:
            r, o = codec.decompress(bytes(b), cap)
            rets.append(r)
            _feed(h, r, o if r >= 0 else b"")
        recs.append([rets, _digest(h)])
    return recs


# ---- frame layer (tests/test_frame.py) ---------------------------------------------------------------------

def frame_cases(gen):
    """(source bytes, block size id, level, content-size flag) of the seeded random frame configurations"""
    rng = np.random.default_rng(4)
    for trial in range(25):
        n = int(rng.choice([0, 1, 100, 65535, 65536, 65537, 150000, 700000]))
        d = gen.datagen(n, float(rng.choice([0.0, 0.5, 0.9])), trial).tobytes() if n else b""
        bsid = int(rng.choice([0, 4, 5, 6, 7]))
        level = int(rng.choice([0, 1, -1, -5]))
        csf = bool(rng.integers(0, 2))
        yield d, bsid, level, csf


def frame_record(frame):
    return [len(frame), hashlib.sha256(frame).hexdigest()]


# ---- the `lz4 -b` tool (tests/test_lz4bench.py) ------------------------------------------------------------

BENCH_FILES = [("p50.bin", 300000, 0.5, 0), ("p90.bin", 70001, 0.9, 1), ("tiny.bin", 40, 0.5, 2), ("p20.bin", 131072, 0.2, 3)]


def write_bench_files(gen, directory):
    paths = []
    for name, n, p, seed in BENCH_FILES:
        path = os.path.join(str(directory), name)
        with open(path, "wb") as f:
            f.write(gen.datagen(n, p, seed).tobytes())
        paths.append(path)
    return paths


def bench_key(args, paths):
    """The command line `lz4 <args> <files>` with the files by name, as the key of its recorded result."""
    return " ".join(list(args) + [os.path.basename(p) for p in paths])


# every command line the tests compare with: (options, indices into BENCH_FILES)
BENCH_COMMANDS = (
    [(["-b1", "-i0", "-B4"], s) for s in ([0], [0, 1, 2, 3])] +
    [(["-b1", "-i0"], s) for s in ([0], [0, 1, 2, 3], [0, 1])] +
    [(["-b0", "-i0", "-B5"], s) for s in ([0], [0, 1, 2, 3])] +
    [(["-b1", "-i0", "-B1000"], s) for s in ([0], [0, 1, 2, 3])] +
    [(["--fast=%d" % f, "-b", "-i0", "-B4"], [0]) for f in (1, 3, 9)] +
    [(["--fast=3", "-b", "-i0", "-B4"], [0, 1, 2, 3])]
)


# ---- fuzz cycles on the drop-in entry points (tests/test_fuzzer_gpu.py) ------------------------------------

FUZZ_SEEDS = (1, 2, 2026)


def fuzz_records(gen, codec, seed, cycles=16):
    """The checks of the fuzz loop of the reference's tests/fuzzer.c (:479-727), one cycle per block of up to
    128 KB: compress at acceleration 1 and at a random one, and with one byte too little room; decode at the exact
    capacity, one byte more, one and ten bytes less; decode the block one byte short and one byte long; decode a
    noisy copy.  Record per cycle: [size, accel, returns, digest of the returns and every successful output]."""
    rng = np.random.default_rng(seed)
    recs = []
    for _ in range(cycles):
        n = int(rng.integers(1, 1 << 17))
        d = gen.datagen(n, float(rng.choice([0.0, 0.2, 0.5, 0.8, 1.0])), int(rng.integers(0, 1 << 30)))
        acc = int(rng.choice([1, 2, 8, 64]))
        h = hashlib.sha256()
        rets = []

        def note(res, ok):
            rets.append(res[0])
            _feed(h, res[0], res[1] if ok(res[0]) else b"")

        c1 = codec.compress(d, 1)
        note(c1, lambda r: r > 0)
        cf = codec.compress(d, acc)
        note(cf, lambda r: r > 0)
        note(codec.compress(d, acc, cf[0] - 1), lambda r: r > 0)
        blk = c1[1]
        for cap in (n, n + 1, n - 1, n - 10):
            if cap >= 0:
                note(codec.decompress(blk, cap), lambda r: r >= 0)
        note(codec.decompress(blk[:-1], n), lambda r: r >= 0)
        note(codec.decompress(blk + b"\0", n), lambda r: r >= 0)
        noisy = bytearray(blk)
        for _ in range(int(rng.integers(1, 4))):
            noisy[int(rng.integers(0, len(noisy)))] = int(rng.integers(0, 256))
        note(codec.decompress(bytes(noisy), n), lambda r: r >= 0)
        recs.append([n, acc, rets, _digest(h)])
    return recs
