#!/usr/bin/env python
"""Generate tests/golden/*.json from the COMPILED REFERENCE (oracle/_ref/libref_lz4.so).

Run where the reference sources exist (oracle/Makefile, REF=<path>):
    make -C oracle ref && python tests/golden/make_golden.py
The reference ships no golden compressed vectors for the block codec (SURVEY.md section 8c), so
these fixtures are outputs of the reference itself: every `ret`, `out` and digest below was
produced by lib/lz4.c (v1.10.0, gcc -O3, x86-64) / tests/datagen.c, never by our own code.
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.pyoracle import Reference  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def hand_built_blocks():
    """Hand-built blocks: SURVEY.md Appendix A.1 (+ tests/fuzzer.c:1108-1120 and :223-249)."""
    tail12 = bytes(range(0x62, 0x6E))
    v = []
    v.append((bytes([0x10, 0x41, 0x00, 0x00, 0xC0]) + tail12, [17, 37]))            # offset 0
    v.append((bytes([0x1F, 0x41, 0x01, 0x00, 0x01, 0xC0]) + tail12, [33, 34, 32]))  # RLE
    v.append((bytes([0x1F, 0x41, 0x01, 0x00, 0x01, 0xC0]) + tail12[:-1], [33]))     # truncated
    v.append((bytes([0x1F, 0x41, 0x01, 0x00, 0x01, 0xC0]) + tail12 + b"\x00", [33]))  # extra byte
    v.append((bytes([0x10, 0x41, 0x02, 0x00, 0xC0]) + tail12, [17]))                # offset before start
    v.append((bytes([0x10, 0x41, 0x01, 0x00, 0x40, 0x77, 0x78, 0x79, 0x7A]), [9, 64]))
    v.append((bytes([0x10, 0x41, 0x01, 0x00, 0x50, 0x76, 0x77, 0x78, 0x79, 0x7A]), [10]))
    v.append((bytes([0x00]), [0, 8]))
    v.append((bytes([0x30, 0x78, 0x79, 0x7A]), [3, 2, 100]))
    v.append((bytes([0xF0, 0xFF, 0xFF, 0x10, 0x61, 0x62]), [200]))
    v.append((bytes([0xEE] + [0x00] * 14 + [0x0E, 0x00]), [200]))                   # fuzzer.c:1110-1119
    v.append((bytes([0xF0] + [0xFF] * 40), [200, 100000]))                          # fuzzer.c:223-249 shape
    v.append((bytes([0x1F, 0x01, 0x01, 0x00]), [200]))
    v.append((b"", [0, 10]))
    # offsets 1..9 overlap patterns, long matches
    for off in range(1, 10):
        lits = bytes(range(0x41, 0x41 + 9))
        blk = bytes([0x9F]) + lits + bytes([off, 0x00, 40]) + bytes([0x50]) + b"vwxyz"
        v.append((blk, [9 + 59 + 5, 9 + 59 + 5 + 70, 9 + 59 + 4]))
    return v


def fuzz_blocks(ref, count=400):
    """Seeded corruptions of small valid blocks (the fuzzer.c:588-622 'noisy source' idea)."""
    rng = np.random.default_rng(20260922)
    out = []
    while len(out) < count:
        n = int(rng.choice([16, 40, 90, 200, 400]))
        p = float(rng.choice([0.2, 0.5, 0.9]))
        d = ref.datagen(n, p, int(rng.integers(0, 1 << 30)))
        _, c = ref.compress(d, 1)
        b = bytearray(c)
        for _ in range(int(rng.integers(1, 5))):
            mode = int(rng.integers(0, 4))
            pos = int(rng.integers(0, len(b))) if b else 0
            if mode == 0 and b:
                b[pos] = int(rng.integers(0, 256))
            elif mode == 1 and b:
                b[pos] = int(rng.choice([0, 0xFF, 0xF0, 0x0F, 0x10, 0x1F]))
            elif mode == 2 and len(b) > 4:
                del b[pos:pos + int(rng.integers(1, 4))]
            else:
                b[pos:pos] = bytes(rng.integers(0, 256, int(rng.integers(1, 4)), dtype=np.uint8))
        caps = [n, n + int(rng.integers(1, 90)), max(n - int(rng.integers(1, 20)), 0)]
        out.append((bytes(b), caps))
    return out


def main():
    ref = Reference()

    decode = []
    for blk, caps in hand_built_blocks() + fuzz_blocks(ref):
        for cap in caps:
            r, o = ref.decompress(blk, cap)
            decode.append({"block": blk.hex(), "cap": cap, "ret": r, "out": o.hex() if r >= 0 else None})
    with open(os.path.join(HERE, "kat_decode.json"), "w") as f:
        json.dump({"source": "lz4 v1.10.0 lib/lz4.c LZ4_decompress_safe, gcc -O3 x86-64", "cases": decode}, f)

    comp = []
    small = [b"", b"x", b"a" * 12, b"a" * 13, b"a" * 20, b"abcd" * 8, bytes(range(256)) * 2, b"\x00" * 1000,
             b"ab" * 40 + b"xyz" + b"ab" * 40]
    for s in small:
        for acc in (1, 8):
            r, c = ref.compress(s, acc)
            comp.append({"src": s.hex(), "accel": acc, "ret": r, "out": c.hex()})
            for cap in (r, r - 1, 0):
                r2, c2 = ref.compress(s, acc, cap)
                comp.append({"src": s.hex(), "accel": acc, "cap": cap, "ret": r2, "out": c2.hex()})
    with open(os.path.join(HERE, "kat_compress.json"), "w") as f:
        json.dump({"source": "lz4 v1.10.0 lib/lz4.c LZ4_compress_fast, gcc -O3 x86-64", "cases": comp}, f)

    # datagen buffers: digests of the generator output, of the reference-compressed bytes
    dg = []
    for (n, p, seed) in [(65536, 0.5, 0), (65536, 0.9, 0), (65536, 0.0, 0), (65536, 1.0, 0), (65547, 0.5, 1),
                         (70000, 0.5, 2), (1 << 20, 0.5, 3), (4 << 20, 0.5, 4), (4 << 20, 0.9, 5), (12345, 0.3, 6),
                         (65546, 0.5, 7), (1000, 0.5, 8)]:
        d = ref.datagen(n, p, seed)
        for acc in (1, 8, 32):
            r, c = ref.compress(d, acc)
            dg.append({"size": n, "proba": p, "seed": seed, "accel": acc, "src_sha256": sha(d),
                       "csize": r, "comp_sha256": sha(c)})
    # 64 KB blocks of a 2 MiB P50 buffer (the BASELINE workload shape), accel 1
    d = ref.datagen(2 << 20, 0.5, 0)
    sizes, h = [], hashlib.sha256()
    for i in range(0, len(d), 65536):
        r, c = ref.compress(d[i:i + 65536], 1)
        sizes.append(r)
        h.update(c)
    stream = {"size": 2 << 20, "proba": 0.5, "seed": 0, "block": 65536, "accel": 1, "src_sha256": sha(d),
              "csizes": sizes, "stream_sha256": h.hexdigest()}
    with open(os.path.join(HERE, "datagen_digests.json"), "w") as f:
        json.dump({"source": "tests/datagen.c RDG_genBuffer + lib/lz4.c LZ4_compress_fast (v1.10.0)",
                   "buffers": dg, "stream": stream}, f, indent=0)

    # frames made by LZ4F_compressFrame (independent blocks, no checksums): digests + one small frame verbatim
    frames = []
    for (n, p, seed, bsid, level, csf) in [(0, 0.5, 0, 4, 0, False), (1, 0.5, 0, 4, 0, True), (1000, 0.5, 1, 4, 0, False),
                                           (65536, 0.5, 2, 4, 0, False), (65537, 0.5, 3, 4, 0, True), (200000, 0.5, 4, 4, 0, False),
                                           (200000, 0.5, 4, 7, -3, True), (1 << 20, 0.9, 5, 5, 0, False), (300000, 0.0, 6, 4, 0, False),
                                           ((4 << 20) + 12345, 0.5, 7, 7, 0, True), (3 << 20, 0.5, 8, 6, -9, False),
                                           (70000, 1.0, 9, 4, 1, False)]:
        d = ref.datagen(n, p, seed) if n else np.zeros(0, dtype=np.uint8)
        f = ref.compress_frame(d, bsid, level, csf)
        row = {"size": n, "proba": p, "seed": seed, "bsid": bsid, "level": level, "content_size": csf,
               "frame_size": len(f), "frame_sha256": sha(f), "src_sha256": sha(d)}
        if len(f) <= 1200:
            row["frame_hex"] = f.hex()
        frames.append(row)
    with open(os.path.join(HERE, "frames.json"), "w") as f:
        json.dump({"source": "lz4 v1.10.0 lib/lz4frame.c LZ4F_compressFrame (blockIndependent, no checksums)",
                   "frames": frames}, f, indent=0)

    # one whole reference-compressed 64 KB P50 block as a binary fixture (BASELINE config 1)
    d = ref.datagen(65536, 0.5, 0)
    _, c = ref.compress(d, 1)
    with open(os.path.join(HERE, "p50_seed0_64k.lz4block"), "wb") as f:
        f.write(c)
    print("decode cases", len(decode), "compress cases", len(comp), "datagen rows", len(dg), "block", len(c), "frames", len(frames))
    reference_answers(ref)


def reference_answers(ref):
    """tests/golden/ref_answers.json: the reference's answers to the seeded cases of tests/ref_answers.py"""
    import re
    import subprocess
    import tempfile
    sys.path.insert(0, os.path.dirname(HERE))
    import ref_answers as ra

    ans = {"source": "lz4 v1.10.0: lib/lz4.c, lib/lz4frame.c, tests/datagen.c (gcc -O3 x86-64) and the programs/ "
                     "command-line tool, run on the cases of tests/ref_answers.py",
           "datagen": ra.datagen_records(ref),
           "compress": ra.compress_records(ref, ref),
           "noisy": ra.noisy_records(ref, ref),
           "frames": [ra.frame_record(ref.compress_frame(d, bsid, level, csf)) for d, bsid, level, csf in ra.frame_cases(ref)],
           "fuzz": {str(s): ra.fuzz_records(ref, ref, s) for s in ra.FUZZ_SEEDS}}
    cli = os.path.join(ROOT, "oracle", "_ref", "lz4")
    bench = {}
    with tempfile.TemporaryDirectory() as tmp:
        paths = ra.write_bench_files(ref, tmp)
        for args, idx in ra.BENCH_COMMANDS:
            sub = [paths[i] for i in idx]
            r = subprocess.run([cli] + args + sub, capture_output=True, text=True, timeout=120)
            text = (r.stdout + r.stderr).replace("\r", "\n")
            m = re.findall(r":\s*(\d+) ->\s*(\d+) \(([\d.]+)\),\s*[\d.]+ MB/s,\s*[\d.]+ MB/s", text)
            assert r.returncode == 0 and m, text
            bench[ra.bench_key(args, sub)] = [int(m[-1][0]), int(m[-1][1]), m[-1][2]]
    ans["lz4_bench"] = bench
    with open(ra.GOLDEN, "w") as f:
        json.dump(ans, f, separators=(",", ":"))
        f.write("\n")
    print("reference answers:", {k: len(v) for k, v in ans.items() if k != "source"})


if __name__ == "__main__":
    main()
