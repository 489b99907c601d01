"""Frame layer (SURVEY.md section 8 f-1).  CPU part: the Python frame restatement (tests/frame_oracle.py,
on the oracle's block codec) reproduces the reference's LZ4F_compressFrame output (golden digests).  GPU part: LZ4B200_compressFrame_host emits the same bytes and
LZ4B200_decompressFrame_host decodes reference frames; unsupported / malformed frames give the
documented error codes."""
import hashlib
import struct

import numpy as np
import pytest

import frame_oracle as fo
import ref_answers as ra
from conftest import load_golden


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


@pytest.fixture(scope="module")
def frames():
    return load_golden("frames.json")["frames"]


def _src(oracle, row):
    return oracle.datagen(row["size"], row["proba"], row["seed"]).tobytes() if row["size"] else b""


def test_xxh32_known_answers():
    # published XXH32 test values for short inputs (seed 0): "" -> 0x02CC5D05, "a" -> 0x550D7456, "abc" -> 0x32D153FF
    assert fo.xxh32_short(b"") == 0x02CC5D05
    assert fo.xxh32_short(b"a") == 0x550D7456
    assert fo.xxh32_short(b"abc") == 0x32D153FF


def test_frame_restatement_matches_reference_golden(oracle, frames):
    for row in frames:
        d = _src(oracle, row)
        assert sha(d) == row["src_sha256"]
        f = fo.compress_frame(oracle, d, row["bsid"], row["level"], row["content_size"])
        assert len(f) == row["frame_size"] and sha(f) == row["frame_sha256"], row
        if "frame_hex" in row:
            assert f.hex() == row["frame_hex"]
        back, used = fo.decompress_frame(oracle, f)
        assert back == d and used == len(f)


def test_frame_restatement_vs_compiled_reference(oracle):
    """seeded random configurations against the reference's LZ4F_compressFrame frames (tests/ref_answers.py)"""
    want = ra.load()["frames"]
    for trial, (d, bsid, level, csf) in enumerate(ra.frame_cases(oracle)):
        f = fo.compress_frame(oracle, d, bsid, level, csf)
        assert ra.frame_record(f) == want[trial], (trial, len(d), bsid, level, csf)
        assert fo.decompress_frame(oracle, f) == (d, len(f))


# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_frames_byte_identical_and_roundtrip(oracle, frames):
    from lz4_b200 import frame
    from oracle.pyoracle import Reference, have_reference
    ref = Reference() if have_reference() else None
    for row in frames:
        d = _src(oracle, row)
        f = frame.compress_frame(d, row["bsid"], row["level"], row["content_size"])
        assert len(f) == row["frame_size"] and sha(f) == row["frame_sha256"], row
        assert frame.decompress_frame(f, max(len(d), 1)) == d
        if ref is not None and ref.have_frame():
            assert ref.decompress_frame(f, max(len(d), 1)) == d
            assert frame.decompress_frame(ref.compress_frame(d, row["bsid"], row["level"], row["content_size"]), len(d) + 5) == d


@pytest.mark.gpu
def test_gpu_frame_random_configs_vs_restatement(oracle):
    from lz4_b200 import frame
    rng = np.random.default_rng(8)
    for trial in range(14):
        n = int(rng.choice([0, 1, 13, 65535, 65536, 65537, 300000, 1 << 20, (1 << 22) + 7]))
        d = oracle.datagen(n, float(rng.choice([0.0, 0.5, 0.9])), 50 + trial).tobytes() if n else b""
        bsid = int(rng.choice([0, 4, 5, 6, 7]))
        level = int(rng.choice([0, 1, -2, -31]))
        csf = bool(rng.integers(0, 2))
        f = frame.compress_frame(d, bsid, level, csf)
        assert f == fo.compress_frame(oracle, d, bsid, level, csf), (n, bsid, level, csf)
        assert frame.decompress_frame(f, max(n, 1)) == d


@pytest.mark.gpu
def test_gpu_frame_irregular_and_rejected_inputs(oracle):
    from lz4_b200 import frame
    from lz4_b200.frame import Lz4FrameError
    d = oracle.datagen(200000, 0.5, 77).tobytes()
    good = fo.compress_frame(oracle, d, 4, 0, True)
    # a frame whose non-final blocks are short (what a flushing streaming compressor produces)
    desc = bytes([(1 << 6) | (1 << 5), 4 << 4])
    hand = bytearray(struct.pack("<I", 0x184D2204) + desc + bytes([(fo.xxh32_short(desc) >> 8) & 0xFF]))
    pieces = [d[:1000], d[1000:70000 - 3], d[70000 - 3:70000], d[70000:]]
    for pce in pieces:
        for i in range(0, len(pce), 65536):
            blk = pce[i:i + 65536]
            r, c = oracle.compress(blk, 1, len(blk) - 1)
            hand += (struct.pack("<I", len(blk) | 0x80000000) + blk) if (r == 0 or r >= len(blk)) else (struct.pack("<I", r) + c)
    hand += struct.pack("<I", 0)
    assert frame.decompress_frame(bytes(hand), len(d)) == d
    # destination too small
    with pytest.raises(Lz4FrameError) as e:
        frame.decompress_frame(good, len(d) - 1)
    assert e.value.code == -5
    # malformed: bad magic, bad header checksum, truncated, content size mismatch, block bigger than the maximum
    for bad in (b"\x00" + good[1:], good[:6] + bytes([good[6] ^ 1]) + good[7:], good[:len(good) // 2], good[:-4]):
        with pytest.raises(Lz4FrameError) as e:
            frame.decompress_frame(bad, len(d))
        assert e.value.code == -3
    wrong = bytearray(fo.compress_frame(oracle, d, 4, 0, True)); wrong[6] ^= 0x10
    wrong[14] = (fo.xxh32_short(bytes(wrong[4:14])) >> 8) & 0xFF       # valid header, wrong content size
    with pytest.raises(Lz4FrameError) as e:
        frame.decompress_frame(bytes(wrong), len(d))
    assert e.value.code == -3
    # unsupported: linked blocks / content checksum / block checksum (frames made by hand-editing the flags)
    for flg in ((1 << 6), (1 << 6) | (1 << 5) | (1 << 2), (1 << 6) | (1 << 5) | (1 << 4)):
        dsc = bytes([flg, 4 << 4])
        fr = struct.pack("<I", 0x184D2204) + dsc + bytes([(fo.xxh32_short(dsc) >> 8) & 0xFF]) + struct.pack("<I", 0)
        with pytest.raises(Lz4FrameError) as e:
            frame.decompress_frame(fr, 10)
        assert e.value.code == -4
    with pytest.raises(Lz4FrameError) as e:
        frame.compress_frame(d, 4, 3, False)                             # LZ4HC level
    assert e.value.code == -4


# ------------------------------------------------------------------------------------------
# host logic of the frame layer that needs no GPU: header validation, error codes, empty frames
# ------------------------------------------------------------------------------------------
def _frame_lib():
    from lz4_b200 import build, _lib
    build.build()
    return _lib.load()


def _decode_rc(lib, frame_bytes, cap=64):
    import ctypes as C
    src = np.frombuffer(bytes(frame_bytes), dtype=np.uint8)
    dst = np.zeros(max(cap, 1), dtype=np.uint8)
    used = C.c_int64(-1)
    return int(lib.LZ4B200_decompressFrame_host(src.ctypes.data, len(src), dst.ctypes.data, cap, C.byref(used))), used.value


def test_frame_header_validation_needs_no_gpu(oracle):
    lib = _frame_lib()
    empty = fo.compress_frame(oracle, b"", 4, 0, False)                   # header + EndMark (lz4frame.c:1222)
    assert _decode_rc(lib, empty) == (0, len(empty))
    assert _decode_rc(lib, empty + b"trailing")[0] == 0                    # bytes after the frame are not consumed
    assert _decode_rc(lib, empty[:6])[0] == -3                             # shorter than minFHSize
    assert _decode_rc(lib, b"\x05" + empty[1:])[0] == -3                   # magic
    assert _decode_rc(lib, empty[:6] + bytes([empty[6] ^ 0xFF]) + empty[7:])[0] == -3     # header checksum
    assert _decode_rc(lib, empty[:7])[0] == -3                             # no EndMark
    assert _decode_rc(lib, struct.pack("<I", 0x184D2A50) + b"\x04\x00\x00\x00abcd")[0] == -4   # skippable frame
    for flg, bd, want in (((1 << 6), 4 << 4, -4),                          # linked blocks
                          ((1 << 6) | (1 << 5) | (1 << 2), 4 << 4, -4),    # content checksum
                          ((1 << 6) | (1 << 5) | (1 << 4), 4 << 4, -4),    # block checksum
                          ((2 << 6) | (1 << 5), 4 << 4, -3),               # version
                          ((1 << 6) | (1 << 5) | 2, 4 << 4, -3),           # reserved FLG bit
                          ((1 << 6) | (1 << 5), 3 << 4, -3),               # block size id < 4 (lz4frame.c:1409)
                          ((1 << 6) | (1 << 5), (4 << 4) | 1, -3)):        # reserved BD bits
        dsc = bytes([flg, bd])
        fr = struct.pack("<I", 0x184D2204) + dsc + bytes([(fo.xxh32_short(dsc) >> 8) & 0xFF]) + struct.pack("<I", 0)
        assert _decode_rc(lib, fr)[0] == want, (flg, bd)
    # a block header announcing more than the maximum block size (lz4frame.c:1745)
    dsc = bytes([(1 << 6) | (1 << 5), 4 << 4])
    fr = struct.pack("<I", 0x184D2204) + dsc + bytes([(fo.xxh32_short(dsc) >> 8) & 0xFF]) + struct.pack("<I", 65537) + b"\0" * 65537
    assert _decode_rc(lib, fr)[0] == -3


def test_frame_compress_argument_rules_need_no_gpu():
    lib = _frame_lib()
    assert lib.LZ4B200_compressFrameBound(0, 0) == 19 + 4 + 4 + 4
    assert lib.LZ4B200_compressFrameBound(65536, 4) >= 7 + 4 + 65536 + 4
    assert lib.LZ4B200_compressFrameBound(100, 3) == -1 and lib.LZ4B200_compressFrameBound(-1, 4) == -1
    src = np.zeros(100, dtype=np.uint8)
    dst = np.zeros(4096, dtype=np.uint8)
    assert lib.LZ4B200_compressFrame_host(src.ctypes.data, 100, dst.ctypes.data, 4096, 4, 2, 0) == -4    # LZ4HC level
    assert lib.LZ4B200_compressFrame_host(src.ctypes.data, 100, dst.ctypes.data, 50, 4, 0, 0) == -5     # dst too small
    assert lib.LZ4B200_compressFrame_host(src.ctypes.data, 100, dst.ctypes.data, 4096, 9, 0, 0) == -1    # block size id
    # an empty input needs no block and therefore no GPU: header + EndMark, content-size flag dropped (lz4frame.c:445)
    r = lib.LZ4B200_compressFrame_host(None, 0, dst.ctypes.data, 4096, 4, 0, 1)
    assert r == 11 and dst[:11].tobytes().hex() == "04224d1860408200000000"
