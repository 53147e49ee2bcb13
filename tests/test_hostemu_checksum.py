"""Frames with content checksums (ZN_CODEC_CHECKSUM) on the CPU: the compressor compiled for the host with a "warp" of
one lane and the frame assembly restated (tests/host_emu/host_compress_checksum.cpp).  Every frame is checked against
stock libzstd and liblz4 with checksum checking on, its stored checksum against the oracle's XXH64 / XXH32, its length
against the packed layout's size and zn_compress_bound.  The read-side row check (xxh_row_bad) is held to liblz4's and
libzstd's verdicts on LZ4 frames with block and content checksums."""
import ctypes as C
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

EMU = os.path.join(os.path.dirname(__file__), "host_emu")
sys.path.insert(0, os.path.dirname(__file__))
from test_hostemu_compress_long import stdlib_text  # noqa: E402

KIB, MIB = 1024, 1 << 20
LENGTHS = [0, 1, 15, 16, 17, 31, 32, 33, 128 * KIB - 1, 128 * KIB, 128 * KIB + 1, 8 * MIB]
CODECS = {"lz4": 2, "zstd-fast": 1, "zstd-mid": 11, "zstd-high": 12}


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu_ck") / "libhostemu_ck.so")
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-x", "c++", os.path.join(EMU, "host_compress_checksum.cpp"),
                    "-o", so, "-Wno-unknown-pragmas"], check=True, capture_output=True)
    L = C.CDLL(so)
    L.zn_hostemu_compress_checksum.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
    L.zn_hostemu_compress_checksum.restype = C.c_long
    L.zn_hostemu_row_bad.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
    L.zn_hostemu_row_bad.restype = C.c_int
    L.zn_hostemu_xxh.argtypes = [C.c_int, C.c_void_p, C.c_uint64]
    L.zn_hostemu_xxh.restype = C.c_uint64
    return L


def emit(emu, fc, d):
    src = np.zeros(d.size + 64, np.uint8)
    src[:d.size] = d
    out = np.zeros(d.size + d.size // 1024 + 4096, np.uint8)
    sz = C.c_uint64(0)
    n = emu.zn_hostemu_compress_checksum(fc, src.ctypes.data, d.size, out.ctypes.data, C.byref(sz))
    return out[:n].tobytes(), sz.value


def row_bad(emu, blob: bytes, content: bytes) -> bool:
    b = np.frombuffer(blob, np.uint8).copy()
    c = np.frombuffer(content, np.uint8).copy() if content else np.zeros(1, np.uint8)
    return bool(emu.zn_hostemu_row_bad(b.ctypes.data, b.size, c.ctypes.data, len(content)))


def lib_accepts(O, blob: bytes, n: int, lz4: bool) -> bool:
    try:
        (O.liblz4().decompress_frame if lz4 else O.libzstd().decompress)(blob, max(n, 1))
        return True
    except RuntimeError:
        return False


@pytest.mark.parametrize("name", list(CODECS))
def test_checksummed_frames_decode_under_stock_libraries(emu, oracle, name):
    from znippy_b200 import codec
    lz4 = CODECS[name] == 2
    base = codec.CODEC_LZ4 if lz4 else codec.CODEC_ZSTD
    for n in LENGTHS:
        d = stdlib_text(n, 77)
        blob, size = emit(emu, CODECS[name], d)
        assert size == len(blob), (name, n)
        assert len(blob) <= codec.compress_bound(n, base | codec.CODEC_CHECKSUM), (name, n)
        stored = struct.unpack_from("<I", blob, len(blob) - 4)[0]
        if lz4:
            assert blob[4] & 0x04 and not blob[4] & 0x10  # content checksum, no block checksums
            assert oracle.liblz4().decompress_frame(blob, max(n, 1)) == d.tobytes()
            assert stored == oracle.xxh32(d)
        else:
            assert blob[4] == (0x24 if n == 0 else 0xE4)
            assert oracle.libzstd().decompress(blob, max(n, 1)) == d.tobytes()
            assert stored == oracle.xxh64(d) & 0xFFFFFFFF
        assert not row_bad(emu, blob, d.tobytes()), (name, n)
        if n:  # one flipped content byte: both libraries reject the frame, and so does the row check
            bad = bytearray(d.tobytes())
            bad[n // 2] ^= 0x20
            assert row_bad(emu, blob, bytes(bad)), (name, n)
            flipped = bytearray(blob)
            flipped[-4] ^= 1
            assert not lib_accepts(oracle, bytes(flipped), n, lz4), (name, n)
            assert row_bad(emu, bytes(flipped), d.tobytes()), (name, n)


def test_empty_zstd_frame_is_libzstds(emu, oracle):
    blob, _ = emit(emu, 1, np.zeros(0, np.uint8))
    assert blob == bytes.fromhex("28b52ffd2400010000 99e9d851".replace(" ", ""))
    assert blob == oracle.libzstd().compress(b"", 3, checksum=True)


@pytest.mark.parametrize("n", LENGTHS)
def test_compress_bound_adds_four_bytes(n):
    from znippy_b200 import codec
    for base in (codec.CODEC_ZSTD, codec.CODEC_LZ4):
        assert codec.compress_bound(n, base | codec.CODEC_CHECKSUM) == codec.compress_bound(n, base) + 4


def test_scalar_hashes_match_the_oracle(emu, oracle):
    for n in LENGTHS + [3, 7, 63, 64, 65]:
        d = np.ascontiguousarray(stdlib_text(n, 5))
        p = d.ctypes.data if n else np.zeros(1, np.uint8).ctypes.data
        assert emu.zn_hostemu_xxh(64, p, n) == oracle.xxh64(d), n
        assert emu.zn_hostemu_xxh(32, p, n) == oracle.xxh32(d), n


@pytest.mark.parametrize("block_checksum,content_checksum,independent,bsid",
                         [(True, False, True, 4), (False, True, False, 5), (True, True, False, 6), (True, True, True, 7)])
def test_lz4_row_check_matches_liblz4(emu, oracle, block_checksum, content_checksum, independent, bsid):
    """liblz4 frames with block and/or content checksums, linked and independent blocks of 64 KiB - 4 MiB: the row check
    accepts them, and under bit flips in either checksum field gives liblz4's verdict."""
    L = oracle.liblz4()
    d = stdlib_text(5 * MIB + 333, 11).tobytes()
    blob = L.compress_frame(d, block_size_id=bsid, independent=independent, content_checksum=content_checksum,
                            block_checksum=block_checksum)
    assert not row_bad(emu, blob, d)
    rng = np.random.default_rng(bsid)
    fields = []
    if content_checksum:
        fields.append(len(blob) - 4)
    if block_checksum:  # the first block's checksum follows its data
        hdr = 7 + (8 if blob[4] & 0x08 else 0)
        n0 = struct.unpack_from("<I", blob, hdr)[0] & 0x7FFFFFFF
        fields.append(hdr + 4 + n0)
    for f in fields:
        for _ in range(4):
            bad = bytearray(blob)
            bad[f + int(rng.integers(4))] ^= 1 << int(rng.integers(8))
            assert not lib_accepts(oracle, bytes(bad), len(d), True)
            assert row_bad(emu, bytes(bad), d)


def test_zstd_row_check_is_unchanged_for_libzstd_frames(emu, oracle):
    z = oracle.libzstd()
    d = stdlib_text(3 * MIB + 5, 3).tobytes()
    one = z.compress(d, 3, checksum=True)
    multi = z.compress(d[:MIB], 3, checksum=True) + z.compress(d[MIB:], 1, checksum=True)
    for blob in (one, multi):
        assert not row_bad(emu, blob, d)
        bad = bytearray(blob)
        bad[-1] ^= 0x80
        assert row_bad(emu, bytes(bad), d)
    plain = z.compress(d, 3)
    assert not row_bad(emu, plain, d[:-1] + b"?")  # no checksum announced: nothing to check
