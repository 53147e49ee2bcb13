"""Seekable zstd blobs (ZN_CODEC_SEEKABLE) on the CPU: the compressor's window efforts compiled for the host with a
"warp" of one lane (tests/host_emu/host_compress_seekable.cpp), every 128 KiB block a frame of its own and the seek
table the device writes (cz::zstd_seek_table).  Each blob is checked against stock libzstd (whole, and every frame
alone), against a restatement of the seekable format's seek table below, against the oracle's XXH64, and against the
size the packed layout computes (cz::zstd_seekable_size) and zn_compress_bound."""
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
BLOCK = 128 * KIB
EFFORTS = {"zstd-fast": 1, "zstd-mid": 11, "zstd-high": 12}  # levels <= 2, 3..9, 10..19


def parse_seek_table(blob: bytes):
    """The Zstandard seekable format's seek table (contrib/seekable_format/zstd_seekable_compression_format.md in the
    zstd tree), restated: a skippable frame (magic 0x184D2A5E, Frame_Size) that ends the blob, holding Number_Of_Frames
    entries {Compressed_Size u32, Decompressed_Size u32[, Checksum u32]} and the footer {Number_Of_Frames u32,
    Seek_Table_Descriptor u8, Seekable_Magic_Number u32 = 0x8F92EAB1}; descriptor bit 7 = checksums present, bits 6-2
    reserved (zero).  Returns ([(csize, dsize, checksum | None)], offset of the table)."""
    assert len(blob) >= 17
    n, desc, magic = struct.unpack_from("<IBI", blob, len(blob) - 9)
    assert magic == 0x8F92EAB1
    assert desc & 0x7C == 0
    esz = 12 if desc & 0x80 else 8
    start = len(blob) - (8 + esz * n + 9)
    assert start >= 0
    skip_magic, frame_size = struct.unpack_from("<II", blob, start)
    assert skip_magic == 0x184D2A5E and frame_size == esz * n + 9
    entries = []
    for k in range(n):
        e = struct.unpack_from("<III" if esz == 12 else "<II", blob, start + 8 + esz * k)
        entries.append((e[0], e[1], e[2] if esz == 12 else None))
    return entries, start


def check_seekable_blob(O, blob: bytes, data: bytes, bound: int):
    """The checks every seekable blob passes, here and on the GPU (test_gpu_seekable.py)."""
    z = O.libzstd()
    assert len(blob) <= bound
    assert z.decompress(blob, max(len(data), 1)) == data  # concatenated frames, the table skipped
    entries, tab = parse_seek_table(blob)
    assert len(entries) == max(1, -(-len(data) // BLOCK))
    assert sum(e[0] for e in entries) == tab and sum(e[1] for e in entries) == len(data)
    c = d = 0
    for cs, ds, ck in entries:
        frame, content = blob[c:c + cs], data[d:d + ds]
        assert ds == min(BLOCK, len(data) - d)
        assert z.decompress(frame, max(ds, 1)) == content, (c, cs)  # every frame alone
        assert ck == O.xxh64(np.frombuffer(content, np.uint8)) & 0xFFFFFFFF
        c, d = c + cs, d + ds
    return entries


def corpora(O) -> dict:
    c = {"real8m": stdlib_text(8 * MIB), "text": O.gen_text(3 * MIB + 5), "binary": O.gen_binary(MIB + 17),
         "random": O.gen_random(300_000)}
    for n in (0, 1, BLOCK - 1, BLOCK, BLOCK + 1, 8 * MIB + 777):
        c[f"len{n}"] = stdlib_text(n, 4321)
    return c


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu_seek") / "libhostemu_seek.so")
    srcs = [os.path.join(EMU, f) for f in ("host_compress_seekable.cpp", "host_compress.cpp")]
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-x", "c++", *srcs, "-o", so, "-Wno-unknown-pragmas"],
                   check=True, capture_output=True)
    L = C.CDLL(so)
    L.zn_hostemu_compress_seekable.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
    L.zn_hostemu_compress_seekable.restype = C.c_long
    L.zn_hostemu_compress.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]
    L.zn_hostemu_compress.restype = C.c_long
    return L


def emit(emu, fn_codec, d, seekable=True):
    src = np.zeros(d.size + 64, np.uint8)
    src[:d.size] = d
    out = np.zeros(d.size + 28 * (d.size // BLOCK + 1) + 4096, np.uint8)
    if seekable:
        sz = C.c_uint64(0)
        n = emu.zn_hostemu_compress_seekable(fn_codec, src.ctypes.data, d.size, out.ctypes.data, C.byref(sz))
        return out[:n].tobytes(), sz.value
    n = emu.zn_hostemu_compress(fn_codec, src.ctypes.data, d.size, out.ctypes.data)
    return out[:n].tobytes(), n


@pytest.mark.parametrize("effort", list(EFFORTS))
def test_seekable_blobs_decode_frame_by_frame(emu, oracle, effort):
    from znippy_b200 import codec
    for name, d in corpora(oracle).items():
        blob, size = emit(emu, EFFORTS[effort], d)
        assert size == len(blob), (effort, name)
        bound = codec.compress_bound(d.size, codec.CODEC_ZSTD | codec.CODEC_SEEKABLE)
        check_seekable_blob(oracle, blob, d.tobytes(), bound)


def test_empty_slice_layout(emu, oracle):
    blob, _ = emit(emu, 1, np.zeros(0, np.uint8))
    assert len(blob) == 38
    assert blob[:9] == bytes([0x28, 0xB5, 0x2F, 0xFD, 0x20, 0x00, 0x01, 0x00, 0x00])
    assert parse_seek_table(blob)[0] == [(9, 0, oracle.xxh64(np.zeros(0, np.uint8)) & 0xFFFFFFFF)]


def test_envelope_parse_sizes_bare_blobs_from_the_table(emu):
    """zn_envelope_parse (the size decompress_frame and the enveloped batch calls use) of a bare seekable blob is the
    seek table's sum, not its first frame's content size; a damaged table leaves the first frame's size."""
    from znippy_b200 import codec
    for n in (0, 1, BLOCK, BLOCK + 1, 8 * MIB + 777):
        blob, _ = emit(emu, 11, stdlib_text(n, 9))
        env = codec.envelope_parse(blob)
        assert env[:4] == (codec.ENV_BARE, codec.PAYLOAD_ZSTD, 0, len(blob)) and env[4] == n, n
        assert codec.frame_content_size(blob) == n
        bad = bytearray(blob)
        bad[-1] ^= 1  # footer magic
        assert codec.envelope_parse(bytes(bad))[4] == min(n, BLOCK)
        bad = bytearray(blob)
        bad[-(12 + 9)] ^= 1  # last entry's compressed size: the entries no longer add up to the blob
        assert codec.envelope_parse(bytes(bad))[4] == min(n, BLOCK)


@pytest.mark.parametrize("n", [0, 1, BLOCK - 1, BLOCK, BLOCK + 1, 8 * MIB + 777])
def test_compress_bound_is_exact(n):
    """zn_compress_bound of the seekable codec: every block stored raw in its own frame, plus the table."""
    from znippy_b200 import codec
    nb = -(-n // BLOCK)
    want = 38 if n == 0 else n + nb * (13 + 3 + 12) + 17
    assert codec.compress_bound(n, codec.CODEC_ZSTD | codec.CODEC_SEEKABLE) == want


def test_ratio_cost_rehearsal(emu, oracle):
    """One-lane rehearsal of what seekable mode costs on real text (the device's 32-lane parse differs; the bound that
    counts is measured on the GPU, test_gpu_seekable.py): each block loses at most its window's history, and gains a
    13-byte frame header and a 12-byte table entry."""
    d = stdlib_text(8 * MIB)
    for effort, fc in EFFORTS.items():
        plain, _ = emit(emu, fc, d, seekable=False)
        seek, _ = emit(emu, fc, d)
        ratio = len(seek) / len(plain)
        print(f"{effort}: plain {len(plain)} seekable {len(seek)} ({ratio:.4f}x)")
        assert 1.0 < ratio < 1.10, (effort, ratio)
