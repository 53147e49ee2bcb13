"""The decoders with a stop point (range reads, zs::StopAt), on the CPU: the same decode_frames / LZ4 frame code the
k_decode<.., true> kernels run, compiled for the host with a team of one (tests/host_emu/host_decode_prefix.cpp).  For
every stop at 0, 1, every block boundary +-1 and the full size: the prefix equals the oracle's full decode, `produced`
lies in [stop, stop + one block], and the bytes past `produced` are untouched.  A corruption after the stop block is
never seen; one at or before it gives the status of the full decode."""
import base64
import ctypes as C
import json
import os
import random
import struct
import subprocess

import numpy as np
import pytest

EMU = os.path.join(os.path.dirname(__file__), "host_emu")
GOLD = os.path.join(os.path.dirname(__file__), "golden")
CANARY = 0xA5
NO_STOP = 0xFFFFFFFF  # the emulator decodes in full, as k_decode without a stop


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu_prefix") / "libhostemu_prefix.so")
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-x", "c++", os.path.join(EMU, "host_decode_prefix.cpp"),
                    "-o", so, "-Wno-unknown-pragmas"], check=True, capture_output=True)
    L = C.CDLL(so)
    L.zn_hostemu_decode_prefix.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_uint32, C.c_void_p, C.c_uint32,
                                           C.POINTER(C.c_uint32)]
    return L


def decode(emu, blob, cap, stop, lz4_block=False):
    a = np.frombuffer(blob, np.uint8)
    out = np.full(cap + 4096, CANARY, np.uint8)
    n = C.c_uint32(0)
    st = emu.zn_hostemu_decode_prefix(a.ctypes.data, a.size, int(lz4_block), stop, out.ctypes.data, cap, C.byref(n))
    assert st != 0 or (out[n.value:] == CANARY).all(), "bytes written past `produced`"
    return st, n.value, out[:n.value].tobytes()


def blocks(blob):
    """(compressed end, decoded size or None when only the decoder knows it) of every data block, in order, across
    Zstandard / LZ4 frames and skippable frames."""
    out, ip = [], 0
    while ip < len(blob):
        magic = struct.unpack_from("<I", blob, ip)[0]
        if magic & 0xFFFFFFF0 == 0x184D2A50:
            ip += 8 + struct.unpack_from("<I", blob, ip + 4)[0]
        elif magic == 0x184D2204:
            flg = blob[ip + 4]
            ip += 7 + (8 if flg & 0x08 else 0)
            while True:
                w = struct.unpack_from("<I", blob, ip)[0]
                ip += 4
                if w == 0:
                    break
                n = w & 0x7FFFFFFF
                ip += n + (4 if flg & 0x10 else 0)
                out.append((ip, n if w >> 31 else None))
            ip += 4 if flg & 0x04 else 0
        else:
            assert magic == 0xFD2FB528
            fhd = blob[ip + 4]
            single, did, fcs = (fhd >> 5) & 1, fhd & 3, fhd >> 6
            ip += 5 + (0 if single else 1) + (0, 1, 2, 4)[did] + ((1 if single else 0), 2, 4, 8)[fcs]
            while True:
                bh = int.from_bytes(blob[ip:ip + 3], "little")
                last, typ, size = bh & 1, (bh >> 1) & 3, bh >> 3
                ip += 3 + (1 if typ == 1 else size)
                out.append((ip, size if typ < 2 else None))
                if last:
                    break
            ip += 4 if fhd & 0x04 else 0
    return out


def block_ends(emu, blob, full):
    """Decoded end of every block: the decoder's own stops, matched against the walker's sizes where it knows them."""
    ends, p = [], 0
    while p < len(full):
        st, p2, out = decode(emu, blob, len(full), p + 1)
        assert st == 0 and p2 > p and out == full[:p2]
        ends.append(p2)
        p = p2
    res, it, cur = [], iter(ends), 0
    for cend, size in blocks(blob):
        if size == 0:
            res.append((cend, cur))
            continue
        prev, cur = cur, next(it)
        assert size is None or cur - prev == size, (cur, size)
        res.append((cend, cur))
    assert next(it, None) is None
    return res  # [(compressed end, decoded end)]


def cases(O):
    z, l = O.libzstd(), O.liblz4()
    rt = O.real_text(1_000_000)
    out = []
    for f in json.load(open(os.path.join(GOLD, "frames.json")))["frames"]:
        blob = base64.b64decode(f["blob_b64"])
        if f["codec"] == "lz4block":
            out.append((f["name"], blob, None, f["out_len"], True))
        else:
            out.append((f["name"], blob, None, f["out_len"], False))
    for lvl in (1, 3, 19, 22):
        out.append((f"realtext_l{lvl}", z.compress(rt, lvl), rt.tobytes(), rt.size, False))
    for indep in (False, True):
        for bsid in (4, 5):
            d = rt[:700_000]
            out.append((f"lz4f_indep{int(indep)}_bs{bsid}", l.compress_frame(d, block_size_id=bsid, independent=indep,
                                                                            block_checksum=True, content_checksum=True),
                        d.tobytes(), d.size, False))
    out.append(("lz4f_incompressible", l.compress_frame(O.gen_random(300_000), block_size_id=4), O.gen_random(300_000).tobytes(),
                300_000, False))
    d = rt[:300_000]
    out.append(("lz4_raw_block", l.compress_block(d), d.tobytes(), d.size, True))
    multi = z.compress(rt[:200_000], 3, checksum=True) + b"\x50\x2a\x4d\x18\x03\x00\x00\x00abc" + \
        z.compress(rt[200_000:500_000], 19) + z.compress(rt[500_000:600_000], 1)
    out.append(("multi_frame_skippable", multi, rt[:600_000].tobytes(), 600_000, False))
    raw_rle = np.concatenate([O.gen_random(300_000), np.zeros(400_000, np.uint8), O.gen_random(50_000)])
    out.append(("raw_and_rle_blocks", z.compress(raw_rle, 3), raw_rle.tobytes(), raw_rle.size, False))
    return out


def full_bytes(O, blob, want, size, lz4_block):
    if want is not None:
        return want
    if lz4_block:
        rc, o = O.lz4_block_decompress(blob, size)
    elif blob[:4] == b"\x04\x22\x4d\x18":
        rc, o = O.lz4_frame_decompress(blob, size)
    else:
        rc, o = O.zstd_decompress(blob, size)
    assert rc == 0 and len(o) == size
    return o


def test_prefix_decode_at_every_block_boundary(emu, oracle):
    O = oracle
    for name, blob, want, size, lz4_block in cases(O):
        full = full_bytes(O, blob, want, size, lz4_block)
        if lz4_block:  # one block: decodes whole whatever the stop
            for stop in (0, 1, size // 2, size):
                st, p, out = decode(emu, blob, size, stop, lz4_block=True)
                assert st == 0 and p == size and out == full, name
            continue
        bmax = 1 << (8 + 2 * ((blob[5] >> 4) & 7)) if blob[:4] == b"\x04\x22\x4d\x18" else 128 << 10
        ends = [e for _, e in block_ends(emu, blob, full)] if size else []
        stops = {0, 1, size} | {e + d for e in ends for d in (-1, 0, 1)}
        for stop in sorted(s for s in stops if 0 <= s <= size):
            st, p, out = decode(emu, blob, size, stop)
            assert st == 0, (name, stop, st)
            assert out == full[:p], (name, stop)
            assert stop <= p <= stop + bmax, (name, stop, p)
            if stop and stop in ends:  # a stop on a block end decodes exactly that far
                assert p == stop, (name, stop, p)


def test_prefix_decode_stops_before_the_frame_ends(emu, oracle):
    """A stop past the end of the frames: S_SIZE_MISMATCH, as the kernel reports a row shorter than the range needs."""
    d = oracle.real_text(100_000)
    blob = oracle.libzstd().compress(d, 3)
    st, p, _ = decode(emu, blob, 200_000, 150_000)
    assert st == 5 and p == d.size


@pytest.mark.parametrize("name", ["realtext_l3", "realtext_l19", "lz4f_indep0_bs4", "multi_frame_skippable"])
def test_corruption_after_the_stop_block_is_unseen(emu, oracle, name):
    O = oracle
    case = next(c for c in cases(O) if c[0] == name)
    _, blob, full, size, _ = case
    bl = block_ends(emu, blob, full)
    rnd = random.Random(7)
    failures = 0
    for k in (0, len(bl) // 2, len(bl) - 2):
        cend, dend = bl[k]
        cstart = bl[k - 1][0] if k else 0
        # after the stop block: never read, so never seen
        for _ in range(20):
            c = bytearray(blob)
            c[rnd.randrange(cend, len(blob))] ^= 1 << rnd.randrange(8)
            st, p, out = decode(emu, bytes(c), size, dend)
            assert st == 0 and p == dend and out == full[:dend], (name, k)
        # at or before it: exactly what the full decode reports, whenever the full decode fails before the stop
        for _ in range(40):
            c = bytearray(blob)
            c[rnd.randrange(cstart, cend)] ^= 1 << rnd.randrange(8)
            st, p, out = decode(emu, bytes(c), size, dend)
            fst, fp, fout = decode(emu, bytes(c), size, NO_STOP)
            assert out[:min(p, fp)] == fout[:min(p, fp)]
            if st != 0:
                assert st == fst, (name, k)
                failures += 1
            if fst != 0 and fp < dend:
                assert st == fst, (name, k)
    assert failures > 0, name
