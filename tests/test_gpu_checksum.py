"""Frame checksums on the GPU.  Write side (ZN_CODEC_CHECKSUM): compress_batch and compress plans end every frame in its
content checksum (k_slice_xxh), judged by stock libzstd / liblz4 and the oracle's XXH64 / XXH32.  Read side: LZ4 block
and content checksums are verified where a row's digest is compared, on both tree kernels and behind every decode class,
with liblz4's verdict; checksummed zstd rows checked by a whole CTA keep libzstd's verdict.  Archives written with
checksums round-trip, and a flipped checksum byte in the file is a decode error on extract."""
import os
import random
import struct
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(__file__))
from test_hostemu_compress_long import stdlib_text  # noqa: E402

KIB, MIB = 1024, 1 << 20
LENGTHS = [0, 1, 15, 16, 17, 31, 32, 33, 128 * KIB - 1, 128 * KIB, 128 * KIB + 1, 8 * MIB]


@pytest.fixture(scope="module")
def codec():
    from znippy_b200 import codec
    codec.default_ctx()
    return codec


def _batch(datas, first=16):
    offs, cur = [], first
    for d in datas:
        offs.append(cur)
        cur += len(d) + 3
    src = np.zeros(cur + 1, np.uint8)
    for o, d in zip(offs, datas):
        src[o:o + len(d)] = np.frombuffer(bytes(d), np.uint8) if not isinstance(d, np.ndarray) else d
    return src, offs, [len(d) for d in datas]


def _pack(blobs):
    offs = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])[:-1].astype(np.uint64)
    return np.frombuffer(b"".join(blobs) or b"\0", np.uint8), offs


def _decode(codec, blobs, lens, comp=None):
    """decode_verify_batch of bare frames -> (status, outputs)"""
    buf, offs = _pack(blobs)
    ooff = np.concatenate([[0], np.cumsum([(x + 15) & ~15 for x in lens])])[:-1]
    out = np.zeros(int(ooff[-1]) + (lens[-1] if lens else 0) + 16, np.uint8)
    st, _ = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], comp or [1] * len(blobs), lens, None, out, ooff)
    return st, [out[ooff[i]:ooff[i] + lens[i]].tobytes() for i in range(len(lens))]


def _corpora(O):
    c = [stdlib_text(n, 31) for n in LENGTHS]
    c += [O.gen_binary(3 * MIB + 7), O.gen_random(300_000), O.real_text(MIB + 5)]
    return c


def _stored_ok(O, blob, d, lz4):
    stored = struct.unpack_from("<I", blob, len(blob) - 4)[0]
    return stored == (O.xxh32(d) if lz4 else O.xxh64(d) & 0xFFFFFFFF)


# ------------------------------------------------------------------------------------------------- write side

@pytest.mark.parametrize("name,level", [("zstd", 1), ("zstd", 3), ("zstd", 19), ("zstd", 22), ("lz4", 1)])
def test_compress_batch_checksummed_frames(codec, oracle, name, level):
    O = oracle
    lz4 = name == "lz4"
    base = codec.CODEC_LZ4 if lz4 else codec.CODEC_ZSTD
    datas = _corpora(O)
    src, offs, lens = _batch(datas)
    blobs, dg, st = codec.compress_batch(src, offs, lens, level, base | codec.CODEC_CHECKSUM)
    plain, pdg, _ = codec.compress_batch(src, offs, lens, level, base)
    assert not st.any() and np.array_equal(dg, pdg)
    for d, b, p in zip(datas, blobs, plain):
        n = d.size
        assert len(b) <= codec.compress_bound(n, base | codec.CODEC_CHECKSUM)
        assert _stored_ok(O, b, d, lz4), (name, n)
        if lz4:
            assert O.liblz4().decompress_frame(b, max(n, 1)) == d.tobytes()
            assert b[4] == 0x6C and b[:4] + b[5:14] == p[:4] + p[5:14] and b[15:-4] == p[15:], n  # same blocks
        else:
            assert O.libzstd().decompress(b, max(n, 1)) == d.tobytes()
            if n:
                assert b[4] == 0xE4 and b[:4] + b[5:-4] == p[:4] + p[5:], n  # the same blocks as without the flag
            else:
                assert b == O.libzstd().compress(b"", 3, checksum=True)
    # and the library's own decode checks what it wrote
    st2, outs = _decode(codec, blobs, lens)
    assert not st2.any() and all(o == d.tobytes() for o, d in zip(outs, datas))


@pytest.mark.parametrize("envelope", [False, True])
@pytest.mark.parametrize("name,level", [("zstd", 1), ("zstd", 19), ("zstd", 22), ("lz4", 1)])
def test_plan_equals_compress_batch(codec, oracle, name, level, envelope):
    import torch
    from test_gpu_compress_plan import _blobs, _check_packed, _run
    base = codec.CODEC_LZ4 if name == "lz4" else codec.CODEC_ZSTD
    datas = _corpora(oracle)
    src, offs, lens = _batch(datas)
    want, wdg, _ = codec.compress_batch(src, offs, lens, level, base | codec.CODEC_CHECKSUM)
    plan = codec.N.Plan.compress(codec.default_ctx(), offs, lens, level=level, codec=base, envelope=envelope, checksum=True)
    blobs, boffs, dst = _blobs(*_run(torch, plan, torch.from_numpy(src).cuda()))
    _check_packed(blobs, boffs, dst)
    st, dg = plan.results()
    assert not st.any() and np.array_equal(dg, wdg)
    pc = codec.PAYLOAD_LZ4_FRAME if name == "lz4" else codec.PAYLOAD_ZSTD
    for d, w, b in zip(datas, want, blobs):
        if envelope:
            w = codec.envelope_wrap(codec.PAYLOAD_RAW, d.size, d.tobytes()) if len(w) >= d.size else codec.envelope_wrap(pc, d.size, w)
        assert b == w
    plain = codec.N.Plan.compress(codec.default_ctx(), offs, lens, level=level, codec=base, envelope=envelope)
    _run(torch, plain, torch.from_numpy(src).cuda())
    assert plan.launches() == plain.launches() + 1  # the slice checksum kernel
    assert plan.last_ms()[1] > 0


def test_envelope_raw_decision_counts_the_checksum(codec, oracle):
    """A slice whose plain frame is 1-4 bytes shorter than the slice is stored as a frame without the flag and RAW with
    it: the packed layout sizes the frame with its 4-byte checksum."""
    import torch
    from test_gpu_compress_plan import _blobs, _run
    n = 20_000
    rng = np.random.default_rng(4)
    cands = []
    for L in range(4, 120):  # random bytes whose tail repeats an earlier run of L bytes: each L saves a little more
        d = rng.integers(0, 256, n, dtype=np.uint8)
        d[n - L:] = d[1000:1000 + L]
        cands.append(d)
    src, offs, lens = _batch(cands)
    plain, _, _ = codec.compress_batch(src, offs, lens, 3, codec.CODEC_ZSTD)
    hit = [i for i, p in enumerate(plain) if n - 4 <= len(p) < n]
    assert hit, sorted({len(p) - n for p in plain})
    i = hit[0]
    s2, o2, l2 = _batch([cands[i]])
    for checksum, payload in ((False, codec.PAYLOAD_ZSTD), (True, codec.PAYLOAD_RAW)):
        plan = codec.N.Plan.compress(codec.default_ctx(), o2, l2, level=3, envelope=True, checksum=checksum)
        blobs, _, _ = _blobs(*_run(torch, plan, torch.from_numpy(s2).cuda()))
        assert codec.envelope_parse(blobs[0])[1] == payload, checksum
        assert codec.decompress_frame(blobs[0]) == cands[i].tobytes()
        assert codec.CompressCtx(3, envelope=True, checksum=checksum).compress(cands[i]) == blobs[0]


def test_checksum_with_seekable_is_refused_everywhere(codec, oracle, tmp_path):
    import ctypes as C

    from znippy_b200 import archive
    from znippy_b200._native import NativeError, Plan, lib, ptr, u64
    d = oracle.gen_text(1000)
    word = codec.CODEC_ZSTD | codec.CODEC_SEEKABLE | codec.CODEC_CHECKSUM
    with pytest.raises(NativeError):
        codec.compress_batch(d, [0], [d.size], 3, word)
    with pytest.raises(ValueError):
        Plan.compress(codec.default_ctx(), [0], [d.size], level=3, seekable=True, checksum=True)
    o, l = u64([0]), u64([d.size])
    for w in (word, word | codec.N.CODEC_ENVELOPE):
        assert not lib().zn_plan_compress(codec.default_ctx().handle, 1, ptr(o), ptr(l), 3, w, 0)
        assert not lib().zn_archive_writer_create(codec.default_ctx().handle, str(tmp_path / "w.znippy").encode(), 0, 3, w, 0)
    with pytest.raises(ValueError):
        codec.CompressCtx(3, seekable=True, checksum=True)
    with pytest.raises(ValueError):
        archive.compress_stream(str(tmp_path / "x.znippy"), False, level=3, seekable=True, checksum=True)
    (tmp_path / "in").mkdir()
    (tmp_path / "in" / "a.txt").write_bytes(d.tobytes())
    with pytest.raises(ValueError):
        archive.compress_dir(str(tmp_path / "in"), str(tmp_path / "y.znippy"), level=3, seekable=True, checksum=True)
    err = C.create_string_buffer(256)
    rep = (C.c_uint64 * 8)()
    assert lib().zn_archive_compress_dir(codec.default_ctx().handle, str(tmp_path / "in").encode(), str(tmp_path / "z.znippy").encode(),
                                         0, 3, word, 0, 1, C.byref(rep), err, 256) == codec.N.ZN_E_ARG
    assert b"SEEKABLE" in err.value
    # the flag alone, on both codecs, is accepted by every layer
    for base in (codec.CODEC_ZSTD, codec.CODEC_LZ4):
        assert codec.CompressCtx(3, codec=base, checksum=True).compress(d)


# ------------------------------------------------------------------------------------------------- read side: LZ4

def _lz4_rows(O):
    """(frame, content) rows of liblz4 frames with block and/or content checksums, linked and independent, 64 KiB - 4 MiB
    blocks, sized for every decode class: pattern rows <= 64 KiB (one-warp teams, small tree), pattern rows of 300 KiB
    (128-thread teams, large tree), incompressible rows >= 512 KiB (block-parallel kernel), large pattern rows (fused
    kernel), text rows (pipeline, handed back)."""
    L = O.liblz4()
    rows = []
    flags = [(True, False), (False, True), (True, True)]
    for k, (bc, cc) in enumerate(flags):
        for indep in (True, False):
            for bsid in (4, 5, 6, 7):
                kw = dict(block_size_id=bsid, independent=indep, content_checksum=cc, block_checksum=bc)
                for d in (O.gen_binary(60 * KIB + k, 7 * k), O.gen_binary(300 * KIB + bsid, bsid), O.gen_random(600 * KIB + bsid),
                          O.gen_binary(2 * MIB + 3, k), stdlib_text(700 * KIB + bsid, k)):
                    c = d.tobytes()
                    rows.append((L.compress_frame(c, **kw), c))
    return rows


def test_lz4_checksums_verified_on_every_class(codec, oracle):
    from znippy_b200._native import Plan
    import torch
    rows = _lz4_rows(oracle)
    blobs, contents = [r[0] for r in rows], [r[1] for r in rows]
    lens = [len(c) for c in contents]
    st, outs = _decode(codec, blobs, lens)
    assert not st.any() and outs == contents
    # route check: the same batch as a device plan
    buf, boffs = _pack(blobs)
    ooff = np.concatenate([[0], np.cumsum([(x + 15) & ~15 for x in lens])])[:-1]
    digests = b"".join(oracle.blake3(c) for c in contents)
    plan = Plan.decode_verify(codec.default_ctx(), boffs, [len(b) for b in blobs], [1] * len(blobs), ooff, lens, digests)
    d_buf = torch.from_numpy(buf.copy()).cuda()
    d_out = torch.zeros(int(ooff[-1]) + lens[-1] + 16, dtype=torch.uint8, device="cuda")
    plan.run(d_buf.data_ptr(), d_out.data_ptr())
    pst, _ = plan.results()
    assert not pst.any()
    counts = plan.class_counts()
    print("class counts [pipeline, fused, big raw, small, mid]:", counts)
    assert counts[2] > 0 and counts[3] > 0 and counts[4] > 0
    assert any(n <= 64 * KIB for n in lens) and any(n > 64 * KIB for n in lens)  # both tree kernels
    # one flipped bit in a checksum field: that row is a decode error, its neighbours are untouched
    rnd = random.Random(3)
    bad, want = list(blobs), []
    for i, b in enumerate(blobs):
        if i % 3:
            want.append(0)
            continue
        flg = b[4]
        fields = ([len(b) - 4] if flg & 0x04 else [])
        if flg & 0x10:
            hdr = 7 + (8 if flg & 0x08 else 0)
            n0 = struct.unpack_from("<I", b, hdr)[0] & 0x7FFFFFFF
            fields.append(hdr + 4 + n0)
        f = rnd.choice(fields)
        bb = bytearray(b)
        bb[f + rnd.randrange(4)] ^= 1 << rnd.randrange(8)
        bad[i] = bytes(bb)
        want.append(codec.S_DECODE_ERROR)
    st, outs = _decode(codec, bad, lens)
    assert st.tolist() == want
    for i in range(len(bad)):
        if want[i] == 0:
            assert outs[i] == contents[i]


@pytest.mark.parametrize("size", [200 * KIB, 8 * MIB])
def test_lz4_bit_flip_fuzz_matches_liblz4(codec, oracle, size):
    L = oracle.liblz4()
    c = stdlib_text(size, 8).tobytes()
    base = L.compress_frame(c, block_size_id=4, independent=False, content_checksum=True, block_checksum=True)
    rnd = random.Random(size)
    fz = [base]
    for _ in range(63 if size > MIB else 255):
        b = bytearray(base)
        b[rnd.randrange(len(b))] ^= 1 << rnd.randrange(8)
        fz.append(bytes(b))
    st, outs = _decode(codec, fz, [len(c)] * len(fz))
    for i, b in enumerate(fz):
        try:
            ok = L.decompress_frame(b, len(c) + 1) == c
        except RuntimeError:
            ok = False
        assert (st[i] == 0) == ok, (i, st[i])
        if st[i] == 0:
            assert outs[i] == c
    assert st[0] == 0


# ------------------------------------------------------------------------------------------------- read side: zstd, CTA check

def test_zstd_large_rows_keep_libzstds_verdict(codec, oracle):
    O = oracle
    z = O.libzstd()
    c = O.real_text(8 * MIB).tobytes()
    one = z.compress(c, 3, checksum=True)
    multi = b"".join(z.compress(c[k:k + 2 * MIB], 1, checksum=True) for k in range(0, len(c), 2 * MIB))
    rnd = random.Random(12)
    rows = [one, multi]
    for base in (one, multi):
        ends = [len(base) - 4] if base is one else []
        if base is multi:
            p = 0
            for k in range(4):
                p += len(z.compress(c[k * 2 * MIB:(k + 1) * 2 * MIB], 1, checksum=True))
                ends.append(p - 4)
        for e in ends:  # each frame's checksum field
            b = bytearray(base)
            b[e + rnd.randrange(4)] ^= 1 << rnd.randrange(8)
            rows.append(bytes(b))
        for _ in range(24):  # anywhere
            b = bytearray(base)
            b[rnd.randrange(len(b))] ^= 1 << rnd.randrange(8)
            rows.append(bytes(b))
    st, outs = _decode(codec, rows, [len(c)] * len(rows))
    for i, b in enumerate(rows):
        rc, _ = O.zstd_decompress(b, len(c))
        assert (st[i] == 0) == (rc == 0), (i, st[i], rc)
    assert st[0] == 0 and st[1] == 0 and st[2] == codec.S_DECODE_ERROR and outs[0] == c and outs[1] == c


# ------------------------------------------------------------------------------------------------- archives

def _files(O):
    files = {f"small/f{i}.txt": O.real_text(6000 + 97 * i).tobytes()[i % 50:] for i in range(20)}
    files["big/huge.txt"] = stdlib_text(8 * MIB + 777_777, 99).tobytes() + O.real_text(8 * MIB).tobytes()
    files["noise.bin"] = O.gen_random(MIB).tobytes()
    files["empty.txt"] = b""
    return files


@pytest.fixture(scope="module")
def archives(oracle, tmp_path_factory):
    from znippy_b200 import archive, codec
    codec.default_ctx()
    files = _files(oracle)
    d = tmp_path_factory.mktemp("ck")
    src = d / "src"
    for p, b in files.items():
        (src / os.path.dirname(p)).mkdir(parents=True, exist_ok=True)
        (src / p).write_bytes(b)
    out = {}
    for name, cid, env in (("zstd", codec.CODEC_ZSTD, False), ("lz4", codec.CODEC_LZ4, False), ("zstdenv", codec.CODEC_ZSTD, True),
                           ("lz4env", codec.CODEC_LZ4, True)):
        sc = archive.compress_stream(str(d / f"s{name}.znippy"), False, level=3, codec_id=cid, envelope=env, checksum=True)
        for p, b in files.items():
            sc.sender().send(archive.ArchiveEntry(p, b))
        sc.finish()
        out["stream" + name] = sc.output
        o = str(d / f"d{name}.znippy")
        archive.compress_dir(str(src), o, level=3, codec_id=cid, envelope=env, checksum=True)
        out["dir" + name] = o
    return out, files


NAMES = [w + n for w in ("stream", "dir") for n in ("zstd", "lz4", "zstdenv", "lz4env")]


@pytest.mark.parametrize("name", NAMES)
def test_archive_round_trip(codec, oracle, archives, name, tmp_path):
    from znippy_b200 import archive
    paths, files = archives
    path = paths[name]
    ar = archive.ZnippyArchive.open(path)
    for p, b in files.items():
        assert ar.extract_file(p) == b, p
    big = files["big/huge.txt"]
    reqs = [("big/huge.txt", 0, len(big)), ("big/huge.txt", 8 * MIB - 100, 5000), ("small/f3.txt", 10, 100)]
    got = ar.read_ranges(reqs)
    for (p, o, n), g in zip(reqs, got):
        assert g == files[p][o:o + n]
    rep = archive.decompress_archive(path, True, str(tmp_path / "out"))
    assert rep.corrupt_files == 0 and rep.verified_files == len(files)
    for p, b in files.items():
        assert (tmp_path / "out" / p).read_bytes() == b, p
    # every compressed row's frame carries its checksum
    raw = open(path, "rb").read()
    t = archive.read_znippy_index(path)
    for r in range(t.num_rows):
        if not t.column("compressed")[r].as_py():
            continue
        bo, bs = t.column("blob_offset")[r].as_py(), t.column("blob_size")[r].as_py()
        blob = raw[bo:bo + bs]
        if blob[:4] == b"ZNB1":
            _, pc, po, pl, _ = codec.envelope_parse(blob)
            if pc == codec.PAYLOAD_RAW:
                continue
            blob = blob[po:po + pl]
        assert blob[4] in (0xE4, 0x24, 0x6C), (r, blob[:6])


@pytest.mark.parametrize("name", ["streamzstd", "dirlz4", "dirzstdenv"])
def test_flipped_checksum_in_archive_is_a_decode_error(codec, archives, name, tmp_path):
    """Before LZ4 checksums were checked (and with no digest compare on extract) this returned the bytes with ZN_S_OK."""
    from znippy_b200 import archive
    paths, files = archives
    path = paths[name]
    t = archive.read_znippy_index(path)
    rows = [r for r in range(t.num_rows) if t.column("relative_path")[r].as_py() == "small/f5.txt"]
    bo, bs = t.column("blob_offset")[rows[0]].as_py(), t.column("blob_size")[rows[0]].as_py()
    raw = bytearray(open(path, "rb").read())
    raw[bo + bs - 2] ^= 0x10  # inside the content checksum, the frame's last 4 bytes
    bad = tmp_path / "bad.znippy"
    bad.write_bytes(bytes(raw))
    ar = archive.ZnippyArchive.open(str(bad))
    with pytest.raises(Exception):
        ar.extract_file("small/f5.txt")
    assert ar.extract_file("small/f4.txt") == files["small/f4.txt"]
