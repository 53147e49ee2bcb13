"""Seekable zstd (ZN_CODEC_SEEKABLE) on the GPU: compress_batch and compress plans emit one frame per 128 KiB block plus
the seek table, checked with libzstd frame by frame; full rows of such blobs decode on every decode class; archives
written seekable serve a range from only the frames it touches, check each against the table's XXH64, and fall back to
the prefix path when the table is damaged."""
import os
import random
import struct
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(__file__))
from test_hostemu_compress_long import stdlib_text  # noqa: E402
from test_hostemu_seekable import BLOCK, check_seekable_blob, parse_seek_table  # noqa: E402

KIB, MIB = 1024, 1 << 20
SLICE = 8 * MIB
# seekable size / plain size on 8 MiB of real text, measured on one B200 (DESIGN §4.3), plus a small margin
RATIO_BOUND = {1: 1.010, 3: 1.015, 19: 1.017}  # measured 1.0060 / 1.0116 / 1.0134


@pytest.fixture(scope="module")
def codec():
    from znippy_b200 import codec
    codec.default_ctx()
    return codec


def _corpora(O):
    c = {"real8m": stdlib_text(8 * MIB), "text": O.gen_text(3 * MIB + 5), "binary": O.gen_binary(MIB + 17),
         "random": O.gen_random(300_000)}
    for n in (0, 1, BLOCK - 1, BLOCK, BLOCK + 1, 8 * MIB + 777):
        c[f"len{n}"] = stdlib_text(n, 4321)
    return c


def _batch(datas, first=16):
    offs, cur = [], first
    for d in datas:
        offs.append(cur)
        cur += len(d) + 3
    src = np.zeros(cur + 1, np.uint8)
    for o, d in zip(offs, datas):
        src[o:o + len(d)] = d
    return src, offs, [len(d) for d in datas]


def _seek(codec):
    return codec.CODEC_ZSTD | codec.CODEC_SEEKABLE


@pytest.mark.parametrize("level", [1, 3, 19])
def test_compress_batch_seekable_blobs(codec, oracle, level):
    cases = _corpora(oracle)
    datas = list(cases.values())
    src, offs, lens = _batch(datas)
    blobs, dg, st = codec.compress_batch(src, offs, lens, level, _seek(codec))
    assert (st == 0).all()
    for name, d, b, g in zip(cases, datas, blobs, dg):
        check_seekable_blob(oracle, b, d.tobytes(), codec.compress_bound(d.size, _seek(codec)))
        assert g.tobytes() == oracle.blake3(d.tobytes()), name
    plain, _, _ = codec.compress_batch(src, offs, lens, level, codec.CODEC_ZSTD)
    i = list(cases).index("real8m")
    ratio = len(blobs[i]) / len(plain[i])
    print(f"level {level}: real text 8 MiB plain {len(plain[i])} seekable {len(blobs[i])} ratio {ratio:.4f}")
    assert 1.0 < ratio <= RATIO_BOUND[level]


@pytest.mark.parametrize("envelope", [False, True])
@pytest.mark.parametrize("level", [1, 19])
def test_plan_equals_compress_batch(codec, oracle, level, envelope):
    import torch
    sys.path.insert(0, os.path.dirname(__file__))
    from test_gpu_compress_plan import _blobs, _check_packed, _run
    datas = list(_corpora(oracle).values())
    src, offs, lens = _batch(datas)
    want, wdg, _ = codec.compress_batch(src, offs, lens, level, _seek(codec))
    plan = codec.N.Plan.compress(codec.default_ctx(), offs, lens, level=level, envelope=envelope, seekable=True)
    blobs, boffs, dst = _blobs(*_run(torch, plan, torch.from_numpy(src).cuda()))
    _check_packed(blobs, boffs, dst)
    st, dg = plan.results()
    assert (st == 0).all() and np.array_equal(dg, wdg)
    for d, w, b in zip(datas, want, blobs):
        if envelope:
            w = (codec.envelope_wrap(codec.PAYLOAD_RAW, d.size, d.tobytes()) if len(w) >= d.size
                 else codec.envelope_wrap(codec.PAYLOAD_ZSTD, d.size, w))
        assert b == w
    # one launch more than the same plan without the flag: the checksum kernel
    plain = codec.N.Plan.compress(codec.default_ctx(), offs, lens, level=level, envelope=envelope)
    _run(torch, plain, torch.from_numpy(src).cuda())
    assert plan.launches() == plain.launches() + 1
    assert plan.last_ms()[1] > 0


@pytest.mark.parametrize("envelope", [False, True])
def test_compress_ctx_round_trip(codec, oracle, envelope):
    """CompressCtx(seekable=True) blobs come back through decompress_frame: a bare blob of several frames is sized
    from its seek table, a ZNB1 blob from its header."""
    for n in (0, 1, BLOCK + 1, 8 * MIB + 777):
        data = stdlib_text(n, 55).tobytes()
        blob = codec.CompressCtx(3, envelope=envelope, seekable=True).compress(data)
        assert codec.decompress_frame(blob) == data, n
        if not envelope:
            assert codec.frame_content_size(blob) == n
            check_seekable_blob(oracle, blob, data, codec.compress_bound(n, _seek(codec)))


def test_full_rows_decode_on_every_class(codec, oracle):
    import torch
    from znippy_b200._native import Plan
    cases = _corpora(oracle)
    datas = [d for d in cases.values()] + [oracle.real_text(SLICE), oracle.gen_text(SLICE)]
    src, offs, lens = _batch(datas)
    blobs, _, st = codec.compress_batch(src, offs, lens, 3, _seek(codec))
    contents = [d.tobytes() for d in datas]
    digests = b"".join(oracle.blake3(c) for c in contents)
    out_off = np.concatenate([[0], np.cumsum([(n + 15) // 16 * 16 for n in lens])])[:-1]
    out = np.zeros(int(out_off[-1]) + lens[-1] + 16, np.uint8)
    buf = np.frombuffer(b"".join(blobs), np.uint8)
    boffs = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])[:-1]
    st, dg = codec.decode_verify_batch(buf, boffs, [len(b) for b in blobs], [1] * len(blobs), lens, digests, out, out_off)
    assert (st == 0).all()
    for i, c in enumerate(contents):
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c and dg[i].tobytes() == oracle.blake3(c)
    ctx = codec.default_ctx()
    counts = None
    for align in range(16):
        d_buf = torch.zeros(buf.size + 64, dtype=torch.uint8, device="cuda")
        d_buf[align:align + buf.size] = torch.from_numpy(buf.copy()).cuda()
        d_out = torch.zeros(out.size, dtype=torch.uint8, device="cuda")
        plan = Plan.decode_verify(ctx, boffs + align, [len(b) for b in blobs], [1] * len(blobs), out_off, lens, digests)
        plan.run(d_buf.data_ptr(), d_out.data_ptr())
        pst, pdg = plan.results()
        assert (pst == 0).all(), (align, pst)
        assert plan.pipeline_fallbacks() == 0, align
        h = d_out.cpu().numpy()
        for i, c in enumerate(contents):
            assert h[out_off[i]:out_off[i] + len(c)].tobytes() == c, (align, i)
        counts = plan.class_counts()
    print("class counts [pipeline, fused, big raw, small, mid]:", counts)
    assert counts[0] > 0 and counts[1] > 0 and counts[3] + counts[4] > 0


def test_refusals(codec, oracle, tmp_path):
    from znippy_b200 import archive
    from znippy_b200._native import NativeError, Plan
    d = oracle.gen_text(1000)
    with pytest.raises(Exception):
        codec.compress_batch(d, [0], [d.size], 3, codec.CODEC_LZ4 | codec.CODEC_SEEKABLE)
    for lvl in (20, 22):
        with pytest.raises(Exception):
            codec.compress_batch(d, [0], [d.size], lvl, _seek(codec))
        with pytest.raises(NativeError):
            Plan.compress(codec.default_ctx(), [0], [d.size], level=lvl, seekable=True)
        with pytest.raises(ValueError):
            archive.compress_stream(str(tmp_path / "x.znippy"), False, level=lvl, seekable=True)
    with pytest.raises(NativeError):
        Plan.compress(codec.default_ctx(), [0], [d.size], codec=codec.CODEC_LZ4, seekable=True)
    with pytest.raises(ValueError):
        archive.compress_stream(str(tmp_path / "x.znippy"), False, codec_id=codec.CODEC_LZ4, seekable=True)
    (tmp_path / "in").mkdir()
    (tmp_path / "in" / "a.txt").write_bytes(d.tobytes())
    with pytest.raises(NativeError, match="seekable"):
        archive.compress_dir(str(tmp_path / "in"), str(tmp_path / "y.znippy"), codec_id=codec.CODEC_LZ4, seekable=True)
    with pytest.raises(NativeError, match="seekable"):
        archive.compress_dir(str(tmp_path / "in"), str(tmp_path / "y.znippy"), level=21, seekable=True)
    # an unknown znippy_seekable value is refused at open
    path = str(tmp_path / "z.znippy")
    archive.compress_dir(str(tmp_path / "in"), path, level=3, seekable=True)
    raw = bytearray(open(path, "rb").read())
    k = raw.find(b"znippy_seekable")
    assert k >= 0
    while k >= 0:  # every copy of the key (one per sub-index): its value, a flatbuffer string, sits close by
        v = raw.find(b"\x04\x00\x00\x00zstd\x00", max(0, k - 256), k + 256)
        assert v >= 0
        raw[v + 4:v + 8] = b"zsxd"
        k = raw.find(b"znippy_seekable", k + 1)
    bad = tmp_path / "bad.znippy"
    bad.write_bytes(bytes(raw))
    with pytest.raises(Exception, match="seekable"):
        archive.ZnippyArchive.open(str(bad))


# ------------------------------------------------------------------------------------------------- archives

def _files(O):
    files = {f"small/f{i}.txt": O.real_text(6000 + 97 * i).tobytes()[i % 50:] for i in range(40)}
    files["big/huge.txt"] = stdlib_text(SLICE + 777_777, 99).tobytes() + O.real_text(7 * SLICE).tobytes()  # 9 chunks
    files["lib/dep.jar"] = O.gen_random(3 * MIB + 123).tobytes()  # skip-listed: store-as-is
    files["noise.bin"] = O.gen_random(MIB).tobytes()  # compressed row of raw blocks
    files["empty.txt"] = b""
    return files


@pytest.fixture(scope="module")
def archives(oracle, tmp_path_factory):
    from znippy_b200 import archive, codec
    codec.default_ctx()
    files = _files(oracle)
    d = tmp_path_factory.mktemp("seek")
    src = d / "src"
    for p, b in files.items():
        (src / os.path.dirname(p)).mkdir(parents=True, exist_ok=True)
        (src / p).write_bytes(b)
    out = {}
    for lvl in (3, 19):
        for env in (False, True):
            sc = archive.compress_stream(str(d / f"s{lvl}{env}.znippy"), False, level=lvl, envelope=env, seekable=True)
            for p, b in files.items():
                sc.sender().send(archive.ArchiveEntry(p, b))
            sc.finish()
            out[f"stream{lvl}{'env' if env else ''}"] = sc.output
            o = str(d / f"d{lvl}{env}.znippy")
            archive.compress_dir(str(src), o, level=lvl, envelope=env, seekable=True)
            out[f"dir{lvl}{'env' if env else ''}"] = o
    return out, files


def _rows(path):
    from znippy_b200 import archive
    t = archive.read_znippy_index(path)
    cols = {k: t.column(k).to_pylist() for k in ("relative_path", "fdata_offset", "uncompressed_size", "compressed",
                                                 "blob_offset", "blob_size")}
    rows = {}
    for i, p in enumerate(cols["relative_path"]):
        rows.setdefault(p, []).append(i)
    for p in rows:
        rows[p].sort(key=lambda i: cols["fdata_offset"][i])
    return cols, rows


def _payload(codec, raw, cols, r):
    """(payload offset in the file, payload bytes) of row r"""
    bo, bs = cols["blob_offset"][r], cols["blob_size"][r]
    blob = bytes(raw[bo:bo + bs])
    if blob[:4] == b"ZNB1":
        _, _, po, pl, _ = codec.envelope_parse(blob)
        return bo + po, blob[po:po + pl]
    return bo, blob


NAMES = [f"{w}{lvl}{e}" for w in ("stream", "dir") for lvl in (3, 19) for e in ("", "env")]


@pytest.mark.parametrize("name", NAMES)
def test_archive_reads(codec, archives, name):
    from znippy_b200 import archive
    paths, files = archives
    path = paths[name]
    assert archive.read_znippy_index(path).schema.metadata[b"znippy_seekable"] == b"zstd"
    ar = archive.ZnippyArchive.open(path)
    for p, b in files.items():
        assert ar.extract_file(p) == b, p
    rep = archive.verify_archive_integrity(path)
    assert rep.corrupt_files == 0 and rep.verified_files == len(files)
    rng = random.Random(name)
    names = list(files)
    for _ in range(6):
        reqs = []
        for _ in range(rng.randint(1, 40)):
            p = rng.choice(names)
            n = len(files[p])
            off = rng.randint(0, n + 10)
            reqs.append((p, off, rng.choice([1, 100, 4096, 65536, 300_000, 3 * MIB])))
        res = ar.read_ranges(reqs)
        for (p, off, ln), r in zip(reqs, res):
            assert r == files[p][off:off + ln], (p, off, ln)
    # counters: the frames a range touches, and the seek table, are all that is read and decoded
    raw = open(path, "rb").read()
    cols, rows = _rows(path)
    big = files["big/huge.txt"]
    r1 = rows["big/huge.txt"][1]
    po, payload = _payload(codec, raw, cols, r1)
    entries, tab = parse_seek_table(payload)
    table = len(payload) - tab
    if name.endswith("env"):  # the ZNB1 header is parsed from the blob's first bytes
        table += min(64, cols["blob_size"][r1])
    fo = cols["fdata_offset"][r1]
    mid = fo + 4 * MIB + 1000  # inside frame 32 of the chunk
    res, st = ar.read_ranges([("big/huge.txt", mid, 4096)], stats=True)
    assert res[0] == big[mid:mid + 4096]
    assert st["rows_decoded"] == 1 and st["bytes_decoded"] <= 256 * KIB
    assert st["blob_bytes_read"] <= table + entries[32][0], st
    res, st = ar.read_ranges([("big/huge.txt", fo + 5 * BLOCK - 100, 200)], stats=True)  # across a frame boundary
    assert res[0] == big[fo + 5 * BLOCK - 100:fo + 5 * BLOCK + 100] and st["bytes_decoded"] == 2 * BLOCK
    assert st["blob_bytes_read"] == table + entries[4][0] + entries[5][0]
    rl = rows["big/huge.txt"][-1]
    _, pl = _payload(codec, raw, cols, rl)
    el, _ = parse_seek_table(pl)
    res, st = ar.read_ranges([("big/huge.txt", len(big) - 4096, 4096)], stats=True)  # the file's tail
    assert res[0] == big[-4096:] and st["rows_decoded"] == 1 and st["bytes_decoded"] == el[-1][1]


def test_table_checksum_and_damaged_tables(codec, archives, tmp_path):
    from znippy_b200 import archive
    paths, files = archives
    path = paths["stream3"]
    raw = open(path, "rb").read()
    cols, rows = _rows(path)
    (r,) = rows["noise.bin"]
    po, payload = _payload(codec, raw, cols, r)
    entries, tab = parse_seek_table(payload)
    assert len(entries) == 8 and all(e[0] == BLOCK + 16 for e in entries)  # every frame one raw block
    noise = files["noise.bin"]
    c = bytearray(raw)
    c[po + 2 * (BLOCK + 16) + 16 + 777] ^= 0x5A  # frame 2's content: the decode still succeeds
    p2 = tmp_path / "flip.znippy"
    p2.write_bytes(bytes(c))
    ar = archive.ZnippyArchive.open(str(p2))
    from znippy_b200.codec import S_DECODE_ERROR, CodecError
    res = ar.read_ranges([("noise.bin", 2 * BLOCK + 100, 4096)])
    assert isinstance(res[0], CodecError) and res[0].status == S_DECODE_ERROR
    res = ar.read_ranges([("noise.bin", 5 * BLOCK + 100, 4096)])  # a frame the range does not touch
    assert res[0] == noise[5 * BLOCK + 100:5 * BLOCK + 4196]
    # a damaged footer, or an entry inconsistent with the index: the row is decoded from its start
    big = files["big/huge.txt"]
    r1 = rows["big/huge.txt"][1]
    po1, pl1 = _payload(codec, raw, cols, r1)
    fo = cols["fdata_offset"][r1]
    for what in ("footer", "entry"):
        c = bytearray(raw)
        if what == "footer":
            c[po1 + len(pl1) - 1] ^= 0xFF
        else:
            e0 = po1 + len(pl1) - (12 * 64 + 17) + 8 + 4
            c[e0:e0 + 4] = struct.pack("<I", BLOCK - 1)
        p3 = tmp_path / f"{what}.znippy"
        p3.write_bytes(bytes(c))
        ar = archive.ZnippyArchive.open(str(p3))
        off = fo + 4 * MIB
        res, st = ar.read_ranges([("big/huge.txt", off, 4096)], stats=True)
        assert res[0] == big[off:off + 4096], what
        assert st["bytes_decoded"] > 4 * MIB, (what, st)  # the prefix path


def test_cache_keeps_full_rows_only(codec, archives):
    from znippy_b200 import archive
    paths, files = archives
    ar = archive.ZnippyArchive.open(paths["stream19env"], cache_bytes=64 * MIB)
    big = files["big/huge.txt"]
    res, st = ar.read_ranges([("big/huge.txt", 3 * MIB, 100)], stats=True)
    assert res[0] == big[3 * MIB:3 * MIB + 100] and ar.cache_stats()["slices"] == 0
    res, st = ar.read_ranges([("big/huge.txt", 0, SLICE)], stats=True)
    assert res[0] == big[:SLICE] and ar.cache_stats()["slices"] == 1
    res, st = ar.read_ranges([("big/huge.txt", 100, 100)], stats=True)
    assert res[0] == big[100:200] and st["rows_from_cache"] == 1 and st["rows_decoded"] == 0
