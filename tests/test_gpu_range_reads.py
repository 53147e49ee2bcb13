"""Byte-range reads (zn_archive_read_ranges / ZnippyArchive.read_ranges) on the GPU: seeded random batches and edge
ranges equal Python slices of the source files on zstd (levels 1 / 3 / 19 / 22), LZ4 and ZNB1-envelope archives with
store-as-is and RAW rows; the counters show that only the chunks a range touches are read and decoded; caller memory
between the output windows is never written; corruption past an edge chunk's stop block goes unseen while corruption
inside a range reports what extract_files reports; the LRU serves ranges and never keeps partial chunks."""
import ctypes as C
import os
import random
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(__file__))
from test_hostemu_range_decode import blocks  # noqa: E402

MIB = 1 << 20
SLICE = 8 * MIB


@pytest.fixture(scope="module")
def A():
    from znippy_b200 import archive, codec
    codec.default_ctx()
    return archive


def _pack(A, path, files, **kw):
    sc = A.compress_stream(str(path), False, **kw)
    for p, d in files.items():
        sc.sender().send(A.ArchiveEntry(p, d))
    sc.finish()
    return sc.output


def _files(O, big: bool):
    files = {f"small/f{i}.txt": O.real_text(6000 + 97 * i).tobytes()[i % 50:] for i in range(120)}
    files["text/mid.txt"] = O.real_text(700_000).tobytes()
    files["lib/dep.jar"] = O.gen_random(3 * MIB + 123).tobytes()  # skip-listed: store-as-is
    files["empty.txt"] = b""
    if big:
        files["big/huge.bin"] = O.real_text(SLICE * 8 + 777_777).tobytes()  # 9 chunks
    return files


@pytest.fixture(scope="module")
def archives(A, oracle, tmp_path_factory):
    from znippy_b200 import codec
    O = oracle
    d = tmp_path_factory.mktemp("ranges")
    out = {}
    for lvl in (1, 3, 19, 22):
        files = _files(O, lvl == 3)
        out[f"zstd{lvl}"] = (_pack(A, d / f"z{lvl}.znippy", files, level=lvl), files)
    files = _files(O, False)
    out["lz4"] = (_pack(A, d / "lz4.znippy", files, codec_id=codec.CODEC_LZ4), files)
    files = _files(O, False)
    files["env/noise.bin"] = O.gen_random(2 * MIB).tobytes()  # compressed row kind, stored RAW inside ZNB1
    files["env/mixed.bin"] = O.real_text(SLICE).tobytes() + O.gen_random(SLICE // 2).tobytes()
    out["envelope"] = (_pack(A, d / "env.znippy", files, envelope=True, level=3), files)
    return out


def _index(A, path):
    t = A.read_znippy_index(path)
    cols = {k: t.column(k).to_pylist() for k in ("relative_path", "fdata_offset", "uncompressed_size", "compressed",
                                                 "blob_offset", "blob_size")}
    rows = {}
    for i, p in enumerate(cols["relative_path"]):
        rows.setdefault(p, []).append(i)
    for p in rows:
        rows[p].sort(key=lambda i: cols["fdata_offset"][i])
    return cols, rows


def _touched(cols, rows, path, off, length, size):
    """index rows a clamped range overlaps"""
    if path not in rows or length == 0 or off >= size:
        return set()
    hi = off + min(length, size - off)
    return {r for r in rows[path]
            if cols["fdata_offset"][r] < hi and cols["fdata_offset"][r] + cols["uncompressed_size"][r] > off}


def _check(res, reqs, files):
    for r, (p, o, n) in zip(res, reqs):
        if p not in files:
            assert isinstance(r, KeyError), (p, o, n)
        else:
            assert r == files[p][o:o + n], (p, o, n, len(r))


@pytest.mark.parametrize("name", ["zstd1", "zstd3", "zstd19", "zstd22", "lz4", "envelope"])
def test_random_batches_equal_python_slices(A, archives, name):
    path, files = archives[name]
    ar = A.ZnippyArchive.open(path)
    rnd = random.Random(sum(name.encode()))
    names = sorted(files)
    for call in range(6):
        reqs = []
        for _ in range(350):
            p = rnd.choice(names)
            sz = len(files[p])
            o = rnd.randrange(0, sz + 100) if rnd.random() < 0.9 else rnd.randrange(0, max(sz, 1))
            n = rnd.choice([0, 1, 17, 4096, 65536, 200_000, 3 * MIB]) if rnd.random() < 0.5 else rnd.randrange(0, 2 * SLICE)
            reqs.append((p, o, n))
        if call == 0:
            reqs.append(("no/such/file", 0, 10))
        _check(ar.read_ranges(reqs), reqs, files)


def test_edge_ranges_and_counters(A, archives):
    from znippy_b200 import codec
    path, files = archives["zstd3"]
    cols, rows = _index(A, path)
    ar = A.ZnippyArchive.open(path)
    big = files["big/huge.bin"]
    reqs = []
    for k in range(1, 9):
        b = k * SLICE
        for d in (-1, 0, 1):
            reqs += [("big/huge.bin", b + d, 4096), ("big/huge.bin", b + d - 4096, 4096), ("big/huge.bin", b + d, 1)]
    reqs += [("big/huge.bin", 3 * SLICE + 5, 1000),            # inside one chunk
             ("big/huge.bin", 2 * SLICE - 10, SLICE + 20),     # spans three chunks
             ("big/huge.bin", 0, 0), ("big/huge.bin", len(big), 10), ("big/huge.bin", len(big) + 5, 10),
             ("big/huge.bin", len(big) - 100, 1000),            # clamped at EOF
             ("empty.txt", 0, 10), ("missing.txt", 0, 10)]
    reqs += [("big/huge.bin", 4 * SLICE + 1000 * i, 3000) for i in range(50)]  # one chunk, many ranges
    res, st = ar.read_ranges(reqs, stats=True)
    _check(res, reqs, files)
    want = set()
    for p, o, n in reqs:
        if p in files:
            want |= {r for r in _touched(cols, rows, p, o, n, len(files[p])) if cols["compressed"][r]}
    assert st["rows_decoded"] == len(want)
    # 4 KiB from the middle of the big file: one chunk, decoded up to the block that holds the range's end
    mid = 4 * SLICE + 3 * MIB
    r, st = ar.read_ranges([("big/huge.bin", mid, 4096)], stats=True)
    assert r[0] == big[mid:mid + 4096]
    assert st["rows_decoded"] == 1 and st["bytes_decoded"] <= (mid - 4 * SLICE) + 4096 + (128 << 10)
    assert st["blob_bytes_read"] == cols["blob_size"][rows["big/huge.bin"][4]]
    # store-as-is rows: only the requested bytes are read, and no kernel runs
    ctx = codec.default_ctx()
    before = ctx.launches()
    jar = files["lib/dep.jar"]
    reqs = [("lib/dep.jar", len(jar) - 22, 22), ("lib/dep.jar", 1000, 65536), ("lib/dep.jar", len(jar) - 5, 100)]
    res, st = ar.read_ranges(reqs, stats=True)
    _check(res, reqs, files)
    assert ctx.launches() == before and st["rows_decoded"] == 0
    assert st["blob_bytes_read"] == sum(len(x) for x in res)


def test_envelope_raw_rows_never_reach_the_gpu(A, archives):
    from znippy_b200 import codec
    path, files = archives["envelope"]
    cols, rows = _index(A, path)
    ar = A.ZnippyArchive.open(path)
    noise = files["env/noise.bin"]
    ctx = codec.default_ctx()
    before = ctx.launches()
    reqs = [("env/noise.bin", 12345, 4096), ("env/noise.bin", len(noise) - 4096, 8192)]
    res, st = ar.read_ranges(reqs, stats=True)
    _check(res, reqs, files)
    assert ctx.launches() == before and st["rows_decoded"] == 0
    assert st["blob_bytes_read"] <= sum(len(x) for x in res) + 64 * len(rows["env/noise.bin"])
    reqs = [("env/mixed.bin", SLICE - 100, 200), ("env/mixed.bin", SLICE + 1000, 50)]
    _check(ar.read_ranges(reqs), reqs, files)


def test_caller_memory_outside_the_windows_is_untouched(A, archives):
    from znippy_b200 import _native as N, codec
    path, files = archives["zstd3"]
    ar = A.ZnippyArchive.open(path)
    ctx = codec.default_ctx()
    reqs = [("big/huge.bin", 5 * SLICE - 3000, 6000), ("text/mid.txt", 100, 5000), ("lib/dep.jar", 7, 300),
            ("small/f3.txt", 0, 1 << 20), ("missing", 0, 100), ("big/huge.bin", 1 << 40, 10)]
    n = len(reqs)
    off = np.array([r[1] for r in reqs], np.uint64)
    ln = np.array([r[2] for r in reqs], np.uint64)
    gap = 64
    outs = np.zeros(n, np.uint64)
    cur = gap
    for i, (p, o, L) in enumerate(reqs):
        outs[i] = cur
        cur += min(L, max(0, len(files.get(p, b"")) - o)) + gap
    out = np.full(cur, 0xEE, np.uint8)
    got = np.zeros(n, np.uint64)
    st = np.zeros(n, np.uint32)
    arr = (C.c_char_p * n)(*[r[0].encode() for r in reqs])
    ctx.check(N.lib().zn_archive_read_ranges(ctx.handle, ar._h, arr, N.ptr(off), N.ptr(ln), n, N.ptr(out), N.ptr(outs),
                                             N.ptr(got), N.ptr(st), None), "zn_archive_read_ranges")
    mask = np.ones(cur, bool)
    for i, (p, o, L) in enumerate(reqs):
        g = int(got[i])
        assert out[int(outs[i]):int(outs[i]) + g].tobytes() == files.get(p, b"")[o:o + L]
        mask[int(outs[i]):int(outs[i]) + g] = False
    assert (out[mask] == 0xEE).all()
    assert list(st) == [0, 0, 0, 0, 1, 0] and got[4] == 0 and got[5] == 0


def test_corruption_inside_and_past_a_range(A, oracle, tmp_path):
    """One 1 MB real-text chunk of 128 KiB blocks.  A reserved block type in the last block is never reached by a range in
    the first block; a reserved type in the first block fails that range with the status extract_files reports."""
    text = oracle.real_text(1_000_000).tobytes()
    path = _pack(A, tmp_path / "c.znippy", {"t.txt": text}, level=3)
    cols, rows = _index(A, path)
    (r,) = rows["t.txt"]
    bo, bs = cols["blob_offset"][r], cols["blob_size"][r]
    raw = bytearray(open(path, "rb").read())
    blob = bytes(raw[bo:bo + bs])
    bl = blocks(blob)
    assert len(bl) >= 6
    last_hdr = bl[-2][0]  # the last block's header follows the block before it
    fhd = blob[4]  # the first block's header follows the frame header
    first_hdr = 5 + (0 if (fhd >> 5) & 1 else 1) + (0, 1, 2, 4)[fhd & 3] + ((1 if (fhd >> 5) & 1 else 0), 2, 4, 8)[fhd >> 6]
    for hdr, stop_block_ok in ((last_hdr, True), (first_hdr, False)):
        c = bytearray(raw)
        c[bo + hdr] |= 0x06  # block type 3: reserved
        p2 = tmp_path / f"c{hdr}.znippy"
        p2.write_bytes(bytes(c))
        ar = A.ZnippyArchive.open(str(p2))
        with pytest.raises(Exception) as full_err:
            ar.extract_file("t.txt")
        # separate calls: in one call the whole-file range would make the first chunk a full row for both
        res = ar.read_ranges([("t.txt", 100, 4096)]) + ar.read_ranges([("t.txt", 0, len(text))])
        assert isinstance(res[1], type(full_err.value)) and res[1].args == full_err.value.args
        if stop_block_ok:
            assert res[0] == text[100:4196]
        else:
            assert isinstance(res[0], type(full_err.value)) and res[0].args == full_err.value.args


def test_cache_serves_ranges_and_never_keeps_partial_chunks(A, archives):
    from znippy_b200 import codec
    path, files = archives["zstd1"]
    ar = A.ZnippyArchive.open(path, cache_bytes=4 * MIB)
    ctx = codec.default_ctx()
    mid = files["text/mid.txt"]
    r, st = ar.read_ranges([("text/mid.txt", 1000, 2000)], stats=True)  # partial: decoded, not cached
    assert r[0] == mid[1000:3000] and st["rows_decoded"] == 1 and ar.cache_stats()["slices"] == 0
    r, st = ar.read_ranges([("text/mid.txt", 0, len(mid)), ("small/f1.txt", 0, 1 << 30)], stats=True)  # full: cached
    assert r == [mid, files["small/f1.txt"]] and st["rows_decoded"] == 2 and ar.cache_stats()["slices"] == 2
    before = ctx.launches()
    reqs = [("text/mid.txt", 500_000, 100), ("small/f1.txt", 10, 20), ("text/mid.txt", 5, 5)]
    res, st = ar.read_ranges(reqs, stats=True)
    _check(res, reqs, files)
    assert ctx.launches() == before and st["rows_from_cache"] == 2 and st["rows_decoded"] == 0
    assert st["blob_bytes_read"] == 0


@pytest.mark.parametrize("name", ["zstd3", "zstd22", "lz4", "envelope"])
def test_whole_file_range_equals_extract_file(A, archives, name):
    path, files = archives[name]
    ar = A.ZnippyArchive.open(path)
    for p in files:
        assert ar.read_range(p, 0, len(files[p])) == ar.extract_file(p) == files[p], p
    with pytest.raises(KeyError):
        ar.read_range("nope", 0, 1)
