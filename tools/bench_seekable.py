#!/usr/bin/env python
"""Seekable zstd archives (ZN_CODEC_SEEKABLE, DESIGN.md §4.3 / §5b) against plain ones.  The same 256 MiB of real text
(the standard library's sources, as tools/bench_range_reads.py builds it) is written at zstd-3 twice, once seekable and
once not, and read back in the same process:
  - ranges of 4 KiB, 64 KiB and 1 MiB, 1 and 256 per call, at seeded random mid-file offsets and at the file's tail:
    per-call wall time (median, p90; each call ends in a device synchronise), bytes decoded per byte returned, rows
    decoded and blob bytes read per call;
  - extract_file of the whole file;
  - compress GB/s (device time of zn_compress_batch) and ratio at levels 1 / 3 / 19, on the real text and on the
    500 MiB binary pattern, seekable and not, and in a separate torch.profiler pass the device time of each compress
    kernel (the checksum kernel k_block_xxh, the block kernel, the assembly).
Prints one JSON line per case, each carrying the card, its power limit and SM clock; `--out FILE` also writes them.

    python tools/bench_seekable.py [--calls 10] [--out profiles/r3_seekable.jsonl]"""
import argparse
import json
import os
import random
import re
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_compress_long import gpu_info  # noqa: E402
from test_hostemu_compress_long import stdlib_text  # noqa: E402
from znippy_b200 import archive as A, codec  # noqa: E402

MiB = 1 << 20


def pack(path, name, data, seekable):
    sc = A.compress_stream(path, False, level=3, seekable=seekable)
    sc.sender().send(A.ArchiveEntry(name, data))
    sc.finish()
    return sc.output


def pct(xs, q):
    return float(np.percentile(np.array(xs), q))


def compress_rate(data: np.ndarray, level: int, cid: int):
    """device GB/s and ratio of 8 MiB slices of `data` through zn_compress_batch (best of 3 runs)"""
    offs = list(range(0, data.size, 8 * MiB))
    lens = [min(8 * MiB, data.size - o) for o in offs]
    ctx = codec.default_ctx()
    best, out = None, 0
    for _ in range(3):
        blobs, _, st = codec.compress_batch(data, offs, lens, level, cid, ctx)
        assert (st == 0).all()
        ms = ctx.last_compress_ms()
        best = ms if best is None else min(best, ms)
        out = sum(len(b) for b in blobs)
    return data.size / best / 1e6, data.size / out


def kernel_ms(data: np.ndarray, level: int, cid: int) -> dict:
    """device ms per compress kernel of one zn_compress_batch of `data` (8 MiB slices), from torch.profiler (after a
    warm-up call; the profiled call is not one of the timed ones)"""
    from torch.profiler import ProfilerActivity, profile
    offs = list(range(0, data.size, 8 * MiB))
    lens = [min(8 * MiB, data.size - o) for o in offs]
    codec.compress_batch(data, offs, lens, level, cid)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        codec.compress_batch(data, offs, lens, level, cid)
    out = {}
    for k in prof.key_averages():
        t = getattr(k, "device_time_total", None)
        if t is None:
            t = k.cuda_time_total
        m = re.search(r"\b(k_[A-Za-z0-9_]+)", k.key)  # e.g. "void zn::k_zstd_blocks<zn::cz::Win<...>, true>(...)"
        if m and t:
            out[m.group(1)] = round(out.get(m.group(1), 0.0) + t / 1e3, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = gpu_info()
    codec.default_ctx()
    tmp = tempfile.mkdtemp(prefix="zn_seek_bench_")
    real = stdlib_text(9 * MiB)
    real = np.concatenate([np.roll(real, -k * 65_537)[:8 * MiB] for k in range(32)])
    size = real.size
    arch = {}
    for seekable in (False, True):
        t = time.perf_counter()
        p = pack(os.path.join(tmp, f"real{int(seekable)}.znippy"), "realtext.txt", real.tobytes(), seekable)
        arch[seekable] = (A.ZnippyArchive.open(p), os.path.getsize(p), time.perf_counter() - t)
    lines = []

    def emit(rec):
        rec.update(info)
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    for seekable, (ar, fsize, build_s) in arch.items():
        whole = []
        for _ in range(3):
            t = time.perf_counter()
            ar.extract_file("realtext.txt")
            whole.append((time.perf_counter() - t) * 1e3)
        emit({"case": "extract_file", "seekable": seekable, "file_bytes": size, "archive_bytes": fsize,
              "ms_median": round(pct(whole, 50), 3), "archive_build_s": round(build_s, 1)})
    for where in ("mid", "tail"):
        for rsize in (4096, 64 << 10, MiB):
            for batch in (1, 256):
                for seekable, (ar, _, _) in arch.items():
                    rnd = random.Random(rsize * 7 + batch)  # the same offsets for both archives
                    times, dec, ret, rows, read = [], 0, 0, 0, 0
                    for call in range(a.calls + 2):
                        reqs = []
                        for _ in range(batch):
                            off = size - rsize if where == "tail" else rnd.randrange(0, size - rsize + 1)
                            reqs.append(("realtext.txt", off, rsize))
                        t = time.perf_counter()
                        res, st = ar.read_ranges(reqs, stats=True)
                        ms = (time.perf_counter() - t) * 1e3
                        assert not any(isinstance(r, Exception) for r in res)
                        if call < 2:
                            continue  # warm-up
                        times.append(ms)
                        dec += st["bytes_decoded"]
                        ret += sum(len(r) for r in res)
                        rows += st["rows_decoded"]
                        read += st["blob_bytes_read"]
                    emit({"case": f"ranges {where}", "seekable": seekable, "range_bytes": rsize, "ranges_per_call": batch,
                          "calls": a.calls, "call_ms_median": round(pct(times, 50), 3),
                          "call_ms_p90": round(pct(times, 90), 3),
                          "bytes_decoded_per_byte_returned": round(dec / ret, 3),
                          "rows_decoded_per_call": rows / a.calls, "blob_bytes_read_per_call": read / a.calls})
    import oracle as O
    corpora = {"real text 256 MiB": real, "binary pattern 500 MiB": O.gen_binary(500 * MiB)}
    for cname, data in corpora.items():
        for level in (1, 3, 19):
            for seekable in (False, True):
                cid = codec.CODEC_ZSTD | (codec.CODEC_SEEKABLE if seekable else 0)
                gbs, ratio = compress_rate(data, level, cid)
                emit({"case": "compress", "corpus": cname, "level": level, "seekable": seekable,
                      "device_GBps": round(gbs, 3), "ratio": round(ratio, 4)})
    for cname, data in corpora.items():  # profiled apart from the timed runs above
        for level in (1, 3, 19):
            for seekable in (False, True):
                cid = codec.CODEC_ZSTD | (codec.CODEC_SEEKABLE if seekable else 0)
                emit({"case": "compress kernels", "corpus": cname, "level": level, "seekable": seekable,
                      "kernel_ms": kernel_ms(data, level, cid)})
    if a.out:
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
