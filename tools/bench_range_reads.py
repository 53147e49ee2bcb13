#!/usr/bin/env python
"""Byte-range reads (zn_archive_read_ranges, DESIGN.md §5b) against extract_file of the whole file.  Two archives:
  - `huge.bin`, the 2 GiB text pattern of bench.py's text2g workload at zstd-19, a 200 MiB skip-listed random `.jar`
    (store-as-is) and 10 000 x 10 KiB text files, also at zstd-19;
  - 256 MiB of real text (the standard library's sources) at zstd-3.
For each file kind, ranges of 4 KiB, 64 KiB and 1 MiB at seeded random offsets, 1 and 256 ranges per call: per-call
wall time (median, p90; each call ends in a device synchronise), the counters of the call (bytes decoded per byte
returned, rows decoded, blob bytes read) and, for comparison, extract_file of the whole file.  Prints one JSON line per
case, each carrying the card and its power limit; `--out FILE` also writes them there.

    python tools/bench_range_reads.py [--calls 30] [--out profiles/r3_range_reads.jsonl]"""
import argparse
import json
import os
import random
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import incompressible, text_slice  # noqa: E402
from bench_compress_long import gpu_info  # noqa: E402
from test_hostemu_compress_long import stdlib_text  # noqa: E402
from znippy_b200 import archive as A, codec  # noqa: E402

MiB = 1 << 20


def pack(path, entries, level):
    sc = A.compress_stream(path, False, level=level)
    for p, d in entries:
        sc.sender().send(A.ArchiveEntry(p, d))
    sc.finish()
    return path


def pct(xs, q):
    return float(np.percentile(np.array(xs), q))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = gpu_info()
    codec.default_ctx()
    tmp = tempfile.mkdtemp(prefix="zn_range_bench_")
    t0 = time.perf_counter()
    small = [(f"small/f{i:05d}.txt", text_slice(i * 131, 10240).tobytes()) for i in range(10_000)]
    p1 = pack(os.path.join(tmp, "text2g.znippy"),
              [("huge.bin", text_slice(0, 2 << 30).tobytes()), ("lib/big.jar", incompressible(7, 200 * MiB).tobytes())]
              + small, 19)
    real = stdlib_text(9 * MiB)
    real = np.concatenate([np.roll(real, -k * 65_537)[:8 * MiB] for k in range(32)]).tobytes()
    p2 = pack(os.path.join(tmp, "realtext.znippy"), [("realtext.txt", real)], 3)
    build_s = time.perf_counter() - t0
    ar1, ar2 = A.ZnippyArchive.open(p1), A.ZnippyArchive.open(p2)
    cases = [("huge.bin zstd-19 (256 x 8 MiB chunks)", ar1, "huge.bin", 2 << 30, None),
             ("real text zstd-3 (32 x 8 MiB chunks)", ar2, "realtext.txt", len(real), None),
             ("skip-listed .jar, 200 MiB store-as-is", ar1, "lib/big.jar", 200 * MiB, None),
             ("10 000 x 10 KiB files zstd-19", ar1, None, 10240, [p for p, _ in small])]
    lines = []
    rnd = random.Random(11)
    for name, ar, path, size, many in cases:
        whole = []
        for _ in range(3 if size > 64 * MiB else 10):
            p = path or rnd.choice(many)
            t = time.perf_counter()
            ar.extract_file(p)
            whole.append((time.perf_counter() - t) * 1e3)
        for rsize in (4096, 64 << 10, MiB):
            if rsize > size:
                continue
            for batch in (1, 256):
                times, dec, ret, rows, read = [], 0, 0, 0, 0
                for call in range(a.calls + 2):
                    reqs = []
                    for _ in range(batch):
                        p = path or rnd.choice(many)
                        reqs.append((p, rnd.randrange(0, size - rsize + 1), rsize))
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
                rec = {"case": name, "range_bytes": rsize, "ranges_per_call": batch, "calls": a.calls,
                       "call_ms_median": round(pct(times, 50), 3), "call_ms_p90": round(pct(times, 90), 3),
                       "extract_file_ms_median": round(pct(whole, 50), 3),
                       "bytes_decoded_per_byte_returned": round(dec / ret, 3),
                       "rows_decoded_per_call": rows / a.calls, "blob_bytes_read_per_call": read / a.calls,
                       "archive_build_s": round(build_s, 1), **info}
                print(json.dumps(rec), flush=True)
                lines.append(rec)
    if a.out:
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
