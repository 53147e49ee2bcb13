#!/usr/bin/env python
"""Frame checksums (ZN_CODEC_CHECKSUM, DESIGN.md §4.3 / §7): what writing and checking them costs.
  - compress GB/s (device time of zn_compress_batch, best of 3) and ratio with and without the flag: 256 MiB of real text
    (the standard library's sources, as tools/bench_seekable.py builds it) at zstd 1 / 3 / 19 and LZ4, and the 500 MiB
    binary pattern at zstd 19; in a separate torch.profiler pass the device time of each compress kernel (k_slice_xxh
    is the checksum kernel);
  - device decode+verify time (zn_plan_last_ms of a decode plan: total and the tree+compare stage, best of 5) of the
    same real text written with and without checksums, 8 MiB rows;
  - the content-checksum check alone on libzstd-checksummed 8 MiB real-text rows (1 row and 32 rows): the tree+compare
    stage of a decode plan over those rows minus the same stage over the same text without checksums.  Run once against
    this tree and once with --pkg-root pointing at another checkout (the one-thread check of earlier versions) to compare.
Prints one JSON line per case, each carrying the card, its power limit and SM clock; `--out FILE` also writes them.

    python tools/bench_checksum.py [--out profiles/r3_checksum.jsonl] [--only check] [--pkg-root DIR]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--only", default=None, choices=["compress", "decode", "check"])
ap.add_argument("--pkg-root", default=ROOT, help="directory whose znippy_b200 package is measured")
ap.add_argument("--label", default="this tree")
A = ap.parse_args()
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.abspath(A.pkg_root))
from bench_compress_long import gpu_info  # noqa: E402
from test_hostemu_compress_long import stdlib_text  # noqa: E402
from znippy_b200 import codec  # noqa: E402
from znippy_b200._native import Plan  # noqa: E402

MiB = 1 << 20
CHECKSUM = 0x800  # ZN_CODEC_CHECKSUM


def compress_rate(data, level, cid):
    offs = list(range(0, data.size, 8 * MiB))
    lens = [min(8 * MiB, data.size - o) for o in offs]
    ctx = codec.default_ctx()
    best, blobs = None, None
    for _ in range(3):
        blobs, _, st = codec.compress_batch(data, offs, lens, level, cid, ctx)
        assert (st == 0).all()
        ms = ctx.last_compress_ms()
        best = ms if best is None else min(best, ms)
    return data.size / best / 1e6, data.size / sum(len(b) for b in blobs), blobs


def decode_ms(blobs, lens, runs=5):
    """best-of-`runs` zn_plan_last_ms [total, decode, hash, tree+compare] of one decode plan over `blobs` (resident)"""
    import torch
    boffs = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])[:-1]
    ooff = np.concatenate([[0], np.cumsum([(n + 15) // 16 * 16 for n in lens])])[:-1]
    d_buf = torch.from_numpy(np.frombuffer(b"".join(blobs), np.uint8).copy()).cuda()
    d_out = torch.zeros(int(ooff[-1]) + lens[-1] + 16, dtype=torch.uint8, device="cuda")
    plan = Plan.decode_verify(codec.default_ctx(), boffs, [len(b) for b in blobs], [1] * len(blobs), ooff, lens, None)
    best = None
    for _ in range(runs + 1):
        plan.run(d_buf.data_ptr(), d_out.data_ptr())
        st, _ = plan.results()
        assert not st.any(), st
        ms = list(plan.last_ms())
        best = ms if best is None else [min(a, b) for a, b in zip(best, ms)]
    return [round(x, 4) for x in best]


def main():
    info = gpu_info()
    info["package"] = A.label
    codec.default_ctx()
    real = stdlib_text(9 * MiB)
    real = np.concatenate([np.roll(real, -k * 65_537)[:8 * MiB] for k in range(32)])
    lines = []

    def emit(rec):
        rec.update(info)
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    cases = [("real text 256 MiB", "zstd", lvl) for lvl in (1, 3, 19)] + [("real text 256 MiB", "lz4", 1),
                                                                          ("binary pattern 500 MiB", "zstd", 19)]
    if A.only in (None, "compress", "decode"):
        import oracle as O
        from bench_seekable import kernel_ms
        corpora = {"real text 256 MiB": real, "binary pattern 500 MiB": O.gen_binary(500 * MiB)}
        for cname, name, level in cases:
            data = corpora[cname]
            base = codec.CODEC_LZ4 if name == "lz4" else codec.CODEC_ZSTD
            lens = [min(8 * MiB, data.size - o) for o in range(0, data.size, 8 * MiB)]
            for ck in (False, True):
                cid = base | (CHECKSUM if ck else 0)
                gbs, ratio, blobs = compress_rate(data, level, cid)
                rec = {"case": "compress", "corpus": cname, "codec": name, "level": level, "checksum": ck,
                       "device_GBps": round(gbs, 3), "ratio": round(ratio, 4)}
                if A.only != "compress" and cname.startswith("real") and level != 19:
                    ms = decode_ms(blobs, lens)
                    rec.update({"decode_verify_ms": ms[0], "decode_ms": ms[1], "hash_ms": ms[2], "tree_ms": ms[3]})
                emit(rec)
        for cname, name, level in cases:
            base = codec.CODEC_LZ4 if name == "lz4" else codec.CODEC_ZSTD
            for ck in (False, True):
                emit({"case": "compress kernels", "corpus": cname, "codec": name, "level": level, "checksum": ck,
                      "kernel_ms": kernel_ms(corpora[cname], level, base | (CHECKSUM if ck else 0))})
    if A.only in (None, "check"):
        import oracle as O
        z = O.libzstd()
        rows = [real[k * 8 * MiB:(k + 1) * 8 * MiB].tobytes() for k in range(32)]
        with_ck = [z.compress(r, 3, checksum=True) for r in rows]
        without = [z.compress(r, 3) for r in rows]
        for n in (1, 32):
            lens = [8 * MiB] * n
            a, b = decode_ms(with_ck[:n], lens), decode_ms(without[:n], lens)
            emit({"case": "libzstd checksummed rows", "rows": n, "row_bytes": 8 * MiB, "tree_ms_checksummed": a[3],
                  "tree_ms_plain": b[3], "check_ms": round(a[3] - b[3], 4), "total_ms_checksummed": a[0],
                  "total_ms_plain": b[0]})
    if A.out:
        with open(A.out, "a") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
