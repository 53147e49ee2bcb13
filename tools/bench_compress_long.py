#!/usr/bin/env python
"""Speed, ratio and scratch of the zstd long effort (levels >= 20, DESIGN.md §4.3) against the level-19 effort, on
batches larger than the 126 MB L2: 256 MiB of real text (32 slices of 8 MiB, each a different rotation of the standard
library's sources, none repeating inside itself) and the 500 MiB binary pattern (BASELINE configs[3]).  Prints one JSON
line per measurement, each carrying the card and its power limit; `--out FILE` also writes them there.

    python tools/bench_compress_long.py [--steps 5] [--out profiles/r3_compress_long.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from test_hostemu_compress_long import stdlib_text  # noqa: E402
from znippy_b200 import Ctx, Plan, codec  # noqa: E402

SL = 8 << 20


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, plim, clk = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}


def free_mem() -> int:
    import torch
    return torch.cuda.mem_get_info()[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = gpu_info()
    lines = []

    def emit(d):
        d = {**d, **info}
        lines.append(d)
        print(json.dumps(d), flush=True)

    z = bench._libzstd()
    ctx = Ctx(0, staging_bytes=(512 << 20) + (1 << 20))
    text = np.concatenate([stdlib_text(SL, k * 65_537) for k in range(32)])
    binary = (np.arange(500 << 20, dtype=np.uint32) % 251).astype(np.uint8)
    frames = {}
    for cname, data in (("real text 256 MiB (32 rotations of the stdlib sources)", text), ("binary pattern 500 MiB", binary)):
        offs = list(range(0, len(data), SL))
        lens = [min(SL, len(data) - o) for o in offs]
        src = ctx.pinned()[:len(data)]
        src[:] = data
        samples = (0, len(offs) // 2)  # libzstd-19 runs at ~2 MB/s a core: two sample slices
        ref = {i: len(bench._zstd_compress(z, np.ascontiguousarray(data[offs[i]:offs[i] + lens[i]]), 19)) for i in samples}
        for level in (19, 22):
            free0 = free_mem()
            codec.compress_batch(src, offs, lens, level, codec.CODEC_ZSTD, ctx)  # warm-up: modules, scratch growth
            grown = free0 - free_mem()
            ms = []
            for _ in range(a.steps):
                blobs, dg, st = codec.compress_batch(src, offs, lens, level, codec.CODEC_ZSTD, ctx)
                assert not st.any()
                ms.append(ctx.last_compress_ms())
            assert all(z_ok(z, blobs[i], data[offs[i]:offs[i] + lens[i]]) for i in samples)
            out = sum(len(b) for b in blobs)
            emit({"what": "compress", "corpus": cname, "level": level, "bytes_in": len(data), "bytes_out": out,
                  "ratio": round(len(data) / out, 3), "steps": a.steps, "device_ms_median": round(float(np.median(ms)), 2),
                  "device_ms_min": round(min(ms), 2), "device_GBps_median": round(len(data) / float(np.median(ms)) / 1e6, 3),
                  "size_vs_libzstd19_on_samples": round(sum(len(blobs[i]) for i in samples) / sum(ref.values()), 4),
                  "ctx_device_memory_growth_MiB_first_call": round(grown / 2**20, 1)})
            frames[(cname, level)] = (blobs, dg, lens)
    # decode of the level-22 real-text frames through Plan, against libzstd-19 frames of the same slices
    tname = "real text 256 MiB (32 rotations of the stdlib sources)"
    with ThreadPoolExecutor(max(1, min(32, os.cpu_count() or 1))) as ex:
        ref19 = list(ex.map(lambda i: bench._zstd_compress(z, np.ascontiguousarray(text[i * SL:(i + 1) * SL]), 19), range(32)))
    blobs22, dg22, lens = frames[(tname, 22)]
    for label, blobs in (("ours level 22", blobs22), ("libzstd 19", ref19)):
        r = decode_plan(ctx, blobs, lens, dg22, a.steps)
        emit({"what": "decode through Plan", "corpus": tname, "frames": label, "bytes_out": int(sum(lens)),
              "bytes_in": sum(len(b) for b in blobs), **r})
    if a.out:
        with open(a.out, "w") as f:
            f.writelines(json.dumps(d) + "\n" for d in lines)


def z_ok(z, blob, want) -> bool:
    import ctypes as C
    z.ZSTD_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    z.ZSTD_decompress.restype = C.c_size_t
    out = np.empty(len(want), np.uint8)
    b = np.frombuffer(blob, np.uint8)
    return z.ZSTD_decompress(out.ctypes.data, len(want), b.ctypes.data, b.size) == len(want) and (out == want).all()


def decode_plan(ctx, blobs, lens, digests, steps) -> dict:
    import torch
    boff = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])[:-1]
    out_len = np.array(lens, np.uint64)
    out_off = np.concatenate([[0], np.cumsum(out_len)])[:-1].astype(np.uint64)
    d_in = torch.from_numpy(np.frombuffer(b"".join(blobs), np.uint8).copy()).cuda()
    d_out = torch.zeros(int(out_len.sum()) + 256, dtype=torch.uint8, device="cuda")
    plan = Plan.decode_verify(ctx, boff.tolist(), [len(b) for b in blobs], [1] * len(blobs), out_off, out_len, digests.tobytes())
    s = torch.cuda.Stream()  # a real stream: the plan's kernels and the timing events share it
    plan.run(d_in.data_ptr(), d_out.data_ptr(), s.cuda_stream)  # warm-up
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(s)
    for _ in range(steps):
        plan.run(d_in.data_ptr(), d_out.data_ptr(), s.cuda_stream)
    ev[1].record(s)
    torch.cuda.synchronize()
    st, _ = plan.results()
    ms = ev[0].elapsed_time(ev[1]) / steps
    return {"statuses_ok": bool((st == 0).all()), "pipeline_fallbacks": plan.pipeline_fallbacks(), "steps": steps,
            "device_ms_per_step": round(ms, 3), "device_GBps": round(float(out_len.sum()) / ms / 1e6, 1)}


if __name__ == "__main__":
    main()
