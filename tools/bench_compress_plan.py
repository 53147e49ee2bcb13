#!/usr/bin/env python
"""Device-resident compress plans (zn_plan_compress, DESIGN.md §4.3) against the host-buffer call zn_compress_batch on the
same data, alternating in one process.  Workloads larger than the 126 MB L2: 256 MiB of real text in 8 MiB slices
(32 rotations of the standard library's sources) at levels 3, 19 and 22, the 500 MiB binary pattern (BASELINE configs[3])
at level 19, and 100 000 generated 10 KiB text files (configs[0]) at level 19.

Per workload: the device time of the plan's compress kernels plus its sizing and packing (comparable with
zn_ctx_last_compress_ms, which covers the block kernels and the frame assembly of zn_compress_batch) and of the whole
run including the source hash, device GB/s of both, launches per run, the host time zn_plan_run_compress takes to
return (the enqueue alone), and the share of the sizing-and-packing stage in the run.  Prints one JSON line per
workload, each carrying the card and its power limit; `--out FILE` also writes them there.

    python tools/bench_compress_plan.py [--steps 5] [--out profiles/r3_compress_plan.jsonl]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import oracle as O  # noqa: E402
from bench_compress_long import gpu_info  # noqa: E402
from test_hostemu_compress_long import stdlib_text  # noqa: E402
from znippy_b200 import Ctx, Plan, codec  # noqa: E402

MiB = 1 << 20


def workloads():
    whole = stdlib_text(9 * MiB)  # 8 MiB windows of rotations of 9 MiB of sources: no slice repeats inside itself
    text = np.concatenate([np.roll(whole, -k * 65_537)[:8 * MiB] for k in range(32)])
    slices = lambda n, sl: ([o for o in range(0, n, sl)], [min(sl, n - o) for o in range(0, n, sl)])  # noqa: E731
    for level in (3, 19, 22):
        yield "real text 256 MiB, 8 MiB slices", level, text, *slices(text.size, 8 * MiB)
    binary = (np.arange(500 * MiB, dtype=np.uint32) % 251).astype(np.uint8)
    yield "binary pattern 500 MiB, 8 MiB slices", 19, binary, *slices(binary.size, 8 * MiB)
    small = O.gen_text(100_000 * 10240)
    yield "100 000 x 10 KiB text files", 19, small, *slices(small.size, 10240)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = gpu_info()
    ctx = Ctx(0)
    lines = []
    for name, level, data, offs, lens in workloads():
        n = len(offs)
        d_src = torch.from_numpy(data).cuda()
        plan = Plan.compress(ctx, offs, lens, level=level)
        d_dst = torch.empty(plan.capacity(), dtype=torch.uint8, device="cuda")
        d_off = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

        def run_plan():
            before = ctx.launches()
            ev[0].record(s)
            t0 = time.perf_counter()
            plan.run_compress(d_src.data_ptr(), d_dst.data_ptr(), d_off.data_ptr(), s.cuda_stream)
            t1 = time.perf_counter()
            ev[1].record(s)
            s.synchronize()
            return (t1 - t0) * 1e3, ev[0].elapsed_time(ev[1]), plan.last_ms(), ctx.launches() - before

        def run_batch():
            before = ctx.launches()
            blobs, dg, st = codec.compress_batch(data, offs, lens, level, codec.CODEC_ZSTD, ctx)
            return ctx.last_compress_ms(), ctx.launches() - before, blobs, dg, st

        run_plan(), run_batch()  # warm-up: modules, the ctx's scratch
        p, b = [], []
        for _ in range(a.steps):
            p.append(run_plan())
            b.append(run_batch())
        # the last runs of both: same blobs and digests
        boffs = d_off.cpu().numpy()
        dst = d_dst[:int(boffs[-1])].cpu().numpy()
        _, _, blobs, dg, st = b[-1]
        pst, pdg = plan.results()
        same = (not st.any() and not pst.any() and np.array_equal(pdg, dg)
                and all(dst[boffs[i]:boffs[i + 1]].tobytes() == blobs[i] for i in range(n)))
        med = lambda xs: float(np.median(xs))  # noqa: E731
        plan_ms = med([m[1] + m[3] for _, _, m, _ in p])  # compress kernels + sizing and packing
        batch_ms = med([x[0] for x in b])
        d = {"what": "compress plan vs compress_batch", "workload": name, "level": level, "slices": n,
             "bytes_in": int(data.size), "bytes_out": int(boffs[-1]), "steps": a.steps, "same_blobs_and_digests": bool(same),
             "plan_device_ms_median": round(plan_ms, 3),
             "plan_device_GBps": round(data.size / plan_ms / 1e6, 2),
             "plan_run_with_hash_ms_median": round(med([m[0] for _, _, m, _ in p]), 3),
             "plan_stream_events_ms_median": round(med([x[1] for x in p]), 3),
             "batch_device_ms_median": round(batch_ms, 3),
             "batch_device_GBps": round(data.size / batch_ms / 1e6, 2),
             "plan_launches_per_run": plan.launches(), "plan_ctx_launch_delta": p[-1][3],
             "batch_launches_per_call": b[-1][1],
             "plan_enqueue_host_ms_median": round(med([x[0] for x in p]), 3),
             "plan_enqueue_host_ms_max": round(max(x[0] for x in p), 3),
             "sizing_packing_ms_median": round(med([m[3] for _, _, m, _ in p]), 3),
             "sizing_packing_share_of_run": round(med([m[3] / m[0] for _, _, m, _ in p]), 4),
             **info}
        lines.append(d)
        print(json.dumps(d), flush=True)
        plan.close()
        del d_src, d_dst, d_off
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            f.writelines(json.dumps(d) + "\n" for d in lines)


if __name__ == "__main__":
    main()
