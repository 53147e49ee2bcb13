"""bench.py --dump-outputs: the arrays a caller of the timed path receives from its last step, written so that two builds
run with the same arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench
    return bench


def test_output_sample_is_seeded_and_leaves_out_padding(monkeypatch):
    import torch
    bench = _bench()
    rng = np.random.default_rng(1)
    lens = np.array([5, 0, 17, 0, 0, 33, 1], np.uint64)
    off = np.concatenate([[0], np.cumsum((lens + np.uint64(15)) & ~np.uint64(15))])[:-1].astype(np.uint64)
    buf = np.full(int(off[-1] + lens[-1]) + 16, 0xEE, np.uint8)  # alignment padding holds a byte no row holds
    rows = [rng.integers(0, 200, int(n), dtype=np.uint8) for n in lens]
    for o, r in zip(off, rows):
        buf[int(o):int(o) + r.size] = r
    st = np.arange(len(lens), dtype=np.uint32)
    dg = rng.integers(0, 256, (len(lens), 32), dtype=np.uint8)
    d = bench.output_sample(torch.from_numpy(buf), off, lens, st, dg)
    assert all(a.dtype == np.float32 for a in d.values())
    assert (d["output"] == np.concatenate(rows)).all() and (d["status"] == st).all() and (d["digest"] == dg).all()
    # beyond the budgets: fixed-size samples at the same positions on every call, never a padding byte
    monkeypatch.setattr(bench, "DUMP_BYTES", 20)
    monkeypatch.setattr(bench, "DUMP_ROWS", 3)
    a = bench.output_sample(torch.from_numpy(buf), off, lens, st, dg)
    b = bench.output_sample(torch.from_numpy(buf), off, lens, st, dg)
    assert a["output"].size == 20 and a["digest"].shape == (3, 32) and a["status"].shape == (3,)
    assert (a["output"] != 0xEE).all()
    assert all((a[k] == b[k]).all() for k in a)


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    bench = _bench()
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gib", "0.0625", "--steps", "2", "--warmup", "0",
                        "--no-cpu", "--sustain", "0", "--no-compress", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == line["e2e"]["steps"] == line["e2e_extract"]["steps"] == 2
    d = {k: np.load(tmp_path / f"{k}.npy") for k in ("status", "digest", "output")}
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    # 64 MiB of the text pattern = 8 rows of 8 MiB; digests as the official blake3 bindings give them
    want = [np.frombuffer(bench._digest(bench.text_slice(k * bench.SLICE % len(bench.PHRASE), bench.SLICE)), np.uint8)
            for k in range(8)]
    assert (d["status"] == 0).all() and (d["digest"] == np.stack(want)).all()
    assert d["output"].size == bench.DUMP_BYTES and set(np.unique(d["output"]).tolist()) <= set(bench.PHRASE)
