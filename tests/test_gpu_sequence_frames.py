"""The frames of tests/test_hostemu_sequence_frames.py (built from chosen sequences, aimed at the branches of k_zexec2) on
the device.  Every batch asserts the decode class of its rows (zn_plan_class_counts), how many rows the device-wide
pipeline handed back to the one-team decoder (0 unless a row is ill-formed or the stated behaviour is a hand-back), and
every status, byte and digest against the content and the oracle's BLAKE3.  Pipeline rows run in both exec shapes:
mean decoded size >= 256 KiB (k_zexec2<512,4,16384,2,8192>) and a batch of many small rows (k_zexec2<512,2,16384,3>,
whose lists alias the literal staging area)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(__file__))
from test_hostemu_sequence_frames import (BIGPAT, KIB, PIPE, SMALL, cases, lz4_cases, route,  # noqa: E402
                                          route_cases, small_window_cases)


@pytest.fixture(scope="module")
def codec():
    from znippy_b200 import codec as c
    c.default_ctx()
    return c


def _run(codec, oracle, rows, want_fallbacks):
    """rows: (name, blob, content, ok).  One Plan over all of them (blob k at an address that is k modulo 16, output
    rows 16-byte aligned in a buffer pre-filled with 0xEE): asserts the routes plan_build chose equal route() of every row,
    the pipeline's hand-backs, and per row the status, bytes and digest.  Returns the class counts."""
    import torch
    from znippy_b200 import Plan
    offs, cur = [], 0
    for k, (_, b, _, _) in enumerate(rows):
        cur = (cur + 15) // 16 * 16 + k % 16
        offs.append(cur)
        cur += len(b)
    buf = np.zeros(cur + 16, np.uint8)
    for o, (_, b, _, _) in zip(offs, rows):
        buf[o:o + len(b)] = np.frombuffer(b, np.uint8)
    out_len = np.array([len(c) for _, _, c, _ in rows], np.uint64)
    out_off = np.concatenate([[0], np.cumsum((out_len + np.uint64(31)) & ~np.uint64(15))])[:-1].astype(np.uint64)
    digs = np.frombuffer(b"".join(oracle.blake3(c) for _, _, c, _ in rows), np.uint8)
    d_in = torch.from_numpy(buf).cuda()
    d_out = torch.full((int(out_off[-1] + out_len[-1]) + 256,), 0xEE, dtype=torch.uint8, device="cuda")
    plan = Plan.decode_verify(codec.default_ctx(), offs, [len(b) for _, b, _, _ in rows], [1] * len(rows), out_off, out_len,
                              digs)
    want = [0] * 5
    for _, b, c, _ in rows:
        want[route(len(c), len(b))] += 1
    counts = plan.class_counts()
    assert counts == want, (counts, want)
    plan.run(d_in.data_ptr(), d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    st, dg = plan.results()
    assert plan.pipeline_fallbacks() == want_fallbacks
    out = d_out.cpu().numpy()
    for i, (name, _, c, ok) in enumerate(rows):
        o = int(out_off[i])
        if ok:
            assert st[i] == codec.S_OK, (name, st[i])
            assert out[o:o + len(c)].tobytes() == c, name
            assert dg[i].tobytes() == oracle.blake3(c), name
        else:
            assert st[i] == codec.S_DECODE_ERROR, (name, st[i])
        assert (out[o + len(c):o + len(c) + 16] == 0xEE).all(), name  # nothing past the row
    return counts


@pytest.mark.parametrize("shape", ["large", "small"])
def test_sequence_frames_through_the_pipeline(codec, oracle, shape):
    """Every pipeline case (longer than a group, every setup branch over Huffman / RLE / raw literals, list overflow and
    full-depth chains, repeat offsets, frame bounds) in one batch per exec shape, beside the blob of a frame compressed
    against a prefix: that blob alone is handed back and gets S_DECODE_ERROR, its neighbours are exact.  The shape
    follows the mean decoded size of the pipeline rows: filler rows of real text set it on the intended side of 256 KiB."""
    O = oracle
    z = O.libzstd()
    rows = [(n, c["blob"], c["content"], c["ok"]) for n, c in cases().items()]
    total = sum(len(r[2]) for r in rows)
    rt = O.real_text(8 << 20)
    if shape == "large":
        need = 256 * KIB * (len(rows) + 1) - total + 64 * KIB
        fill = [rt[:max(need, 64 * KIB)].tobytes()]
    else:
        fill = [rt[k * 7001:k * 7001 + 6000 + 37 * k].tobytes() for k in range(64)]
    rows += [(f"filler_{k}", z.compress(c, 3), c, True) for k, c in enumerate(fill)]
    mean = sum(len(r[2]) for r in rows) // len(rows)
    assert (mean >= 256 * KIB) == (shape == "large")
    counts = _run(codec, O, rows, want_fallbacks=1)
    assert counts[PIPE] == len(rows)


def test_sequence_frames_through_the_other_decode_classes(codec, oracle):
    """The same shapes as rows of the other classes: pattern rows (offset-1 runs appended until compressed <= 1/64) of
    512 KiB and more (k_decode_ws) and below (k_decode<128,4>), rows under 4 KiB (k_decode<32,2>), and a frame at least as
    large as its content, of raw blocks and one Huffman / FSE block (k_decode_par)."""
    rows = [(n, c["blob"], c["content"], True) for n, c in route_cases().items()]
    counts = _run(codec, oracle, rows, want_fallbacks=0)
    assert counts == [0, 1, 1, 3, 1]


def test_small_window_frames_are_handed_back(codec, oracle):
    """Frames without a content size at windowLog 10 and 12 have blocks of at most 1-4 KiB, more than the pipeline's slot
    budget (decoded size / 16 KiB + 8, DESIGN §4.4) allows: the pipeline hands exactly those two rows back and the
    one-team decoder decodes them exactly; windowLog 14 and 16 stay in the pipeline."""
    rows = [(n, b, d, True) for n, (b, d, _) in small_window_cases().items()]
    _run(codec, oracle, rows, want_fallbacks=sum(p for _, _, p in small_window_cases().values()))


def test_lz4_frames_with_1_and_4_mib_blocks(codec, oracle):
    """LZ4 frames of block size ids 6 and 7, linked and independent: text rows reach the pipeline, which hands every one
    back to the one-team decoder; pattern rows take k_decode_ws; rows under 4 KiB take k_decode<32,2>."""
    rows = [(n, b, d, True) for n, (b, d, _) in lz4_cases().items()]
    counts = _run(codec, oracle, rows, want_fallbacks=4)
    assert counts[PIPE] == 4 and counts[BIGPAT] == 4 and counts[SMALL] == 4


def test_sequence_frames_as_partial_rows(codec, oracle):
    """The pipeline cases decoded up to a stop (zn_decode_windows, the range-read decoder): stops up to 64 KiB run
    k_decode<32,2,true>, larger ones k_decode<128,4,true>; the window [0, stop) of every row equals the content's prefix,
    and the ill-formed blob is rejected exactly when its bad match lies before the stop."""
    from znippy_b200 import _native as N
    L = N.lib()
    L.zn_decode_windows.argtypes = [C.c_void_p] + [C.c_void_p] * 6 + [C.c_uint32] + [C.c_void_p] * 3 + [C.c_uint32] + \
        [C.c_void_p] * 3
    rows = []
    for n, c in cases().items():
        for stop in (1000, 40_000, 100_000, len(c["content"]) - 1):
            if stop < len(c["content"]):
                rows.append((n, c["blob"], c["content"], c["ok"], stop))
    blobs = b"".join(r[1] for r in rows)
    bo = np.cumsum([0] + [len(r[1]) for r in rows])[:-1].astype(np.uint64)
    bl = np.array([len(r[1]) for r in rows], np.uint64)
    cf = np.ones(len(rows), np.uint8)
    ol = np.array([len(r[2]) for r in rows], np.uint64)
    stop = np.array([r[4] for r in rows], np.uint64)
    w_row = np.arange(len(rows), dtype=np.uint32)
    w_off = np.zeros(len(rows), np.uint64)
    pack = np.zeros(int(stop.sum()) + 1, np.uint8)
    st = np.zeros(len(rows), np.uint32)
    produced = np.zeros(len(rows), np.uint64)
    ctx = codec.default_ctx()
    base = np.frombuffer(blobs, np.uint8)
    p = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    rc = L.zn_decode_windows(ctx.handle, p(base), p(bo), p(bl), p(cf), p(ol), p(stop), len(rows), p(w_row), p(w_off),
                             p(stop), len(rows), p(pack), p(st), p(produced))
    assert rc == 0, L.zn_last_error(ctx.handle)
    cur = 0
    for i, (name, _, content, ok, s) in enumerate(rows):
        # the ill-formed blob's bad match opens its second frame: a stop before that frame decodes a good prefix
        if ok or s <= cases()[name]["frames"][-1][2]:
            assert st[i] == codec.S_OK, (name, s, st[i])
            assert pack[cur:cur + s].tobytes() == content[:s], (name, s)
            assert s <= produced[i] <= len(content), (name, s, produced[i])
        else:
            assert st[i] == codec.S_DECODE_ERROR, (name, s, st[i])
        cur += s
