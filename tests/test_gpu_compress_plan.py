"""Device-resident compress plans (zn_plan_compress / zn_plan_run_compress): slices already in HBM compressed into packed
blobs on the caller's stream.  Every blob must equal what the host-buffer calls give for its slice (compress_batch's
frame, or CompressCtx(envelope=True)'s ZNB1 blob), the offsets must be the prefix sum of the blob sizes, and a run must
only enqueue work."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(__file__))
MiB = 1 << 20
LEVELS = [("zstd", 1), ("zstd", 3), ("zstd", 19), ("zstd", 22), ("lz4", 1)]


@pytest.fixture(scope="module")
def env():
    import torch
    from znippy_b200 import codec
    codec.default_ctx()
    return torch, codec


def _cid(codec, name):
    return codec.CODEC_ZSTD if name == "zstd" else codec.CODEC_LZ4


def _corpora(O):
    from test_gpu_compress import _cases
    from test_hostemu_compress_long import stdlib_text
    c = dict(_cases(O))
    c["stdlib8m+17"] = stdlib_text(8 * MiB + 17, 777)  # two units of the long effort
    return c


def _batch(datas, first=16, gap=3, align=1):
    """datas in one host buffer, the first at `first`, then `gap` bytes between slices, offsets rounded up to `align`.
    The window efforts' frames depend on a slice's 16-byte phase in device memory; compress_batch mirrors a compact
    host span from its first byte, so with `first` a multiple of 16 both calls see every slice at the same phase."""
    offs, cur = [], first
    for d in datas:
        offs.append(cur)
        cur = (cur + len(d) + gap + align - 1) // align * align
    src = np.zeros(cur + 1, np.uint8)
    for o, d in zip(offs, datas):
        src[o:o + len(d)] = d
    return src, offs, [len(d) for d in datas]


def _run(torch, plan, d_src, stream=None, sync=True):
    """run_compress on `stream` (a new one by default) into a d_dst offset by 3 bytes; returns (d_dst, d_offsets)"""
    cap = plan.capacity()
    d_dst = torch.full((cap + 3 + 64,), 0xAA, dtype=torch.uint8, device="cuda")
    d_off = torch.full((plan.n + 1,), -1, dtype=torch.int64, device="cuda")
    s = stream if stream is not None else torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())  # the buffers above are written on the current stream
    plan.run_compress(d_src.data_ptr(), d_dst.data_ptr() + 3, d_off.data_ptr(), s.cuda_stream)
    if sync:
        torch.cuda.synchronize()
    return d_dst, d_off


def _blobs(d_dst, d_off):
    offs = d_off.cpu().numpy().astype(np.uint64)
    dst = d_dst.cpu().numpy()
    return [dst[3 + int(offs[i]): 3 + int(offs[i + 1])].tobytes() for i in range(offs.size - 1)], offs, dst


def _check_packed(blobs, offs, dst):
    assert offs[0] == 0 and np.array_equal(offs, np.concatenate([[0], np.cumsum([len(b) for b in blobs])]).astype(np.uint64))
    assert (dst[:3] == 0xAA).all() and (dst[3 + int(offs[-1]):] == 0xAA).all()  # nothing written outside the blobs


@pytest.mark.parametrize("codec_name,level", LEVELS)
def test_plan_blobs_equal_compress_batch_frames(env, oracle, codec_name, level):
    torch, codec = env
    O = oracle
    cid = _cid(codec, codec_name)
    cs = _corpora(O)
    names, datas = list(cs), list(cs.values())
    src, offs, lens = _batch(datas)
    want, want_dg, want_st = codec.compress_batch(src, offs, lens, level, cid)
    assert not want_st.any()
    plan = codec.N.Plan.compress(codec.default_ctx(), offs, lens, level=level, codec=cid)
    assert plan.capacity() == sum(codec.compress_bound(n, cid) for n in lens)
    d_src = torch.from_numpy(src).cuda()
    blobs, boffs, dst = _blobs(*_run(torch, plan, d_src))
    _check_packed(blobs, boffs, dst)
    st, dg = plan.results()
    assert not st.any()
    assert np.array_equal(dg, want_dg)
    for name, d, b, w in zip(names, datas, blobs, want):
        assert b == w, (name, len(b), len(w))
        if codec_name == "zstd":
            assert O.libzstd().decompress(b, len(d)) == d.tobytes(), name
        else:
            assert O.liblz4().decompress_frame(b, len(d)) == d.tobytes(), name
    ms = plan.last_ms()
    assert ms[0] > 0 and ms[1] > 0 and ms[3] > 0 and ms[0] >= max(ms[1:])


@pytest.mark.parametrize("codec_name,level", [("zstd", 3), ("zstd", 22), ("lz4", 1)])
def test_plan_envelope_blobs_equal_archive_rows(env, oracle, codec_name, level):
    torch, codec = env
    O = oracle
    cid = _cid(codec, codec_name)
    cs = _corpora(O)
    names, datas = list(cs), list(cs.values())
    src, offs, lens = _batch(datas, gap=7, align=16)  # CompressCtx.compress stages each slice 16-byte aligned
    plan = codec.N.Plan.compress(codec.default_ctx(), offs, lens, level=level, codec=cid, envelope=True)
    assert plan.capacity() == sum(n + len(codec.envelope_wrap(0, n, b"")) for n in lens)
    d_src = torch.from_numpy(src).cuda()
    blobs, boffs, dst = _blobs(*_run(torch, plan, d_src))
    _check_packed(blobs, boffs, dst)
    st, dg = plan.results()
    assert not st.any()
    cc = codec.CompressCtx(level, cid, envelope=True)
    kinds = {}
    for name, d, b in zip(names, datas, blobs):
        assert b == cc.compress(d), name
        kinds[name] = codec.envelope_parse(b)[1]
    for name in ("empty", "rand", "inc"):  # incompressible slices are stored RAW
        assert kinds[name] == codec.PAYLOAD_RAW, name
    assert kinds["text3m"] == (codec.PAYLOAD_ZSTD if codec_name == "zstd" else codec.PAYLOAD_LZ4_FRAME)
    buf = np.frombuffer(b"".join(blobs), np.uint8)
    out = np.zeros(sum(lens) + 1, np.uint8)
    ooff = np.concatenate([[0], np.cumsum(lens)])[:-1]
    st2, dg2 = codec.decode_verify_batch(buf, boffs[:-1], [len(b) for b in blobs], [codec.COMPRESSED_ENVELOPED] * len(blobs), lens,
                                         dg.tobytes(), out, ooff)
    assert not st2.any() and np.array_equal(dg2, dg)
    for i, d in enumerate(datas):
        assert out[ooff[i]:ooff[i] + len(d)].tobytes() == d.tobytes(), names[i]
    for i, d in enumerate(datas):
        assert dg[i].tobytes() == O.blake3(d.tobytes()), names[i]


def test_plan_round_trip_in_hbm(env):
    """256 MiB of real text in 8 MiB slices: compressed by a plan, decoded by a decode plan from the returned offsets, on
    the same device buffers, checked against the compress plan's digests."""
    torch, codec = env
    from test_hostemu_compress_long import stdlib_text
    Plan = codec.N.Plan
    ctx = codec.default_ctx()
    whole = stdlib_text(9 * MiB)  # each 8 MiB window of a rotation: no slice repeats inside itself
    text = np.concatenate([np.roll(whole, -k * 65_537)[:8 * MiB] for k in range(32)])
    offs, lens = [k * 8 * MiB for k in range(32)], [8 * MiB] * 32
    d_src = torch.from_numpy(text).cuda()
    plan = Plan.compress(ctx, offs, lens, level=19)
    d_dst, d_off = _run(torch, plan, d_src)
    st, dg = plan.results()
    assert not st.any()
    boffs = d_off.cpu().numpy().astype(np.uint64)
    d_out = torch.zeros(len(text) + 256, dtype=torch.uint8, device="cuda")
    dplan = Plan.decode_verify(ctx, boffs[:-1] + 3, np.diff(boffs), [1] * 32, offs, lens, dg.tobytes())
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    dplan.run(d_dst.data_ptr(), d_out.data_ptr(), s.cuda_stream)
    torch.cuda.synchronize()
    st2, dg2 = dplan.results()
    assert not st2.any() and np.array_equal(dg2, dg)
    assert dplan.pipeline_fallbacks() == 0
    assert torch.equal(d_out[:len(text)], d_src)


def test_plan_run_returns_before_the_work_is_done(env, oracle):
    torch, codec = env
    cs = _corpora(oracle)
    datas = [cs["text3m"], cs["real"], cs["rand"]]
    src, offs, lens = _batch(datas)
    want, want_dg, _ = codec.compress_batch(src, offs, lens, 3)
    plan = codec.N.Plan.compress(codec.default_ctx(), offs, lens, level=3)
    d_src = torch.from_numpy(src).cuda()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(1_000_000_000)  # holds the stream for ~0.5 s
    d_dst, d_off = _run(torch, plan, d_src, stream=s, sync=False)
    done = torch.cuda.Event()
    done.record(s)
    assert not done.query()  # the call returned while the stream was still busy
    torch.cuda.synchronize()
    blobs, _, _ = _blobs(d_dst, d_off)
    assert blobs == want
    assert np.array_equal(plan.results()[1], want_dg)


def test_plan_reuse_concurrency_and_isolation(env, oracle):
    torch, codec = env
    ctx = codec.default_ctx()
    cs = _corpora(oracle)
    a = [cs["text3m"], cs["real"], cs["bin1m+17"], cs["exe"], cs["one"]]
    b = [np.roll(x, 1000) for x in a]
    src_a, offs, lens = _batch(a)
    src_b, offs_b, _ = _batch(b)
    assert offs_b == offs
    p3 = codec.N.Plan.compress(ctx, offs, lens, level=3)
    p22 = codec.N.Plan.compress(ctx, offs, lens, level=22, codec=codec.CODEC_ZSTD)
    # a host-buffer call on the same ctx between plan creation and run, with other sizes and another effort
    other = cs["stdlib8m+17"]
    codec.compress_batch(other, [0, 17], [other.size - 17, 17], 22)
    codec.compress_batch(other, [0], [other.size], 1, codec.CODEC_LZ4)
    want = {(lvl, k): codec.compress_batch(s, offs, lens, lvl) for lvl in (3, 22) for k, s in (("a", src_a), ("b", src_b))}
    d_a, d_b = torch.from_numpy(src_a).cuda(), torch.from_numpy(src_b).cuda()
    # the same plan over two different sources of the same sizes
    for k, d in (("a", d_a), ("b", d_b)):
        blobs, _, _ = _blobs(*_run(torch, p3, d))
        assert blobs == want[(3, k)][0], k
        assert np.array_equal(p3.results()[1], want[(3, k)][1]), k
    # two plans at once on two streams
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    r3 = _run(torch, p3, d_b, stream=s1, sync=False)
    r22 = _run(torch, p22, d_a, stream=s2, sync=False)
    torch.cuda.synchronize()
    assert _blobs(*r3)[0] == want[(3, "b")][0]
    assert _blobs(*r22)[0] == want[(22, "a")][0]
    assert np.array_equal(p22.results()[1], want[(22, "a")][1])


@pytest.mark.parametrize("codec_name,level,digests", [("zstd", 1, True), ("zstd", 22, True), ("lz4", 1, False)])
def test_plan_launch_count(env, oracle, codec_name, level, digests):
    torch, codec = env
    ctx = codec.default_ctx()
    cs = _corpora(oracle)
    src, offs, lens = _batch([cs["stdlib8m+17"], cs["text10k"], cs["empty"]])
    plan = codec.N.Plan.compress(ctx, offs, lens, level=level, codec=_cid(codec, codec_name), digests=digests)
    d_src = torch.from_numpy(src).cuda()
    before = ctx.launches()
    _run(torch, plan, d_src)
    assert ctx.launches() - before == plan.launches() > 0


def test_plan_bookkeeping_and_refusals(env):
    torch, codec = env
    N = codec.N
    L = N.lib()
    ctx = codec.default_ctx()
    # n = 0: a valid plan whose run writes d_offsets[0] = 0
    p0 = N.Plan.compress(ctx, [], [])
    assert p0.capacity() == 0
    d_off = torch.full((2,), 123, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    p0.run_compress(0, 0, d_off.data_ptr())
    torch.cuda.synchronize()
    assert d_off.tolist() == [0, 123]
    st, dg = p0.results()
    assert st.size == 0 and p0.launches() == 0
    # wrong kinds: ZN_E_STATE, nothing touched
    plan = N.Plan.compress(ctx, [0, 5], [5, 100], level=3)
    hplan = N.Plan.hash(ctx, [0], [5])
    d_src = torch.zeros(256, dtype=torch.uint8, device="cuda")
    d_dst = torch.zeros(plan.capacity() + 16, dtype=torch.uint8, device="cuda")
    d_off = torch.zeros(4, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    vp = C.c_void_p
    assert L.zn_plan_run(plan._h, vp(d_src.data_ptr()), vp(d_dst.data_ptr()), None) == N.ZN_E_STATE
    assert L.zn_plan_run_compress(hplan._h, vp(d_src.data_ptr()), vp(d_dst.data_ptr()), vp(d_off.data_ptr()), None) == N.ZN_E_STATE
    assert L.zn_plan_class_counts(plan._h, (C.c_uint32 * 5)()) == N.ZN_E_STATE
    assert L.zn_plan_pipeline_fallbacks(plan._h, C.byref(C.c_uint32())) == N.ZN_E_STATE
    assert L.zn_plan_results(plan._h, None, None) == N.ZN_E_STATE  # not run yet
    # d_offsets must be 8-byte aligned
    assert L.zn_plan_run_compress(plan._h, vp(d_src.data_ptr()), vp(d_dst.data_ptr()), vp(d_off.data_ptr() + 4), None) == N.ZN_E_ARG
    torch.cuda.synchronize()
    assert not d_dst.any() and not d_off.any()
    # refused at creation: a slice of 4 GiB or more (sizes only, no buffer), codecs other than ZSTD / LZ4 (+ ENVELOPE)
    with pytest.raises(N.NativeError, match="slice too large"):
        N.Plan.compress(ctx, [0, 0], [10, 4 << 30])
    for bad in (0, 3, N.CODEC_ENVELOPE, 0x200 | N.CODEC_ZSTD):
        with pytest.raises(N.NativeError, match="codec"):
            N.Plan.compress(ctx, [0], [10], codec=bad)
    N.Plan.compress(ctx, [0], [10], codec=N.CODEC_LZ4, envelope=True).close()
