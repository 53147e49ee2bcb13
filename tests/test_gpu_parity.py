"""GPU parity tests proper: the CUDA path (through the C ABI of libznippy_cuda.so) against the CPU oracle and the
committed golden fixtures.  Reference items: a1 codec::decompress_into (codec.rs:67-78), a2/a6 blake3::hash
(decompress.rs:172, stream_packer.rs:219), a3 read-loop status rules (decompress.rs:156-184), a7 store-as-is rows.
Bar: bit-exact bytes and digests."""
import base64
import json
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def codec():
    from znippy_b200 import codec as c
    c.default_ctx()  # raises loudly when the CUDA library or device is missing
    return c


def _pack(blobs, align=1, lead=0):
    offs, cur = [], lead
    for b in blobs:
        cur = (cur + align - 1) // align * align
        offs.append(cur)
        cur += len(b)
    buf = np.zeros(cur + 1, np.uint8)
    for o, b in zip(offs, blobs):
        buf[o:o + len(b)] = np.frombuffer(b, np.uint8)
    return buf, offs


def _run(codec, blobs, comp, contents, expect=True, want_out=True, align=1, lead=0, out_lens=None):
    buf, offs = _pack(blobs, align, lead)
    out_len = out_lens or [len(c) for c in contents]
    out_off = np.concatenate([[0], np.cumsum([(n + 15) // 16 * 16 + 3 for n in out_len])])[:-1] + 1  # odd alignment
    out = np.zeros(int(out_off[-1]) + out_len[-1] + 64 if len(out_len) else 1, np.uint8) if want_out else None
    import oracle as O
    ex = b"".join(O.blake3(c) for c in contents) if expect else None
    st, dg = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], comp, out_len, ex, out,
                                       out_off if want_out else None)
    return st, dg, out, out_off


def _classes(codec, blobs, contents):
    """rows per decode class plan_build gives these rows (zn_plan_class_counts; the plan is not run)"""
    from znippy_b200 import Plan
    lens = [len(c) for c in contents]
    return Plan.decode_verify(codec.default_ctx(), np.cumsum([0] + [len(b) for b in blobs])[:-1], [len(b) for b in blobs],
                              [1] * len(blobs), np.cumsum([0] + lens)[:-1], lens).class_counts()


def test_blake3_kats(codec, oracle):
    O = oracle
    kats = json.load(open(os.path.join(GOLD, "blake3_kat.json")))
    datas = []
    for k in kats:
        g = {"text": O.gen_text, "binary": O.gen_binary, "random": O.gen_random}.get(k["gen"])
        datas.append(g(k["n"]).tobytes() if g else O.gen_incompressible(k["n"], k.get("seed", 0)).tobytes())
    for lead in (0, 1, 5):  # aligned (cp.async path) and misaligned (assembled path) sources
        buf, offs = _pack(datas, align=16, lead=lead)
        offs = [o for o in offs]
        dg = codec.hash_batch(buf, offs, [len(d) for d in datas])
        for k, d in zip(kats, dg):
            assert d.tobytes().hex() == k["blake3"], (k["gen"], k["n"], lead)


def test_blake3_random_lengths_vs_oracle(codec, oracle):
    rng = np.random.default_rng(7)
    lens = [0, 1, 63, 64, 65, 1023, 1024, 1025] + [int(x) for x in rng.integers(0, 300000, 200)]
    datas = [rng.integers(0, 256, n, dtype=np.uint8).tobytes() for n in lens]
    buf, offs = _pack(datas, align=1, lead=3)
    dg = codec.hash_batch(buf, offs, lens)
    for d, data in zip(dg, datas):
        assert d.tobytes() == oracle.blake3(data)


def test_golden_frames(codec, oracle):
    frames = [f for f in json.load(open(os.path.join(GOLD, "frames.json")))["frames"] if f["codec"] != "lz4block"]
    blobs = [base64.b64decode(f["blob_b64"]) for f in frames]
    buf, offs = _pack(blobs)
    out_len = [f["out_len"] for f in frames]
    out_off = np.concatenate([[0], np.cumsum(out_len)])[:-1]
    out = np.zeros(sum(out_len) + 1, np.uint8)
    ex = b"".join(bytes.fromhex(f["out_blake3"]) for f in frames)
    st, dg = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [1] * len(blobs), out_len, ex, out, out_off)
    for i, f in enumerate(frames):
        assert st[i] == 0, (f["name"], st[i])
        assert dg[i].tobytes().hex() == f["out_blake3"], f["name"]
        assert oracle.blake3_official(out[out_off[i]:out_off[i] + out_len[i]]).hex() == f["out_blake3"], f["name"]


@pytest.mark.parametrize("level", [-5, 1, 3, 7, 19])
def test_zstd_entropy_paths_vs_oracle(codec, oracle, level):
    O = oracle
    z = O.libzstd()
    contents = [O.real_text(1_200_000).tobytes(), O.gen_small_alphabet(300_000).tobytes(),
                O.gen_periodic_noise(2000, 200, 12).tobytes(), O.gen_rle_literals().tobytes(),
                O.gen_text(3 << 20).tobytes(), O.gen_binary(1 << 20).tobytes(), O.gen_random(200_000).tobytes(), b"",
                bytes([7]) * 70000 + O.real_text(3000).tobytes() + bytes([9]) * 200000]
    blobs = [z.compress(c, level) for c in contents]
    # the last row, runs around real text, is compressed to under 1/64 and is below 512 KiB: it takes k_decode<128,4>,
    # not the device-wide pipeline
    assert _classes(codec, blobs[-1:], contents[-1:]) == [0, 0, 0, 0, 1]
    for b, c in zip(blobs, contents):  # the oracle agrees with libzstd on these frames
        rc, o = O.zstd_decompress(b, len(c))
        assert rc == 0 and o == c
    st, dg, out, out_off = _run(codec, blobs, [1] * len(blobs), contents)
    assert st.tolist() == [0] * len(blobs)
    for i, c in enumerate(contents):
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c, i
        assert dg[i].tobytes() == O.blake3(c)


def test_lz4_frames_vs_oracle(codec, oracle):
    O = oracle
    l = O.liblz4()
    contents = [O.real_text(900_000).tobytes(), O.gen_text(1 << 20).tobytes(), O.gen_random(100_000).tobytes(), b"",
                O.gen_binary(300_000).tobytes()]
    blobs = [l.compress_frame(c) for c in contents]
    blobs += [l.compress_frame(c, block_size_id=5, independent=False, content_checksum=True, block_checksum=True, level=9)
              for c in contents]
    contents = contents + contents
    st, dg, out, out_off = _run(codec, blobs, [1] * len(blobs), contents)
    assert st.tolist() == [0] * len(blobs)
    for i, c in enumerate(contents):
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c, i


def test_small_files_batch_and_store_as_is(codec, oracle):
    """config 1 shape (many 10 KiB text files, one blob each) mixed with store-as-is rows (a7)."""
    O = oracle
    z = O.libzstd()
    n = 3000
    contents, blobs, comp = [], [], []
    frame = z.compress(O.gen_text(10240).tobytes(), 19)
    rng = np.random.default_rng(3)
    for i in range(n):
        if i % 7 == 3:
            c = rng.integers(0, 256, int(rng.integers(0, 5000)), dtype=np.uint8).tobytes()
            contents.append(c); blobs.append(c); comp.append(0)
        else:
            contents.append(O.gen_text(10240).tobytes()); blobs.append(frame); comp.append(1)
    st, dg, out, out_off = _run(codec, blobs, comp, contents)
    assert not st.any()
    text_digest = O.blake3(contents[0])
    for i, c in enumerate(contents):
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c, i
        assert dg[i].tobytes() == (text_digest if comp[i] else O.blake3(c))
    # verify-only (save_data=false): no output buffer, same statuses
    st2, dg2, _, _ = _run(codec, blobs, comp, contents, want_out=False)
    assert not st2.any() and (dg2 == dg).all()


def test_full_slice_8mib_property(codec, oracle):
    """BASELINE-size slices (8 MiB, stream_packer.rs:31): digest of the decoded slice equals the SURVEY KATs."""
    O = oracle
    z = O.libzstd()
    text, binary = O.gen_text(8 << 20), O.gen_binary(8 << 20)
    rnd = O.gen_random(8 << 20)
    blobs = [z.compress(text, 19), z.compress(binary, 19), z.compress(rnd, 19), rnd.tobytes()]
    contents = [text.tobytes(), binary.tobytes(), rnd.tobytes(), rnd.tobytes()]
    st, dg, out, out_off = _run(codec, blobs, [1, 1, 1, 0], contents)
    assert st.tolist() == [0, 0, 0, 0]
    assert dg[0].tobytes().hex() == "350a3bb730dfa2c4fa41d9a68b80c605fe0bc65c4fa60d1f60ab8fa85830976c"
    assert dg[1].tobytes().hex() == "1adedad9735f565ac6e22dab203db63b960c27098f2c0f0fda9adf9238d4c0c9"
    for i, c in enumerate(contents):
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c


def test_status_rules(codec, oracle):
    """decompress.rs:156-184: codec error -> row skipped; digest mismatch counted; one bad blob never fails the batch."""
    O = oracle
    z = O.libzstd()
    good = O.real_text(100_000).tobytes()
    frame = z.compress(good, 3)
    trunc = frame[:len(frame) // 2]
    notframe = b"\x00\x01\x02\x03" + good[:100]
    contents = [good, good, good, good, good]
    blobs = [frame, trunc, notframe, frame, good]
    buf, offs = _pack(blobs)
    ex = bytearray(b"".join(O.blake3(c) for c in contents))
    ex[3 * 32] ^= 1  # wrong expectation for row 3
    out = np.zeros(5 * 100_016, np.uint8)
    out_off = [i * 100_016 for i in range(5)]
    st, dg = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [1, 1, 1, 1, 0], [len(good)] * 5, bytes(ex),
                                       out, out_off)
    assert st.tolist() == [codec.S_OK, codec.S_DECODE_ERROR, codec.S_UNSUPPORTED, codec.S_DIGEST_MISMATCH, codec.S_OK]
    assert out[:100_000].tobytes() == good and out[4 * 100_016:4 * 100_016 + 100_000].tobytes() == good
    # capacity below the frame's content: DST_TOO_SMALL / SIZE_MISMATCH, never an overrun
    canary = np.full(200_000, 0xAB, np.uint8)
    st, _ = codec.decode_verify_batch(buf, offs[:1], [len(frame)], [1], [50_000], None, canary, [0])
    assert st[0] in (codec.S_DST_TOO_SMALL, codec.S_SIZE_MISMATCH)
    assert (canary[50_000:] == 0xAB).all()
    st, _ = codec.decode_verify_batch(buf, offs[:1], [len(frame)], [1], [100_001], None, canary, [0])
    assert st[0] == codec.S_SIZE_MISMATCH


def test_bitflip_fuzz_matches_oracle_verdict(codec, oracle):
    """Injected corruption: for every flipped frame the GPU agrees with the oracle on accept/reject, and on the bytes
    when both accept."""
    O = oracle
    z = O.libzstd()
    data = O.real_text(60_000).tobytes()
    base = z.compress(data, 3)
    rnd = random.Random(5)
    blobs = []
    for _ in range(400):
        c = bytearray(base)
        for _ in range(rnd.choice([1, 1, 2])):
            c[rnd.randrange(len(c))] ^= 1 << rnd.randrange(8)
        blobs.append(bytes(c))
    buf, offs = _pack(blobs)
    cap = 60_000
    out = np.zeros(len(blobs) * 60_016, np.uint8)
    out_off = [i * 60_016 for i in range(len(blobs))]
    st, _ = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [1] * len(blobs), [cap] * len(blobs), None, out,
                                      out_off)
    for i, b in enumerate(blobs):
        rc, o = O.zstd_decompress(b, cap)
        ok_ref = rc == 0 and len(o) == cap
        assert (st[i] == 0) == ok_ref, (i, st[i], rc, len(o))
        if ok_ref:
            assert out[out_off[i]:out_off[i] + cap].tobytes() == o


def test_codec_rs_unit_tests(codec, oracle):
    """The reference's own codec tests (codec.rs:84-123), against frames from libzstd (decode side) — the GPU
    compressor's round trips live in test_gpu_compress.py."""
    z = oracle.libzstd()
    inp = (b"Hello world! This is a test of compression roundtrip. Repeated data helps compression. "
           b"Repeated data helps compression. Repeated data helps compression.")
    assert codec.decompress_frame(z.compress(inp, 3)) == inp
    for i in range(10):
        d = bytes((x + i) % 251 for x in range(4096))
        out = bytearray()
        assert codec.decompress_into(z.compress(d, 3), out) == 4096 and bytes(out) == d
    assert codec.blake3_hash(b"").hex() == "af1349b9f5f9a1a6a0404dea36dcc9499bcb25c9adc112b7cc9a93cae41f3262"


def test_block_parallel_path_levels_and_fuzz(codec, oracle):
    """Large entropy-coded blobs (compressed above 1/64 of their content) take the device-wide pipeline, whatever the
    name says: k_decode_par only gets rows whose frame is at least as large as their content.  All levels (treeless
    literals / repeat-mode tables appear at >= 7), multi-frame blobs, and injected corruption: the verdict must match the
    oracle's and nothing may hang."""
    O = oracle
    z = O.libzstd()
    rt = O.real_text(3_000_000)
    contents, blobs = [], []
    for lvl in (-5, 1, 3, 7, 12, 19):
        contents.append(rt.tobytes()); blobs.append(z.compress(rt, lvl))
    contents.append(O.gen_rle_literals().tobytes() * 4); blobs.append(z.compress(contents[-1], 19))
    two = rt[:1_200_000].tobytes()
    contents.append(two + two[:700_000]); blobs.append(z.compress(two, 3) + z.compress(two[:700_000], 19))
    assert _classes(codec, blobs, contents) == [len(blobs), 0, 0, 0, 0]
    st, dg, out, out_off = _run(codec, blobs, [1] * len(blobs), contents)
    assert st.tolist() == [0] * len(blobs)
    for i, c in enumerate(contents):
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c, i
        assert dg[i].tobytes() == O.blake3(c)
    # corruption
    base = z.compress(rt[:1_500_000], 3)
    rnd = random.Random(11)
    bad = []
    for _ in range(48):
        c = bytearray(base)
        for _ in range(rnd.choice([1, 2, 3])):
            c[rnd.randrange(len(c))] ^= 1 << rnd.randrange(8)
        bad.append(bytes(c))
    cap = 1_500_000
    buf, offs = _pack(bad)
    outb = np.zeros(len(bad) * (cap + 16), np.uint8)
    ooff = [i * (cap + 16) for i in range(len(bad))]
    st, _ = codec.decode_verify_batch(buf, offs, [len(b) for b in bad], [1] * len(bad), [cap] * len(bad), None, outb, ooff)
    for i, b in enumerate(bad):
        rc, o = O.zstd_decompress(b, cap)
        ok_ref = rc == 0 and len(o) == cap
        assert (st[i] == 0) == ok_ref, (i, st[i], rc, len(o))
        if ok_ref:
            assert outb[ooff[i]:ooff[i] + cap].tobytes() == o


def test_raw_lz4_blocks(codec, oracle):
    """compressed[i] == 2: one raw LZ4 block per blob (LZ4_compress_default / _HC output, no frame), sizes from the index."""
    O = oracle
    l = O.liblz4()
    frames = [f for f in json.load(open(os.path.join(GOLD, "frames.json")))["frames"] if f["codec"] == "lz4block"]
    blobs = [base64.b64decode(f["blob_b64"]) for f in frames]
    lens = [f["out_len"] for f in frames]
    want = [bytes.fromhex(f["out_blake3"]) for f in frames]
    for d in (O.real_text(700_000), O.gen_text(2 << 20), O.gen_binary(100_000), O.gen_random(50_000), O.gen_text(13)):
        blobs.append(l.compress_block(d)); lens.append(len(d)); want.append(O.blake3(d))
        blobs.append(l.compress_block(d, 9)); lens.append(len(d)); want.append(O.blake3(d))
    buf, offs = _pack(blobs)
    ooff = np.concatenate([[0], np.cumsum(lens)])[:-1]
    out = np.zeros(sum(lens) + 1, np.uint8)
    st, dg = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [2] * len(blobs), lens, b"".join(want), out, ooff)
    assert not st.any(), st
    # a truncated block and a too-small destination are per-blob errors
    st, _ = codec.decode_verify_batch(buf, offs[:1], [len(blobs[0]) - 3], [2], lens[:1], None, out, [0])
    assert st[0] != 0
    st, _ = codec.decode_verify_batch(buf, offs[:1], [len(blobs[0])], [2], [lens[0] - 1], None, out, [0])
    assert st[0] in (codec.S_DST_TOO_SMALL, codec.S_DECODE_ERROR, codec.S_SIZE_MISMATCH)


def test_block_parallel_mixed_batch_with_small_sources(codec, oracle):
    """A big-blob batch that also holds blobs whose compressed form is small, with short-sequence blocks and long-match
    blocks interleaved.  Every row is entropy-coded above 1/64 and at least 4 KiB, so the device-wide pipeline takes them
    all (not the block-parallel kernel the name recalls)."""
    O = oracle
    z = O.libzstd()
    rt = O.real_text(2_500_000)
    small_real = O.real_text(20_000)                     # ~6 KB compressed: staged source + lane executor
    mix = np.concatenate([O.gen_text(400_000), rt[:300_000], O.gen_binary(300_000), rt[300_000:500_000]])
    contents = [rt.tobytes(), small_real.tobytes(), mix.tobytes(), rt[:1_000_000].tobytes(), small_real[:5000].tobytes(),
                rt[100:2_200_100].tobytes()]
    blobs = [z.compress(c, 3) for c in contents]
    assert _classes(codec, blobs, contents) == [len(blobs), 0, 0, 0, 0]
    st, dg, out, out_off = _run(codec, blobs, [1] * len(blobs), contents)
    assert st.tolist() == [0] * len(blobs)
    for i, c in enumerate(contents):
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c, i


@pytest.mark.parametrize("mode", ["ws"])
def test_fused_decode_hash_kernels(codec, oracle, mode, monkeypatch):
    """Large, highly compressible blobs through the fused decode+hash kernel (`ws` = warp-specialised, k_decode_ws): same
    bytes, same digests, same status rules as the oracle; a small grid makes every decode team take several blobs."""
    O = oracle
    z, l = O.libzstd(), O.liblz4()
    monkeypatch.setenv("ZN_WS_GRID", "3")
    datas = [O.gen_text(8 << 20), O.gen_binary(8 << 20), O.gen_text((1 << 20) + 17), O.gen_binary(700_000),
             np.zeros(3 << 20, np.uint8), O.gen_text(5_000_001), O.gen_binary((4 << 20) - 1), O.gen_text(2 << 20),
             O.gen_binary(6 << 20), O.gen_text(1_234_567), O.gen_text(4 << 20)]
    blobs = [z.compress(d, 19 if i % 2 == 0 else 3) for i, d in enumerate(datas)]
    blobs[7] = l.compress_frame(datas[7])
    contents = [d.tobytes() for d in datas]
    st, dg, out, out_off = _run(codec, blobs, [1] * len(blobs), contents)
    assert st.tolist() == [0] * len(blobs)
    for i, c in enumerate(contents):
        assert dg[i].tobytes() == O.blake3(c), i
        assert out[out_off[i]:out_off[i] + len(c)].tobytes() == c, i
    # 16-byte aligned rows (the bench layout), digest only compared on the device
    buf, offs = _pack(blobs)
    lens = [len(c) for c in contents]
    ooff = np.concatenate([[0], np.cumsum([(n + 15) // 16 * 16 for n in lens])])[:-1]
    out2 = np.zeros(int(ooff[-1]) + lens[-1] + 16, np.uint8)
    st, dg2 = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [1] * len(blobs), lens,
                                        b"".join(O.blake3(c) for c in contents), out2, ooff)
    assert st.tolist() == [0] * len(blobs) and (dg2 == dg).all()
    # one corrupted blob, one wrong expectation: only those rows fail
    bad = bytearray(blobs[2]); bad[len(bad) // 2] ^= 0x10
    blobs2 = list(blobs); blobs2[2] = bytes(bad)
    buf, offs = _pack(blobs2)
    ex = [O.blake3(c) for c in contents]; ex[5] = bytes(32)
    st, _ = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs2], [1] * len(blobs2), lens, b"".join(ex), out2, ooff)
    assert st[5] == codec.S_DIGEST_MISMATCH and st[2] != 0
    assert [int(x) for i, x in enumerate(st) if i not in (2, 5)] == [0] * (len(blobs) - 2)


def test_fused_kernel_survives_corrupt_blobs(codec, oracle):
    """Bit flips in large pattern blobs through the default (warp-specialised fused) path: the call returns, damaged rows
    report an error or a digest mismatch, every other row stays bit-exact (a producer that fails must still queue all of
    its tiles, or the hash warps would wait for ever — the kernel's watchdog would turn that into an error return)."""
    O = oracle
    z = O.libzstd()
    datas = [O.gen_text(4 << 20), O.gen_binary(3 << 20), O.gen_text((2 << 20) + 5), O.gen_binary(5 << 20), O.gen_text(1 << 20),
             O.gen_binary(2 << 20)]
    good = [z.compress(d, 19) for d in datas]
    want = [O.blake3(d.tobytes()) for d in datas]
    lens = [d.size for d in datas]
    ooff = np.concatenate([[0], np.cumsum([(n + 15) // 16 * 16 for n in lens])])[:-1]
    out = np.zeros(int(ooff[-1]) + lens[-1] + 16, np.uint8)
    rng = random.Random(11)
    for trial in range(16):
        victim = rng.randrange(len(good))
        bad = bytearray(good[victim])
        pos = rng.randrange(4, len(bad))
        bad[pos] ^= 1 << rng.randrange(8)
        blobs = list(good)
        blobs[victim] = bytes(bad)
        buf, offs = _pack(blobs)
        st, dg = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [1] * len(blobs), lens, b"".join(want), out, ooff)
        for i in range(len(blobs)):
            if i != victim:
                assert st[i] == 0 and dg[i].tobytes() == want[i], (trial, i)
        ref_rc, ref_out = O.zstd_decompress(bytes(bad), lens[victim])
        if ref_rc == 0 and ref_out == datas[victim].tobytes():
            assert st[victim] == 0  # the flip hit a bit that does not matter (e.g. the unverified frame checksum)
        else:
            assert st[victim] != 0, (trial, victim, pos)


def test_caller_memory_between_output_ranges_is_left_alone(codec, oracle):
    """ADVICE r1 (low): the D2H copy used to return one span whenever the ranges were 'compact', overwriting caller
    bytes that lie between two declared ranges with stale device memory.  Gaps of 16 bytes or more are never written;
    alignment padding (< 16 bytes) is the only documented exception (include/znippy_cuda.h)."""
    O = oracle
    z = O.libzstd()
    contents = [O.real_text(50_000 + 777 * i).tobytes() for i in range(6)]
    blobs = [z.compress(c, 3) for c in contents]
    buf, offs = _pack(blobs)
    gaps = [0, 16, 100, 4000, 17, 64]
    out_off, cur = [], 0
    for c, g in zip(contents, gaps):
        cur += g
        out_off.append(cur)
        cur += len(c)
    out = np.full(cur + 64, 0x5A, np.uint8)
    st, _ = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [1] * 6, [len(c) for c in contents],
                                       b"".join(O.blake3(c) for c in contents), out, out_off)
    assert not st.any()
    keep = np.ones(out.size, bool)
    for o, c in zip(out_off, contents):
        assert out[o:o + len(c)].tobytes() == c
        keep[o:o + len(c)] = False
    assert (out[keep] == 0x5A).all()


def test_zstd_content_checksums_are_verified(codec, oracle):
    """RFC 8878 §3.1.1 Content_Checksum (low 32 bits of XXH64 of the frame's content): libzstd — and so the reference's
    decode — rejects a frame whose stored checksum is wrong; so does the GPU path (k_xxh64_verify).  Same accept/reject
    verdict as the oracle and libzstd for every flipped bit of checksummed frames, tails of 0..31 bytes, a multi-frame
    blob, and a frame the pipeline / pattern / small-blob classes decode."""
    O = oracle
    z = O.libzstd()
    rnd = random.Random(9)
    contents = [O.real_text(n).tobytes() for n in (0, 1, 5, 31, 32, 33, 63, 64, 1000, 65_537, 300_000, 3 << 20)]
    contents += [O.gen_text(2 << 20).tobytes(), O.gen_binary(10_240).tobytes()]
    blobs = [z.compress(c, 3, checksum=True) for c in contents]
    contents.append(contents[8] + contents[9])            # two checksummed frames back to back
    blobs.append(blobs[8] + blobs[9])
    for c, b in zip(contents[:10], blobs[:10]):            # the oracle's XXH64 is what the frames carry
        assert int.from_bytes(b[-4:], "little") == O.xxh64(c) & 0xFFFFFFFF
    n = len(blobs)
    buf, offs = _pack(blobs)
    lens = [len(c) for c in contents]
    ooff = np.concatenate([[0], np.cumsum([(x + 15) & ~15 for x in lens])])[:-1]
    out = np.zeros(int(ooff[-1]) + lens[-1] + 16, np.uint8)
    st, dg = codec.decode_verify_batch(buf, offs, [len(b) for b in blobs], [1] * n, lens, None, out, ooff)
    assert not st.any()
    for i, c in enumerate(contents):
        assert out[ooff[i]:ooff[i] + len(c)].tobytes() == c and dg[i].tobytes() == O.blake3(c)
    # a wrong stored checksum (any of its 32 bits) is a decode error; the neighbours are untouched
    bad = list(blobs)
    for i in range(n):
        b = bytearray(blobs[i])
        b[len(b) - 1 - rnd.randrange(4)] ^= 1 << rnd.randrange(8)
        bad[i] = bytes(b)
    bad[3] = blobs[3]
    buf, offs = _pack(bad)
    st, _ = codec.decode_verify_batch(buf, offs, [len(b) for b in bad], [1] * n, lens, None, out, ooff)
    for i in range(n):
        rc, _o = O.zstd_decompress(bad[i], lens[i])
        assert (st[i] == 0) == (rc == 0), (i, st[i], rc)
    assert st[3] == 0 and st[0] == codec.S_DECODE_ERROR and st[n - 1] == codec.S_DECODE_ERROR
    # bit-flip fuzz over whole checksummed frames: verdict equality with the oracle, with no exception left
    base = blobs[9]
    fz = []
    for _ in range(300):
        c = bytearray(base)
        c[rnd.randrange(len(c))] ^= 1 << rnd.randrange(8)
        fz.append(bytes(c))
    buf, offs = _pack(fz)
    cap = lens[9]
    o2 = np.zeros(len(fz) * (cap + 16), np.uint8)
    st, _ = codec.decode_verify_batch(buf, offs, [len(b) for b in fz], [1] * len(fz), [cap] * len(fz), None, o2,
                                      [i * (cap + 16) for i in range(len(fz))])
    for i, b in enumerate(fz):
        rc, o = O.zstd_decompress(b, cap)
        assert (st[i] == 0) == (rc == 0 and len(o) == cap), (i, st[i], rc)


def test_fused_kernel_watchdog_ends_a_stalled_queue(codec, oracle, monkeypatch):
    """VERDICT r1: the consumer-side watchdog of the fused decode+hash kernel (fused_ws.cuh) was never made to fire.  With
    ZN_WS_TEST_STALL the host announces one tile more than the producers will ever publish; a hash warp then waits for an
    entry that never comes, the spin limit (~3 s) trips, every other waiter sees the flag, the kernel ENDS, and the call
    reports an error instead of results — the GPU is not left spinning, and the next call works."""
    import time
    from znippy_b200 import Ctx
    O = oracle
    z = O.libzstd()
    data = O.gen_text(2 << 20).tobytes()
    blob = z.compress(data, 19)
    blobs = [blob] * 4
    buf, offs = _pack(blobs)
    ctx = Ctx(0)
    args = (buf, offs, [len(b) for b in blobs], [1] * 4, [len(data)] * 4, O.blake3(data) * 4, None, None, ctx)
    st, _ = codec.decode_verify_batch(*args)
    assert not st.any()
    monkeypatch.setenv("ZN_WS_TEST_STALL", "1")
    t0 = time.time()
    with pytest.raises(Exception, match="stalled"):
        codec.decode_verify_batch(*args)
    assert 1.0 < time.time() - t0 < 30.0
    monkeypatch.delenv("ZN_WS_TEST_STALL")
    st, dg = codec.decode_verify_batch(*args)
    assert not st.any() and dg[0].tobytes() == O.blake3(data)


def test_store_as_is_row_with_disagreeing_sizes_is_refused(codec, oracle):
    """ADVICE r1 (medium): a store-as-is row whose blob_size differs from its uncompressed_size used to be gathered with
    blob_size bytes into an output slot sized for uncompressed_size — an out-of-bounds device write into the neighbours.
    Such a row now gets SIZE_MISMATCH, nothing of it is written, and its neighbours come out intact."""
    O = oracle
    a, b, c = O.real_text(50_000).tobytes(), O.gen_random(70_000).tobytes(), O.real_text(30_000).tobytes()
    blobs = [a, b, c]
    buf, offs = _pack(blobs)
    out_len = [len(a), 1_000, len(c)]            # the middle row claims 1 000 bytes for a 70 000-byte blob
    out_off = [0, 50_016, 51_024]
    out = np.full(51_024 + 30_000 + 64, 0xCD, np.uint8)
    st, dg = codec.decode_verify_batch(buf, offs, [len(x) for x in blobs], [0, 0, 0], out_len, None, out, out_off)
    assert st.tolist() == [codec.S_OK, codec.S_SIZE_MISMATCH, codec.S_OK]
    assert out[:50_000].tobytes() == a and out[51_024:51_024 + 30_000].tobytes() == c
    assert (out[51_024 + 30_000:] == 0xCD).all()  # (the refused row's own 1 000-byte range is unspecified, nothing beyond the rows is touched)
    assert dg[0].tobytes() == O.blake3(a) and dg[2].tobytes() == O.blake3(c)


def test_pipeline_keeps_well_formed_frames_at_every_alignment(codec, oracle):
    """The device-wide pipeline hands a blob back to the one-team decoder only when something is off; a silent hand-back
    of well-formed frames would keep every parity test green and cost the whole speed-up.  Entropy-coded frames of several
    levels at all 16 byte alignments of the blob (the sequence stage stages its bit stream in 16-byte units and hands bit
    positions from one kernel to the next): bytes and digests bit-exact, and zn_plan_pipeline_fallbacks reports 0."""
    import torch
    from znippy_b200 import Plan
    O, z = oracle, oracle.libzstd()
    rt = O.real_text(2_500_000)
    contents, blobs = [], []
    for k in range(16):
        c = rt[k * 100_000: k * 100_000 + 300_000 + 4099 * k].tobytes()
        contents.append(c)
        blobs.append(z.compress(c, [1, 3, 7, 19][k % 4]))
    offs, cur = [], 0
    for k, b in enumerate(blobs):  # blob k starts at an address that is k modulo 16
        cur = (cur + 15) // 16 * 16 + k
        offs.append(cur)
        cur += len(b)
    buf = np.zeros(cur + 16, np.uint8)
    for o, b in zip(offs, blobs):
        buf[o:o + len(b)] = np.frombuffer(b, np.uint8)
    out_len = np.array([len(c) for c in contents], np.uint64)
    out_off = np.concatenate([[0], np.cumsum((out_len + np.uint64(15)) & ~np.uint64(15))])[:-1].astype(np.uint64)
    digs = np.frombuffer(b"".join(O.blake3(c) for c in contents), np.uint8)
    ctx = codec.default_ctx()
    d_in = torch.from_numpy(buf).cuda()
    d_out = torch.zeros(int(out_off[-1] + out_len[-1]) + 256, dtype=torch.uint8, device="cuda")
    plan = Plan.decode_verify(ctx, offs, [len(b) for b in blobs], [1] * 16, out_off, out_len, digs)
    assert plan.class_counts()[0] == 16
    plan.run(d_in.data_ptr(), d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    st, dg = plan.results()
    assert st.tolist() == [0] * 16
    assert plan.pipeline_fallbacks() == 0
    out = d_out.cpu().numpy()
    for i, c in enumerate(contents):
        assert out[int(out_off[i]): int(out_off[i]) + len(c)].tobytes() == c, i
        assert dg[i].tobytes() == O.blake3(c)


def test_entropy_coded_slices_at_baseline_size(codec, oracle):
    """The realistic shape of the metric: 8 MiB slices (stream_packer.rs:31) of real text, entropy-coded (Huffman literals,
    FSE tables, repeat offsets) at a fast level and at the reference's 19, decoded by the device-wide pipeline with the
    two-phase sequence stage (mean decoded size >= 256 KiB).  Size-independent property at full slice size: every digest
    equals the oracle's blake3 of the content, every byte equals the content, no slice is handed back."""
    import torch
    from znippy_b200 import Plan
    O, z = oracle, oracle.libzstd()
    rt = O.real_text((8 << 20) + 24 * 4099)
    contents = [rt[k * 4099: k * 4099 + (8 << 20)] for k in range(24)]  # 24 distinct slices (shifted windows of the corpus)
    blobs = [z.compress(c, 19 if k == 7 else (1 if k % 3 == 0 else 3)) for k, c in enumerate(contents)]
    offs, cur = [], 0
    for k, b in enumerate(blobs):
        cur = (cur + 15) // 16 * 16 + (5 * k) % 16
        offs.append(cur)
        cur += len(b)
    buf = np.zeros(cur + 16, np.uint8)
    for o, b in zip(offs, blobs):
        buf[o:o + len(b)] = np.frombuffer(b, np.uint8)
    out_len = np.array([c.size for c in contents], np.uint64)
    out_off = (np.arange(24, dtype=np.uint64) * np.uint64(8 << 20))
    digs = np.frombuffer(b"".join(O.blake3(c.tobytes()) for c in contents), np.uint8)
    ctx = codec.default_ctx()
    d_in = torch.from_numpy(buf).cuda()
    d_out = torch.zeros(24 * (8 << 20) + 256, dtype=torch.uint8, device="cuda")
    plan = Plan.decode_verify(ctx, offs, [len(b) for b in blobs], [1] * 24, out_off, out_len, digs)
    assert plan.class_counts()[0] == 24
    for _ in range(2):  # a second run reuses the pipeline's pools
        plan.run(d_in.data_ptr(), d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    st, dg = plan.results()
    assert st.tolist() == [0] * 24
    assert plan.pipeline_fallbacks() == 0
    assert (dg.reshape(-1) == digs).all()
    out = d_out.cpu().numpy()
    for k, c in enumerate(contents):
        assert (out[k * (8 << 20): (k + 1) * (8 << 20)] == c).all(), k


def test_pipeline_one_pass_sequence_stage(codec, oracle):
    """Batches of very many small entropy-coded rows take the one-pass sequence stage (k_zseq_g): more blocks than two
    rounds of phase-1 lanes (2 x SMs x kSeq1Lanes, kSeq1Lanes = 56) and a mean decoded size below 256 KiB.  Real-text rows
    of 4-12 KiB at levels 1 / 3 / 19: every status, byte and digest equals the oracle's, no row is handed back, and the run
    launches one kernel less than a 64-row slice of the same rows, which takes the two-phase form (k_zseq1 + k_zseq2)."""
    import torch
    from znippy_b200 import Plan
    O, z = oracle, oracle.libzstd()
    ctx = codec.default_ctx()
    n = 2 * torch.cuda.get_device_properties(0).multi_processor_count * 56 + 512
    rng = np.random.default_rng(17)
    rt = O.real_text(8 << 20)
    lens = rng.integers(4096, 12289, n)
    starts = rng.integers(0, rt.size - 12288, n)
    contents = [rt[s:s + k].tobytes() for s, k in zip(starts, lens)]
    blobs = [z.compress(c, (1, 3, 19)[i % 3]) for i, c in enumerate(contents)]
    offs, cur = [], 0
    for k, b in enumerate(blobs):
        cur = (cur + 15) // 16 * 16 + k % 16
        offs.append(cur)
        cur += len(b)
    buf = np.zeros(cur + 16, np.uint8)
    for o, b in zip(offs, blobs):
        buf[o:o + len(b)] = np.frombuffer(b, np.uint8)
    out_len = np.array([len(c) for c in contents], np.uint64)
    out_off = np.concatenate([[0], np.cumsum((out_len + np.uint64(15)) & ~np.uint64(15))])[:-1].astype(np.uint64)
    digs = np.frombuffer(b"".join(O.blake3(c) for c in contents), np.uint8)
    d_in = torch.from_numpy(buf).cuda()
    d_out = torch.zeros(int(out_off[-1] + out_len[-1]) + 256, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def run(m):
        plan = Plan.decode_verify(ctx, offs[:m], [len(b) for b in blobs[:m]], [1] * m, out_off[:m], out_len[:m], digs[:m * 32])
        assert plan.class_counts()[0] == m
        plan.run(d_in.data_ptr(), d_out.data_ptr(), stream)
        torch.cuda.synchronize()
        st, dg = plan.results()
        assert st.tolist() == [0] * m
        assert plan.pipeline_fallbacks() == 0
        assert (dg.reshape(-1) == digs[:m * 32]).all()
        return plan.launches()

    two_phase = run(64)
    one_pass = run(n)
    assert one_pass == two_phase - 1
    out = d_out.cpu().numpy()
    for i, c in enumerate(contents):
        assert out[int(out_off[i]): int(out_off[i]) + len(c)].tobytes() == c, i
