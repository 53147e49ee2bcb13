"""Pins the CPU oracle (oracle/) against the golden vectors and the independent libraries in the image.

Reference items checked (SURVEY.md §8a): a1 codec::decompress_into (codec.rs:67-78) payload formats,
a2/a6 blake3::hash (decompress.rs:172, stream_packer.rs:219), a3 worker-loop counters (decompress.rs:135-190).
"""
import base64
import json
import os

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

GOLD = os.path.join(os.path.dirname(__file__), "golden")

# KAT table from SURVEY.md §8(c) (computed there with the official blake3 bindings)
SURVEY_KATS = [
    ("text", 0, "af1349b9f5f9a1a6a0404dea36dcc9499bcb25c9adc112b7cc9a93cae41f3262"),
    ("text", 1024, "3224bc8e92b73e84c9fcb9e4ada53239e32ad26ba68b5beb6e36e0b64ff46981"),
    ("text", 1025, "5b3e0e8dfde4b8ffd77f11c0e821ef158017cd112448744237470436608b9b95"),
    ("text", 10240, "c22424898e1f1cb805cc292109097f2438ace28d14f77dddea39037f082aed01"),
    ("text", 8 << 20, "350a3bb730dfa2c4fa41d9a68b80c605fe0bc65c4fa60d1f60ab8fa85830976c"),
    ("binary", 4096, "015094013f57a5277b59d8475c0501042c0b642e531b0a1c8f58d2163229e969"),
    ("binary", 8 << 20, "1adedad9735f565ac6e22dab203db63b960c27098f2c0f0fda9adf9238d4c0c9"),
    ("random", 1 << 20, "245e108ab7b7624dd4a00f9046e1caad2d4e57ae6691214c6e08c1b1e98d8b89"),
]


def _gen(O, kind, n, seed=0):
    return {"text": lambda: O.gen_text(n), "binary": lambda: O.gen_binary(n), "random": lambda: O.gen_random(n),
            "incompressible": lambda: O.gen_incompressible(n, seed), "realtext": lambda: O.real_text(n)}[kind]()


def test_generators_match_reference_definitions(oracle):
    O = oracle
    phrase = b"The quick brown fox jumps over the lazy dog. "
    assert O.gen_text(200).tobytes() == (phrase * 5)[:200]
    assert O.gen_text(100, phase=7).tobytes() == (phrase * 5)[7:107]
    assert O.gen_binary(600).tolist() == [i % 251 for i in range(600)]
    assert O.gen_binary(10, start=249).tolist() == [(249 + i) % 251 for i in range(10)]
    val, exp = 12345, []
    for _ in range(64):
        val = (val * 6364136223846793005 + 1) % (1 << 64)
        exp.append((val >> 33) & 0xFF)
    assert O.gen_random(64).tolist() == exp
    v, exp = (5 * 0x9E3779B97F4A7C15 + 1) % (1 << 64), []
    for _ in range(64):
        v = (v * 6364136223846793005 + 1442695040888963407) % (1 << 64)
        exp.append((v >> 33) & 0xFF)
    assert O.gen_incompressible(64, 5).tolist() == exp


@pytest.mark.parametrize("kind,n,hexd", SURVEY_KATS)
def test_blake3_survey_kats(oracle, kind, n, hexd):
    data = _gen(oracle, kind, n)
    assert oracle.blake3(data).hex() == hexd
    assert oracle.blake3(data, fast=True).hex() == hexd


def test_blake3_golden_file(oracle):
    for k in json.load(open(os.path.join(GOLD, "blake3_kat.json"))):
        data = _gen(oracle, k["gen"], k["n"], k.get("seed", 0))
        assert oracle.blake3(data).hex() == k["blake3"], k
        assert oracle.blake3(data, fast=True).hex() == k["blake3"], k


@settings(max_examples=60, deadline=None)
@given(st.binary(min_size=0, max_size=70000))
def test_blake3_vs_official(data):
    import oracle as O
    assert O.blake3(data) == O.blake3_official(data)


def test_xxhash_vs_python_xxhash(oracle):
    import xxhash
    rng = np.random.default_rng(1)
    for n in [0, 1, 3, 4, 7, 8, 15, 16, 31, 32, 33, 63, 64, 100, 1000, 4097]:
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert oracle.xxh64(b) == xxhash.xxh64(b).intdigest()
        assert oracle.xxh32(b) == xxhash.xxh32(b).intdigest()
        assert oracle.xxh64(b, 77) == xxhash.xxh64(b, seed=77).intdigest()


def _frames():
    return json.load(open(os.path.join(GOLD, "frames.json")))


def test_golden_frames_decode(oracle):
    O = oracle
    for f in _frames()["frames"]:
        blob = base64.b64decode(f["blob_b64"])
        if f["codec"] == "zstd":
            rc, out = O.zstd_decompress(blob, f["out_len"])
            assert O.zstd_frame_content_size(blob) == (0, f["out_len"])
        elif f["codec"] == "lz4f":
            rc, out = O.lz4_frame_decompress(blob, f["out_len"])
            # liblz4 treats contentSize == 0 as "unknown", so the empty frame carries no size field
            assert O.lz4_frame_content_size(blob) == ((0, f["out_len"]) if f["out_len"] else (1, 0))
        else:
            rc, out = O.lz4_block_decompress(blob, f["out_len"])
        assert rc == 0, f["name"]
        assert len(out) == f["out_len"], f["name"]
        assert O.blake3_official(out).hex() == f["out_blake3"], f["name"]


def test_golden_frame_facts_match_survey():
    facts = _frames()["facts"]
    assert facts["zstd_text_10k_l19_len"] == 64 and facts["zstd_text_8m_l19_len"] == 762
    assert facts["zstd_binary_8m_l19_len"] == 968 and facts["zstd_random_1m_l19_len"] == 1048609
    assert facts["zstd_empty_hex"] == "28b52ffd2000010000"
    assert facts["lz4block_text_10k_len"] == 95 and facts["lz4block_text_8m_len"] == 32952


@pytest.mark.parametrize("level", [-5, 1, 3, 7, 12, 19])
def test_zstd_realtext_levels_cover_entropy_paths(oracle, level):
    O = oracle
    data = O.real_text(1_500_000)
    blob = O.libzstd().compress(data, level)
    rc, out, stats = O.zstd_decompress(blob, len(data), want_stats=True)
    assert rc == 0 and out == data.tobytes()
    assert stats["sequences"] > 1000 and stats["mode_fse"] > 0
    if level >= 1:
        assert stats["lit_huf_4stream"] > 0 and stats["huf_weights_fse"] > 0


def test_zstd_path_coverage_union(oracle):
    """Across the test corpora every literal mode, table mode and block type of RFC 8878 is exercised."""
    O, z = oracle, oracle.libzstd()
    rt = O.real_text(600_000)
    corpora = [
        (O.gen_text(300_000), 19), (O.gen_random(300_000), 3), (O.real_text(3 << 20), 19), (rt, 1),
        (np.concatenate([np.full(200_000, 65, np.uint8), rt[:5000], np.full(150_000, 66, np.uint8)]), 3),
        (rt[:300], 3), (rt[:2000], 19),
        (np.frombuffer(bytes(np.random.default_rng(3).choice([97, 98, 99, 100], 50000).astype(np.uint8)), np.uint8), 3),
        (np.tile(rt[:50], 40), 1), (O.gen_rle_literals(), 19),
        (O.gen_small_alphabet(300), 1), (O.gen_small_alphabet(3000), 1),
        (O.gen_periodic_noise(2000, 200, 12), 3), (O.gen_periodic_noise(20000, 64, 8), 19),
    ]
    tot = {}
    for data, lvl in corpora:
        blob = z.compress(data, lvl)
        rc, out, s = O.zstd_decompress(blob, len(data), want_stats=True)
        assert rc == 0 and out == data.tobytes()
        for k, v in s.items():
            tot[k] = tot.get(k, 0) + v
    for need in ("blocks_raw", "blocks_rle", "blocks_compressed", "lit_raw", "lit_rle", "lit_huf_1stream",
                 "lit_huf_4stream", "lit_treeless", "huf_weights_direct", "huf_weights_fse", "mode_predefined",
                 "mode_rle", "mode_fse", "mode_repeat", "repcode_uses", "overlap_matches"):
        assert tot.get(need, 0) > 0, (need, tot)


def test_zstd_checksum_and_multiframe_and_skippable(oracle):
    O, z = oracle, oracle.libzstd()
    a, b = O.real_text(70_000), O.gen_text(5000)
    blob = z.compress(a, 3, checksum=True)
    rc, out, s = O.zstd_decompress(blob, len(a), want_stats=True)
    assert rc == 0 and out == a.tobytes() and s["checksums_verified"] == 1
    bad = bytearray(blob)
    bad[-1] ^= 1
    assert O.zstd_decompress(bytes(bad), len(a))[0] == O.ERR_CHECKSUM
    skip = (0x184D2A53).to_bytes(4, "little") + (5).to_bytes(4, "little") + b"hello"
    multi = blob + skip + z.compress(b, 19)
    rc, out, s = O.zstd_decompress(multi, len(a) + len(b), want_stats=True)
    assert rc == 0 and out == a.tobytes() + b.tobytes() and s["frames"] == 2 and s["skippable_frames"] == 1
    assert z.decompress(multi, len(a) + len(b)) == out


def test_zstd_window_frames_without_single_segment(oracle):
    O, z = oracle, oracle.libzstd()
    data = O.real_text(400_000)
    blob = z.compress(data, 3, params={101: 17, 200: 0})  # windowLog=17, no content size -> Window_Descriptor present
    assert O.zstd_frame_content_size(blob)[0] == 1
    rc, out = O.zstd_decompress(blob, len(data))
    assert rc == 0 and out == data.tobytes()


def test_zstd_error_cases(oracle):
    O, z = oracle, oracle.libzstd()
    data = O.real_text(50_000)
    blob = z.compress(data, 3)
    assert O.zstd_decompress(blob, len(data) - 1)[0] in (O.ERR_DST_TOO_SMALL,)
    assert O.zstd_decompress(blob[:-7], len(data))[0] != 0
    assert O.zstd_decompress(b"\x00\x01\x02\x03\x04\x05", 10)[0] == O.ERR_BAD_MAGIC
    assert O.zstd_decompress(b"", 10)[0] == O.ERR_SRC_TRUNCATED
    rng = np.random.default_rng(5)
    for _ in range(300):  # bit flips never crash; they give an error or different bytes
        bad = bytearray(blob)
        i = int(rng.integers(4, len(bad)))
        bad[i] ^= 1 << int(rng.integers(0, 8))
        rc, out = O.zstd_decompress(bytes(bad), len(data))
        assert rc != 0 or len(out) == len(data)


@settings(max_examples=80, deadline=None)
@given(st.binary(min_size=0, max_size=5000), st.sampled_from([1, 3, 19]), st.integers(1, 60))
def test_zstd_roundtrip_hypothesis(data, level, rep):
    import oracle as O
    data = data * rep
    blob = O.libzstd().compress(data, level)
    rc, out = O.zstd_decompress(blob, len(data))
    assert rc == 0 and out == data


@settings(max_examples=80, deadline=None)
@given(st.binary(min_size=0, max_size=5000), st.integers(1, 40))
def test_lz4_roundtrip_hypothesis(data, rep):
    import oracle as O
    data = data * rep
    l = O.liblz4()
    if data:
        rc, out = O.lz4_block_decompress(l.compress_block(data), len(data))
        assert rc == 0 and out == data
        rc, out = O.lz4_block_decompress(l.compress_block(data, 9), len(data))
        assert rc == 0 and out == data
    for kw in ({}, {"content_checksum": True, "block_checksum": True}):
        rc, out = O.lz4_frame_decompress(l.compress_frame(data, **kw), len(data))
        assert rc == 0 and out == data


def test_lz4_errors(oracle):
    O, l = oracle, oracle.liblz4()
    data = O.real_text(30000)
    blk = l.compress_block(data)
    assert O.lz4_block_decompress(blk, len(data) - 1)[0] == O.ERR_DST_TOO_SMALL
    assert O.lz4_block_decompress(blk[:-3], len(data))[0] != 0
    fr = bytearray(l.compress_frame(data))
    fr[5] ^= 0x10
    assert O.lz4_frame_decompress(bytes(fr), len(data))[0] != 0


def test_cpu_pipeline_counters_follow_reference_rules(oracle):
    """decompress.rs:140,168-184: total_chunks always; written/verified/corrupt only when decode succeeded."""
    O, z = oracle, oracle.libzstd()
    slices = [O.gen_text(10240), O.gen_binary(5000), O.gen_random(3000), np.zeros(0, np.uint8), O.real_text(20000)]
    comp = [True, True, False, True, True]
    blobs = [z.compress(s, 3) if c else s.tobytes() for s, c in zip(slices, comp)]
    sums = np.stack([np.frombuffer(O.blake3_official(s), np.uint8) for s in slices])
    blobs[1] = blobs[1][:-2] + b"\xff\xff"          # row 1: corrupt frame -> decode error
    sums[4, 0] ^= 1                                  # row 4: digest mismatch
    off = np.cumsum([0] + [len(b) for b in blobs])[:-1]
    arch = np.frombuffer(b"".join(blobs), np.uint8)
    usz = [len(s) for s in slices]
    for use_lib in (True, False):
        r = O.decompress_rows(arch, off, [len(b) for b in blobs], [0] * 5, comp, usz, sums, 3, use_libzstd=use_lib)
        assert r.total_chunks == 5 and r.decode_errors == 1 and r.corrupt_rows == 1
        assert r.total_written_bytes == 10240 + 3000 + 0 + 20000
        assert r.verified_bytes == 10240 + 3000 and r.corrupt_bytes == 20000
    blobs2, dig = O.compress_slices(np.concatenate(slices), np.cumsum([0] + usz)[:-1], usz, 3, 2)
    for s, b, d in zip(slices, blobs2, dig):
        assert z.decompress(b, len(s)) == s.tobytes() and d.tobytes() == O.blake3_official(s)


def test_frames_from_chosen_sequences(oracle):
    """compress_sequences: libzstd writes a frame carrying exactly the given parse (explicit block delimiters, validated
    sequences), which libzstd and the oracle decode to the expanded content, with one sequence per tuple given; repeated
    distances become repeat codes; an invalid tuple is refused."""
    O, z = oracle, oracle.libzstd()
    rt = O.real_text(400_000)
    blocks = [[(5000, 100_000, 1), (2000, 20_000, 3)],
              [(100, 40, 7)] * 600 + [(10, 30_000, 17_000), (55, 0, 0)],
              [(3, 5, 4)] * 5000]
    content, frame = z.compress_sequences(blocks, rt)
    assert len(content) == 127_000 + 600 * 140 + 30_010 + 55 + 5000 * 8
    assert content[:5000] == rt[:5000].tobytes() and content[5000:105_000] == content[4999:5000] * 100_000
    assert z.decompress(frame, len(content)) == content
    rc, out, st = O.zstd_decompress(frame, len(content), want_stats=True)
    assert rc == 0 and out == content
    assert st["sequences"] == sum(1 for b in blocks for t in b if t[1]) and st["blocks_compressed"] == 3
    assert st["repcode_uses"] >= 5000
    with pytest.raises(RuntimeError):
        z.compress_sequences([[(10, 2, 5)]], rt)  # shorter than the minimum match
    with pytest.raises(ValueError):
        z.compress_sequences([[(10, 5, 11)]], rt)  # reaches before the content
