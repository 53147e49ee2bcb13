"""Zstandard frames built from chosen sequences (oracle `compress_sequences`: libzstd writes every frame byte from an exact
(literal length, match length, offset) list), aimed at the branches of the pipeline's execution kernel `k_zexec2` and at
the routing of rows to decode classes.  On the CPU: every frame decodes to its content through the host emulation of the
pipeline (every stage up to exec, at several blob alignments), of the one-team decoder and of the block-parallel
decoder, with libzstd's verdict; the branch witness shows that the cases reach every branch they are meant to in both
exec shapes; the route mirror shows which kernel each row is meant for.  tests/test_gpu_sequence_frames.py runs the same
cases on the device."""
import functools
import os
import sys
from collections import Counter

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(__file__))
from test_host_logic import emu  # noqa: E402,F401  (emu: the host emulation fixture)
from test_hostemu_range_decode import blocks as frame_blocks  # noqa: E402

GB = 16384        # k_zexec2's group buffer
LIT_LANE = 8      # kLitLane: literal runs up to this length are stored by the owning lane, longer ones are warp jobs
MATCH_LANE = 16   # kMatchLane: likewise for matches
# exec shapes (zpipe_tu.cu): sequences per group (K * NT) and entries per list of unknown bytes (LC)
SHAPES = {"large": (4 * 512, 8192), "small": (2 * 512, 4096)}
PIPE, BIGPAT, BIGRAW, SMALL, MID = range(5)  # decode classes, in zn_plan_class_counts order
KIB = 1024


def route(dst_cap, src_len, lz4_block=False):
    """The decode class plan_build (znippy_cuda.cu) gives a compressed row, from its index sizes alone."""
    big, pat = dst_cap >= 512 * KIB, src_len * 64 <= dst_cap
    if big and pat and not lz4_block:
        return BIGPAT
    if not lz4_block and not pat and src_len < dst_cap and dst_cap >= 4096:
        return PIPE
    if big:
        return BIGRAW
    return SMALL if dst_cap <= 64 * KIB else MID


def witness(frames, kseqs, lc):
    """Replays the group and setup logic of k_zexec2 (zpipe_kernels.cuh:547-822) over the sequences given to
    compress_sequences.  `frames`: (frame bytes, blocks of (ll, ml, off), output position of the frame) per frame of one
    blob.  Returns (hits, groups):
    * hits counts, per sequence, the branch it takes: `alone` (count == 0, lines 572-594: longer than a group in output or
      literals), `lit_lane` / `lit_job` (lines 627-635), `{lane|job}_{before|inside|straddle|self}` (the three setup
      branches of lines 644-666 for matches up to MATCH_LANE, and the same placement for warp jobs, lines 699-710;
      `self` = distance below length), `to_frame_start` (a match that reaches exactly to its frame's first byte) and
      `bad_offset` (the `off > dabs - frame_start` check, lines 581 and 639, after which the blob is handed back); per
      group `list_rescan` (more unknown bytes after round 0 than a list holds: line 808 sends round 1 back to a scan) and
      `full_group` (the group holds K * NT sequences);
    * groups lists (sequences, bytes, unknown bytes after round 0, longest parent chain) per group.
    A byte's parent is the byte it copies (window position `i mod off`); bytes whose source lies before the group, and
    literals, are known at setup (depth 0); round 0 resolves exactly the bytes of depth 1."""
    hits, groups = Counter(), []
    for frame, blks, frame_start in frames:
        kinds = frame_blocks(frame)
        assert len(kinds) == len(blks), "libzstd wrote a different number of blocks than it was given"
        blk0 = frame_start
        for blk, (_, raw_size) in zip(blks, kinds):
            seqs = [t for t in blk if t[1]]
            tail = blk[-1][0] if blk and blk[-1][1] == 0 else 0
            if raw_size is None and not _block(seqs, blk0, frame_start, kseqs, lc, hits, groups):
                return hits, groups  # the blob is handed back at its first bad offset
            blk0 += sum(ll + ml for ll, ml, _ in seqs) + tail
    return hits, groups


def _block(seqs, blk0, frame_start, kseqs, lc, hits, groups):
    n = len(seqs)
    out = np.zeros(n + 1, np.int64)
    lit = np.zeros(n + 1, np.int64)
    for i, (ll, ml, _) in enumerate(seqs):
        out[i + 1] = out[i] + ll + ml
        lit[i + 1] = lit[i] + ll
    s0, gpos, lit_next = 0, blk0, 0
    while s0 < n:
        cnt = 0
        while (cnt < kseqs and s0 + cnt < n and blk0 + out[s0 + cnt + 1] - gpos <= GB
               and lit[s0 + cnt + 1] - lit_next <= GB):
            cnt += 1
        if cnt == 0:
            ll, ml, off = seqs[s0]
            da = blk0 + out[s0] + ll
            hits["alone"] += 1
            if off > da - frame_start:
                hits["bad_offset"] += 1
                return False
            hits["to_frame_start"] += int(off == da - frame_start)
            gpos, lit_next, s0 = da + ml, lit[s0 + 1], s0 + 1
            continue
        gend = blk0 + out[s0 + cnt]
        depth = np.zeros(gend - gpos, np.int64)
        bad = False
        for i in range(s0, s0 + cnt):
            ll, ml, off = seqs[i]
            if ll:
                hits["lit_lane" if ll <= LIT_LANE else "lit_job"] += 1
            dabs = blk0 + out[i] + ll
            if off > dabs - frame_start:
                hits["bad_offset"] += 1
                bad = True
                continue
            hits["to_frame_start"] += int(off == dabs - frame_start)
            sabs = dabs - off
            where = ("self" if off < ml else "before" if sabs + ml <= gpos else "inside" if sabs >= gpos else "straddle")
            hits[("lane_" if ml <= MATCH_LANE else "job_") + where] += 1
            src = sabs + np.arange(ml) % off - gpos
            depth[dabs - gpos: dabs - gpos + ml] = np.where(src >= 0, depth[np.maximum(src, 0)] + 1, 0)
        if bad:
            return False
        unknown = int((depth >= 2).sum())
        groups.append((cnt, int(gend - gpos), unknown, int(depth.max(initial=0))))
        hits["list_rescan"] += unknown > lc
        hits["full_group"] += cnt == kseqs
        gpos, lit_next, s0 = gend, lit[s0 + cnt], s0 + cnt
    return True


# ---------------------------------------------------------------------------------------------------------- the cases

class _Seqs:
    """Builds blocks of (ll, ml, off) tuples while tracking the output position, so every offset stays inside the frame."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.pos = 0
        self.lits = 0

    def add(self, blk, ll, ml, off):
        assert 0 < off <= self.pos + ll, (off, self.pos, ll)
        blk.append((int(ll), int(ml), int(off)))
        self.pos += ll + ml
        self.lits += ll

    def text(self, blk, n):
        """n sequences shaped like LZ77 over text: literal runs of 3-40 bytes, matches of 4-30 bytes at 20-2000"""
        r = self.rng
        for _ in range(n):
            ll = int(r.integers(3, 41))
            hi = min(2000, self.pos + ll)
            self.add(blk, ll, int(r.integers(4, 31)), int(r.integers(min(20, hi), hi + 1)))

    def mixed(self, blk, n):
        """n sequences drawn to land in every setup branch: literal runs up to and above LIT_LANE; matches up to and above
        MATCH_LANE that are far (before any group), near (inside), just behind their literals (straddling the start of a
        group when they open one) or self-feeding at distances 1-17, 31, 32 and 33"""
        r = self.rng
        for _ in range(n):
            if sum(ll + ml for ll, ml, _ in blk[-200:]) and sum(ll + ml for ll, ml, _ in blk) > 120_000:
                break  # a block holds at most 128 KiB
            ll = int(r.integers(0, 9)) if r.random() < 0.5 else int(r.integers(9, 61))
            ml = int(r.integers(3, 17)) if r.random() < 0.5 else int(r.integers(17, 81))
            kind = r.integers(0, 10)
            if kind < 2 and self.pos > 40000:
                off = int(r.integers(20000, 40001))
            elif kind < 5:
                off = int(r.integers(ml, 401))
            elif kind < 8:  # ll < off < ll + ml, off >= ml: straddles when the sequence opens a group
                lo = max(ml, ll + 1)
                off = int(r.integers(lo, ll + ml)) if lo < ll + ml else int(r.integers(ml, 401))
            else:
                off = int(r.choice(list(range(1, 18)) + [31, 32, 33]))
                ml = max(ml, off + int(r.integers(1, 40)))
            if self.pos + ll == 0:
                ll = 1
            self.add(blk, ll, ml, min(off, self.pos + ll))


def _frame(O, blks, lits, params=None, **kw):
    """compress_sequences with minMatch 3 (ZSTD_c_minMatch = 105), so that 3-byte matches pass libzstd's validation"""
    return O.libzstd().compress_sequences(blks, lits, params={105: 3, **(params or {})}, **kw)


@functools.lru_cache(maxsize=None)
def cases():
    """name -> dict(blob, content, frames (for the witness), route, pipe (0: the pipeline keeps the row, 1: hands it
    back), ok (well-formed), stats (the oracle's, when a zstd frame))"""
    import oracle as O
    z = O.libzstd()
    rt = O.real_text(4 << 20).tobytes()
    out = {}

    def put(name, frames, lits, ok=True, parts=None, **kw):
        """frames: list of blocks lists; returns nothing, stores the case (one blob of one or more frames)"""
        blob, content, wf = b"", b"", []
        for k, blks in enumerate(frames):
            c, f = _frame(O, blks, lits[k] if isinstance(lits, list) else lits, **kw)
            wf.append((f, blks, len(content)))
            blob += f + (parts[k] if parts and k < len(parts) else b"")
            content += c
        out[name] = dict(blob=blob, content=content, frames=wf, ok=ok)

    # longer than a group: a literal run over 16 KiB, and matches over 16 KiB at distances 1, 3, 16, 16 385 and beyond
    # 64 KiB, each opening a block and right after a partly filled group
    s = _Seqs(1)
    b0 = []
    s.add(b0, 30000, 4, 9)
    s.text(b0, 60)
    blks = [b0]
    for off in (1, 3, 16, 16385, 70000):
        b = []
        s.add(b, 5, 17000, off)
        s.text(b, 40)
        s.add(b, 7, 17000, off)
        s.text(b, 20)
        blks.append(b)
    put("long", [blks], rt)

    # every setup branch, lane and warp job, with Huffman literals
    s = _Seqs(2)
    blks = [[] for _ in range(3)]
    for b in blks:
        s.mixed(b, 2500)
    put("setup_huffman", [blks], rt)

    # the same shapes over RLE literals (every literal byte the same) after a block of text they copy from
    s = _Seqs(3)
    b0 = []
    s.text(b0, 2000)
    n0 = s.lits
    b1, b2 = [], []
    s.mixed(b1, 2000)
    s.mixed(b2, 2000)
    put("setup_rle_literals", [[b0, b1, b2]], rt[:n0] + b"a" * (s.lits - n0))

    # and over raw literals (literalCompressionMode = uncompressed)
    s = _Seqs(4)
    blks = [[], []]
    for b in blks:
        s.mixed(b, 2500)
    put("setup_raw_literals", [blks], rt, params={O._Zstd.C_LITERAL_COMPRESSION_MODE: 2})

    # list overflow and depth: a chain through a whole 16 KiB group (16 352 bytes unknown after round 0), and one match
    # level per sequence for as many sequences as a group holds
    s = _Seqs(5)
    b0, b1, b2, b3 = [], [], [], []
    s.text(b0, 1500)
    s.add(b1, 16, 16, 16)
    for _ in range(1023):
        s.add(b1, 0, 16, 16)
    s.add(b2, 3, 3, 3)
    for _ in range(5000):
        s.add(b2, 0, 3, 3)
    s.text(b3, 800)
    put("deep", [[b0, b1, b2, b3]], rt)

    # repeat offsets: distances equal to one of the last three, the ll == 0 shift ("repeat 1 minus one" included), and a
    # repeat code in the first sequence of the next block (resolved symbolically in k_zchain)
    s = _Seqs(6)
    r = s.rng
    b0, b1, b2 = [], [], []
    s.text(b0, 1000)
    hist = [b0[-1][2], b0[-2][2], b0[-3][2]]
    for blk in (b1, b2):
        if blk is b2:
            s.add(b2, 3, 8, hist[0])
        for _ in range(1500):
            ll = int(r.integers(0, 12)) if r.random() < 0.7 else 0
            u = r.random()
            if u < 0.5:
                off = hist[int(r.integers(0, 3))]
            elif u < 0.65 and ll == 0 and hist[0] > 1:
                off = hist[0] - 1
            else:
                off = int(r.integers(8, 3000))
            off = min(off, s.pos + ll)
            s.add(blk, ll, int(r.integers(3, 24)), off)
            if off in hist:
                hist.remove(off)
            hist = [off] + hist[:2]
    put("repeat_offsets", [[b0, b1, b2]], rt)

    # frame bounds: a second frame at an output position that is not a multiple of 16, after a skippable frame, whose
    # matches reach exactly to its own first byte
    s = _Seqs(7)
    b0 = []
    s.text(b0, 2000)
    b0.append(((7 - s.pos) % 16 + 16, 0, 0))  # trailing literals: the frame's content ends at 7 mod 16
    lits1 = rt[:s.lits + b0[-1][0]]
    s2 = _Seqs(8)
    c0 = []
    s2.add(c0, 50, 10, 50)   # copies the frame's first bytes
    s2.add(c0, 10, 20, 70)   # ll + previous output = 70: again exactly the frame start
    s2.text(c0, 1500)
    put("multi_frame", [[b0], [c0]], [lits1, rt[500_000:]], parts=[O.libzstd().skippable_frame(b"zn" * 20)])
    mf = out["multi_frame"]
    assert len(mf["frames"][0][0]) + 48 + len(mf["frames"][1][0]) == len(mf["blob"]) and mf["frames"][1][2] % 16 == 7

    # a frame compressed against a prefix (the first frame's content) stored after that frame: its first match reaches
    # before its own start, which a frame on its own cannot do — every decoder must reject the blob
    s = _Seqs(9)
    a0 = []
    s.text(a0, 2000)
    ca, fa = _frame(O, [a0], rt)
    sb = _Seqs(10)
    sb.pos = len(ca)  # the offsets below may reach into the prefix
    bb = []
    sb.add(bb, 10, 40, 5000)
    sb.text(bb, 400)
    cb, fb = _frame(O, [bb], rt[1_000_000:], prefix=ca, params={O._Zstd.C_VALIDATE_SEQUENCES: 0})
    out["ref_prefix"] = dict(blob=fa + fb, content=ca + cb, ok=False,
                             frames=[(fa, [a0], 0), (fb, [bb], len(ca))])

    for v in out.values():
        v["route"] = route(len(v["content"]), len(v["blob"]))
        v["pipe"] = 0 if v["ok"] else 1
    return out


@functools.lru_cache(maxsize=None)
def route_cases():
    """The same shapes as rows of the other decode classes: name -> dict(blob, content, route)"""
    import oracle as O
    z = O.libzstd()
    rt = O.real_text(1 << 20).tobytes()
    out = {}
    rle_block = [(1, 128 * KIB - 1, 1)]  # one byte and 128 KiB - 1 of offset 1: libzstd writes an RLE block

    def padded(name, blks, want):
        """blks plus offset-1 runs until compressed <= decoded / 64"""
        n = 0
        while True:
            c, f = _frame(O, blks + [rle_block] * n, rt)
            if len(f) * 64 <= len(c):
                break
            n += 1
        out[name] = dict(blob=f, content=c, route=want)

    s = _Seqs(11)
    blks = [[], []]
    for b in blks:
        s.mixed(b, 1500)
    padded("pattern_big", blks, BIGPAT)
    s = _Seqs(12)
    b = []
    s.mixed(b, 60)
    padded("pattern_mid", [b], MID)
    for k in range(3):  # under 4 KiB: one-warp teams
        s = _Seqs(13 + k)
        b = []
        s.add(b, 20, 12, 15)
        s.mixed(b, 30 + 10 * k)
        c, f = _frame(O, [b], rt[k * 5000:])
        out[f"small_{k}"] = dict(blob=f, content=c, route=SMALL)
    # at least as large as its content: 1 KiB blocks of random literals (raw blocks, 3 header bytes each) and one
    # Huffman / FSE block of skewed literals
    rnd = O.gen_random(530 * KIB).tobytes()
    skew = O.gen_small_alphabet(4000).tobytes()
    s = _Seqs(16)
    blks = [[(KIB, 0, 0)] for _ in range(530)]
    s.pos = 530 * KIB
    hb = []
    for _ in range(20):
        s.add(hb, 10, int(s.rng.integers(4, 20)), int(s.rng.integers(1, 600)))
    c, f = _frame(O, blks[:300] + [hb] + blks[300:], rnd[:300 * KIB] + skew[:200] + rnd[300 * KIB:])
    out["raw_blocks_and_one_entropy_block"] = dict(blob=f, content=c, route=BIGRAW)
    return out


def small_window_cases():
    """libzstd frames without a content size at windowLog 10 / 12 / 14 / 16: name -> (blob, content, pipe)"""
    import oracle as O
    d = O.real_text(300_000)
    return {f"wlog{wl}": (O.libzstd().compress(d, 3, params={101: wl, 200: 0}), d.tobytes(), int(wl <= 12))
            for wl in (10, 12, 14, 16)}


def lz4_cases():
    """LZ4 frames with 1 MiB and 4 MiB blocks (ids 6, 7), linked and independent: name -> (blob, content, route)"""
    import oracle as O
    l = O.liblz4()
    datas = {"text": O.real_text(1_200_000), "pattern": O.gen_text(5 << 20), "small": O.real_text(3000)}
    out = {}
    for bsid in (6, 7):
        for indep in (False, True):
            for k, d in datas.items():
                b = l.compress_frame(d, block_size_id=bsid, independent=indep, content_checksum=True)
                out[f"lz4_bs{bsid}_{'indep' if indep else 'linked'}_{k}"] = (b, d.tobytes(), route(d.size, len(b)))
    return out


# ---------------------------------------------------------------------------------------------------------- the tests

def test_cases_decode_with_libzstd_and_the_oracle(oracle):
    z = oracle.libzstd()
    for name, c in {**cases(), **route_cases()}.items():
        rc, o, st = oracle.zstd_decompress(c["blob"], len(c["content"]), want_stats=True)
        if c.get("ok", True):
            assert rc == 0 and o == c["content"], name
            assert z.decompress(c["blob"], len(c["content"])) == c["content"], name
        else:
            assert rc != 0, name
            with pytest.raises(RuntimeError):
                z.decompress(c["blob"], len(c["content"]))
        c["stats"] = st
    st = cases()
    assert st["repeat_offsets"]["stats"]["repcode_uses"] > 1000
    assert st["setup_rle_literals"]["stats"]["lit_rle"] >= 2 and st["setup_raw_literals"]["stats"]["lit_raw"] >= 2
    assert st["setup_huffman"]["stats"]["lit_huf_4stream"] >= 3 and st["multi_frame"]["stats"]["skippable_frames"] == 1
    rb = route_cases()["raw_blocks_and_one_entropy_block"]["stats"]
    assert rb["blocks_raw"] == 530 and rb["blocks_compressed"] == 1 and rb["lit_huf_1stream"] + rb["lit_huf_4stream"] == 1
    for name, (b, d, _) in small_window_cases().items():
        assert z.decompress(b, len(d) + 1) == d, name
    for name, (b, d, _) in lz4_cases().items():
        assert oracle.liblz4().decompress_frame(b, len(d)) == d, name


@pytest.mark.parametrize("mis", [0, 5, 13])
def test_cases_through_the_host_emulation(emu, mis):  # noqa: F811
    """Every decoder's host build against the content: the pipeline up to exec (hands back exactly the ill-formed blob),
    the one-team decoder and the block-parallel decoder (reject it)."""
    for name, c in {**cases(), **route_cases()}.items():
        d = c["content"]
        if "pipe" in c:  # rows of the other classes never reach the pipeline
            rc, out, _ = emu.decode_pipe(c["blob"], len(d), mis)
            assert rc == c["pipe"], (name, rc)
            assert rc or out == d, name
        st, out = emu.decode(c["blob"], len(d), mis % 8)
        st2, out2 = emu.decode_par(c["blob"], len(d))
        if c.get("ok", True):
            assert st == 0 and out == d, (name, st)
            assert st2 == 0 and out2 == d, (name, st2)
        else:
            assert st != 0 and st2 != 0, name
    for name, (b, d, pipe) in small_window_cases().items():
        rc, out, _ = emu.decode_pipe(b, len(d), mis)
        assert rc == pipe, name
        assert rc or out == d
        st, out = emu.decode(b, len(d), mis % 8)
        assert st == 0 and out == d, name


def test_routes():
    for name, c in cases().items():
        assert c["route"] == PIPE, name
    for name, c in route_cases().items():
        assert route(len(c["content"]), len(c["blob"])) == c["route"], name
    lz = Counter(r for _, _, r in lz4_cases().values())
    assert lz == {PIPE: 4, BIGPAT: 4, SMALL: 4}, lz  # LZ4 text rows reach the pipeline, which hands them back
    for name, (b, d, _) in small_window_cases().items():
        assert route(len(d), len(b)) == PIPE, name


def witness_hits(shape):
    kseqs, lc = SHAPES[shape]
    total, groups = Counter(), []
    for name, c in cases().items():
        h, g = witness(c["frames"], kseqs, lc)
        assert ("bad_offset" in h) == (not c["ok"]), name
        total += h
        groups += g
    return total, groups


BRANCHES = ["alone", "lit_lane", "lit_job", "lane_before", "lane_inside", "lane_straddle", "lane_self", "job_before",
            "job_inside", "job_straddle", "job_self", "to_frame_start", "bad_offset", "list_rescan", "full_group"]


@pytest.mark.parametrize("shape", list(SHAPES))
def test_witness_reaches_every_branch(shape):
    """Each branch of k_zexec2's group logic is reached by at least one sequence or group of the cases, in both exec
    shapes; the deepest chain is one level per sequence of a full group."""
    kseqs, lc = SHAPES[shape]
    hits, groups = witness_hits(shape)
    print(shape, dict(hits), "groups", len(groups), "max unknown after round 0", max(g[2] for g in groups),
          "deepest chain", max(g[3] for g in groups))
    assert all(hits[b] > 0 for b in BRANCHES), {b: hits[b] for b in BRANCHES}
    assert max(g[3] for g in groups) == kseqs
    assert max(g[2] for g in groups) > 8192
    # self-feeding distances 1-17, 31, 32, 33 as warp jobs, 1-15 in the lane
    seen_lane, seen_job = set(), set()
    for c in cases().values():
        for _, blks, _ in c["frames"]:
            for blk in blks:
                for ll, ml, off in blk:
                    if 0 < off < ml:
                        (seen_lane if ml <= MATCH_LANE else seen_job).add(off)
    assert seen_job >= set(range(1, 18)) | {31, 32, 33} and seen_lane >= set(range(1, 16))

