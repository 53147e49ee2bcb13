// Zstandard frame decoder (RFC 8878), one team (CTA) per blob.
//
// Replaces codec::decompress_into (znippy-common/src/codec.rs:67-78: zl_get_decompressed_size -> zl_decompress) for
// blobs whose payload is a Zstandard frame.  The arithmetic on the reference path lives in openzl-sys-rs 0.2.0 ->
// facebook/openzl -> zstd (not vendored); this is written from the format specification.
//
// Execution model.  All header parsing is team-uniform scalar code that every thread executes redundantly (the
// loads are broadcasts), so no control state is ever communicated.  Serial work is done by single threads:
//   thread 0            builds the Huffman / FSE decoding tables in shared memory and runs the three interleaved
//                       FSE state machines, emitting resolved sequences {literal offset, ll, ml, match offset} into a
//                       shared-memory batch (repeat-offset history, literal and output cursors and every bounds check
//                       live here, so executors never see an invalid sequence);
//   threads 0..3        decode the (up to) four Huffman literal streams into the per-CTA literal scratch.
// Bandwidth work is done by the whole team: each batch of sequences is executed with 128-bit cooperative copies
// (coop.cuh).  A barrier is taken only when a match reads bytes written since the previous barrier (tracked with a
// watermark), so literal-heavy and long-match data run barrier-free.
#pragma once
#include "coop.cuh"
#include "zstd_tables.cuh"

namespace zn {

constexpr uint32_t kSeqBatch = 256;

struct SeqRec {
  uint32_t lit;  // offset of this sequence's literals inside the block's literal source
  uint32_t ll;
  uint32_t ml;
  uint32_t off;  // resolved match distance (>= 1) when ml > 0
};

// Everything a team shares while decoding one blob (lives in shared memory on the device).
struct DecShared {
  zs::HufTable huf;
  zs::FseTable ll, of, ml, wt;  // wt: scratch table for FSE-compressed Huffman weights
  SeqRec ring[kSeqBatch];
  uint8_t* tile;  // kTileBytes of 128-byte aligned shared memory, bulk-store source of long periodic matches; may be null
  uint32_t pat[kPatWords];
  uint16_t next[256];    // scratch of the Huffman-weights FSE table build (literal decoder)
  uint16_t next_seq[64]; // scratch of the sequence-table builds (sequence decoder; the two may run concurrently)
  int16_t norm[64];
  uint8_t weights[256];
  uint32_t lut_ll[36], lut_ml[53];  // length code -> baseline | extra bits << 24 (shared-memory copy: LDS, not indexed LDC)
  // single-writer mailboxes (thread 0 -> team); each has its own slot so that a fast thread 0 can never overwrite
  // one before a slow thread has read it (there is at least one barrier between a read and the slot's next write)
  uint32_t huf_used;    // bytes of the Huffman tree description, ~0u = malformed
  uint32_t err_lit;     // literal streams
  uint32_t err_tab;     // sequence tables + initial FSE states
  uint32_t err_seq;     // sequence batch
  uint32_t rep_pub[3];  // repeat-offset history after the block's last sequence
  uint32_t lit_pub;     // literals consumed by the block's sequences
};

// Prebuilt decoding tables for the predefined distributions (built once per context with zs::fse_build).
struct PredefTables {
  uint32_t ll[64], of[32], ml[64];
};

#if defined(__CUDACC__)
__device__ PredefTables g_predef;  // filled by zn_ctx_create
#endif
#if defined(__CUDA_ARCH__)
ZN_D const PredefTables* predef_tables() { return &g_predef; }
#else
inline const PredefTables* predef_tables() {
  static PredefTables p;
  static bool init = false;
  if (!init) {
    zs::FseTable t;
    uint16_t next[64];
    zs::fse_build(&t, zs::kLLDefault, 36, 6, next);
    for (int i = 0; i < 64; i++) p.ll[i] = t.e[i];
    zs::fse_build(&t, zs::kOFDefault, 29, 5, next);
    for (int i = 0; i < 32; i++) p.of[i] = t.e[i];
    zs::fse_build(&t, zs::kMLDefault, 53, 6, next);
    for (int i = 0; i < 64; i++) p.ml[i] = t.e[i];
    init = true;
  }
  return &p;
}
#endif

namespace zs {

// Fills the length-code lookup tables of `sh`; strided over the team (call before the first block, then barrier).
ZN_HD void init_luts(const Team& t, DecShared* sh) {
  for (uint32_t i = t.tid; i < 36; i += t.n) sh->lut_ll[i] = kLLBase[i] | ((uint32_t)kLLBits[i] << 24);
  for (uint32_t i = t.tid; i < 53; i += t.n) sh->lut_ml[i] = kMLBase[i] | ((uint32_t)kMLBits[i] << 24);
}

// cursors of one frame that thread 0's sequence decoder and the executors both advance
struct ExecState {
  uint32_t pos;   // next output byte (relative to the blob's output start)
  uint32_t wm;    // bytes below wm were written, and are visible to the team, since its last memory barrier
  uint32_t bulk;  // bulk (async-proxy) stores are in flight: they cover bytes at or above wm only
};

// Barrier after which every byte written so far is visible to the whole team (and tile / pat may be rewritten).
ZN_HD void mem_sync(const Team& t, ExecState& es) {
  if (es.bulk) {
    if (t.tid < kBulkIssuers) bulk_wait_all();
    es.bulk = 0;
  }
  team_sync(t);
  es.wm = es.pos;
}

// Executes ring[0..n): literal copy then match copy per sequence.  Team-uniform.
ZN_HD void exec_batch(const Team& t, DecShared* sh, uint32_t n, uint8_t* out, const uint8_t* lit_base, int lit_rle,
                      ExecState& es) {
  for (uint32_t i = 0; i < n; i++) {
    const SeqRec s = sh->ring[i];
    if (s.ll) {
      if (lit_rle >= 0) team_fill(t, out + es.pos, (uint32_t)lit_rle, s.ll);
      else team_copy(t, out + es.pos, lit_base + s.lit, s.ll);
      es.pos += s.ll;
    }
    if (s.ml) {
      const uint32_t src_lo = es.pos - s.off;
      const uint32_t src_hi = s.off >= s.ml ? src_lo + s.ml : es.pos;
      ZN_TP(6);
      if (src_hi > es.wm) mem_sync(t, es);
      ZN_TP(7);
      if (team_match(t, out + es.pos, s.off, s.ml, sh->pat, sh->tile)) es.bulk = 1;
      es.pos += s.ml;
    }
  }
}

// One Huffman stream of `n` symbols, decoded by the calling thread. Returns false when the stream is malformed.
ZN_HD bool huf_decode_stream(const HufTable* h, const uint8_t* p, uint32_t len, uint8_t* out, uint32_t n) {
  BackBits b;
  if (!b.init(p, len)) return false;
  const uint32_t mb = h->max_bits;
  uint32_t i = 0;
  // two symbols per refill (2 x 11 bits <= 32)
  for (; i + 2 <= n; i += 2) {
    b.refill();
    const uint32_t e0 = h->e[b.peek(mb)];
    b.skip(e0 >> 8);
    const uint32_t e1 = h->e[b.peek(mb)];
    b.skip(e1 >> 8);
    out[i] = (uint8_t)e0;
    out[i + 1] = (uint8_t)e1;
  }
  if (i < n) {
    b.refill();
    const uint32_t e0 = h->e[b.peek(mb)];
    b.skip(e0 >> 8);
    out[i] = (uint8_t)e0;
  }
  return b.bits_left == 0;
}

struct LitInfo {
  const uint8_t* base;  // literal source (compressed input for raw, scratch for Huffman)
  int rle;              // >= 0: every literal is this byte
  uint32_t len;         // regenerated size
  uint32_t consumed;    // bytes of the block taken by the literals section
};

// Literals section (RFC 8878 §3.1.1.3.1).  Team-uniform; returns S_OK or S_DECODE_ERROR.
ZN_HD uint32_t decode_literals(const Team& t, DecShared* sh, const uint8_t* p, uint32_t len, uint8_t* lit_scratch,
                               LitInfo& li) {
  if (len < 1) return S_DECODE_ERROR;
  const uint32_t b0 = p[0], type = b0 & 3, sf = (b0 >> 2) & 3;
  if (type < 2) {
    uint32_t hdr, regen;
    if ((sf & 1) == 0) { hdr = 1; regen = b0 >> 3; }
    else if (sf == 1) { if (len < 2) return S_DECODE_ERROR; hdr = 2; regen = (b0 >> 4) | ((uint32_t)p[1] << 4); }
    else { if (len < 3) return S_DECODE_ERROR; hdr = 3; regen = (b0 >> 4) | ((uint32_t)p[1] << 4) | ((uint32_t)p[2] << 12); }
    if (regen > kZstdBlockMax) return S_DECODE_ERROR;
    li.len = regen;
    if (type == 0) {
      if (hdr + regen > len) return S_DECODE_ERROR;
      li.base = p + hdr; li.rle = -1; li.consumed = hdr + regen;
    } else {
      if (hdr + 1 > len) return S_DECODE_ERROR;
      li.base = nullptr; li.rle = (int)p[hdr]; li.consumed = hdr + 1;
    }
    return S_OK;
  }
  uint32_t hdr, regen, comp, streams;
  if (sf <= 1) {
    if (len < 3) return S_DECODE_ERROR;
    const uint32_t v = ld24le(p);
    hdr = 3; regen = (v >> 4) & 0x3FF; comp = (v >> 14) & 0x3FF; streams = sf == 0 ? 1 : 4;
  } else if (sf == 2) {
    if (len < 4) return S_DECODE_ERROR;
    const uint32_t v = ld32le(p);
    hdr = 4; regen = (v >> 4) & 0x3FFF; comp = v >> 18; streams = 4;
  } else {
    if (len < 5) return S_DECODE_ERROR;
    const uint64_t v = (uint64_t)ld32le(p) | ((uint64_t)p[4] << 32);
    hdr = 5; regen = (uint32_t)(v >> 4) & 0x3FFFF; comp = (uint32_t)(v >> 22); streams = 4;
  }
  if (regen > kZstdBlockMax || hdr + comp > len) return S_DECODE_ERROR;
  const uint8_t* q = p + hdr;
  uint32_t qlen = comp;
  // -- Huffman table (thread 0), result published through sh->huf_used
  if (type == 2) {
    if (t.tid == 0) {
      const int used = huf_read_table(&sh->huf, q, qlen, sh->weights, &sh->wt, sh->next);
      sh->huf_used = used < 0 ? 0xFFFFFFFFu : (uint32_t)used;
    }
    team_sync(t);
    const uint32_t used = sh->huf_used;
    if (used == 0xFFFFFFFFu || used > qlen) return S_DECODE_ERROR;
    q += used; qlen -= used;
  } else {
    if (!sh->huf.valid) return S_DECODE_ERROR;
  }
  // -- streams
  uint32_t s_off[4], s_len[4], o_off[4], o_len[4];
  if (streams == 1) {
    s_off[0] = 0; s_len[0] = qlen; o_off[0] = 0; o_len[0] = regen;
  } else {
    if (qlen < 6) return S_DECODE_ERROR;
    const uint32_t s1 = ld16le(q), s2 = ld16le(q + 2), s3 = ld16le(q + 4);
    if (6 + s1 + s2 + s3 > qlen) return S_DECODE_ERROR;
    const uint32_t seg = (regen + 3) / 4;
    if (seg * 3 > regen) return S_DECODE_ERROR;
    s_off[0] = 6; s_len[0] = s1;
    s_off[1] = 6 + s1; s_len[1] = s2;
    s_off[2] = 6 + s1 + s2; s_len[2] = s3;
    s_off[3] = 6 + s1 + s2 + s3; s_len[3] = qlen - s_off[3];
    for (int k = 0; k < 4; k++) { o_off[k] = seg * k; o_len[k] = k < 3 ? seg : regen - 3 * seg; }
  }
  if (t.tid == 0) sh->err_lit = 0;
  team_sync(t);
#if defined(__CUDA_ARCH__)
  if (t.tid < streams) {
    const uint32_t k = t.tid;
    uint32_t so = s_off[0], sl = s_len[0], oo = o_off[0], ol = o_len[0];
#pragma unroll
    for (uint32_t j = 1; j < 4; j++)
      if (k == j) { so = s_off[j]; sl = s_len[j]; oo = o_off[j]; ol = o_len[j]; }
    if (!huf_decode_stream(&sh->huf, q + so, sl, lit_scratch + oo, ol)) sh->err_lit = 1;
  }
#else
  for (uint32_t k = 0; k < streams; k++)
    if (!huf_decode_stream(&sh->huf, q + s_off[k], s_len[k], lit_scratch + o_off[k], o_len[k])) sh->err_lit = 1;
#endif
  team_sync(t);
  if (sh->err_lit) return S_DECODE_ERROR;
  li.base = lit_scratch; li.rle = -1; li.len = regen; li.consumed = hdr + comp;
  return S_OK;
}

// One of the three sequence tables (RFC 8878 §3.1.1.3.2.1).  Called by thread 0 only.  Returns false on error.
ZN_HD bool setup_seq_table(FseTable* t, uint32_t mode, const uint8_t*& q, const uint8_t* end, int max_log, int max_sym,
                           const uint32_t* predef, int predef_log, DecShared* sh) {
  if (mode == 0) {  // entries were copied by the whole team (decode_block)
    (void)predef;
    t->log = (uint32_t)predef_log;
    t->valid = 1;
    return true;
  }
  if (mode == 1) {
    if (q >= end) return false;
    const uint32_t sym = *q++;
    if ((int)sym > max_sym) return false;
    fse_build_rle(t, sym);
    return true;
  }
  if (mode == 2) {
    int log, nsym;
    const int used = fse_read_ncount(q, (uint32_t)(end - q), max_log, max_sym, sh->norm, &log, &nsym);
    if (used < 0) return false;
    fse_build(t, sh->norm, nsym, log, sh->next_seq);
    q += used;
    return true;
  }
  return t->valid != 0;  // repeat
}

// Per-block sequence decoder state, meaningful in thread 0 only.
struct SeqDecoder {
  BackBits b;
  uint32_t sl, so, sm;   // FSE states
  uint32_t rep0, rep1, rep2;
  uint32_t lit_pos;      // literals consumed so far in this block
  uint32_t out_pos;      // output cursor as the decoder sees it (ahead of the executors by one batch)
};

// Decodes up to kSeqBatch sequences (the last one being sequence `nseq-1` of the block) into sh->ring.
// Thread 0 only.  Returns S_OK / S_DECODE_ERROR / S_DST_TOO_SMALL.
ZN_HD uint32_t decode_seq_batch(DecShared* sh, SeqDecoder& d, uint32_t first, uint32_t count, uint32_t nseq,
                                uint32_t lit_len, uint32_t cap, uint32_t frame_start) {
  const uint32_t* tl = sh->ll.e;
  const uint32_t* to = sh->of.e;
  const uint32_t* tm = sh->ml.e;
  for (uint32_t i = 0; i < count; i++) {
    const uint32_t el = tl[d.sl], eo = to[d.so], em = tm[d.sm];
    const uint32_t lc = fse_sym(el), oc = fse_sym(eo), mc = fse_sym(em);
    if (oc > 31 || mc > 52 || lc > 35) return S_DECODE_ERROR;
    d.b.refill();
    const uint32_t obits = d.b.read(oc);
    const uint64_t ov = ((uint64_t)1 << oc) + obits;
    d.b.refill();
    const uint32_t xm = sh->lut_ml[mc], xl = sh->lut_ll[lc];
    const uint32_t ml = (xm & 0xFFFFFFu) + d.b.read(xm >> 24);
    const uint32_t ll = (xl & 0xFFFFFFu) + d.b.read(xl >> 24);
    if (first + i + 1 < nseq) {
      d.b.refill();
      d.sl = fse_base(el) + d.b.read(fse_nbits(el));
      d.sm = fse_base(em) + d.b.read(fse_nbits(em));
      d.so = fse_base(eo) + d.b.read(fse_nbits(eo));
    }
    if (d.b.bits_left < 0) return S_DECODE_ERROR;
    uint64_t offset;
    if (ov > 3) {
      offset = ov - 3;
      d.rep2 = d.rep1; d.rep1 = d.rep0; d.rep0 = (uint32_t)offset;
    } else {
      const uint32_t idx = (uint32_t)ov - 1 + (ll == 0 ? 1u : 0u);
      if (idx == 0) offset = d.rep0;
      else {
        offset = idx == 3 ? (uint64_t)d.rep0 - 1 : (idx == 1 ? d.rep1 : d.rep2);
        if (offset == 0) return S_DECODE_ERROR;
        if (idx != 1) d.rep2 = d.rep1;
        d.rep1 = d.rep0;
        d.rep0 = (uint32_t)offset;
      }
    }
    if (ll > lit_len - d.lit_pos) return S_DECODE_ERROR;
    if ((uint64_t)ll + ml > (uint64_t)(cap - d.out_pos)) return S_DST_TOO_SMALL;
    if (offset > (uint64_t)(d.out_pos + ll - frame_start)) return S_DECODE_ERROR;
    SeqRec r;
    r.lit = d.lit_pos; r.ll = ll; r.ml = ml; r.off = (uint32_t)offset;
    sh->ring[i] = r;
    d.lit_pos += ll;
    d.out_pos += ll + ml;
  }
  return S_OK;
}

// rep[] = repeat-offset history carried across the blocks of a frame (team-uniform copy in every thread)
struct FrameState {
  uint32_t rep0, rep1, rep2;
  uint32_t predef;  // bit0/1/2: the LL/OF/ML table in shared memory currently holds the predefined distribution
};

// Compressed block.  Team-uniform.  Advances es.pos.
ZN_HD uint32_t decode_block(const Team& t, DecShared* sh, const uint8_t* p, uint32_t len, uint8_t* out, uint32_t cap,
                            uint32_t frame_start, FrameState& fs, ExecState& es, uint8_t* lit_scratch) {
  ZN_TP(1);
  LitInfo li;
  uint32_t rc = decode_literals(t, sh, p, len, lit_scratch, li);
  if (rc != S_OK) return rc;
  const uint8_t* q = p + li.consumed;
  const uint8_t* end = p + len;
  const uint32_t block_start = es.pos;
  if (q >= end) return S_DECODE_ERROR;
  uint32_t nseq = *q++;
  if (nseq >= 128) {
    if (nseq == 255) { if (end - q < 2) return S_DECODE_ERROR; nseq = (uint32_t)q[0] + ((uint32_t)q[1] << 8) + 0x7F00u; q += 2; }
    else { if (end - q < 1) return S_DECODE_ERROR; nseq = ((nseq - 128) << 8) + q[0]; q += 1; }
  }
  uint32_t lit_pos = 0;
  if (nseq > 0) {
    if (q >= end) return S_DECODE_ERROR;
    const uint32_t modes = *q++;
    if (modes & 3) return S_DECODE_ERROR;
    SeqDecoder d;
    const PredefTables* pd = predef_tables();
    // -- predefined tables: copied by the whole team, and only when the table does not already hold them
    {
      const uint32_t mll = modes >> 6, mof = (modes >> 4) & 3, mml = (modes >> 2) & 3;
      if (mll == 0 && !(fs.predef & 1u)) for (uint32_t i = t.tid; i < 64; i += t.n) sh->ll.e[i] = pd->ll[i];
      if (mof == 0 && !(fs.predef & 2u)) for (uint32_t i = t.tid; i < 32; i += t.n) sh->of.e[i] = pd->of[i];
      if (mml == 0 && !(fs.predef & 4u)) for (uint32_t i = t.tid; i < 64; i += t.n) sh->ml.e[i] = pd->ml[i];
      if (mll != 3) fs.predef = (fs.predef & ~1u) | (mll == 0 ? 1u : 0u);
      if (mof != 3) fs.predef = (fs.predef & ~2u) | (mof == 0 ? 2u : 0u);
      if (mml != 3) fs.predef = (fs.predef & ~4u) | (mml == 0 ? 4u : 0u);
    }
    // -- other table modes + initial states (thread 0); outcome in sh->err_tab
    if (t.tid == 0) {
      uint32_t e = S_OK;
      const uint8_t* qq = q;
      if (!setup_seq_table(&sh->ll, modes >> 6, qq, end, 9, 35, pd->ll, 6, sh) ||
          !setup_seq_table(&sh->of, (modes >> 4) & 3, qq, end, 8, 31, pd->of, 5, sh) ||
          !setup_seq_table(&sh->ml, (modes >> 2) & 3, qq, end, 9, 52, pd->ml, 6, sh))
        e = S_DECODE_ERROR;
      if (e == S_OK && !d.b.init(qq, (uint32_t)(end - qq))) e = S_DECODE_ERROR;
      if (e == S_OK) {
        d.b.refill();
        d.sl = d.b.read(sh->ll.log);
        d.so = d.b.read(sh->of.log);
        d.sm = d.b.read(sh->ml.log);
        if (d.b.bits_left < 0) e = S_DECODE_ERROR;
        d.rep0 = fs.rep0; d.rep1 = fs.rep1; d.rep2 = fs.rep2;
        d.lit_pos = 0;
        d.out_pos = es.pos;
      }
      sh->err_tab = e;
    }
    ZN_TP(2);
    team_sync(t);
    ZN_TP(3);
    if (sh->err_tab != S_OK) return sh->err_tab;
    for (uint32_t first = 0; first < nseq; first += kSeqBatch) {
      const uint32_t count = nseq - first < kSeqBatch ? nseq - first : kSeqBatch;
      if (t.tid == 0) {
        uint32_t e = decode_seq_batch(sh, d, first, count, nseq, li.len, cap, frame_start);
        if (e == S_OK && first + count == nseq && d.b.bits_left != 0) e = S_DECODE_ERROR;
        sh->err_seq = e;
        if (first + count == nseq) {  // publish the block's final history and literal cursor
          sh->rep_pub[0] = d.rep0; sh->rep_pub[1] = d.rep1; sh->rep_pub[2] = d.rep2;
          sh->lit_pub = d.lit_pos;
        }
      }
      ZN_TP(4);
      team_sync(t);
      ZN_TP(5);
      if (sh->err_seq != S_OK) return sh->err_seq;
      exec_batch(t, sh, count, out, li.base, li.rle, es);
      ZN_TP(9);
      team_sync(t);  // ring and err_seq are rewritten by the next batch
      if (!es.bulk) es.wm = es.pos;
    }
    fs.rep0 = sh->rep_pub[0]; fs.rep1 = sh->rep_pub[1]; fs.rep2 = sh->rep_pub[2];
    lit_pos = sh->lit_pub;
  }
  const uint32_t rest = li.len - lit_pos;
  if (rest > cap - es.pos) return S_DST_TOO_SMALL;
  if (rest) {
    if (li.rle >= 0) team_fill(t, out + es.pos, (uint32_t)li.rle, rest);
    else team_copy(t, out + es.pos, li.base + lit_pos, rest);
    es.pos += rest;
  }
  if (es.pos - block_start > kZstdBlockMax) return S_DECODE_ERROR;
  return S_OK;
}


// Hook called (team-uniform) after every block and once at the end; the fused decode+hash kernel hashes the chunks that
// have become final (below es.wm) while later blocks' bulk stores are still in flight.
struct NoHook {
  ZN_HD void after_block(const Team&, ExecState&) {}
  ZN_HD void finish(const Team&, ExecState&) {}
};

// Range reads: ends the decode after the first block whose end reaches `stop` (block-granular, so at most one block is
// written past it).  Every other hook decodes to the end; stop_here is then a constant false and compiles away.
struct StopAt : NoHook {
  uint32_t stop;
};
template <class Hook>
ZN_HD bool stop_here(const Hook&, uint32_t) { return false; }
ZN_HD bool stop_here(const StopAt& h, uint32_t pos) { return pos >= h.stop; }

// All concatenated frames of one blob (skippable frames are skipped).  Team-uniform.
// Returns the blob's status; *produced = bytes written to out.  With a StopAt hook the decode returns S_OK as soon as a
// block ends at or past the stop, without the frame-content-size comparison or the checksum of that frame.
template <class Hook>
ZN_HD uint32_t decode_frames(const Team& t, DecShared* sh, const uint8_t* src, uint32_t src_len, uint8_t* out,
                             uint32_t cap, uint8_t* lit_scratch, uint32_t& predef, uint32_t* produced, Hook& hook) {
  uint32_t ip = 0;
  ExecState es;
  es.pos = 0;
  es.wm = 0;
  es.bulk = 0;
  *produced = 0;
  if (src_len == 0) return S_DECODE_ERROR;
  while (ip < src_len) {
    if (src_len - ip >= 8) {
      const uint32_t magic = ld32le(src + ip);
      if ((magic & 0xFFFFFFF0u) == 0x184D2A50u) {
        const uint32_t sz = ld32le(src + ip + 4);
        if (sz > src_len - ip - 8) return S_DECODE_ERROR;
        ip += 8 + sz;
        continue;
      }
    }
    // ---- frame header
    if (src_len - ip < 5) return S_DECODE_ERROR;
    if (ld32le(src + ip) != 0xFD2FB528u) return ip == 0 ? S_UNSUPPORTED : S_DECODE_ERROR;
    const uint32_t fhd = src[ip + 4], fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, did_flag = fhd & 3;
    if (fhd & 0x08) return S_UNSUPPORTED;
    const uint32_t checksum = (fhd >> 2) & 1;
    uint32_t hp = ip + 5;
    uint64_t window = 0;
    if (!single) {
      if (src_len < hp + 1) return S_DECODE_ERROR;
      const uint32_t wd = src[hp++], e = wd >> 3, m = wd & 7;
      const uint64_t base = 1ull << (10 + e);
      window = base + (base >> 3) * m;
    }
    const uint32_t db = did_flag == 3 ? 4u : did_flag;
    if (src_len < hp + db) return S_DECODE_ERROR;
    uint32_t did = 0;
    for (uint32_t i = 0; i < db; i++) did |= (uint32_t)src[hp + i] << (8 * i);
    hp += db;
    if (did != 0) return S_UNSUPPORTED;
    const uint32_t fb = fcs_flag == 0 ? single : (fcs_flag == 1 ? 2u : (fcs_flag == 2 ? 4u : 8u));
    if (src_len < hp + fb) return S_DECODE_ERROR;
    uint64_t fcs = 0;
    for (uint32_t i = 0; i < fb; i++) fcs |= (uint64_t)src[hp + i] << (8 * i);
    if (fb == 2) fcs += 256;
    hp += fb;
    if (single) window = fcs;
    ip = hp;
    const uint32_t frame_start = es.pos;
    const uint32_t block_max = window < kZstdBlockMax ? (uint32_t)window : kZstdBlockMax;
    FrameState fs;
    fs.rep0 = 1; fs.rep1 = 4; fs.rep2 = 8;
    fs.predef = predef;  // table CONTENT survives the per-frame validity reset below
    team_sync(t);  // nobody may still be using the previous frame's tables
    if (t.tid == 0) sh->huf.valid = sh->ll.valid = sh->of.valid = sh->ml.valid = 0;
    team_sync(t);
    // ---- blocks
    for (;;) {
      if (src_len - ip < 3) return S_DECODE_ERROR;
      const uint32_t bh = ld24le(src + ip);
      ip += 3;
      const uint32_t last = bh & 1, type = (bh >> 1) & 3, bsize = bh >> 3;
      if (type == 3) return S_DECODE_ERROR;
      if (type == 0) {
        if (bsize > src_len - ip) return S_DECODE_ERROR;
        if (bsize > cap - es.pos) return S_DST_TOO_SMALL;
        team_copy(t, out + es.pos, src + ip, bsize);
        es.pos += bsize;
        ip += bsize;
      } else if (type == 1) {
        if (src_len - ip < 1) return S_DECODE_ERROR;
        if (bsize > cap - es.pos) return S_DST_TOO_SMALL;
        team_fill(t, out + es.pos, src[ip], bsize);
        es.pos += bsize;
        ip += 1;
      } else {
        if (bsize > src_len - ip) return S_DECODE_ERROR;
        if (bsize > block_max || bsize < 2) return S_DECODE_ERROR;
        const uint32_t rc = decode_block(t, sh, src + ip, bsize, out, cap, frame_start, fs, es, lit_scratch);
        predef = fs.predef;
        if (rc != S_OK) return rc;
        ip += bsize;
      }
      *produced = es.pos;
      hook.after_block(t, es);
      if (stop_here(hook, es.pos)) return S_OK;
      if (last) break;
    }
    if (fb != 0 && (uint64_t)(es.pos - frame_start) != fcs) return S_SIZE_MISMATCH;
    if (checksum) {  // XXH64 content checksum: present but not verified here (blake3 of the content is; DESIGN.md)
      if (src_len - ip < 4) return S_DECODE_ERROR;
      ip += 4;
    }
  }
  *produced = es.pos;
  hook.finish(t, es);
  return S_OK;
}

}  // namespace zs
}  // namespace zn
