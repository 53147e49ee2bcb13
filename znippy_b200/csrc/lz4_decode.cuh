// LZ4 frame decoder (LZ4 Frame format 1.6.x + LZ4 block format), one team (CTA) per blob.
//
// Second payload codec of codec::decompress_into (znippy-common/src/codec.rs:67-78; OpenZL "wraps zstd+lz4",
// README.md:10).  Written from the public format descriptions.  Thread 0 walks the token stream of a block and emits
// sequences {literal offset, ll, ml, distance} into the shared batch; the team executes them with the same
// cooperative copy engine as the Zstandard path (zstd_decode.cuh: exec_batch).  Linked blocks need nothing special:
// the whole output of the blob is the window.  The header checksum byte is verified here; block / content checksums
// (XXH32) are stepped over and verified where the row's digest is compared (xxh_verify.cuh).
#pragma once
#include "zstd_decode.cuh"

namespace zn {
namespace lz {

// XXH32 of a short input (len < 16), as needed for the frame-descriptor checksum
ZN_HD uint32_t xxh32_short(const uint8_t* p, uint32_t len) {
  const uint32_t P1 = 2654435761u, P2 = 2246822519u, P3 = 3266489917u, P4 = 668265263u, P5 = 374761393u;
  (void)P1;
  uint32_t h = P5 + len;
  uint32_t i = 0;
  for (; i + 4 <= len; i += 4) {
    h += ld32le(p + i) * P3;
    h = ((h << 17) | (h >> 15)) * P4;
  }
  for (; i < len; i++) {
    h += (uint32_t)p[i] * P5;
    h = ((h << 11) | (h >> 21)) * P1;
  }
  h ^= h >> 15; h *= P2;
  h ^= h >> 13; h *= P3;
  h ^= h >> 16;
  return h;
}

struct BlockCursor {  // thread 0 only
  uint32_t ip;       // next input byte inside the block
  uint32_t out_pos;  // output cursor (blob-relative), ahead of the executors by one batch
  uint32_t done;
};

// Parses up to kSeqBatch sequences of the block p[0..len).  Thread 0 only.
ZN_HD uint32_t parse_batch(DecShared* sh, const uint8_t* p, uint32_t len, BlockCursor& c, uint32_t out_limit,
                           uint32_t win_start, uint32_t* count_out) {
  uint32_t n = 0;
  while (n < kSeqBatch && !c.done) {
    if (c.ip >= len) return S_DECODE_ERROR;
    const uint32_t token = p[c.ip++];
    uint32_t ll = token >> 4;
    if (ll == 15) {
      uint32_t b;
      do {
        if (c.ip >= len) return S_DECODE_ERROR;
        b = p[c.ip++];
        ll += b;
        if (ll > 0x7FFFFFFFu) return S_DECODE_ERROR;
      } while (b == 255);
    }
    if (ll > len - c.ip) return S_DECODE_ERROR;
    if (ll > out_limit - c.out_pos) return S_DST_TOO_SMALL;
    SeqRec r;
    r.lit = c.ip; r.ll = ll; r.ml = 0; r.off = 0;
    c.ip += ll;
    c.out_pos += ll;
    if (c.ip == len) {  // last sequence: literals only
      c.done = 1;
      sh->ring[n++] = r;
      break;
    }
    if (len - c.ip < 2) return S_DECODE_ERROR;
    const uint32_t off = ld16le(p + c.ip);
    c.ip += 2;
    if (off == 0 || off > c.out_pos - win_start) return S_DECODE_ERROR;
    uint32_t ml = token & 15;
    if (ml == 15) {
      uint32_t b;
      do {
        if (c.ip >= len) return S_DECODE_ERROR;
        b = p[c.ip++];
        ml += b;
        if (ml > 0x7FFFFFFFu) return S_DECODE_ERROR;
      } while (b == 255);
    }
    ml += 4;
    if (ml > out_limit - c.out_pos) return S_DST_TOO_SMALL;
    r.ml = ml; r.off = off;
    c.out_pos += ml;
    sh->ring[n++] = r;
  }
  *count_out = n;
  return S_OK;
}

// One LZ4 block.  Team-uniform.  `win_start` = lowest output position a match may reach.
ZN_HD uint32_t decode_block(const Team& t, DecShared* sh, const uint8_t* p, uint32_t len, uint8_t* out,
                            uint32_t out_limit, uint32_t win_start, zs::ExecState& es) {
  if (len == 0) return S_DECODE_ERROR;
  BlockCursor c;
  c.ip = 0; c.out_pos = es.pos; c.done = 0;
  for (;;) {
    if (t.tid == 0) {
      uint32_t n = 0;
      sh->err_seq = parse_batch(sh, p, len, c, out_limit, win_start, &n);
      sh->rep_pub[0] = n;
      sh->rep_pub[1] = c.done;
    }
    team_sync(t);
    if (sh->err_seq != S_OK) return sh->err_seq;
    const uint32_t n = sh->rep_pub[0], done = sh->rep_pub[1];
    zs::exec_batch(t, sh, n, out, p, -1, es);
    team_sync(t);
    if (!es.bulk) es.wm = es.pos;
    if (done) break;
  }
  return S_OK;
}

// `hook` only decides where to stop (zs::stop_here): after the data block that reaches a StopAt's stop, S_OK without
// the content-size comparison.
template <class Hook>
ZN_HD uint32_t decode_frame(const Team& t, DecShared* sh, const uint8_t* src, uint32_t src_len, uint8_t* out,
                            uint32_t cap, uint32_t* produced, const Hook& hook) {
  *produced = 0;
  if (src_len < 7) return S_DECODE_ERROR;
  if (ld32le(src) != 0x184D2204u) return S_UNSUPPORTED;
  const uint32_t flg = src[4], bd = src[5];
  if ((flg >> 6) != 1 || (flg & 0x02)) return S_UNSUPPORTED;
  const uint32_t indep = (flg >> 5) & 1, bchk = (flg >> 4) & 1, has_csize = (flg >> 3) & 1, cchk = (flg >> 2) & 1;
  if (flg & 1) return S_UNSUPPORTED;  // dictionary id
  if (bd & 0x8F) return S_UNSUPPORTED;
  const uint32_t bs = (bd >> 4) & 7;
  if (bs < 4) return S_UNSUPPORTED;
  const uint32_t bmax = 1u << (8 + 2 * bs);
  uint32_t ip = 6;
  uint64_t csize = 0;
  if (has_csize) {
    if (src_len < ip + 8) return S_DECODE_ERROR;
    csize = (uint64_t)ld32le(src + ip) | ((uint64_t)ld32le(src + ip + 4) << 32);
    ip += 8;
  }
  if (src_len < ip + 1) return S_DECODE_ERROR;
  if ((uint8_t)(xxh32_short(src + 4, ip - 4) >> 8) != src[ip]) return S_DECODE_ERROR;
  ip += 1;
  zs::ExecState es;
  es.pos = 0; es.wm = 0; es.bulk = 0;
  for (;;) {
    if (src_len - ip < 4) return S_DECODE_ERROR;
    const uint32_t w = ld32le(src + ip);
    ip += 4;
    if (w == 0) break;
    const uint32_t raw = w >> 31, n = w & 0x7FFFFFFFu;
    if (n > bmax || n > src_len - ip) return S_DECODE_ERROR;
    if (raw) {
      if (n > cap - es.pos) return S_DST_TOO_SMALL;
      team_copy(t, out + es.pos, src + ip, n);
      es.pos += n;
    } else {
      const uint32_t room = cap - es.pos;
      const uint32_t limit = es.pos + (room < bmax ? room : bmax);
      const uint32_t rc = decode_block(t, sh, src + ip, n, out, limit, indep ? es.pos : 0u, es);
      if (rc != S_OK) return rc;
    }
    *produced = es.pos;
    if (zs::stop_here(hook, es.pos)) return S_OK;
    ip += n;
    if (bchk) {
      if (src_len - ip < 4) return S_DECODE_ERROR;
      ip += 4;
    }
  }
  if (cchk) {
    if (src_len - ip < 4) return S_DECODE_ERROR;
    ip += 4;
  }
  *produced = es.pos;
  if (has_csize && csize != (uint64_t)es.pos) return S_SIZE_MISMATCH;
  return S_OK;
}
ZN_HD uint32_t decode_frame(const Team& t, DecShared* sh, const uint8_t* src, uint32_t src_len, uint8_t* out,
                            uint32_t cap, uint32_t* produced) {
  return decode_frame(t, sh, src, src_len, out, cap, produced, zs::NoHook{});
}

}  // namespace lz

// Entry point of the codec for one blob: picks the payload format by its magic number.
// `predef` (team-uniform, owned by the caller across blobs) records which sequence tables in `sh` hold the
// predefined distributions, so consecutive blobs do not copy them again.
template <class Hook>
ZN_HD uint32_t decode_blob(const Team& t, DecShared* sh, const uint8_t* src, uint32_t src_len, uint8_t* out,
                           uint32_t cap, uint8_t* lit_scratch, uint32_t& predef, uint32_t* produced, Hook& hook) {
  *produced = 0;
  if (src_len >= 4 && ld32le(src) == 0x184D2204u) {
    const uint32_t rc = lz::decode_frame(t, sh, src, src_len, out, cap, produced, hook);
    if (rc == S_OK) {  // the LZ4 path has no per-block hook: everything is hashed at the end
      zs::ExecState es;
      es.pos = *produced; es.wm = 0; es.bulk = 1;  // force a full memory barrier (and bulk drain) in finish()
      hook.finish(t, es);
    }
    return rc;
  }
  return zs::decode_frames(t, sh, src, src_len, out, cap, lit_scratch, predef, produced, hook);
}
ZN_HD uint32_t decode_blob(const Team& t, DecShared* sh, const uint8_t* src, uint32_t src_len, uint8_t* out,
                           uint32_t cap, uint8_t* lit_scratch, uint32_t& predef, uint32_t* produced) {
  zs::NoHook h;
  return decode_blob(t, sh, src, src_len, out, cap, lit_scratch, predef, produced, h);
}

// A raw LZ4 block (LZ4_compress_default output): no header at all, the index supplies both sizes.
ZN_HD uint32_t decode_lz4_block(const Team& t, DecShared* sh, const uint8_t* src, uint32_t src_len, uint8_t* out,
                                uint32_t cap, uint32_t* produced) {
  zs::ExecState es;
  es.pos = 0; es.wm = 0; es.bulk = 0;
  *produced = 0;
  const uint32_t rc = lz::decode_block(t, sh, src, src_len, out, cap, 0u, es);
  *produced = es.pos;
  return rc;
}

}  // namespace zn
