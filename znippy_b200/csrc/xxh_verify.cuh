// Content and block checksums of Zstandard and LZ4 frames, on both sides of the codec.
//
// Read side: libzstd and liblz4 reject a frame whose stored checksum disagrees with its bytes; so does this path.  Right
// before a row's blake3 digest is compared (the tree kernels) the frames of a decoded row are walked exactly as the
// decoder consumed them (xxh_row_walk), and every stored checksum the walk meets is checked:
//   Zstandard (RFC 8878 §3.1.1): Content_Checksum = low 32 bits of XXH64(frame content, 0), per frame that sets the flag;
//   LZ4 (frame format 1.6.x):    Block_Checksum = XXH32(stored block bytes, 0) when FLG.B.Checksum is set, and
//                                Content_Checksum = XXH32(decoded content, 0) when FLG.C.Checksum is set.
// A mismatch turns the row's status into S_DECODE_ERROR.  Rows whose frame announces no checksum cost one header read and
// no launch.  k_b3_tree_small checks its rows on one thread each (xxh_row_bad); k_b3_tree_large checks a row with its
// whole CTA: one thread lists the spans, the warps hash them (xxh_warp), so the block checksums of an LZ4 frame are
// hashed in parallel.
//
// Write side (ZN_CODEC_CHECKSUM): k_slice_xxh hashes every source slice with one warp (xxh_warp) and the assembly
// kernels store the result behind the frame.
//
// XXH64 / XXH32 are four independent accumulator chains over 32 / 16-byte stripes and strictly serial along the
// stripes: the chains are all the parallelism one hashed span has.
#pragma once
#include "common.cuh"

namespace zn {

namespace xx {
constexpr uint64_t P1 = 0x9E3779B185EBCA87ull, P2 = 0xC2B2AE3D27D4EB4Full, P3 = 0x165667B19E3779F9ull, P4 = 0x85EBCA77C2B2AE63ull,
                   P5 = 0x27D4EB2F165667C5ull;
constexpr uint32_t Q1 = 2654435761u, Q2 = 2246822519u, Q3 = 3266489917u, Q4 = 668265263u, Q5 = 374761393u;  // XXH32
ZN_D uint64_t rotl(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
ZN_D uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
ZN_D uint64_t round(uint64_t acc, uint64_t in) { return rotl(acc + in * P2, 31) * P1; }
ZN_D uint32_t round32(uint32_t acc, uint32_t in) { return rotl32(acc + in * Q2, 13) * Q1; }
ZN_D uint64_t merge(uint64_t h, uint64_t v) { return (h ^ round(0, v)) * P1 + P4; }
ZN_D uint64_t rd64(const uint8_t* p) {
  if ((reinterpret_cast<uintptr_t>(p) & 7u) == 0) return *reinterpret_cast<const uint64_t*>(p);
  uint64_t v = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) v |= (uint64_t)p[i] << (8 * i);
  return v;
}
ZN_D uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

// Initial accumulator k (0..3) of the four chains, seed 0
ZN_D uint64_t init64(uint32_t k) { return k == 0 ? P1 + P2 : k == 1 ? P2 : k == 2 ? 0ull : 0ull - P1; }
ZN_D uint32_t init32(uint32_t k) { return k == 0 ? Q1 + Q2 : k == 1 ? Q2 : k == 2 ? 0u : 0u - Q1; }
// The four chains merged into the hash state (input of at least one stripe)
ZN_D uint64_t converge64(uint64_t v1, uint64_t v2, uint64_t v3, uint64_t v4) {
  uint64_t h = rotl(v1, 1) + rotl(v2, 7) + rotl(v3, 12) + rotl(v4, 18);
  h = merge(h, v1); h = merge(h, v2); h = merge(h, v3); h = merge(h, v4);
  return h;
}
ZN_D uint32_t converge32(uint32_t v1, uint32_t v2, uint32_t v3, uint32_t v4) {
  return rotl32(v1, 1) + rotl32(v2, 7) + rotl32(v3, 12) + rotl32(v4, 18);
}

// The bytes [q, end) behind the last stripe, then the avalanche.  `h` already holds the input length; r.rd64 / rd32 /
// rd8 read the input at a byte position.
template <class R>
ZN_D uint64_t finish64(uint64_t h, uint64_t q, uint64_t end, const R& r) {
  while (q + 8 <= end) { h ^= round(0, r.rd64(q)); h = rotl(h, 27) * P1 + P4; q += 8; }
  if (q + 4 <= end) { h ^= (uint64_t)r.rd32(q) * P1; h = rotl(h, 23) * P2 + P3; q += 4; }
  while (q < end) { h ^= (uint64_t)r.rd8(q++) * P5; h = rotl(h, 11) * P1; }
  h ^= h >> 33; h *= P2; h ^= h >> 29; h *= P3; h ^= h >> 32;
  return h;
}
template <class R>
ZN_D uint32_t finish32(uint32_t h, uint64_t q, uint64_t end, const R& r) {
  while (q + 4 <= end) { h += r.rd32(q) * Q3; h = rotl32(h, 17) * Q4; q += 4; }
  while (q < end) { h += (uint32_t)r.rd8(q++) * Q5; h = rotl32(h, 11) * Q1; }
  h ^= h >> 15; h *= Q2; h ^= h >> 13; h *= Q3; h ^= h >> 16;
  return h;
}

struct PtrRd {  // input in (global) memory
  const uint8_t* p;
  ZN_D uint64_t rd64(uint64_t i) const { return xx::rd64(p + i); }
  ZN_D uint32_t rd32(uint64_t i) const { return xx::rd32(p + i); }
  ZN_D uint32_t rd8(uint64_t i) const { return p[i]; }
};

}  // namespace xx

// XXH64(p[0..len), 0) by ONE thread: the four accumulators are independent chains, so one thread interleaving them is as
// fast as four lanes with one each.
ZN_D uint64_t xxh64_1(const uint8_t* p, uint64_t len) {
  uint64_t h = xx::P5;
  const uint64_t done = len / 32 * 32;
  if (len >= 32) {
    uint64_t v1 = xx::init64(0), v2 = xx::init64(1), v3 = xx::init64(2), v4 = xx::init64(3);
    for (const uint8_t* q = p; q < p + done; q += 32) {
      v1 = xx::round(v1, xx::rd64(q));
      v2 = xx::round(v2, xx::rd64(q + 8));
      v3 = xx::round(v3, xx::rd64(q + 16));
      v4 = xx::round(v4, xx::rd64(q + 24));
    }
    h = xx::converge64(v1, v2, v3, v4);
  }
  return xx::finish64(h + len, done, len, xx::PtrRd{p});
}
// XXH32(p[0..len), 0) by one thread
ZN_D uint32_t xxh32_1(const uint8_t* p, uint64_t len) {
  uint32_t h = xx::Q5;
  const uint64_t done = len / 16 * 16;
  if (len >= 16) {
    uint32_t v1 = xx::init32(0), v2 = xx::init32(1), v3 = xx::init32(2), v4 = xx::init32(3);
    for (const uint8_t* q = p; q < p + done; q += 16) {
      v1 = xx::round32(v1, xx::rd32(q));
      v2 = xx::round32(v2, xx::rd32(q + 4));
      v3 = xx::round32(v3, xx::rd32(q + 8));
      v4 = xx::round32(v4, xx::rd32(q + 12));
    }
    h = xx::converge32(v1, v2, v3, v4);
  }
  return xx::finish32(h + (uint32_t)len, done, len, xx::PtrRd{p});
}

#if defined(__CUDACC__)
// ---- staged hash: one warp, the input streamed into a shared-memory ring by coalesced 16-byte cp.async copies, three
// tiles in flight.  Lanes 0..3 each run one accumulator chain over the staged stripes (a chain is serial, so more
// lanes cannot help one span; the loads no longer sit on the chain's critical path).  The tail and the avalanche run
// on every lane from the ring, so the result is warp-uniform.
constexpr uint32_t kXxhTile = 512;            // bytes per pipeline stage: one 16-byte copy per lane
constexpr uint32_t kXxhRing = 4 * kXxhTile;   // shared memory per warp: the tile being hashed, the one before it (a
                                              // stripe may straddle the two) and two in flight

namespace xx {
struct RingRd {  // logical byte i of the span sits at ring byte (a + i) mod kXxhRing
  const uint32_t* w;
  uint32_t a;
  ZN_D uint32_t rd32(uint64_t i) const {
    const uint32_t x = a + (uint32_t)i, k = x >> 2;
    const uint32_t lo = w[k & (kXxhRing / 4 - 1)], hi = w[(k + 1) & (kXxhRing / 4 - 1)];
    return __funnelshift_r(lo, hi, (x & 3u) * 8u);
  }
  ZN_D uint64_t rd64(uint64_t i) const { return (uint64_t)rd32(i) | (uint64_t)rd32(i + 4) << 32; }
  ZN_D uint32_t rd8(uint64_t i) const { return reinterpret_cast<const uint8_t*>(w)[(a + (uint32_t)i) & (kXxhRing - 1)]; }
};
}  // namespace xx

// XXH<Bits>(p[0..len), 0), Bits = 64 or 32, by one warp: all 32 lanes call with the same arguments and get the hash.
// ring = this warp's kXxhRing bytes of shared memory, 16-byte aligned.  p may have any alignment: the copies cover the
// 16-byte granules the span touches, never a byte outside them.
template <int Bits>
ZN_D uint64_t xxh_warp(const uint8_t* p, uint64_t len, uint8_t* ring, uint32_t lane) {
  constexpr uint32_t S = Bits == 64 ? 32u : 16u, W = S / 4;  // stripe bytes, bytes per chain per stripe
  const uint32_t a = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 15u);
  const uint8_t* base = p - a;
  const uint64_t span = a + len, tiles = (span + kXxhTile - 1) / kXxhTile, full = len / S * S;
  const xx::RingRd rd{reinterpret_cast<const uint32_t*>(ring), a};
  auto issue = [&](uint64_t t) {
    const uint64_t off = t * kXxhTile + lane * 16u;
    if (t < tiles && off < span) cp_async16(ring + (off & (kXxhRing - 1)), base + off);
    cp_async_commit();
  };
  __syncwarp();  // the ring's previous span is fully read
  issue(0); issue(1); issue(2);
  uint64_t v = Bits == 64 ? xx::init64(lane & 3u) : xx::init32(lane & 3u);
  uint64_t pos = 0;  // stripes before pos are in the chains
#pragma unroll 1
  for (uint64_t t = 0; t < tiles; t++) {
    cp_async_wait<2>();
    __syncwarp();
    const uint64_t landed = (t + 1) * kXxhTile < span ? (t + 1) * kXxhTile - a : len;
    const uint64_t stop = landed < full ? landed / S * S : full;
    if (lane < 4) {
#pragma unroll 4
      for (uint64_t s = pos; s < stop; s += S) {
        if (Bits == 64) v = xx::round(v, rd.rd64(s + lane * W));
        else v = xx::round32((uint32_t)v, rd.rd32(s + lane * W));
      }
    }
    if (stop > pos) pos = stop;
    __syncwarp();  // tile t - 1 is no longer read: its slot takes tile t + 3
    issue(t + 3);
  }
  cp_async_wait<0>();
  __syncwarp();
  const uint64_t v1 = __shfl_sync(0xFFFFFFFFu, v, 0), v2 = __shfl_sync(0xFFFFFFFFu, v, 1), v3 = __shfl_sync(0xFFFFFFFFu, v, 2),
                 v4 = __shfl_sync(0xFFFFFFFFu, v, 3);
  uint64_t h;
  if (Bits == 64) h = xx::finish64((len >= S ? xx::converge64(v1, v2, v3, v4) : xx::P5) + len, full, len, rd);
  else h = xx::finish32((len >= S ? xx::converge32((uint32_t)v1, (uint32_t)v2, (uint32_t)v3, (uint32_t)v4) : xx::Q5) + (uint32_t)len,
                        full, len, rd);
  __syncwarp();  // every lane is done with the ring
  return h;
}
#endif

// ---- read side: the checksums of one decoded row
// Calls emit(p, len, bits, want) for every stored checksum of the row's frames, in frame order, as long as emit returns
// true: XXH<bits>(p[0..len)) must have the low 32 bits `want`.  The walk follows what the decoder consumed: for a
// Zstandard row every frame (skippable frames skipped) up to the first one that does not parse, walked only when the
// first frame announces a checksum (libzstd writes the flag per stream, not per frame); for an LZ4 row its one frame.
template <class Emit>
ZN_D void xxh_row_walk(const BlobDesc& d, const uint8_t* __restrict__ blobs_base, const uint8_t* __restrict__ out_base, Emit& emit) {
  if (!(d.flags & F_COMPRESSED) || (d.flags & F_LZ4_BLOCK)) return;  // raw LZ4 blocks carry no checksum
  if (d.src_len < 9 || d.src_len >= 0xFFFFFFF0ull) return;
  const uint8_t* src = blobs_base + d.src_off;
  const uint32_t src_len = (uint32_t)d.src_len;
  const uint8_t* out = out_base + d.dst_off;
  if (xx::rd32(src) == 0x184D2204u) {  // LZ4 frame (lz::decode_frame)
    const uint32_t flg = src[4], bchk = (flg >> 4) & 1, cchk = (flg >> 2) & 1;
    if (!bchk && !cchk) return;
    uint32_t ip = 6 + ((flg >> 3) & 1 ? 8u : 0u) + 1u;
    for (;;) {
      if (ip > src_len || src_len - ip < 4) return;
      const uint32_t w = xx::rd32(src + ip), n = w & 0x7FFFFFFFu;
      ip += 4;
      if (w == 0) break;
      if (n > src_len - ip) return;
      ip += n;
      if (bchk) {
        if (src_len - ip < 4) return;
        if (!emit(src + ip - n, (uint64_t)n, 32u, xx::rd32(src + ip))) return;
        ip += 4;
      }
    }
    if (cchk && src_len - ip >= 4) emit(out, d.dst_cap, 32u, xx::rd32(src + ip));
    return;
  }
  uint32_t ip = 0, frames = 0;
  uint64_t opos = 0;
  while (ip + 5 <= src_len) {
    const uint32_t magic = xx::rd32(src + ip);
    if ((magic & 0xFFFFFFF0u) == 0x184D2A50u) {  // skippable frame
      if (src_len - ip < 8) break;
      const uint32_t sz = xx::rd32(src + ip + 4);
      if (sz > src_len - ip - 8) break;
      ip += 8 + sz;
      continue;
    }
    if (magic != 0xFD2FB528u) break;  // not a frame: nothing to do here
    const uint32_t fhd = src[ip + 4], fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, did_flag = fhd & 3;
    const bool checksum = (fhd >> 2) & 1;
    if (frames == 0 && !checksum) break;  // the common case ends here
    uint32_t hp = ip + 5 + (single ? 0u : 1u) + (did_flag == 3 ? 4u : did_flag);
    const uint32_t fb = fcs_flag == 0 ? single : (fcs_flag == 1 ? 2u : (fcs_flag == 2 ? 4u : 8u));
    if (hp + fb > src_len) break;
    uint64_t fcs = ~0ull;
    if (fb) {
      fcs = 0;
      for (uint32_t i = 0; i < fb; i++) fcs |= (uint64_t)src[hp + i] << (8 * i);
      if (fb == 2) fcs += 256;
    }
    hp += fb;
    bool ok = false;
    for (;;) {  // block headers
      if (hp + 3 > src_len) break;
      const uint32_t bh = (uint32_t)src[hp] | (uint32_t)src[hp + 1] << 8 | (uint32_t)src[hp + 2] << 16;
      const uint32_t type = (bh >> 1) & 3u, size = bh >> 3;
      hp += 3;
      const uint32_t adv = type == 1 ? 1u : size;
      if (adv > src_len - hp) break;
      hp += adv;
      if (bh & 1u) { ok = true; break; }
    }
    if (!ok) break;
    uint32_t stored = 0;
    if (checksum) {
      if (hp + 4 > src_len) break;
      stored = xx::rd32(src + hp);
      hp += 4;
    }
    // content range of this frame: from its header, or — a lone frame without one — everything the row decoded to
    uint64_t flen;
    if (fcs != ~0ull) flen = fcs;
    else if (frames == 0 && hp == src_len) flen = d.dst_cap;
    else break;
    if (opos + flen > d.dst_cap) break;
    if (checksum && !emit(out + opos, flen, 64u, stored)) return;
    opos += flen;
    ip = hp;
    frames++;
  }
}

// One thread, one decoded row: true when a checksum of the row's frames disagrees with its bytes.
struct XxhScalarCheck {
  bool bad = false;
  ZN_D bool operator()(const uint8_t* p, uint64_t len, uint32_t bits, uint32_t want) {
    bad = (bits == 64 ? (uint32_t)xxh64_1(p, len) : xxh32_1(p, len)) != want;
    return !bad;
  }
};
ZN_D bool xxh_row_bad(const BlobDesc& d, const uint8_t* __restrict__ blobs_base, const uint8_t* __restrict__ out_base) {
  XxhScalarCheck c;
  xxh_row_walk(d, blobs_base, out_base, c);
  return c.bad;
}

}  // namespace zn
