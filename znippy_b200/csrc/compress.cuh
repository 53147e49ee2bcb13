// Per-slice compressors (write side): LZ4 blocks and Zstandard compressed blocks, one warp per block.
//
// Replaces CompressCtx::compress_into (znippy-common/src/codec.rs:43-55) as called from the barrel / worker bodies
// (znippy-compress/src/stream_packer.rs:230, slot_packer.rs:570).  The reference reaches zstd level 19 through OpenZL
// (not vendored); this is a GPU-shaped design written from the LZ4 block/frame and RFC 8878 formats:
//
//   * a slice is cut into independent blocks (LZ4: 64 KiB frame blocks; zstd: 128 KiB blocks) and every block of
//     every slice of the batch is compressed by its own warp — 8 MiB slices give 64-128 blocks each, so a 500 MiB
//     batch is ~4-8 k warps of work;
//   * match finder: the 32 lanes hash 32 consecutive positions at once into a shared-memory table, ballot picks the
//     first lane with a verified 4-byte match, and the match is extended 128 bytes per step across the warp;
//   * zstd blocks carry raw literals and sequences coded with the PREDEFINED FSE tables (modes byte 0), never a
//     repeat-offset code, so blocks do not depend on each other and stock libzstd decodes the frame;
//     the match window of a block is primed with the tail of the previous block (the window is the whole slice),
//     except in seekable slices, where every block is a frame of its own and starts without history;
//   * every block lands in a scratch slot; a second kernel lays the blocks out back to back behind the frame header.
//
// Everything here is warp-uniform code over a `Warp` abstraction (32 lanes on the device, 1 lane on the host) so the
// format logic is exercised on the CPU against stock libzstd / liblz4 (tests/host_emu).
#pragma once
#include <cmath>
#ifndef ZN_CP
#define ZN_CP_BEGIN() do {} while (0)
#define ZN_CP(i) do {} while (0)
#endif
#include "bitio.cuh"
#include "zstd_tables.cuh"

namespace zn {
namespace cz {

struct Warp {
  uint32_t lane, n;
};

#if defined(__CUDA_ARCH__)
ZN_D uint32_t w_ballot(const Warp&, bool p) { return __ballot_sync(0xFFFFFFFFu, p); }
ZN_D uint32_t w_shfl(const Warp&, uint32_t v, uint32_t src) { return __shfl_sync(0xFFFFFFFFu, v, src); }
ZN_D void w_sync(const Warp&) { __syncwarp(); }
ZN_D uint32_t w_shfl_xor(const Warp&, uint32_t v, uint32_t d) { return __shfl_xor_sync(0xFFFFFFFFu, v, d); }
ZN_D uint32_t ffs32(uint32_t v) { return (uint32_t)__ffs((int)v); }
ZN_D void w_count(uint32_t* p) { atomicAdd(p, 1u); }
ZN_D void w_or(uint32_t* p, uint32_t v) { if (v) atomicOr(p, v); }
ZN_D uint32_t w_max(const Warp&, uint32_t v) { return __reduce_max_sync(0xFFFFFFFFu, v); }
ZN_D uint32_t w_min(const Warp&, uint32_t v) { return __reduce_min_sync(0xFFFFFFFFu, v); }
ZN_D uint32_t w_shfl_up(const Warp&, uint32_t v, uint32_t d) { return __shfl_up_sync(0xFFFFFFFFu, v, d); }
// unaligned 32-bit little-endian load from shared memory through two aligned words (the buffer has slack behind it)
ZN_D uint32_t ld32s(const uint8_t* p) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
  return __funnelshift_r(w[0], w[1], ((uint32_t)reinterpret_cast<uintptr_t>(p) & 3u) * 8u);
}
// exclusive prefix sum over the lanes; *total = sum over the warp
ZN_D uint32_t w_excl_scan(const Warp& w, uint32_t v, uint32_t* total) {
  uint32_t x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d); if ((int)w.lane >= d) x += y; }
  *total = __shfl_sync(0xFFFFFFFFu, x, 31);
  return x - v;
}
constexpr bool kOnDevice = true;
ZN_D uint32_t w_sum(const Warp&, uint32_t v) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
  return v;
}
#else
inline uint32_t w_ballot(const Warp&, bool p) { return p ? 1u : 0u; }
inline uint32_t w_shfl(const Warp&, uint32_t v, uint32_t) { return v; }
inline void w_sync(const Warp&) {}
inline uint32_t w_shfl_xor(const Warp&, uint32_t v, uint32_t) { return v; }
inline uint32_t ffs32(uint32_t v) { return v ? (uint32_t)__builtin_ffs((int)v) : 0u; }
inline void w_count(uint32_t* p) { (*p)++; }
inline uint32_t w_sum(const Warp&, uint32_t v) { return v; }
inline void w_or(uint32_t* p, uint32_t v) { *p |= v; }
inline uint32_t w_max(const Warp&, uint32_t v) { return v; }
inline uint32_t w_min(const Warp&, uint32_t v) { return v; }
inline uint32_t w_shfl_up(const Warp&, uint32_t v, uint32_t) { return v; }
inline uint32_t ld32s(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline uint32_t w_excl_scan(const Warp&, uint32_t v, uint32_t* total) { *total = v; return 0; }
constexpr bool kOnDevice = false;
#endif

ZN_HD uint32_t hash4(uint32_t v, uint32_t hlog) { return (v * 2654435761u) >> (32 - hlog); }

constexpr uint32_t kLz4Block = 64u * 1024u;
constexpr uint32_t kLz4Slot = kLz4Block + kLz4Block / 255u + 32u;  // worst-case LZ4 block
constexpr uint32_t kLz4HashLog = 12;                                 // 4096 x u16 = 8 KiB per warp
constexpr uint32_t kZstdHashLog = 12;                                // default table: 4096 x u16 = 8 KiB per warp (Win::kHashLog)
#ifndef ZN_LAZY_MATCH_W
#define ZN_LAZY_MATCH_W 4
#define ZN_LAZY_SKIP_W 16
#endif
constexpr uint32_t kLazyMatchWeight = ZN_LAZY_MATCH_W, kLazySkipWeight = ZN_LAZY_SKIP_W;
#ifndef ZN_MIN_MATCH
#define ZN_MIN_MATCH 4
#endif
constexpr uint32_t kZstdMinMatch = ZN_MIN_MATCH;                     // shortest match the zstd parser emits
#ifndef ZN_INSERT_SPAN
#define ZN_INSERT_SPAN 64
#endif
constexpr uint32_t kZstdInsertSpan = ZN_INSERT_SPAN;                 // positions of a long match entered beyond the round
constexpr uint32_t kLazyProbeWords = 5;                              // words compared beyond the 4 verified bytes
constexpr uint32_t kLazyProbe = 4u + 4u * kLazyProbeWords;                                  // bytes each candidate lane compares before the warp votes
// Window geometry of the zstd match finder (see zstd_compress_block): W fresh bytes per window, H bytes of history
// kept when it slides.  Shared memory per warp = H + W + 80 bytes + the 8 KiB table, which sets how many warps an
// SM holds — the compressor is latency-bound, so speed follows the warp count and ratio follows W + H.
#ifndef ZN_FAST_HASHLOG
#define ZN_FAST_HASHLOG 12
#endif
template <uint32_t W, uint32_t H, uint32_t HL>
struct Win {
  static constexpr uint32_t kBytes = W, kHist = H;
  static constexpr uint32_t kHashLog = HL;           // 2^HL u16 table entries
  static constexpr uint32_t kData = H + W + 16u;   // staged bytes (multiple of 16; + alignment slop)
  static constexpr uint32_t kSmem = kData + 64u;   // + slack for the word-wise probes
  static_assert(kData % 16u == 0 && kData < 65535u && H + 160u < W, "window geometry");
};
using WinFast = Win<16384, 4096, ZN_FAST_HASHLOG>;    // levels <= 2
using WinMid = Win<32768, 8192, 12>;     // levels 3..9
using WinHigh = Win<49152, 14336, 12>;   // levels >= 10
constexpr uint32_t kZstdMaxSeq = 32768;                              // sequences per 128 KiB block (min match 4)
#ifndef ZN_CBLOCK
#define ZN_CBLOCK kZstdBlockMax
#endif
constexpr uint32_t kZstdCBlock = ZN_CBLOCK;                          // input bytes per compressed block (<= 128 KiB)
constexpr uint32_t kZstdHalf = kZstdCBlock + 64u;                  // one staging region
constexpr uint32_t kZstdSlot = 2u * kZstdHalf;                       // region A: raw literals (+ sequences); region B: Huffman payload

// Length of the common prefix of a[0..max) and b[0..max), found 4 bytes per lane per step.
ZN_HD uint32_t match_extend(const Warp& w, const uint8_t* a, const uint8_t* b, uint32_t max) {
  uint32_t len = 0;
  for (;;) {
    const uint32_t idx = len + 4u * w.lane;
    uint32_t neq;  // number of equal leading bytes in this lane's word, 0..4
    if (idx + 4u <= max) {
      const uint32_t x = ld32le(a + idx) ^ ld32le(b + idx);
      neq = x == 0 ? 4u : ((ffs32(x) - 1u) >> 3);
    } else {
      neq = 0;
      while (idx + neq < max && a[idx + neq] == b[idx + neq]) neq++;
    }
    const uint32_t stop = w_ballot(w, neq < 4u);
    if (stop) {
      const uint32_t first = ffs32(stop) - 1u;
      return len + 4u * first + w_shfl(w, neq, first);
    }
    len += 4u * w.n;
  }
}


// Common prefix length of a[0..lim) and b[0..lim), lim <= 4*K, one lane.  The device version works on aligned words
// (K+1 loads per side, all in flight together) and may read up to 4*K+7 bytes past a / b: the caller guarantees slack.
template <int K>
ZN_HD uint32_t prefix_words(const uint8_t* a, const uint8_t* b, uint32_t lim) {
#if defined(__CUDA_ARCH__)
  const uint32_t* wa = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(a) & ~(uintptr_t)3);
  const uint32_t* wb = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(b) & ~(uintptr_t)3);
  const uint32_t sa = ((uint32_t)reinterpret_cast<uintptr_t>(a) & 3u) * 8u, sb = ((uint32_t)reinterpret_cast<uintptr_t>(b) & 3u) * 8u;
  uint32_t ra[K + 1], rb[K + 1];
#pragma unroll
  for (int k = 0; k <= K; k++) { ra[k] = wa[k]; rb[k] = wb[k]; }
  uint32_t n = 4u * K;
#pragma unroll
  for (int k = K - 1; k >= 0; k--) {
    const uint32_t x = __funnelshift_r(ra[k], ra[k + 1], sa) ^ __funnelshift_r(rb[k], rb[k + 1], sb);
    if (x) n = 4u * k + (((uint32_t)__ffs((int)x) - 1u) >> 3);
  }
  return n < lim ? n : lim;
#else
  uint32_t n = 0;
  while (n < lim && a[n] == b[n]) n++;
  return n;
#endif
}

// dst[0..n) = src[0..n), spread over the warp (byte granular; the compressed side is small by construction)
ZN_HD void w_copy(const Warp& w, uint8_t* dst, const uint8_t* src, uint32_t n) {
  for (uint32_t i = w.lane; i < n; i += w.n) dst[i] = src[i];
}

// LZ4 length extension: value v (>= 0) as 255,255,...,rest.  Returns bytes written.
ZN_HD uint32_t lz4_put_len(const Warp& w, uint8_t* dst, uint32_t v) {
  const uint32_t n255 = v / 255u;
  for (uint32_t i = w.lane; i < n255; i += w.n) dst[i] = 255;
  if (w.lane == 0) dst[n255] = (uint8_t)(v - n255 * 255u);
  return n255 + 1u;
}

// ------------------------------------------------------------------------------------------------- LZ4 block
// Compresses in[0..n) (n <= 64 KiB) into out (capacity kLz4Slot).  tab = 4096 x u16 (shared memory), zeroed here.
// Returns the compressed size (may exceed n for incompressible input; the caller then stores the block raw).
ZN_HD uint32_t lz4_compress_block(const Warp& w, const uint8_t* in, uint32_t n, uint8_t* out, uint16_t* tab) {
  for (uint32_t i = w.lane; i < (1u << kLz4HashLog); i += w.n) tab[i] = 0;
  w_sync(w);
  uint32_t op = 0, anchor = 0, pos = 0;
  if (n >= 13) {
    const uint32_t mflimit = n - 12, matchlimit = n - 5;
    while (pos < mflimit) {
      const uint32_t p = pos + w.lane;
      const bool valid = p < mflimit;
      const uint32_t v = valid ? ld32le(in + p) : 0u;
      const uint32_t h = hash4(v, kLz4HashLog);
      const uint32_t cand = valid ? tab[h] : 0u;
      const bool ok = valid && cand < p && ld32le(in + cand) == v;
      const uint32_t m = w_ballot(w, ok);
      const uint32_t f = m ? ffs32(m) - 1u : w.n;
      // insert only the positions up to the match: later lanes are looked up again next step (or lie inside the
      // match) and must not find themselves in the table instead of their real candidate
      w_sync(w);
      if (valid && w.lane <= f) tab[h] = (uint16_t)p;
      w_sync(w);
      if (!m) {
        pos += w.n;
        continue;
      }
      const uint32_t mp = pos + f, mc = w_shfl(w, cand, f);
      const uint32_t ml = 4u + match_extend(w, in + mp + 4, in + mc + 4, matchlimit - (mp + 4));
      // ---- emit: token, literal length, literals, offset, match length
      const uint32_t ll = mp - anchor, mlc = ml - 4u;
      if (w.lane == 0) out[op] = (uint8_t)(((ll < 15u ? ll : 15u) << 4) | (mlc < 15u ? mlc : 15u));
      op += 1;
      if (ll >= 15u) op += lz4_put_len(w, out + op, ll - 15u);
      w_copy(w, out + op, in + anchor, ll);
      op += ll;
      if (w.lane == 0) {
        out[op] = (uint8_t)(mp - mc);
        out[op + 1] = (uint8_t)((mp - mc) >> 8);
      }
      op += 2;
      if (mlc >= 15u) op += lz4_put_len(w, out + op, mlc - 15u);
      pos = anchor = mp + ml;
    }
  }
  // last sequence: literals only
  const uint32_t ll = n - anchor;
  if (w.lane == 0) out[op] = (uint8_t)((ll < 15u ? ll : 15u) << 4);
  op += 1;
  if (ll >= 15u) op += lz4_put_len(w, out + op, ll - 15u);
  w_copy(w, out + op, in + anchor, ll);
  op += ll;
  w_sync(w);
  return op;
}

// LZ4 frame header for a slice of `content` bytes (15 bytes): independent 64 KiB blocks, content size present, and
// with `checksum` (ZN_CODEC_CHECKSUM) the content checksum flag.
ZN_HD uint32_t lz4_frame_header(uint8_t* dst, uint64_t content, bool checksum = false) {
  dst[0] = 0x04; dst[1] = 0x22; dst[2] = 0x4D; dst[3] = 0x18;
  dst[4] = checksum ? 0x6C : 0x68;  // version 01, B.Indep, C.Size[, C.Checksum]
  dst[5] = 0x40;  // 64 KiB blocks
  for (int i = 0; i < 8; i++) dst[6 + i] = (uint8_t)(content >> (8 * i));
  // XXH32 of the 10 descriptor bytes (len < 16 path)
  const uint32_t P1 = 2654435761u, P2 = 2246822519u, P3 = 3266489917u, P4 = 668265263u, P5 = 374761393u;
  uint32_t h = P5 + 10u;
  for (int i = 0; i < 8; i += 4) {
    h += ld32le(dst + 4 + i) * P3;
    h = ((h << 17) | (h >> 15)) * P4;
  }
  for (int i = 8; i < 10; i++) {
    h += (uint32_t)dst[4 + i] * P5;
    h = ((h << 11) | (h >> 21)) * P1;
  }
  h ^= h >> 15; h *= P2;
  h ^= h >> 13; h *= P3;
  h ^= h >> 16;
  dst[14] = (uint8_t)(h >> 8);
  return 15;
}

// ------------------------------------------------------------------------------------------------- FSE encoding
// Compression tables for the three predefined distributions (RFC 8878 §3.1.1.3.2.2.1), built once on the host.
struct FseCTable {
  uint16_t state[512];     // next-state table (table log <= 9)
  int32_t delta_nb[53];    // per symbol: (maxBitsOut << 16) - minStatePlus
  int32_t delta_state[53]; // per symbol: first state slot - count
  uint32_t log;
};
struct PredefCTables {
  FseCTable ll, of, ml;
};
struct FseBuildScratch {
  int32_t cumul[54];
  uint8_t symtab[512];
};

// One thread.  norm sums to 1 << log (entries of -1 count as 1); log 0 with a single symbol of count 1 gives the
// zero-bit table the RLE mode needs.
ZN_HD void fse_build_ctable(FseCTable* ct, const int16_t* norm, int nsym, int log, FseBuildScratch* sc) {
  const int size = 1 << log, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
  int32_t* cumul = sc->cumul;
  uint8_t* symtab = sc->symtab;
  int high = size - 1;
  cumul[0] = 0;
  for (int s = 0; s < nsym; s++) {
    if (norm[s] == -1) { cumul[s + 1] = cumul[s] + 1; symtab[high--] = (uint8_t)s; }
    else cumul[s + 1] = cumul[s] + norm[s];
  }
  int pos = 0;
  for (int s = 0; s < nsym; s++)
    for (int i = 0; i < norm[s]; i++) {
      symtab[pos] = (uint8_t)s;
      do pos = (pos + step) & mask; while (pos > high);
    }
  for (int u = 0; u < size; u++) { const int s = symtab[u]; ct->state[cumul[s]++] = (uint16_t)(size + u); }
  int total = 0;
  for (int s = 0; s < nsym; s++) {
    const int n = norm[s];
    if (n == 0) { ct->delta_nb[s] = ((log + 1) << 16) - (1 << log); ct->delta_state[s] = 0; }
    else if (n == -1 || n == 1) { ct->delta_nb[s] = (log << 16) - (1 << log); ct->delta_state[s] = total - 1; total++; }
    else {
      const int max_bits = log - hibit32((uint32_t)(n - 1));
      const int min_plus = n << max_bits;
      ct->delta_nb[s] = (max_bits << 16) - min_plus;
      ct->delta_state[s] = total - n;
      total += n;
    }
  }
  ct->log = (uint32_t)log;
}

inline void build_predef_ctables(PredefCTables* p) {
  FseBuildScratch sc;
  fse_build_ctable(&p->ll, zs::kLLDefault, 36, 6, &sc);
  fse_build_ctable(&p->of, zs::kOFDefault, 29, 5, &sc);
  fse_build_ctable(&p->ml, zs::kMLDefault, 53, 6, &sc);
}

#if defined(__CUDACC__)
__device__ PredefCTables g_predef_c;  // filled by zn_ctx_create
#endif
#if defined(__CUDA_ARCH__)
ZN_D const PredefCTables* predef_ctables() { return &g_predef_c; }
#else
inline const PredefCTables* predef_ctables() {
  static PredefCTables p;
  static bool init = false;
  if (!init) { build_predef_ctables(&p); init = true; }
  return &p;
}
#endif

// forward bit writer (the decoder reads it backwards): bits accumulate LSB first
struct BitWriter {
  uint8_t* p;
  uint64_t acc;
  uint32_t nbits;
  ZN_HD void add(uint32_t v, uint32_t n) {  // n <= 32
    acc |= (uint64_t)(v & (n >= 32 ? 0xFFFFFFFFu : ((1u << n) - 1u))) << nbits;
    nbits += n;
  }
  ZN_HD void flush() {  // keeps < 8 bits pending
    while (nbits >= 8) { *p++ = (uint8_t)acc; acc >>= 8; nbits -= 8; }
  }
  ZN_HD void close() {  // end mark
    add(1, 1);
    flush();
    if (nbits) { *p++ = (uint8_t)acc; acc = 0; nbits = 0; }
  }
};

// code of a literal length / match length: the code c with base[c] <= v < base[c] + 2^bits[c]
ZN_HD uint32_t len_code(uint32_t v, const uint32_t* base, const uint8_t* bits, uint32_t direct, uint32_t ncodes) {
  if (v < direct + base[0]) return v - base[0];
  uint32_t c = direct;
  while (c + 1 < ncodes && v >= base[c + 1]) c++;
  (void)bits;
  return c;
}

struct FseCState {
  uint32_t value;
  ZN_HD void init(const FseCTable* ct, uint32_t sym) {
    const int32_t dnb = ct->delta_nb[sym];
    const uint32_t nb = (uint32_t)(dnb + (1 << 15)) >> 16;
    const uint32_t v = (nb << 16) - (uint32_t)dnb;
    value = ct->state[(int32_t)(v >> nb) + ct->delta_state[sym]];
  }
  ZN_HD void encode(BitWriter& bw, const FseCTable* ct, uint32_t sym) {
    const uint32_t nb = (uint32_t)((int32_t)value + ct->delta_nb[sym]) >> 16;
    bw.add(value, nb);
    value = ct->state[(int32_t)(value >> nb) + ct->delta_state[sym]];
  }
  ZN_HD void flush(BitWriter& bw, const FseCTable* ct) { bw.add(value, ct->log); }
};

// packed sequence: ll | ml << 20 | off << 40 (ll, ml < 2^20; off < 2^24: the long effort reaches back 8 MiB)
ZN_HD uint64_t seq_pack(uint32_t ll, uint32_t ml, uint32_t off) { return (uint64_t)ll | ((uint64_t)ml << 20) | ((uint64_t)off << 40); }

// ---- FSE table description (RFC 8878 §4.1.1): the writer mirroring fse_read_ncount of the decoder.
// alphabet = index of the last symbol with a non-zero count + 1.  Returns bytes written (< 96).
ZN_HD uint32_t fse_write_ncount(uint8_t* out, const int16_t* norm, uint32_t alphabet, uint32_t log) {
  uint8_t* p = out;
  const int size = 1 << log;
  uint32_t bits = log - 5u, nacc = 4;
  int remaining = size + 1, threshold = size, nb = (int)log + 1;
  uint32_t sym = 0;
  bool prev0 = false;
  while (sym < alphabet && remaining > 1) {
    if (prev0) {  // run of zero-probability symbols: 2-bit repeat counts
      uint32_t start = sym;
      while (sym < alphabet && !norm[sym]) sym++;
      if (sym == alphabet) break;
      while (sym >= start + 24) {
        start += 24;
        bits += 0xFFFFu << nacc;
        p[0] = (uint8_t)bits; p[1] = (uint8_t)(bits >> 8); p += 2;
        bits >>= 16;
      }
      while (sym >= start + 3) { start += 3; bits += 3u << nacc; nacc += 2; }
      bits += (sym - start) << nacc;
      nacc += 2;
      if (nacc > 16) { p[0] = (uint8_t)bits; p[1] = (uint8_t)(bits >> 8); p += 2; bits >>= 16; nacc -= 16; }
    }
    int count = norm[sym++];
    const int mx = (2 * threshold - 1) - remaining;
    remaining -= count < 0 ? -count : count;
    count++;
    if (count >= threshold) count += mx;
    bits += (uint32_t)count << nacc;
    nacc += (uint32_t)nb;
    nacc -= (count < mx) ? 1u : 0u;
    prev0 = (count == 1);
    while (remaining < threshold) { nb--; threshold >>= 1; }
    if (nacc > 16) { p[0] = (uint8_t)bits; p[1] = (uint8_t)(bits >> 8); p += 2; bits >>= 16; nacc -= 16; }
  }
  p[0] = (uint8_t)bits; p[1] = (uint8_t)(bits >> 8);
  p += (nacc + 7) / 8;
  return (uint32_t)(p - out);
}

// Scales a histogram (total > 0, >= 2 symbols present) to sum 1 << log with every present symbol >= 1.
ZN_HD void fse_normalize(int16_t* norm, const uint32_t* cnt, uint32_t nsym, uint32_t total, uint32_t log) {
  const uint32_t size = 1u << log;
  uint32_t sum = 0, largest = 0;
  for (uint32_t s = 0; s < nsym; s++) {
    uint32_t q = 0;
    if (cnt[s]) {
      const uint64_t scaled = (uint64_t)cnt[s] * size;
      q = (uint32_t)(scaled / total);
      const uint32_t rem = (uint32_t)(scaled % total);
      if (q == 0) q = 1;
      else if (q < 8 && 2u * rem > total + total / (q + 1)) q++;  // small shares round to nearest-ish
      if (cnt[s] > cnt[largest]) largest = s;
    }
    norm[s] = (int16_t)q;
    sum += q;
  }
  if (sum <= size) { norm[largest] = (int16_t)(norm[largest] + (size - sum)); return; }
  for (uint32_t excess = sum - size; excess; excess--) {  // shave the biggest shares
    uint32_t big = 0;
    for (uint32_t s = 1; s < nsym; s++) if (norm[s] > norm[big]) big = s;
    norm[big]--;
  }
}

// cost in bits of coding the histogram with a normalised table (-1 entries count as 1)
ZN_HD float fse_cost(const uint32_t* cnt, const int16_t* norm, uint32_t nsym, uint32_t log) {
  float c = (float)log;  // final state flush
  for (uint32_t s = 0; s < nsym; s++)
    if (cnt[s]) { const int q = norm[s] < 0 ? 1 : norm[s]; c += (float)cnt[s] * ((float)log - log2f((float)q)); }
  return c;
}

struct SeqScratch {
  FseCTable ct[3];
  FseBuildScratch bs[3];
  uint32_t cnt[3][53];
  int16_t norm[3][54];
  uint8_t hdr[3][96];
  uint32_t mode[3], hlen[3];
  uint32_t sbits[3][32];   // per chunk: FSE state bits of each sequence, value << 8 | count
  int32_t dnb[3][32];      // per chunk: delta_nb / delta_state of each sequence's three codes, fetched by the lanes so
  int32_t dst[3][32];      //            that the serial state chains only wait for the state table itself
  uint32_t bitbuf[88];     // per chunk: the assembled bitstream (<= 31 carried bits + 32 x 81: state bits 9 + 8 + 9,
                           // extra bits 16 + 16 + 23 for an offset value < 2^24), 2 623 of 2 816 bits
};

// packed sequence after pass 1: ll:17 | ml - 4:17 | offset value:24 | ll code:6   (ml is 4 .. 131072; the ml code is
// recomputed in pass 2, which leaves room for offset values up to 8 MiB + 3)
ZN_HD uint64_t seq_pack2(uint32_t ll, uint32_t ml, uint32_t ofv, uint32_t lc) {
  return (uint64_t)ll | ((uint64_t)(ml - 4u) << 17) | ((uint64_t)ofv << 34) | ((uint64_t)lc << 58);
}

// Sequences section, called by the whole warp.  Offsets become repeat codes where the history written by THIS block
// allows it (blocks are compressed independently, so the history inherited from the previous block is treated as
// unknown); each of the three code tables is sent FSE-compressed, RLE or predefined, whichever is estimated cheapest.
// The lanes load 32 sequences at a time (one coalesced access) and hand them to the serial parts through shuffles;
// lanes 0-2 build one table each; lane 0 writes the bitstream.  Rewrites seqs[] in place.  Returns (on every lane)
// bytes written, or 0 when the section would exceed `limit` bytes (the block is then stored raw); the writer
// overshoots `limit` by < 16 bytes.
ZN_HD uint32_t zstd_encode_sequences(const Warp& w, uint8_t* dst, uint64_t* seqs, uint32_t nseq, uint32_t limit, SeqScratch* sc) {
  uint8_t* p = dst;
  if (w.lane == 0) {
    if (nseq < 128) *p++ = (uint8_t)nseq;
    else if (nseq < 0x7F00) { *p++ = (uint8_t)((nseq >> 8) + 128); *p++ = (uint8_t)nseq; }
    else { *p++ = 255; *p++ = (uint8_t)(nseq - 0x7F00); *p++ = (uint8_t)((nseq - 0x7F00) >> 8); }
  }
  if (nseq == 0) return w_shfl(w, (uint32_t)(p - dst), 0);
  // pass 1: offset values + code histograms
  for (uint32_t i = w.lane; i < 3 * 53; i += w.n) sc->cnt[i / 53][i % 53] = 0;
  w_sync(w);
  uint32_t r0 = 0, r1 = 0, r2 = 0;  // 0 = not known to this block; tracked identically by every lane
  for (uint32_t base = 0; base < nseq; base += w.n) {
    const uint32_t k = base + w.lane;
    const uint64_t s = k < nseq ? seqs[k] : 0ull;
    const uint32_t ll = (uint32_t)(s & 0xFFFFF), ml = (uint32_t)((s >> 20) & 0xFFFFF), off = (uint32_t)(s >> 40);
    const uint32_t here = nseq - base < w.n ? nseq - base : w.n;
    uint32_t v = 0;
    // Fast path: a repeat code needs an offset equal to one of the three before it (r0 - 1 included), which is rare
    // and which every lane can test against its three predecessors at once.
    bool maybe = false;
    if (w.n > 1) {
      const uint32_t o1 = w_shfl_up(w, off, 1), o2 = w_shfl_up(w, off, 2), o3 = w_shfl_up(w, off, 3);
      const uint32_t q1 = w.lane >= 1 ? o1 : (w.lane == 0 ? r0 : 0u);
      const uint32_t q2 = w.lane >= 2 ? o2 : (w.lane == 1 ? r0 : r1);
      const uint32_t q3 = w.lane >= 3 ? o3 : (w.lane == 2 ? r0 : (w.lane == 1 ? r1 : r2));
      maybe = k < nseq && (off == q1 || off == q2 || off == q3 || off + 1u == q1);
    }
    if (w.n > 1 && !w_ballot(w, maybe)) {
      v = off + 3u;
      if (here >= 3) { r0 = w_shfl(w, off, here - 1); r1 = w_shfl(w, off, here - 2); r2 = w_shfl(w, off, here - 3); }
      else if (here == 2) { r2 = r0; r0 = w_shfl(w, off, 1); r1 = w_shfl(w, off, 0); }
      else { r2 = r1; r1 = r0; r0 = w_shfl(w, off, 0); }
    } else
    for (uint32_t j = 0; j < here; j++) {
      const uint32_t llj = w_shfl(w, ll, j), offj = w_shfl(w, off, j);
      uint32_t vj;
      if (llj) {
        if (offj == r0) vj = 1;
        else if (offj == r1) { vj = 2; r1 = r0; r0 = offj; }
        else if (offj == r2) { vj = 3; r2 = r1; r1 = r0; r0 = offj; }
        else { vj = offj + 3u; r2 = r1; r1 = r0; r0 = offj; }
      } else {
        if (offj == r1) { vj = 1; r1 = r0; r0 = offj; }
        else if (offj == r2) { vj = 2; r2 = r1; r1 = r0; r0 = offj; }
        else if (r0 > 1 && offj == r0 - 1u) { vj = 3; r2 = r1; r1 = r0; r0 = offj; }
        else { vj = offj + 3u; r2 = r1; r1 = r0; r0 = offj; }
      }
      if (j == w.lane) v = vj;
    }
    if (k < nseq) {
      const uint32_t lc = len_code(ll, zs::kLLBase, zs::kLLBits, 16, 36), mc = len_code(ml, zs::kMLBase, zs::kMLBits, 32, 53);
      seqs[k] = seq_pack2(ll, ml, v, lc);
      w_count(&sc->cnt[0][lc]);
      w_count(&sc->cnt[1][hibit32(v)]);
      w_count(&sc->cnt[2][mc]);
    }
  }
  w_sync(w);
  // table choice: lane t builds table t
  const PredefCTables* pd = predef_ctables();
  const FseCTable* dct[3] = {&pd->ll, &pd->of, &pd->ml};
  for (uint32_t t = w.lane; t < 3; t += w.n) {
    const int16_t* dnorm = t == 0 ? zs::kLLDefault : (t == 1 ? zs::kOFDefault : zs::kMLDefault);
    const uint32_t dsym = t == 0 ? 36u : (t == 1 ? 29u : 53u), dlog = t == 1 ? 5u : 6u, maxlog = t == 1 ? 8u : 9u;
    sc->mode[t] = 0;
    sc->hlen[t] = 0;
    uint32_t present = 0, last = 0;
    for (uint32_t q = 0; q < 53; q++) if (sc->cnt[t][q]) { present++; last = q; }
    const float c_pre = last < dsym ? fse_cost(sc->cnt[t], dnorm, dsym, dlog) : 1e30f;
    if (present == 1) {
      if (c_pre <= 8.f) continue;
      for (uint32_t q = 0; q <= last; q++) sc->norm[t][q] = 0;
      sc->norm[t][last] = 1;
      fse_build_ctable(&sc->ct[t], sc->norm[t], (int)last + 1, 0, &sc->bs[t]);
      sc->hdr[t][0] = (uint8_t)last;
      sc->hlen[t] = 1;
      sc->mode[t] = 1;
      continue;
    }
    uint32_t log = nseq > 1 ? (uint32_t)hibit32(nseq - 1) : 0u;
    log = log > 7 ? log - 2 : 5;
    if (log > maxlog) log = maxlog;
    while ((1u << log) < 2u * present && log < maxlog) log++;
    fse_normalize(sc->norm[t], sc->cnt[t], last + 1, nseq, log);
    const uint32_t hl = fse_write_ncount(sc->hdr[t], sc->norm[t], last + 1, log);
    const float c_fse = 8.f * (float)hl + fse_cost(sc->cnt[t], sc->norm[t], last + 1, log);
    if (c_fse >= c_pre) continue;
    fse_build_ctable(&sc->ct[t], sc->norm[t], (int)last + 1, (int)log, &sc->bs[t]);
    sc->hlen[t] = hl;
    sc->mode[t] = 2;
  }
  w_sync(w);
  const FseCTable* ct[3];
  for (int t = 0; t < 3; t++) ct[t] = sc->mode[t] ? &sc->ct[t] : dct[t];
  if (w.lane == 0) {
    *p++ = (uint8_t)((sc->mode[0] << 6) | (sc->mode[1] << 4) | (sc->mode[2] << 2));
    for (int t = 0; t < 3; t++) for (uint32_t i = 0; i < sc->hlen[t]; i++) *p++ = sc->hdr[t][i];
  }
  // pass 2: the bitstream, last sequence first, 32 sequences per step.  Lanes 0-2 each advance one FSE state chain
  // (the only serial dependence); then every lane assembles the bits of its own sequence — state bits of OF, ML, LL,
  // then the extra bits of LL, ML, OF — at the bit offset given by a warp prefix sum, and the finished words leave
  // as a byte-coalesced store.
  uint32_t over = 0;
  if (w.lane == 0) over = (uint32_t)(p - dst) > limit ? 1u : 0u;
  over = w_shfl(w, over, 0);
  p = dst + w_shfl(w, (uint32_t)(p - dst), 0);
  for (uint32_t i = w.lane; i < 88; i += w.n) sc->bitbuf[i] = 0;
  uint32_t stv[kOnDevice ? 1 : 3] = {0};
  uint32_t carry = 0;  // bits pending in bitbuf[0]
  w_sync(w);
  for (uint32_t chunk = (nseq + w.n - 1) / w.n; chunk-- > 0 && !over;) {
    const uint32_t base = chunk * w.n;
    const uint32_t here = nseq - base < w.n ? nseq - base : w.n;
    const bool mine = w.lane < here;
    const uint64_t sj = mine ? seqs[base + (here - 1u - w.lane)] : 0ull;  // lane i takes the i-th sequence in coding order
    const uint32_t ll = (uint32_t)(sj & 0x1FFFF), ml = 4u + (uint32_t)((sj >> 17) & 0x1FFFF), ofv = (uint32_t)((sj >> 34) & 0xFFFFFF);
    const uint32_t lc = (uint32_t)(sj >> 58), mc = len_code(ml, zs::kMLBase, zs::kMLBits, 32, 53);
    const uint32_t oc = mine ? (uint32_t)hibit32(ofv) : 0u;
    if (mine) {
      sc->dnb[0][w.lane] = ct[0]->delta_nb[lc]; sc->dst[0][w.lane] = ct[0]->delta_state[lc];
      sc->dnb[1][w.lane] = ct[1]->delta_nb[oc]; sc->dst[1][w.lane] = ct[1]->delta_state[oc];
      sc->dnb[2][w.lane] = ct[2]->delta_nb[mc]; sc->dst[2][w.lane] = ct[2]->delta_state[mc];
    }
    w_sync(w);
    for (uint32_t t = w.lane; t < 3; t += w.n) {
      const uint16_t* stt = ct[t]->state;
      uint32_t v = stv[kOnDevice ? 0 : t];
      uint32_t i = 0;
      if (base + here == nseq) {  // the very first sequence coded only seeds the state (FseCState::init)
        const int32_t dnb = sc->dnb[t][0];
        const uint32_t nb = (uint32_t)(dnb + (1 << 15)) >> 16;
        v = stt[(int32_t)(((nb << 16) - (uint32_t)dnb) >> nb) + sc->dst[t][0]];
        sc->sbits[t][0] = 0;
        i = 1;
      }
      for (; i < here; i++) {
        const uint32_t nb = (uint32_t)((int32_t)v + sc->dnb[t][i]) >> 16;
        sc->sbits[t][i] = ((v & ((1u << nb) - 1u)) << 8) | nb;
        v = stt[(int32_t)(v >> nb) + sc->dst[t][i]];
      }
      stv[kOnDevice ? 0 : t] = v;
    }
    w_sync(w);
    uint64_t a = 0, b = 0;
    uint32_t na = 0, nbx = 0;
    if (mine) {
      const uint32_t so_ = sc->sbits[1][w.lane], sm_ = sc->sbits[2][w.lane], sl_ = sc->sbits[0][w.lane];
      a = (uint64_t)(so_ >> 8);
      na = so_ & 255u;
      a |= (uint64_t)(sm_ >> 8) << na;
      na += sm_ & 255u;
      a |= (uint64_t)(sl_ >> 8) << na;
      na += sl_ & 255u;
      const uint32_t llb = zs::kLLBits[lc], mlb = zs::kMLBits[mc];
      b = (uint64_t)(ll - zs::kLLBase[lc]);
      b |= (uint64_t)(ml - zs::kMLBase[mc]) << llb;
      b |= (uint64_t)(ofv - (1u << oc)) << (llb + mlb);
      nbx = llb + mlb + oc;
    }
    uint32_t tot = 0;
    const uint32_t at = carry + w_excl_scan(w, na + nbx, &tot);
    if (mine) {
      for (int part = 0; part < 2; part++) {
        const uint64_t v = part ? b : a;
        const uint32_t n = part ? nbx : na, off = part ? at + na : at;
        if (!n) continue;
        const uint32_t wi = off >> 5, sh = off & 31u;
        const uint64_t lo = v << sh;
        w_or(&sc->bitbuf[wi], (uint32_t)lo);
        if (n + sh > 32) w_or(&sc->bitbuf[wi + 1], (uint32_t)(lo >> 32));
        if (n + sh > 64) w_or(&sc->bitbuf[wi + 2], (uint32_t)(v >> (64u - sh)));
      }
    }
    w_sync(w);
    const uint32_t bits = carry + tot, nw = bits >> 5;
    if ((uint32_t)(p - dst) + 4u * nw > limit) { over = 1; break; }
    for (uint32_t i = w.lane; i < 4u * nw; i += w.n) p[i] = (uint8_t)(sc->bitbuf[i >> 2] >> (8u * (i & 3u)));
    const uint32_t keep = sc->bitbuf[nw];
    w_sync(w);
    for (uint32_t i = w.lane; i <= nw; i += w.n) sc->bitbuf[i] = i == 0 ? keep : 0u;
    w_sync(w);
    p += 4u * nw;
    carry = bits & 31u;
  }
  // final states: ML, OF, LL, then the end mark
  const uint32_t st_ll = kOnDevice ? w_shfl(w, stv[0], 0) : stv[0];
  const uint32_t st_of = kOnDevice ? w_shfl(w, stv[0], 1) : stv[kOnDevice ? 0 : 1];
  const uint32_t st_ml = kOnDevice ? w_shfl(w, stv[0], 2) : stv[kOnDevice ? 0 : 2];
  uint32_t total = 0;
  if (w.lane == 0 && !over) {
    BitWriter bw{p, (uint64_t)sc->bitbuf[0], carry};
    bw.add(st_ml, ct[2]->log);
    bw.flush();
    bw.add(st_of, ct[1]->log);
    bw.flush();
    bw.add(st_ll, ct[0]->log);
    bw.close();
    total = (uint32_t)(bw.p - dst);
  }
  return w_shfl(w, total, 0);
}


// ------------------------------------------------------------------------------------------------- Huffman literals
// Literals section with Huffman-compressed literals (RFC 8878 §3.1.1.3.1, type 2): tree described by direct 4-bit
// weights, 1 or 4 streams.  scratch = >= 1024 words of shared memory (the idle match-finder table).
// Returns the section size written at dst, or 0 when Huffman coding is not applicable / does not pay.
constexpr uint32_t kHufMaxBits = 11;

// Code lengths (<= 11 bits) and canonical codes from the histogram, whole warp; fills nb[256], code[256] and
// res[0] = max_bits (0 = not applicable), res[1] = last symbol present.  The merge loop finds the two lightest
// roots with two warp min-reductions per step.
ZN_HD void huf_build(const Warp& w, const uint32_t* cnt, uint8_t* nb, uint16_t* code, uint32_t* work, uint32_t* res) {
  uint32_t my_present = 0, my_last = 0;
  for (uint32_t s = w.lane; s < 256; s += w.n) { nb[s] = 0; if (cnt[s]) { my_present++; my_last = s; } }
  const uint32_t present = w_sum(w, my_present), last = w_max(w, my_last);
  if (w.lane == 0) { res[0] = 0; res[1] = last; }
  w_sync(w);
  if (present < 2) return;
  uint32_t* wt = work;                                         // 512 entries
  uint16_t* parent = reinterpret_cast<uint16_t*>(work + 512);  // 512 entries
  uint16_t* leaf_of = parent + 512;                            // present entries: symbol of leaf i
  if (w.lane == 0) {
    uint32_t k = 0;
    for (uint32_t s = 0; s <= last; s++) if (cnt[s]) { wt[k] = cnt[s]; parent[k] = 0xFFFF; leaf_of[k] = (uint16_t)s; k++; }
  }
  w_sync(w);
  const uint32_t nleaf = present;
  uint32_t nn = nleaf;
  for (uint32_t step = 0; step + 1 < nleaf; step++) {
    uint32_t k1 = 0xFFFFFFFFu, k2 = 0xFFFFFFFFu;  // this lane's two lightest roots, as weight << 9 | node
    for (uint32_t i = w.lane; i < nn; i += w.n) {
      if (parent[i] != 0xFFFF) continue;
      const uint32_t key = (wt[i] << 9) | i;
      if (key < k1) { k2 = k1; k1 = key; }
      else if (key < k2) k2 = key;
    }
    const uint32_t ka = w_min(w, k1);
    const uint32_t kb = w_min(w, k1 == ka ? k2 : k1);
    w_sync(w);
    if (w.lane == 0) {
      wt[nn] = (ka >> 9) + (kb >> 9);
      parent[nn] = 0xFFFF;
      parent[ka & 511u] = parent[kb & 511u] = (uint16_t)nn;
    }
    nn++;
    w_sync(w);
  }
  uint32_t my_maxd = 0;
  for (uint32_t i = w.lane; i < nleaf; i += w.n) {
    uint32_t d = 0;
    for (uint32_t j = i; parent[j] != 0xFFFF; j = parent[j]) d++;
    nb[leaf_of[i]] = (uint8_t)(d > 255 ? 255 : d);
    my_maxd = d > my_maxd ? d : my_maxd;
  }
  uint32_t maxd = w_max(w, my_maxd);
  w_sync(w);
  if (w.lane != 0) return;
  if (maxd > kHufMaxBits) {  // length-limit: clamp, then repair the Kraft sum (units of 2^-11)
    int32_t total = 0;
    for (uint32_t s = 0; s <= last; s++)
      if (nb[s]) { if (nb[s] > kHufMaxBits) nb[s] = kHufMaxBits; total += 1 << (kHufMaxBits - nb[s]); }
    while (total > (1 << kHufMaxBits)) {  // lengthen the cheapest code that is not yet at the limit
      uint32_t best = 256;
      for (uint32_t s = 0; s <= last; s++)
        if (nb[s] && nb[s] < kHufMaxBits && (best == 256 || nb[s] > nb[best] || (nb[s] == nb[best] && cnt[s] < cnt[best]))) best = s;
      if (best == 256) return;
      total -= 1 << (kHufMaxBits - nb[best] - 1);
      nb[best]++;
    }
    while (total < (1 << kHufMaxBits)) {  // give the slack back to the most frequent symbol it fits
      uint32_t best = 256;
      for (uint32_t s = 0; s <= last; s++)
        if (nb[s] > 1 && total + (1 << (kHufMaxBits - nb[s])) <= (1 << kHufMaxBits) && (best == 256 || cnt[s] > cnt[best])) best = s;
      if (best == 256) return;
      total += 1 << (kHufMaxBits - nb[best]);
      nb[best]--;
    }
    maxd = 0;
    for (uint32_t s = 0; s <= last; s++) maxd = nb[s] > maxd ? nb[s] : maxd;
  }
  // canonical codes in the decoder's order: ascending weight (longest codes first), ascending symbol within a weight
  uint32_t pos = 0;
  for (uint32_t wgt = 1; wgt <= maxd; wgt++) {
    const uint32_t len = maxd + 1 - wgt;
    for (uint32_t s = 0; s <= last; s++)
      if (nb[s] == len) { code[s] = (uint16_t)(pos >> (wgt - 1)); pos += 1u << (wgt - 1); }
  }
  res[0] = pos == (1u << maxd) ? maxd : 0u;
}

// Huffman weights, FSE-compressed (RFC 8878 §4.2.1.1: table log <= 6, two interleaved states, header byte = size of the
// stream < 128).  One thread.  Writes header byte + table description + stream at `out` and returns the byte count, or 0
// when this form is not possible (fewer than two distinct weights, or 128 bytes and more).
ZN_HD uint32_t huf_write_weights_fse(uint8_t* out, const uint8_t* wts, uint32_t n, uint32_t* scratch) {
  if (n < 2) return 0;
  uint32_t* cnt = scratch;                                    // 16 words
  int16_t* norm = reinterpret_cast<int16_t*>(scratch + 16);   // 16 entries
  FseCTable* ct = reinterpret_cast<FseCTable*>(scratch + 32);
  FseBuildScratch* bs = reinterpret_cast<FseBuildScratch*>(scratch + 32 + (sizeof(FseCTable) + 3) / 4);
  for (int k = 0; k < 16; k++) cnt[k] = 0;
  uint32_t maxw = 0, present = 0;
  for (uint32_t k = 0; k < n; k++) { if (!cnt[wts[k]]++) present++; if (wts[k] > maxw) maxw = wts[k]; }
  if (present < 2) return 0;
  int hb = hibit32(n - 1) - 2;
  const uint32_t log = hb < 5 ? 5u : (hb > 6 ? 6u : (uint32_t)hb);
  fse_normalize(norm, cnt, maxw + 1, n, log);
  const uint32_t hdr = fse_write_ncount(out + 1, norm, maxw + 1, log);
  fse_build_ctable(ct, norm, (int)maxw + 1, (int)log, bs);
  BitWriter bw{out + 1 + hdr, 0, 0};
  FseCState s1, s2;
  uint32_t k = n;
  if (n & 1u) {
    s1.init(ct, wts[--k]);
    s2.init(ct, wts[--k]);
    s1.encode(bw, ct, wts[--k]);
    bw.flush();
  } else {
    s2.init(ct, wts[--k]);
    s1.init(ct, wts[--k]);
  }
  while (k > 0) {
    s2.encode(bw, ct, wts[--k]);
    s1.encode(bw, ct, wts[--k]);
    bw.flush();
  }
  s2.flush(bw, ct);
  bw.flush();
  s1.flush(bw, ct);
  bw.close();
  const uint32_t size = (uint32_t)(bw.p - (out + 1));
  if (size == 0 || size >= 128) return 0;
  out[0] = (uint8_t)size;
  return 1 + size;
}

ZN_HD uint32_t zstd_huf_literals(const Warp& w, const uint8_t* lit, uint32_t nlit, uint8_t* dst, uint32_t* scratch) {
  if (nlit < 64) return 0;
  uint32_t* cnt = scratch;                                        // [0, 256)
  uint8_t* nb = reinterpret_cast<uint8_t*>(scratch + 256);        // 256 bytes
  uint16_t* code = reinterpret_cast<uint16_t*>(scratch + 320);    // 256 x u16
  uint32_t* pub = scratch + 448;                                  // mailbox: [0] max_bits, [1] last_sym, [2..5] stream bits
  uint32_t* work = scratch + 464;                                 // tree construction (< 1100 words)
  for (uint32_t i = w.lane; i < 256; i += w.n) cnt[i] = 0;
  w_sync(w);
  for (uint32_t i = w.lane; i < nlit; i += w.n) w_count(&cnt[lit[i]]);
  w_sync(w);
  huf_build(w, cnt, nb, code, work, pub);
  w_sync(w);
  const uint32_t maxbits = pub[0], last = pub[1];
  if (!maxbits) return 0;
  const uint32_t ns = nlit >= 256 ? 4u : 1u;
  const uint32_t seg = ns == 4 ? (nlit + 3) / 4 : nlit;
  uint32_t sbytes[4] = {0, 0, 0, 0};
  for (uint32_t k = 0; k < ns; k++) {  // exact stream sizes first, so that every stream is encoded in place
    const uint32_t lo = k * seg, hi = (k == ns - 1) ? nlit : lo + seg;
    uint32_t bits = 0;
    for (uint32_t i = lo + w.lane; i < hi; i += w.n) bits += nb[lit[i]];
    bits = w_sum(w, bits);
    sbytes[k] = (bits + 8) >> 3;  // + end marker, rounded up
  }
  const uint32_t nweights = last;  // symbols 0..last-1 explicit, `last` implied
  // tree description: direct 4-bit weights (<= 128 of them) or FSE-compressed weights, whichever is smaller
  uint8_t* tdesc = reinterpret_cast<uint8_t*>(scratch + 1600);  // <= 130 bytes
  if (w.lane == 0) {
    uint8_t* wts = reinterpret_cast<uint8_t*>(scratch + 1640);  // 256 bytes
    for (uint32_t i = 0; i < nweights; i++) wts[i] = nb[i] ? (uint8_t)(maxbits + 1 - nb[i]) : (uint8_t)0;
    const uint32_t direct = nweights <= 128 ? 1 + (nweights + 1) / 2 : 0u;
    uint32_t sz = huf_write_weights_fse(tdesc, wts, nweights, scratch + 1712);
    if (!sz || (direct && direct <= sz)) {
      sz = direct;
      if (direct) {
        tdesc[0] = (uint8_t)(127 + nweights);
        for (uint32_t i = 0; i < nweights; i += 2)
          tdesc[1 + i / 2] = (uint8_t)((wts[i] << 4) | (i + 1 < nweights ? wts[i + 1] : 0));
      }
    }
    pub[6] = sz;
  }
  w_sync(w);
  const uint32_t tree = pub[6];
  if (!tree) return 0;
  const uint32_t comp = tree + (ns == 4 ? 6u : 0u) + sbytes[0] + sbytes[1] + sbytes[2] + sbytes[3];
  uint32_t hdr, sf;
  if (ns == 1) { if (comp >= 1024) return 0; hdr = 3; sf = 0; }
  else if (nlit < 1024 && comp < 1024) { hdr = 3; sf = 1; }
  else if (nlit < 16384 && comp < 16384) { hdr = 4; sf = 2; }
  else { hdr = 5; sf = 3; }
  if (hdr + comp + 8 >= nlit) return 0;  // does not pay
  if (ns == 4 && (sbytes[0] > 0xFFFF || sbytes[1] > 0xFFFF || sbytes[2] > 0xFFFF)) return 0;
  if (w.lane == 0) {
    if (hdr == 3) { const uint32_t v = 2u | (sf << 2) | (nlit << 4) | (comp << 14); dst[0] = (uint8_t)v; dst[1] = (uint8_t)(v >> 8); dst[2] = (uint8_t)(v >> 16); }
    else if (hdr == 4) { const uint32_t v = 2u | (sf << 2) | (nlit << 4) | (comp << 18); dst[0] = (uint8_t)v; dst[1] = (uint8_t)(v >> 8); dst[2] = (uint8_t)(v >> 16); dst[3] = (uint8_t)(v >> 24); }
    else { const uint64_t v = 2ull | ((uint64_t)sf << 2) | ((uint64_t)nlit << 4) | ((uint64_t)comp << 22); for (int i = 0; i < 5; i++) dst[i] = (uint8_t)(v >> (8 * i)); }
    uint8_t* t = dst + hdr;
    for (uint32_t i = 0; i < tree; i++) t[i] = tdesc[i];
    if (ns == 4) {
      uint8_t* j = t + tree;
      j[0] = (uint8_t)sbytes[0]; j[1] = (uint8_t)(sbytes[0] >> 8); j[2] = (uint8_t)sbytes[1]; j[3] = (uint8_t)(sbytes[1] >> 8);
      j[4] = (uint8_t)sbytes[2]; j[5] = (uint8_t)(sbytes[2] >> 8);
    }
  }
  uint32_t soff[4];
  soff[0] = hdr + tree + (ns == 4 ? 6u : 0u);
  for (int k = 1; k < 4; k++) soff[k] = soff[k - 1] + sbytes[k - 1];
  for (uint32_t k = w.lane; k < ns; k += w.n) {  // one lane per stream; symbols go in last-to-first
    const uint32_t lo = k * seg, hi = (k == ns - 1) ? nlit : lo + seg;
    BitWriter bw{dst + soff[k], 0, 0};
    if (hi > lo) {  // aligned words, the next one fetched while the current one is coded
      const uintptr_t first = reinterpret_cast<uintptr_t>(lit + lo), lastb = reinterpret_cast<uintptr_t>(lit + hi - 1);
      const uint32_t* wp = reinterpret_cast<const uint32_t*>(lastb & ~(uintptr_t)3);
      const uint32_t* wlo = reinterpret_cast<const uint32_t*>(first & ~(uintptr_t)3);
      uint32_t cur = *wp;
      for (;;) {
        const uint32_t nxt = wp > wlo ? wp[-1] : 0u;
        const uintptr_t wb = reinterpret_cast<uintptr_t>(wp);
        const int top = (int)((lastb < wb + 3 ? lastb : wb + 3) - wb), bot = (int)((first > wb ? first : wb) - wb);
        for (int j = top; j >= bot; j--) {
          const uint32_t s = (cur >> (8 * j)) & 255u;
          bw.add(code[s], nb[s]);
          if (bw.nbits >= 32) bw.flush();
        }
        if (wp == wlo) break;
        wp--;
        cur = nxt;
      }
    }
    bw.close();
  }
  w_sync(w);
  return hdr + comp;
}

// ------------------------------------------------------------------------------------------------- zstd block payload
// Literals + sequences sections of one compressed block, whole warp: the block's nlit literals sit at stage + 3 and
// its nseq sequences in seqs (seq_pack).  scratch = shared memory of >= kPayloadScratch bytes (Huffman tables, then
// SeqScratch).  Huffman-compressed literals go to region B when that pays, raw literals stay in place (region A).
// Returns the payload size (the payload starts at stage + *payload_off), or 0 when the block should be stored raw.
constexpr uint32_t kPayloadScratch = 10240;
static_assert(sizeof(SeqScratch) <= kPayloadScratch, "SeqScratch outgrew the payload scratch");

ZN_HD uint32_t zstd_block_payload(const Warp& w, uint8_t* stage, uint32_t nlit, uint64_t* seqs, uint32_t nseq, uint32_t n,
                                  uint32_t* scratch, uint32_t* payload_off) {
  uint8_t* lit = stage + 3;
  uint8_t* regB = stage + kZstdHalf;
  const uint32_t hsz = zstd_huf_literals(w, lit, nlit, regB, scratch);
  if (hsz) {
    uint32_t total = 0;
    if (hsz + 16u < n) {
      const uint32_t ss = zstd_encode_sequences(w, regB + hsz, seqs, nseq, n - hsz - 16u, reinterpret_cast<SeqScratch*>(scratch));
      if (ss) total = hsz + ss;
    }
    w_sync(w);
    *payload_off = kZstdHalf;
    return (total && total < n) ? total : 0u;
  }
  // literals section header (raw literals), placed right before the literal bytes
  const uint32_t hs = nlit < 32 ? 1u : (nlit < 4096 ? 2u : 3u);
  uint8_t* hp = stage + 3 - hs;
  uint32_t total = 0;
  if (w.lane == 0) {
    if (hs == 1) hp[0] = (uint8_t)(nlit << 3);
    else if (hs == 2) { hp[0] = (uint8_t)(0x04 | ((nlit & 0xF) << 4)); hp[1] = (uint8_t)(nlit >> 4); }
    else { hp[0] = (uint8_t)(0x0C | ((nlit & 0xF) << 4)); hp[1] = (uint8_t)(nlit >> 4); hp[2] = (uint8_t)(nlit >> 12); }
  }
  // the block must beat its raw form, which also keeps the section inside the slot
  if (hs + nlit + 16u < n) {
    const uint32_t ss = zstd_encode_sequences(w, lit + nlit, seqs, nseq, n - (hs + nlit) - 16u, reinterpret_cast<SeqScratch*>(scratch));
    if (ss) total = hs + nlit + ss;
  }
  w_sync(w);
  *payload_off = 3 - hs;
  return (total && total < n) ? total : 0u;
}

// ------------------------------------------------------------------------------------------------- zstd block
// Compresses slice[bstart .. bstart+n) (n <= 128 KiB) into the payload of one compressed block.
//   stage   kZstdSlot bytes: literals are written from stage+3, the block payload ends up at stage + *payload_off
//   seqs    kZstdMaxSeq packed sequences (global scratch)
//   D       WN::kSmem bytes of shared memory, 16-byte aligned: the input window the match finder works in
//   tab     2^WN::kHashLog x u16 (shared memory): window position of the latest occurrence of each hash
// The match finder never touches global memory: the input slides through D in windows of WN::kBytes, each keeping the
// last WN::kHist bytes of history (16-byte copies, the window keeps the source's alignment).  Offsets therefore stay
// below WN::kHist + WN::kBytes.  A match cut by a window edge is picked up again by the next window and merged back
// into one sequence, so periodic data still costs one sequence per block.
// Returns the payload size, or 0 when the block should be stored raw.
struct alignas(16) V16 { uint32_t a, b, c, d; };

template <class WN>
ZN_HD uint32_t zstd_compress_block(const Warp& w, const uint8_t* slice, uint32_t bstart, uint32_t n, uint8_t* stage,
                                   uint64_t* seqs, uint8_t* D, uint16_t* tab, uint32_t* payload_off) {
  constexpr uint32_t kWinHist = WN::kHist, kWinData = WN::kData, kHashLog = WN::kHashLog;
  const uint32_t hist = bstart < kWinHist ? bstart : kWinHist;
  const uint8_t* g = slice + bstart - hist;  // global address of D[0] (made 16-byte aligned just below)
  const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(g) & 15u);
  g -= mis;
  uint32_t dlo = mis;                  // first valid byte of D
  uint32_t pos = mis + hist, anchor = pos;
  uint32_t bend = pos + n;             // block end in window coordinates (beyond the window until the last one)
  uint32_t filled = 0;                 // bytes of D staged so far (multiple of 16)
  uint8_t* lit = stage + 3;
  uint32_t nlit = 0, nseq = 0, ll_carry = 0;
  uint32_t p_ll = 0, p_ml = 0, p_off = 0;  // the sequence not yet written out (it may still grow across a window edge)
  uint32_t cont_off = 0;                   // offset of a match that ran into the window edge
  bool have = false, first = true;
  ZN_CP_BEGIN();
  for (;;) {
    // ---- stage D[filled .. target)
    const uint32_t want = (bend + 15u) & ~15u;
    const uint32_t target = want < kWinData ? want : kWinData;
    for (uint32_t c = filled / 16u + w.lane; c < target / 16u; c += w.n) {
      const uint32_t lo = c * 16u;
      if (lo >= dlo && lo + 16u <= bend) *reinterpret_cast<V16*>(D + lo) = *reinterpret_cast<const V16*>(g + lo);
      else for (uint32_t i = lo < dlo ? dlo : lo; i < lo + 16u && i < bend; i++) D[i] = g[i];
    }
    filled = target;
    const uint32_t dend = bend < filled ? bend : filled;
    w_sync(w);
    if (first) {  // empty table, then the history of the previous block
      for (uint32_t i = w.lane; i < (1u << kHashLog); i += w.n) tab[i] = 0xFFFFu;
      w_sync(w);
      for (uint32_t p = dlo + w.lane; p + 4u <= pos; p += w.n) tab[hash4(ld32s(D + p), kHashLog)] = (uint16_t)p;
      w_sync(w);
      first = false;
    }
    const bool final = dend == bend;
    if (cont_off) {  // carry the cut match on (the table has no entry for the bytes a match covered)
      if (cont_off <= pos - dlo && pos < dend) {
        const uint32_t more = match_extend(w, D + pos, D + pos - cont_off, dend - pos);
        p_ml += more;
        pos = anchor = pos + more;
        if (!final && pos == dend && more) { /* still running: keep cont_off */ } else cont_off = 0;
      } else cont_off = 0;
    }
    ZN_CP(0);
    // positions below plimit are parsed in this window: a match needs 4 bytes to verify, and a window that is not
    // the last keeps 64 bytes of look-ahead for the probes
    const uint32_t plimit = final ? (n >= 8 ? bend - 7u : pos) : dend - 64u;
    while (pos < plimit) {
      const uint32_t p = pos + w.lane;
      const bool valid = p < plimit;
      const uint32_t v = valid ? ld32s(D + p) : 0u;
      const uint32_t h = hash4(v, kHashLog);
      const uint32_t cand = valid ? tab[h] : 0xFFFFu;
      bool ok = valid && cand < p && ld32s(D + cand) == v;
      ZN_CP(1);
      // Parallel lazy matching: every lane that found a candidate measures its own match (up to kLazyProbe bytes), and
      // the warp takes the lane with the best gain — bytes matched minus the positions skipped to get there — instead
      // of the first lane with any 4-byte match.  Fewer, longer sequences; the window is 32 positions, where a serial
      // lazy parser looks 1-2 ahead.
      uint32_t probe = 0;
      if (ok) {
        const uint32_t lim = dend - p < kLazyProbe ? dend - p : kLazyProbe;
        probe = 4u + prefix_words<kLazyProbeWords>(D + p + 4, D + cand + 4, lim - 4u);
        // Minimum match (tunable, ZN_MIN_MATCH): a sequence costs ~21 bits once entropy coded, so on skewed small-alphabet
        // data 6-7 pays (78 -> 54 KB on the test corpus), while on source text the host emulation measures 4 best.
        ok = probe >= kZstdMinMatch;
      }
      const uint32_t m = w_ballot(w, ok);
      ZN_CP(2);
      if (!m) {
        if (valid) tab[h] = (uint16_t)p;
        w_sync(w);
        pos += w.n;
        ZN_CP(3);
        continue;
      }
      // One look-up round serves every match that starts inside these 32 positions: pick the best lane, emit its
      // sequence, then pick again among the lanes behind the end of that match.
      uint32_t lo = 0, f = 0, next = pos + w.n;
      for (;;) {
        const uint32_t mm = lo < 32u ? (m >> lo) << lo : 0u;
        if (!mm) { f = w.n - 1u; break; }  // nothing more starts here: the rest of the window is literals
        const uint32_t f0 = ffs32(mm) - 1u;
        // score: matched bytes x 4 - skipped positions x 16 (measured optimum; a literal costs less than a byte once Huffman coded)
        const uint32_t score = (ok && w.lane >= lo) ? probe * kLazyMatchWeight + kLazySkipWeight * (w.n - 1u - (w.lane - f0)) : 0u;
        // warp arg-max in one reduction: key = score : (31 - lane), so the earliest lane wins ties
        const uint32_t key = w_max(w, (score << 5) | (31u - w.lane));
        f = w.n == 1 ? 0u : 31u - (key & 31u);
        const uint32_t mp = pos + f, mc = w_shfl(w, cand, f);
        uint32_t ml = w_shfl(w, probe, f);  // a probe that stopped short of its cap already is the match length
        if (ml == kLazyProbe) ml += match_extend(w, D + mp + ml, D + mc + ml, dend - (mp + ml));
        const uint32_t run = mp - anchor, ll = ll_carry + run, off = mp - mc;
        w_copy(w, lit + nlit, D + anchor, run);
        nlit += run;
        ll_carry = 0;
        if (have && ll == 0 && off == p_off) p_ml += ml;  // the continuation of the match a window edge cut
        else {
          if (have) {
            if (w.lane == 0) seqs[nseq] = seq_pack(p_ll, p_ml, p_off);
            nseq++;
          }
          p_ll = ll; p_ml = ml; p_off = off;
          have = true;
        }
        anchor = mp + ml;
        if (!final && anchor == dend) cont_off = off;
        if (anchor >= pos + w.n) { next = anchor; break; }
        lo = anchor - pos;
      }
      ZN_CP(4);
      // Every position of the round enters the table, the ones covered by matches included (most bytes of compressible
      // data lie inside matches: leaving them out hides them from every later look-up).  The next round starts at `next`,
      // so none of these lanes is looked up again and can find itself.  The part of a long match that reaches beyond the
      // round is entered too, up to kZstdInsertSpan positions.
      (void)f;
      if (valid && p < next) tab[h] = (uint16_t)p;
      if (next > pos + w.n) {
        const uint32_t lim = next < pos + w.n + kZstdInsertSpan ? next : pos + w.n + kZstdInsertSpan;
        for (uint32_t q = pos + w.n + w.lane; q < lim && q + 4u <= dend; q += w.n) tab[hash4(ld32s(D + q), kHashLog)] = (uint16_t)q;
      }
      w_sync(w);
      pos = next;
      ZN_CP(5);
    }
    if (final) break;
    // ---- slide: the literals seen so far leave, the last kWinHist bytes stay
    if (pos > anchor) {
      w_copy(w, lit + nlit, D + anchor, pos - anchor);
      nlit += pos - anchor;
      ll_carry += pos - anchor;
      anchor = pos;
    }
    const uint32_t S = (pos - kWinHist) & ~15u;  // pos >= kWinData - 64 - 32 > kWinHist here
    w_sync(w);
    for (uint32_t c = w.lane; c < (filled - S) / 16u; c += w.n)  // source and destination never overlap: S > filled - S
      *reinterpret_cast<V16*>(D + 16u * c) = *reinterpret_cast<const V16*>(D + S + 16u * c);
    for (uint32_t i = w.lane; i < (1u << kHashLog); i += w.n) {
      const uint32_t e = tab[i];
      tab[i] = (e != 0xFFFFu && e >= S) ? (uint16_t)(e - S) : (uint16_t)0xFFFFu;
    }
    g += S;
    pos -= S; anchor -= S; bend -= S; filled -= S;
    dlo = dlo > S ? dlo - S : 0u;
    w_sync(w);
  }
  if (have) {
    if (w.lane == 0) seqs[nseq] = seq_pack(p_ll, p_ml, p_off);
    nseq++;
  }
  uint32_t* tabw = reinterpret_cast<uint32_t*>(D);  // the window is idle from here on: scratch for the entropy stages
  const uint32_t end = bend;
  const uint8_t* in = D;
  const uint32_t rest = end - anchor;
  w_copy(w, lit + nlit, in + anchor, rest);
  nlit += rest;
  w_sync(w);
  if (nseq == 0) return 0;  // nothing found: raw block
  ZN_CP(6);
  const uint32_t total = zstd_block_payload(w, stage, nlit, seqs, nseq, n, tabw, payload_off);
  ZN_CP(8);
  return total;
}

// ------------------------------------------------------------------------------------------------- zstd long effort
// Levels >= 20.  The match finder sees the whole slice (up to kLongReach back) through a candidate index built per
// round of slices:
//   * every position q of a round (the round's units laid back to back) gets the key bucket << kLongPosBits | q,
//     bucket = a hash of the kLongK bytes at q; a radix sort of the keys puts the earlier positions with q's bucket
//     right before q, nearest first, and rank[q] says where q landed;
//   * a unit is the part of a slice one index covers: slices are parsed in pieces of kLongPiece bytes, each indexed
//     together with the kLongReach bytes before it, so a round holds whole units and no key reaches another slice;
//   * one warp parses each 128 KiB block: the best of the kLongD nearest candidates of a position (probes capped at
//     kLongProbe bytes), the last offset as a repeat candidate, and a two-step lazy rule (zstd's lazy2 gains).
// The best match of a position depends only on the slice's bytes, and the parse itself is serial code every lane
// runs alike, so the sequences do not depend on the lane count: the host emulation (one lane) emits the GPU's bytes.
constexpr uint32_t kLongReach = 8u << 20;                   // largest offset (the reference's slice, libzstd-19's window)
constexpr uint32_t kLongPiece = 8u << 20;                   // slice bytes parsed per unit (a multiple of kZstdCBlock)
constexpr uint32_t kLongPosBits = 27;                       // positions per round < 2^27 (units are <= 16 MiB)
constexpr uint32_t kLongRound = 1u << kLongPosBits;
constexpr uint32_t kLongHashBits = 29;
constexpr uint32_t kLongKeyBits = kLongPosBits + kLongHashBits;  // key bits the sort orders
#ifndef ZN_LONG_K
#define ZN_LONG_K 5
#define ZN_LONG_D 16
#endif
constexpr uint32_t kLongK = ZN_LONG_K;                      // bytes hashed into a bucket (4 .. 8)
constexpr uint32_t kLongD = ZN_LONG_D;                      // candidates probed per position
constexpr uint32_t kLongProbe = 256;                        // bytes a probe measures; a chosen match is extended beyond
constexpr uint32_t kLongBatch = kOnDevice ? 32u : 4u;       // positions evaluated together (one per lane on the device)
static_assert(kLongPiece % kZstdCBlock == 0 && kLongK >= 4 && kLongK <= 8, "long effort geometry");

// Slice positions [lo, hi) of a unit occupy round positions [q0, q0 + hi - lo).
struct LongIndex {
  const uint64_t* sk;    // the round's keys, sorted
  const uint32_t* rank;  // rank[q]: index of q's key in sk
  uint32_t q0, lo;
};

ZN_HD uint64_t long_key(const uint8_t* slice, uint32_t pos, uint32_t hi, uint32_t q) {
  uint64_t b = (1ull << kLongHashBits) - 1u;  // the last kLongK - 1 positions share one bucket (matches are verified)
  if (hi - pos >= kLongK) {
    uint64_t v = 0;
    for (uint32_t i = 0; i < kLongK; i++) v |= (uint64_t)slice[pos + i] << (8u * i);
    b = (v * 0x9E3779B185EBCA87ull) >> (64u - kLongHashBits);
  }
  return (b << kLongPosBits) | q;
}

// unaligned little-endian 32-bit load that touches only the aligned words holding p[0..4)
ZN_HD uint32_t ld32g(const uint8_t* p) {
#if defined(__CUDA_ARCH__)
  const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
  const uint32_t sh = ((uint32_t)reinterpret_cast<uintptr_t>(p) & 3u) * 8u;
  return sh ? __funnelshift_r(w[0], w[1], sh) : w[0];
#else
  return ld32le(p);
#endif
}

// common prefix length of a[0..lim) and b[0..lim), one lane
ZN_HD uint32_t long_prefix(const uint8_t* a, const uint8_t* b, uint32_t lim) {
  uint32_t n = 0;
  for (; n + 4u <= lim; n += 4u) {
    const uint32_t x = ld32g(a + n) ^ ld32g(b + n);
    if (x) return n + ((ffs32(x) - 1u) >> 3);
  }
  while (n < lim && a[n] == b[n]) n++;
  return n;
}

// Longest match for slice position p among its kLongD nearest candidates, measured up to min(kLongProbe, end - p);
// the nearest candidate wins a tie.  *len = 0 when no candidate matches at all.
ZN_HD void long_best(const uint8_t* s, const LongIndex& ix, uint32_t p, uint32_t end, uint32_t* len, uint32_t* off) {
  const uint32_t i = ix.rank[ix.q0 + (p - ix.lo)];
  const uint64_t bucket = ix.sk[i] >> kLongPosBits;
  const uint32_t lim = end - p < kLongProbe ? end - p : kLongProbe;
  uint32_t bl = 0, bo = 0;
  for (uint32_t d = 1; d <= kLongD && d <= i; d++) {
    const uint64_t k = ix.sk[i - d];
    const uint32_t cq = (uint32_t)k & (kLongRound - 1u);
    if ((k >> kLongPosBits) != bucket || cq < ix.q0) break;  // bucket or unit exhausted
    const uint32_t c = cq - ix.q0 + ix.lo;
    if (p - c > kLongReach) break;
    if (s[c + bl] != s[p + bl]) continue;  // cannot beat the best so far
    const uint32_t l = long_prefix(s + p, s + c, lim);
    if (l > bl) {
      bl = l;
      bo = p - c;
      if (l == lim) break;
    }
  }
  *len = bl;
  *off = bo;
}

// lazy2's gain of a match: 4 per byte minus the bits of its offset value (a repeat of the last offset codes as 1)
ZN_HD int32_t long_gain(uint32_t ml, uint32_t off, uint32_t rep) {
  return 4 * (int32_t)ml - (int32_t)hibit32(off == rep ? 1u : off + 3u);
}

// Compresses slice s[bstart .. bstart+n) (n <= 128 KiB) into the payload of one compressed block, whole warp.
//   ix       the candidate index of the unit holding the block
//   stage    kZstdSlot bytes: literals are written from stage+3, the payload ends up at stage + *payload_off
//   seqs     kZstdMaxSeq packed sequences (global scratch)
//   bl, bo   kLongBatch words each (shared memory): match length / offset of the positions being evaluated
//   scratch  kPayloadScratch bytes of shared memory for the entropy stages
// Returns the payload size, or 0 when the block should be stored raw.
ZN_HD uint32_t zstd_long_block(const Warp& w, const uint8_t* s, const LongIndex& ix, uint32_t bstart, uint32_t n,
                               uint8_t* stage, uint64_t* seqs, uint32_t* bl, uint32_t* bo, uint32_t* scratch,
                               uint32_t* payload_off) {
  const uint32_t bend = bstart + n;
  uint8_t* lit = stage + 3;
  uint32_t nlit = 0, nseq = 0, anchor = bstart, pos = bstart, rep = 0;
  uint32_t base = bend;  // first position of the evaluated batch (none yet)
  // best match at p: the index's candidates, then the last offset of this block as a repeat candidate
  auto best = [&](uint32_t p, uint32_t* ml, uint32_t* off) {
    if (p - base >= kLongBatch) {
      w_sync(w);
      for (uint32_t i = w.lane; i < kLongBatch; i += w.n) {
        uint32_t l = 0, o = 0;
        if (p + i + 4u <= bend) long_best(s, ix, p + i, bend, &l, &o);
        bl[i] = l;
        bo[i] = o;
      }
      w_sync(w);
      base = p;
    }
    *ml = bl[p - base];
    *off = bo[p - base];
    if (rep && rep <= p) {
      const uint32_t lim = bend - p < kLongProbe ? bend - p : kLongProbe;
      const uint32_t rl = long_prefix(s + p, s + p - rep, lim);
      if (rl >= 4u && (*ml < 4u || long_gain(rl, rep, rep) >= long_gain(*ml, *off, rep))) { *ml = rl; *off = rep; }
    }
  };
  while (pos + 4u <= bend) {
    uint32_t ml, off;
    best(pos, &ml, &off);
    if (ml < 4u) { pos++; continue; }
    uint32_t start = pos;
    for (uint32_t ip = pos;;) {  // lazy2: a later start wins when it gains 4 (one step on) or 7 (two steps on) more
      bool moved = false;
      for (uint32_t step = 1; step <= 2 && ip + 1u + 4u <= bend; step++) {
        ip++;
        uint32_t ml2, off2;
        best(ip, &ml2, &off2);
        if (ml2 >= 4u && long_gain(ml2, off2, rep) > long_gain(ml, off, rep) + (step == 1 ? 4 : 7)) {
          ml = ml2; off = off2; start = ip;
          moved = true;
          break;
        }
      }
      if (!moved) break;
    }
    if (ml == kLongProbe && start + ml < bend) ml += match_extend(w, s + start + ml, s + start - off + ml, bend - (start + ml));
    w_copy(w, lit + nlit, s + anchor, start - anchor);
    if (w.lane == 0) seqs[nseq] = seq_pack(start - anchor, ml, off);
    nlit += start - anchor;
    nseq++;
    rep = off;
    pos = anchor = start + ml;
  }
  w_copy(w, lit + nlit, s + anchor, bend - anchor);
  nlit += bend - anchor;
  w_sync(w);
  if (nseq == 0) return 0;
  return zstd_block_payload(w, stage, nlit, seqs, nseq, n, scratch, payload_off);
}

// Zstandard frame header: single segment, 8-byte content size (13 bytes), and with `checksum` (ZN_CODEC_CHECKSUM) the
// content checksum flag; empty content uses the 1-byte form (zstd_empty_frame).
ZN_HD uint32_t zstd_frame_header(uint8_t* dst, uint64_t content, bool checksum = false) {
  dst[0] = 0x28; dst[1] = 0xB5; dst[2] = 0x2F; dst[3] = 0xFD;
  dst[4] = checksum ? 0xE4 : 0xE0;
  for (int i = 0; i < 8; i++) dst[5 + i] = (uint8_t)(content >> (8 * i));
  return 13;
}
ZN_HD void zstd_block_header(uint8_t* dst, uint32_t last, uint32_t type, uint32_t size) {
  const uint32_t v = last | (type << 1) | (size << 3);
  dst[0] = (uint8_t)v; dst[1] = (uint8_t)(v >> 8); dst[2] = (uint8_t)(v >> 16);
}

// ---- sizes of what the assemble kernels (compress_kernels.cuh) write for a slice of n bytes, from the per-block
// results alone: a packed layout is computed on the device before any frame byte exists.
// zstd: meta = the slice's first {payload offset, size} pair (size 0 = raw block); the empty frame is 9 bytes.
// `checksum`: 4 more bytes, the content checksum behind the last block.
ZN_HD uint64_t zstd_frame_size(uint64_t n, const uint32_t* meta, bool checksum = false) {
  if (n == 0) return checksum ? 13 : 9;
  uint64_t sz = checksum ? 17 : 13;
  for (uint64_t o = 0, j = 0; o < n; o += kZstdCBlock, j++) {
    const uint32_t bn = (uint32_t)(n - o < kZstdCBlock ? n - o : kZstdCBlock), c = meta[2 * j + 1];
    sz += 3 + (c ? c : bn);
  }
  return sz;
}
// The empty frame, as libzstd writes it: single segment, 1-byte content size 0, empty raw last block (9 bytes); with
// `checksum` as libzstd writes it with ZSTD_c_checksumFlag: descriptor 0x24 and XXH64("") behind the block (13 bytes).
ZN_HD uint32_t zstd_empty_frame(uint8_t* dst, bool checksum = false) {
  const uint8_t e[13] = {0x28, 0xB5, 0x2F, 0xFD, 0x20, 0x00, 0x01, 0x00, 0x00, 0x99, 0xE9, 0xD8, 0x51};
  for (int k = 0; k < 9; k++) dst[k] = e[k];
  if (!checksum) return 9;
  dst[4] = 0x24;
  for (int k = 9; k < 13; k++) dst[k] = e[k];
  return 13;
}

// ---- seekable layout (ZN_CODEC_SEEKABLE): every kZstdCBlock block of the slice is a frame of its own (the 13-byte
// header, one last block), then the seek table of the Zstandard seekable format (contrib/seekable_format in the zstd
// tree): a skippable frame, magic 0x184D2A5E and Frame_Size = 12 N + 9, holding per frame {compressed size, decompressed
// size, low 32 bits of XXH64(content, 0)}, then the footer {N, descriptor 0x80 = checksums present, 0x8F92EAB1}, all
// little-endian.  An empty slice is the empty frame and a table with one entry.
constexpr uint32_t kSeekEntry = 12, kSeekFixed = 17;  // bytes per entry; skippable header (8) + footer (9)
constexpr uint32_t kSeekSkipMagic = 0x184D2A5Eu, kSeekFooterMagic = 0x8F92EAB1u, kSeekChecksums = 0x80u;
constexpr uint32_t kXxhEmpty = 0x51D8E999u;  // low 32 bits of XXH64("", 0)
ZN_HD void put_le32(uint8_t* d, uint32_t v) { d[0] = (uint8_t)v; d[1] = (uint8_t)(v >> 8); d[2] = (uint8_t)(v >> 16); d[3] = (uint8_t)(v >> 24); }
// meta as for zstd_frame_size
ZN_HD uint64_t zstd_seekable_size(uint64_t n, const uint32_t* meta) {
  if (n == 0) return 9 + kSeekEntry + kSeekFixed;
  uint64_t sz = kSeekFixed;
  for (uint64_t o = 0, j = 0; o < n; o += kZstdCBlock, j++) {
    const uint32_t bn = (uint32_t)(n - o < kZstdCBlock ? n - o : kZstdCBlock), c = meta[2 * j + 1];
    sz += 13 + 3 + (c ? c : bn) + kSeekEntry;
  }
  return sz;
}
// The seek table of a slice of n bytes at dst; returns its length.  meta as for zstd_frame_size, xxh = the checksum of
// the slice's first frame (unused when n == 0).
ZN_HD uint32_t zstd_seek_table(uint8_t* dst, uint64_t n, const uint32_t* meta, const uint32_t* xxh) {
  const uint32_t nf = n ? (uint32_t)((n + kZstdCBlock - 1) / kZstdCBlock) : 1u;
  put_le32(dst, kSeekSkipMagic);
  put_le32(dst + 4, kSeekEntry * nf + 9);
  uint8_t* e = dst + 8;
  if (n == 0) {
    put_le32(e, 9); put_le32(e + 4, 0); put_le32(e + 8, kXxhEmpty);
    e += kSeekEntry;
  }
  for (uint64_t o = 0, j = 0; o < n; o += kZstdCBlock, j++, e += kSeekEntry) {
    const uint32_t bn = (uint32_t)(n - o < kZstdCBlock ? n - o : kZstdCBlock), c = meta[2 * j + 1];
    put_le32(e, 13 + 3 + (c ? c : bn)); put_le32(e + 4, bn); put_le32(e + 8, xxh[j]);
  }
  put_le32(e, nf);
  e[4] = (uint8_t)kSeekChecksums;
  put_le32(e + 5, kSeekFooterMagic);
  return kSeekFixed + kSeekEntry * nf;
}

// LZ4: csize = the slice's first block size (>= the block's input size means stored); 15-byte header, 4-byte EndMark,
// and with `checksum` the 4-byte content checksum
ZN_HD uint64_t lz4_frame_size(uint64_t n, const uint32_t* csize, bool checksum = false) {
  uint64_t sz = 15 + 4 + (checksum ? 4 : 0);
  for (uint64_t o = 0, j = 0; o < n; o += kLz4Block, j++) {
    const uint32_t bn = (uint32_t)(n - o < kLz4Block ? n - o : kLz4Block), c = csize[j];
    sz += 4 + (c < bn ? c : bn);
  }
  return sz;
}

// ZNB1 envelope header (csrc/envelope.cpp, zn_envelope_znb1_header): "ZNB1", payload codec, LEB128 decoded size
constexpr uint32_t kZnb1Raw = 0, kZnb1Zstd = 1, kZnb1Lz4Frame = 3;  // ZN_PAYLOAD_* of include/znippy_cuda.h
ZN_HD uint32_t znb1_header_len(uint64_t n) {
  uint32_t l = 6;
  for (; n >= 128; n >>= 7) l++;
  return l;
}
ZN_HD uint32_t znb1_header(uint8_t* dst, uint32_t codec, uint64_t n) {
  dst[0] = 'Z'; dst[1] = 'N'; dst[2] = 'B'; dst[3] = '1';
  dst[4] = (uint8_t)codec;
  uint32_t p = 5;
  do {
    uint8_t b = (uint8_t)(n & 0x7F);
    n >>= 7;
    if (n) b |= 0x80;
    dst[p++] = b;
  } while (n);
  return p;
}

}  // namespace cz
}  // namespace zn
