// BLAKE3 batch kernels: chunk chaining values (flat over every 1 KiB chunk of every blob in the batch) and the
// tree merge + digest compare.  Replaces blake3::hash + the 32-byte compare of the reference's read loop
// (znippy-common/src/decompress.rs:172-184) and the write-side hash (stream_packer.rs:219, slot_packer.rs:553).
//
// Roofline note (DESIGN.md): BLAKE3 is bound by the integer ALU pipe, not by HBM — 7 rounds x 8 G x 12 ops per
// 64-byte block ~ 10.5 ops/byte.  The chunk kernel therefore keeps the ALU pipe fed: one lane per chunk, message
// words staged through shared memory by coalesced 16-byte cp.async copies (double buffered per warp, no CTA
// barriers), conflict-free 128-bit shared loads (odd row stride), and a full 32-lane tile even when a batch is
// 100 000 ten-chunk blobs, because lanes are assigned over the flat (blob, chunk) index space.
#pragma once
#include "blake3.cuh"
#include "xxh_verify.cuh"

namespace zn {

// Where a blob's content lives: decoded rows in the output buffer, store-as-is rows in the blobs buffer.
ZN_D const uint8_t* content_ptr(const BlobDesc& d, const uint8_t* blobs_base, const uint8_t* out_base) {
  return (d.flags & F_COMPRESSED) ? out_base + d.dst_off : blobs_base + d.src_off;
}

constexpr int kB3Warps = 8;                      // warps per CTA
constexpr int kB3RowBytes = 128;                 // bytes of each chunk staged per pipeline stage (2 blocks)
constexpr int kB3RowStride = kB3RowBytes + 16;   // 9 quads: odd -> conflict-free LDS.128 across lanes
constexpr int kB3Stages = 2;
constexpr int kB3StageBytes = 32 * kB3RowStride;
constexpr int kB3SmemPerWarp = kB3Stages * kB3StageBytes;
constexpr int kB3RowsPerIssue = 32 / (kB3RowBytes / 16);  // rows covered by one warp-wide 16-byte copy (4)

// Stage `stage_idx` (bytes [stage_idx*128, +128) of each of the warp's 32 chunks) -> shared memory.
// ptr/len are this lane's chunk; rows are other lanes' chunks, fetched by shuffle.  `regular` (warp-uniform) = the 32
// chunks are full, 16-byte aligned and contiguous in memory (the common case inside a large blob): rows are then
// addressed from lane 0's pointer without any shuffle.
ZN_D void b3_issue_stage(uint8_t* buf, const uint8_t* ptr, uint32_t len, uint32_t stage_idx, uint32_t lane, bool regular,
                         const uint8_t* base0) {
  const uint32_t q = lane & 7u;          // quad inside the row
  const uint32_t sub = lane >> 3;        // row inside the issue group
  const uint32_t base = stage_idx * kB3RowBytes + q * 16u;
  if (regular) {
#pragma unroll
    for (int it = 0; it < 32 / kB3RowsPerIssue; it++) {
      const uint32_t row = it * kB3RowsPerIssue + sub;
      cp_async16(buf + row * kB3RowStride + q * 16u, base0 + (size_t)row * kChunk + base);
    }
    return;
  }
  const uint32_t ptr_lo = (uint32_t)reinterpret_cast<uintptr_t>(ptr);
  const uint32_t ptr_hi = (uint32_t)(reinterpret_cast<uintptr_t>(ptr) >> 32);
#pragma unroll
  for (int it = 0; it < 32 / kB3RowsPerIssue; it++) {
    const uint32_t row = it * kB3RowsPerIssue + sub;
    const uint32_t rlo = __shfl_sync(0xFFFFFFFFu, ptr_lo, row);
    const uint32_t rhi = __shfl_sync(0xFFFFFFFFu, ptr_hi, row);
    const uint32_t rlen = __shfl_sync(0xFFFFFFFFu, len, row);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(((uintptr_t)rhi << 32) | rlo) + base;
    uint8_t* dst = buf + row * kB3RowStride + q * 16u;
    if (base + 16u <= rlen && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
      cp_async16(dst, src);
    } else if (base < rlen) {  // unaligned source or the blob's last, partial quad: assemble from byte loads
      const uint32_t nb = min(16u, rlen - base);
      uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
#pragma unroll
      for (uint32_t j = 0; j < 4; j++) {
        // L2 loads (never the non-coherent path, never L1): the fused decoders hash their own output, and a sector that
        // straddles two tiles must not be served from an L1 copy taken before its second half was written
        if (j < nb) w0 |= (uint32_t)__ldcg(src + j) << (8 * j);
        if (j + 4 < nb) w1 |= (uint32_t)__ldcg(src + j + 4) << (8 * j);
        if (j + 8 < nb) w2 |= (uint32_t)__ldcg(src + j + 8) << (8 * j);
        if (j + 12 < nb) w3 |= (uint32_t)__ldcg(src + j + 12) << (8 * j);
      }
      *reinterpret_cast<uint4*>(dst) = make_uint4(w0, w1, w2, w3);
    }
  }
}

// Chaining values of one warp tile: lane L hashes the (<= 1 KiB) chunk at `ptr` (len bytes, chunk counter ctr).
// wbuf = this warp's kB3SmemPerWarp bytes of shared memory.  All 32 lanes must call (act = lane has a chunk).
ZN_D void b3_warp_tile(uint8_t* wbuf, const uint8_t* ptr, uint32_t len, uint32_t ctr, bool root, bool act, uint32_t lane,
                       uint32_t one, uint32_t (&cv)[8]) {
  const uint32_t nblocks = act ? (len == 0 ? 1u : (len + 63u) >> 6) : 0u;
  b3::set_iv(cv);
  // ---- software pipeline over the 8 stages of a chunk
  const uint8_t* base0 = reinterpret_cast<const uint8_t*>(
      ((uintptr_t)__shfl_sync(0xFFFFFFFFu, (uint32_t)(reinterpret_cast<uintptr_t>(ptr) >> 32), 0) << 32) |
      __shfl_sync(0xFFFFFFFFu, (uint32_t)reinterpret_cast<uintptr_t>(ptr), 0));
  const bool regular = __all_sync(0xFFFFFFFFu, act && len == kChunk && ptr == base0 + (size_t)lane * kChunk) &&
                       (reinterpret_cast<uintptr_t>(base0) & 15) == 0;
  __syncwarp();
  b3_issue_stage(wbuf, ptr, len, 0, lane, regular, base0);
  cp_async_commit();
#pragma unroll 1
  for (uint32_t s = 0; s < kChunk / kB3RowBytes; s++) {
    uint8_t* cur = wbuf + (s & 1u) * kB3StageBytes;
    if (s + 1 < kChunk / kB3RowBytes) b3_issue_stage(wbuf + ((s + 1) & 1u) * kB3StageBytes, ptr, len, s + 1, lane, regular, base0);
    cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
    const uint4* row = reinterpret_cast<const uint4*>(cur + lane * kB3RowStride);
    // NOT unrolled: one copy of the 7-round compression (~13 KB of code) instead of two.  Instruction fetch is what
    // limits the hash warps once other code runs on the SM too: in the fused kernel (fused_ws.cuh) 15 % of the warp
    // samples were "no instruction" stalls with the unrolled body, and the kernel went from 1.22 to 1.08 ms without it.
#pragma unroll 1
    for (uint32_t j = 0; j < kB3RowBytes / 64; j++) {
      const uint32_t b = s * (kB3RowBytes / 64) + j;
      if (b < nblocks) {
        uint32_t m[16];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const uint4 v = row[j * 4 + k];
          m[4 * k] = v.x; m[4 * k + 1] = v.y; m[4 * k + 2] = v.z; m[4 * k + 3] = v.w;
        }
        const uint32_t n = min(64u, len - b * 64u);
        if (n < 64u) {
#pragma unroll
          for (int k = 0; k < 16; k++) {
            const int vb = (int)n - 4 * k;  // valid bytes in word k
            m[k] = vb >= 4 ? m[k] : (vb <= 0 ? 0u : (m[k] & (0xFFFFFFFFu >> (8 * (4 - vb)))));
          }
        }
        uint32_t flags = (b == 0 ? b3::CHUNK_START : 0u);
        if (b + 1 == nblocks) flags |= b3::CHUNK_END | (root ? b3::ROOT : 0u);
        b3::compress(cv, m, ctr, 0u, n, flags, one);
      }
    }
    __syncwarp();  // everyone is done with `cur` before the next iteration's copies land in it
  }
}

// K3a: chunk chaining values of the flat chunks [chunk_lo, chunk_hi).  chunk_prefix[b] = first flat chunk index of
// blob b (n_blobs+1 entries).
__global__ void __launch_bounds__(kB3Warps * 32) k_b3_chunks(const BlobDesc* __restrict__ blobs,
                                                              const uint32_t* __restrict__ chunk_prefix,
                                                              uint32_t n_blobs, uint32_t chunk_lo, uint32_t chunk_hi,
                                                              const uint8_t* __restrict__ blobs_base,
                                                              const uint8_t* __restrict__ out_base,
                                                              uint32_t* cvs, uint32_t one) {
  extern __shared__ __align__(16) uint8_t b3_smem[];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint8_t* wbuf = b3_smem + warp * kB3SmemPerWarp;
  const uint32_t n_tiles = (chunk_hi - chunk_lo + 31u) >> 5;
  const uint32_t warps_total = gridDim.x * kB3Warps;
  for (uint32_t tile = blockIdx.x * kB3Warps + warp; tile < n_tiles; tile += warps_total) {
    const uint32_t g = chunk_lo + tile * 32u + lane;
    const bool act = g < chunk_hi;
    // ---- which chunk of which blob is mine
    const uint8_t* ptr = nullptr;
    uint32_t len = 0, ctr = 0;
    bool root = false, skip = false;
    if (act) {
      uint32_t lo = 0, hi = n_blobs;
      while (hi - lo > 1) {  // largest b with chunk_prefix[b] <= g
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(chunk_prefix + mid) <= g) lo = mid; else hi = mid;
      }
      const BlobDesc d = blobs[lo];
      skip = (d.flags & F_HASHED) != 0;  // chaining values already produced by the fused decode kernel
      ctr = g - __ldg(chunk_prefix + lo);
      ptr = content_ptr(d, blobs_base, out_base) + (uint64_t)ctr * kChunk;
      const uint64_t remain = d.dst_cap - (uint64_t)ctr * kChunk;
      len = remain < kChunk ? (uint32_t)remain : kChunk;
      root = d.n_chunks == 1;
    }
    if (__all_sync(0xFFFFFFFFu, !act || skip)) continue;
    uint32_t cv[8];
    b3_warp_tile(wbuf, ptr, len, ctr, root, act && !skip, lane, one, cv);
    if (act && !skip) b3::store_cv(cvs + (uint64_t)g * 8, cv);
  }
}

// digest = cv words little-endian; compare with expect and fold into status (decode errors win).  xxh_bad: a checksum of
// the row's frames disagrees with its bytes (xxh_verify.cuh), a decode error.
ZN_D void finish_blob(const BlobDesc& d, uint32_t blob, const uint32_t (&cv)[8], uint32_t* __restrict__ digests,
                      const uint32_t* __restrict__ expect, uint32_t* __restrict__ status, bool xxh_bad) {
  b3::store_cv(digests + (uint64_t)blob * 8, cv);
  if (xxh_bad && status[blob] == S_OK) status[blob] = S_DECODE_ERROR;
  if ((d.flags & F_HAS_EXPECT) && status[blob] == S_OK) {
    bool eq = true;
#pragma unroll
    for (int i = 0; i < 8; i++) eq &= (__ldg(expect + (uint64_t)blob * 8 + i) == cv[i]);
    if (!eq) status[blob] = S_DIGEST_MISMATCH;
  }
}

// K3b: small blobs (<= kTreeSmallMax chunks): one lane walks the levels of its own blob in place.
__global__ void __launch_bounds__(128) k_b3_tree_small(const BlobDesc* __restrict__ blobs,
                                                       const uint32_t* __restrict__ list, uint32_t n_list,
                                                       uint32_t* cvs, uint32_t* __restrict__ digests,
                                                       const uint32_t* __restrict__ expect,
                                                       uint32_t* __restrict__ status, uint32_t one,
                                                       const uint8_t* blobs_base, const uint8_t* out_base) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_list) return;
  const uint32_t blob = list[t];
  const BlobDesc d = blobs[blob];
  uint32_t* base = cvs + d.cv_base * 8;
  uint32_t n = d.n_chunks;
  uint32_t l[8], r[8], o[8];
  while (n > 1) {
    const uint32_t pairs = n >> 1;
    for (uint32_t j = 0; j < pairs; j++) {
      b3::load_cv(base + (uint64_t)(2 * j) * 8, l);
      b3::load_cv(base + (uint64_t)(2 * j + 1) * 8, r);
      b3::parent(l, r, n == 2, o, one);
      b3::store_cv(base + (uint64_t)j * 8, o);
    }
    if (n & 1) {
      b3::load_cv(base + (uint64_t)(n - 1) * 8, l);
      b3::store_cv(base + (uint64_t)pairs * 8, l);
    }
    n = pairs + (n & 1);
  }
  b3::load_cv(base, o);
  finish_blob(d, blob, o, digests, expect, status, out_base && status[blob] == S_OK && xxh_row_bad(d, blobs_base, out_base));
}

// Checksums of one decoded row by a whole CTA (xxh_verify.cuh): thread 0 walks the frame and block headers into a list
// of spans in shared memory, the warps hash the spans (xxh_warp).  A row with more spans than the list holds is walked
// again for each further part of the list.
constexpr uint32_t kRowSpans = 256;
struct XxhSpan {
  const uint8_t* p;
  uint64_t len;
  uint32_t bits, want;
};
struct XxhSpanList {  // emit() of xxh_row_walk: keeps spans [first, first + kRowSpans), counts them all
  XxhSpan* list;
  uint32_t first, total = 0;
  ZN_D bool operator()(const uint8_t* p, uint64_t len, uint32_t bits, uint32_t want) {
    if (total >= first && total - first < kRowSpans) list[total - first] = XxhSpan{p, len, bits, want};
    total++;
    return true;
  }
};
template <int kThreads>
ZN_D bool xxh_row_bad_cta(const BlobDesc& d, bool ok, const uint8_t* blobs_base, const uint8_t* out_base) {
  __shared__ XxhSpan spans[kRowSpans];
  __shared__ uint32_t n_spans, more, bad;
  __shared__ __align__(16) uint8_t ring[kThreads / 32][kXxhRing];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  for (uint32_t first = 0;; first += kRowSpans) {
    if (threadIdx.x == 0) {
      XxhSpanList l{spans, first};
      if (ok) xxh_row_walk(d, blobs_base, out_base, l);
      n_spans = l.total > first ? min(l.total - first, kRowSpans) : 0u;
      more = l.total > first + kRowSpans;
      if (first == 0) bad = 0;
    }
    __syncthreads();
    for (uint32_t k = warp; k < n_spans; k += kThreads / 32) {
      const XxhSpan sp = spans[k];
      const uint32_t h = sp.bits == 64 ? (uint32_t)xxh_warp<64>(sp.p, sp.len, ring[warp], lane)
                                       : (uint32_t)xxh_warp<32>(sp.p, sp.len, ring[warp], lane);
      if (lane == 0 && h != sp.want) bad = 1;
    }
    __syncthreads();
    const bool stop = !more || bad;
    __syncthreads();  // everyone has read `more` and `bad` before thread 0 walks again
    if (stop) return bad;
  }
}

// K3c: large blobs: one CTA per blob, every level spread over the CTA.  Levels ping-pong between the blob's slots in
// `cvs` and in `cvs2` (same layout), so a level needs no barrier between its items — the 8 warps run their (load, load,
// compress, store) items independently and hide each other's L2 round trips — only one barrier per level.  Then the
// CTA checks the row's frame checksums.
__global__ void __launch_bounds__(512) k_b3_tree_large(const BlobDesc* __restrict__ blobs,
                                                       const uint32_t* __restrict__ list,
                                                       uint32_t* cvs, uint32_t* cvs2, uint32_t* __restrict__ digests,
                                                       const uint32_t* __restrict__ expect,
                                                       uint32_t* __restrict__ status, uint32_t one,
                                                       const uint8_t* blobs_base, const uint8_t* out_base) {
  const uint32_t blob = list[blockIdx.x];
  const BlobDesc d = blobs[blob];
  uint32_t* src = cvs + d.cv_base * 8;
  uint32_t* dst = cvs2 + d.cv_base * 8;
  uint32_t n = d.n_chunks;
  uint32_t l[8], r[8], o[8];
  while (n > 1) {
    const uint32_t pairs = n >> 1, items = pairs + (n & 1);  // the odd tail is a pass-through item
    for (uint32_t j = threadIdx.x; j < items; j += blockDim.x) {
      b3::load_cv(src + (uint64_t)(2 * j) * 8, l);
      if (j < pairs) {
        b3::load_cv(src + (uint64_t)(2 * j + 1) * 8, r);
        b3::parent(l, r, n == 2, o, one);
      } else {
#pragma unroll
        for (int i = 0; i < 8; i++) o[i] = l[i];
      }
      b3::store_cv(dst + (uint64_t)j * 8, o);
    }
    __syncthreads();
    uint32_t* t = src; src = dst; dst = t;
    n = items;
  }
  const bool bad = out_base && xxh_row_bad_cta<512>(d, status[blob] == S_OK, blobs_base, out_base);
  if (threadIdx.x == 0) {
    b3::load_cv(src, o);
    finish_blob(d, blob, o, digests, expect, status, bad);
  }
}

constexpr uint32_t kTreeSmallMax = 64;

}  // namespace zn
