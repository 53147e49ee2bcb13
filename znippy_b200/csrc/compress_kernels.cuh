// K6/K7: batched per-slice compression kernels (one warp per block) and frame assembly; host launcher.
// See compress.cuh for the algorithms and the reference call sites this replaces.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <string>
#include <vector>

#include "compress.cuh"
#include "coop.cuh"

namespace zn {

struct SliceDesc {
  uint64_t src_off, src_len;
  uint64_t dst_off;     // frame goes to dst_base + dst_off
  uint32_t blk_first;   // first global block index of this slice
  uint32_t n_blocks;
};

constexpr int kLz4WarpsPerCta = 4;
constexpr int kZstdWarpsPerCta = 1;
template <class WN>
struct ZstdLaunch {
  static constexpr uint32_t kWindow = (WN::kSmem + 127u) & ~127u;
  static constexpr uint32_t kSmemBytes = kWindow + (2u << WN::kHashLog);
  static constexpr uint32_t kCtasPerSm = (228u * 1024u) / (kSmemBytes + 1024u);
};

// which slice owns global block j (slices' blk_first ascending)
ZN_D uint32_t slice_of_block(const SliceDesc* __restrict__ s, uint32_t n_slices, uint32_t j) {
  uint32_t lo = 0, hi = n_slices;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (s[mid].blk_first <= j) lo = mid; else hi = mid;
  }
  return lo;
}

// ---- LZ4: every 64 KiB block of every slice -> tmp slot; csize[j] = compressed size (>= n means "store raw")
__global__ void __launch_bounds__(kLz4WarpsPerCta * 32) k_lz4_blocks(const SliceDesc* __restrict__ slices, uint32_t n_slices,
                                                                     uint32_t total_blocks, const uint8_t* __restrict__ src_base,
                                                                     uint8_t* tmp, uint32_t* csize) {
  __shared__ uint16_t tabs[kLz4WarpsPerCta][1u << cz::kLz4HashLog];
  const uint32_t warp = threadIdx.x >> 5;
  const cz::Warp w{threadIdx.x & 31u, 32u};
  for (uint32_t j = blockIdx.x * kLz4WarpsPerCta + warp; j < total_blocks; j += gridDim.x * kLz4WarpsPerCta) {
    const uint32_t si = slice_of_block(slices, n_slices, j);
    const SliceDesc s = slices[si];
    const uint64_t o = (uint64_t)(j - s.blk_first) * cz::kLz4Block;
    const uint32_t n = (uint32_t)(s.src_len - o < cz::kLz4Block ? s.src_len - o : cz::kLz4Block);
    const uint32_t c = cz::lz4_compress_block(w, src_base + s.src_off + o, n, tmp + (size_t)j * cz::kLz4Slot, tabs[warp]);
    if (w.lane == 0) csize[j] = c;
    __syncwarp();
  }
}

// ---- LZ4 frame assembly: the CTA writes slice i's frame at dst_base + dst_off (k_lz4_assemble: one CTA per slice)
ZN_D void lz4_assemble(const SliceDesc* __restrict__ slices, uint32_t i, const uint8_t* __restrict__ src_base, const uint8_t* tmp,
                       const uint32_t* __restrict__ csize, uint8_t* dst_base, uint64_t* dst_len) {
  const SliceDesc s = slices[i];
  uint8_t* dst = dst_base + s.dst_off;
  const Team t{threadIdx.x, blockDim.x};
  if (threadIdx.x == 0) cz::lz4_frame_header(dst, s.src_len);
  uint64_t op = 15;
  for (uint32_t b = 0; b < s.n_blocks; b++) {
    const uint32_t j = s.blk_first + b;
    const uint64_t o = (uint64_t)b * cz::kLz4Block;
    const uint32_t n = (uint32_t)(s.src_len - o < cz::kLz4Block ? s.src_len - o : cz::kLz4Block);
    const uint32_t c = csize[j];
    const bool raw = c >= n;
    const uint32_t sz = raw ? n : c;
    if (threadIdx.x == 0) {
      const uint32_t word = sz | (raw ? 0x80000000u : 0u);
      dst[op] = (uint8_t)word; dst[op + 1] = (uint8_t)(word >> 8); dst[op + 2] = (uint8_t)(word >> 16); dst[op + 3] = (uint8_t)(word >> 24);
    }
    team_copy(t, dst + op + 4, raw ? src_base + s.src_off + o : tmp + (size_t)j * cz::kLz4Slot, sz);
    op += 4 + sz;
  }
  if (threadIdx.x == 0) {
    dst[op] = dst[op + 1] = dst[op + 2] = dst[op + 3] = 0;  // EndMark
    dst_len[i] = op + 4;
  }
}
__global__ void __launch_bounds__(256) k_lz4_assemble(const SliceDesc* __restrict__ slices, const uint8_t* __restrict__ src_base,
                                                      const uint8_t* tmp, const uint32_t* __restrict__ csize, uint8_t* dst_base,
                                                      uint64_t* dst_len) {
  lz4_assemble(slices, blockIdx.x, src_base, tmp, csize, dst_base, dst_len);
}

// ---- zstd: every 128 KiB block of every slice -> staged payload; meta[2j] = payload offset in the slot, meta[2j+1] = size (0 = raw)
template <class WN>
__global__ void __launch_bounds__(32) k_zstd_blocks(const SliceDesc* __restrict__ slices, uint32_t n_slices, uint32_t total_blocks,
                                                    const uint8_t* __restrict__ src_base, uint8_t* tmp, uint64_t* seq_scratch,
                                                    uint32_t* meta) {
  extern __shared__ __align__(16) uint8_t zsm[];  // one warp per CTA: the input window, then the hash table
  uint8_t* D = zsm;
  uint16_t* tab = reinterpret_cast<uint16_t*>(zsm + ZstdLaunch<WN>::kWindow);
  const cz::Warp w{threadIdx.x, 32u};
  uint64_t* seqs = seq_scratch + (size_t)blockIdx.x * cz::kZstdMaxSeq;
  for (uint32_t j = blockIdx.x; j < total_blocks; j += gridDim.x) {
    const uint32_t si = slice_of_block(slices, n_slices, j);
    const SliceDesc s = slices[si];
    const uint64_t o = (uint64_t)(j - s.blk_first) * cz::kZstdCBlock;
    const uint32_t n = (uint32_t)(s.src_len - o < cz::kZstdCBlock ? s.src_len - o : cz::kZstdCBlock);
    uint32_t poff = 0;
    const uint32_t c = cz::zstd_compress_block<WN>(w, src_base + s.src_off, (uint32_t)o, n, tmp + (size_t)j * cz::kZstdSlot, seqs, D, tab,
                                               &poff);
    if (w.lane == 0) { meta[2 * j] = poff; meta[2 * j + 1] = c; }
    __syncwarp();
  }
}

// ---- zstd long effort (levels >= 20): candidate index per round of units, then one warp per 128 KiB block
// A unit: slice positions [lo, hi) indexed, [parse_lo, hi) parsed (cz::zstd_long_block); q0 = round position of lo.
struct LongUnit {
  uint64_t src_off;    // slice start in the source
  uint32_t lo, parse_lo, hi, q0;
  uint32_t blk_first;  // global block index of the block at parse_lo
};
constexpr int kLongCtasPerSm = 8;  // one warp per CTA; bounds the per-CTA sequence scratch

// keys[q] for every position q < n_pos of the round (units ascending in q0)
__global__ void __launch_bounds__(256) k_long_keys(const LongUnit* __restrict__ units, uint32_t n_units, uint32_t n_pos,
                                                   const uint8_t* __restrict__ src_base, uint64_t* keys) {
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_pos; q += gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = n_units;
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (units[mid].q0 <= q) lo = mid; else hi = mid;
    }
    const LongUnit u = units[lo];
    keys[q] = cz::long_key(src_base + u.src_off, u.lo + (q - u.q0), u.hi, q);
  }
}

// rank[q] = where q's key landed in the sorted order
__global__ void __launch_bounds__(256) k_long_rank(const uint64_t* __restrict__ sk, uint32_t n_pos, uint32_t* rank) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pos; i += gridDim.x * blockDim.x)
    rank[(uint32_t)sk[i] & (cz::kLongRound - 1u)] = i;
}

// blocks [blk0, blk0 + n_blk) of the round (its units ascending in blk_first); meta as k_zstd_blocks writes it
__global__ void __launch_bounds__(32) k_long_blocks(const LongUnit* __restrict__ units, uint32_t n_units, uint32_t blk0,
                                                    uint32_t n_blk, const uint8_t* __restrict__ src_base,
                                                    const uint64_t* __restrict__ sk, const uint32_t* __restrict__ rank,
                                                    uint8_t* tmp, uint64_t* seq_scratch, uint32_t* meta) {
  __shared__ __align__(16) uint32_t scratch[cz::kPayloadScratch / 4];
  __shared__ uint32_t bl[cz::kLongBatch], bo[cz::kLongBatch];
  const cz::Warp w{threadIdx.x, 32u};
  uint64_t* seqs = seq_scratch + (size_t)blockIdx.x * cz::kZstdMaxSeq;
  for (uint32_t j = blk0 + blockIdx.x; j < blk0 + n_blk; j += gridDim.x) {
    uint32_t lo = 0, hi = n_units;
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (units[mid].blk_first <= j) lo = mid; else hi = mid;
    }
    const LongUnit u = units[lo];
    const uint32_t bstart = u.parse_lo + (j - u.blk_first) * cz::kZstdCBlock;
    const uint32_t n = u.hi - bstart < cz::kZstdCBlock ? u.hi - bstart : cz::kZstdCBlock;
    const cz::LongIndex ix{sk, rank, u.q0, u.lo};
    uint32_t poff = 0;
    const uint32_t c = cz::zstd_long_block(w, src_base + u.src_off, ix, bstart, n, tmp + (size_t)j * cz::kZstdSlot, seqs, bl, bo,
                                           scratch, &poff);
    if (w.lane == 0) { meta[2 * j] = poff; meta[2 * j + 1] = c; }
    __syncwarp();
  }
}

// ---- zstd frame assembly: the CTA writes slice i's frame at dst_base + dst_off (k_zstd_assemble: one CTA per slice)
ZN_D void zstd_assemble(const SliceDesc* __restrict__ slices, uint32_t i, const uint8_t* __restrict__ src_base, const uint8_t* tmp,
                        const uint32_t* __restrict__ meta, uint8_t* dst_base, uint64_t* dst_len) {
  const SliceDesc s = slices[i];
  uint8_t* dst = dst_base + s.dst_off;
  const Team t{threadIdx.x, blockDim.x};
  if (s.src_len == 0) {  // same bytes as libzstd: single-segment, 1-byte content size 0, empty raw last block
    if (threadIdx.x == 0) {
      const uint8_t e[9] = {0x28, 0xB5, 0x2F, 0xFD, 0x20, 0x00, 0x01, 0x00, 0x00};
      for (int k = 0; k < 9; k++) dst[k] = e[k];
      dst_len[i] = 9;
    }
    return;
  }
  if (threadIdx.x == 0) cz::zstd_frame_header(dst, s.src_len);
  uint64_t op = 13;
  for (uint32_t b = 0; b < s.n_blocks; b++) {
    const uint32_t j = s.blk_first + b;
    const uint64_t o = (uint64_t)b * cz::kZstdCBlock;
    const uint32_t n = (uint32_t)(s.src_len - o < cz::kZstdCBlock ? s.src_len - o : cz::kZstdCBlock);
    const uint32_t poff = meta[2 * j], c = meta[2 * j + 1];
    const uint32_t last = b + 1 == s.n_blocks ? 1u : 0u;
    if (c == 0) {
      if (threadIdx.x == 0) cz::zstd_block_header(dst + op, last, 0, n);
      team_copy(t, dst + op + 3, src_base + s.src_off + o, n);
      op += 3 + n;
    } else {
      if (threadIdx.x == 0) cz::zstd_block_header(dst + op, last, 2, c);
      team_copy(t, dst + op + 3, tmp + (size_t)j * cz::kZstdSlot + poff, c);
      op += 3 + c;
    }
  }
  if (threadIdx.x == 0) dst_len[i] = op;
}
__global__ void __launch_bounds__(256) k_zstd_assemble(const SliceDesc* __restrict__ slices, const uint8_t* __restrict__ src_base,
                                                       const uint8_t* tmp, const uint32_t* __restrict__ meta, uint8_t* dst_base,
                                                       uint64_t* dst_len) {
  zstd_assemble(slices, blockIdx.x, src_base, tmp, meta, dst_base, dst_len);
}

// ---- packed layout (device-resident compress plans): blob i = [ZNB1 header] + frame, or header + the slice's bytes when
// the envelope stores it RAW; blobs back to back.  One CTA: per tile of slices, every thread sizes one slice from the
// block results (cz::zstd_frame_size / lz4_frame_size), the CTA scans the sizes, and each thread writes its slice's
// offset, its frame's destination (past the header) into slices[i].dst_off, the RAW decision and the header.
constexpr int kLayoutThreads = 1024;
__global__ void __launch_bounds__(kLayoutThreads) k_pack_layout(SliceDesc* slices, uint32_t n, const uint32_t* __restrict__ res,
                                                                uint32_t lz4, uint32_t envelope, uint8_t* dst_base,
                                                                uint64_t* offsets, uint32_t* raw) {
  __shared__ uint64_t warp_sum[kLayoutThreads / 32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint64_t carry = 0;  // bytes of the tiles before this one (every thread keeps the same value)
  for (uint32_t base = 0; base < n; base += kLayoutThreads) {
    const uint32_t i = base + threadIdx.x;
    uint64_t sz = 0, len = 0;
    uint32_t hl = 0, r = 0;
    if (i < n) {
      const SliceDesc s = slices[i];
      len = s.src_len;
      sz = lz4 ? cz::lz4_frame_size(len, res + s.blk_first) : cz::zstd_frame_size(len, res + 2 * (size_t)s.blk_first);
      if (envelope) {
        r = sz >= len;
        hl = cz::znb1_header_len(len);
        sz = hl + (r ? len : sz);
      }
    }
    uint64_t incl = sz;  // inclusive scan inside the warp, then over the warps' sums
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) {
      const uint64_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if (lane >= d) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    uint64_t before = 0, tile = 0;
    for (uint32_t k = 0; k < kLayoutThreads / 32; k++) {
      const uint64_t v = warp_sum[k];
      before += k < warp ? v : 0;
      tile += v;
    }
    const uint64_t off = carry + before + incl - sz;
    if (i < n) {
      offsets[i] = off;
      slices[i].dst_off = off + hl;
      raw[i] = r;
      if (envelope) cz::znb1_header(dst_base + off, r ? cz::kZnb1Raw : (lz4 ? cz::kZnb1Lz4Frame : cz::kZnb1Zstd), len);
    }
    carry += tile;
    __syncthreads();  // warp_sum is rewritten by the next tile
  }
  if (threadIdx.x == 0) offsets[n] = carry;
}

// Frames straight into the packed layout (one CTA per slice); a RAW row gets the slice's bytes instead of its frame.
// dst_len receives the frame lengths, as from k_zstd_assemble / k_lz4_assemble.
template <bool LZ4>
__global__ void __launch_bounds__(256) k_assemble_packed(const SliceDesc* __restrict__ slices, const uint8_t* __restrict__ src_base,
                                                         const uint8_t* tmp, const uint32_t* __restrict__ res,
                                                         const uint32_t* __restrict__ raw, uint8_t* dst_base, uint64_t* dst_len) {
  if (raw[blockIdx.x]) {
    const SliceDesc s = slices[blockIdx.x];
    team_copy(Team{threadIdx.x, blockDim.x}, dst_base + s.dst_off, src_base + s.src_off, (uint32_t)s.src_len);
    return;
  }
  if (LZ4) lz4_assemble(slices, blockIdx.x, src_base, tmp, res, dst_base, dst_len);
  else zstd_assemble(slices, blockIdx.x, src_base, tmp, res, dst_base, dst_len);
}

}  // namespace zn
