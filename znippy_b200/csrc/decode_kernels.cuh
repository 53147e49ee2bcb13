// K1/K2: batched blob decode.  A persistent grid of CTAs pulls blobs from a work counter (largest first, so the
// tail of the batch is made of small blobs); each CTA is the "team" of zstd_decode.cuh / lz4_decode.cuh.
// Replaces the codec call of the reference's read loop (znippy-common/src/decompress.rs:156-166) and of
// ZnippyArchive::extract_file (archive.rs:159-164) for a whole batch of index rows at once.
#pragma once
#include "lz4_decode.cuh"

namespace zn {

constexpr uint32_t kLitStride = kZstdBlockMax + 256;  // per-CTA Huffman literal scratch
constexpr uint32_t kSrcStage = 8192;                  // blobs up to this size are parsed out of shared memory

constexpr uint32_t kSrcSmall = 2048;                  // ... and blobs up to this size are staged K at a time

// Warp-wide copy global -> shared (any alignment), used to stage the next small blobs while nobody else waits.
ZN_D void warp_stage(uint8_t* dst, const uint8_t* src, uint32_t n, uint32_t lane) {
  for (uint32_t i = lane; i < n; i += 32) dst[i] = __ldg(src + i);
}

// `only_if` (nullable): word only_if[i * only_stride] != 0 selects list item i; null = every item.
// NT threads per team; the CTA claims KB work items per atomic and its first KB warps fetch their descriptors (and
// stage blobs <= kSrcSmall) in parallel, so the three dependent global round trips (counter -> list -> descriptor ->
// bytes) are paid once per KB blobs instead of once per blob.  This is what bounds the 100 000 x 10 KiB-file corpus.
// kStop (range reads): blob i is decoded only up to the block that reaches stop[i] (zs::StopAt) into its full-size
// output; it fails with S_SIZE_MISMATCH when its frames end before stop[i].
template <int NT, int KB, bool kStop = false>
__global__ void __launch_bounds__(NT, NT == 32 ? 16 : 512 / NT) k_decode(const BlobDesc* __restrict__ blobs, const uint32_t* __restrict__ list,
                                                         uint32_t n_list, const uint8_t* blobs_base, uint8_t* out_base,
                                                         uint8_t* lit_scratch, uint32_t* status, uint32_t* produced,
                                                         uint32_t* work_counter, uint32_t* cvs, uint32_t one,
                                                         const uint32_t* only_if, uint32_t only_stride,
                                                         const uint32_t* __restrict__ stop = nullptr) {
  __shared__ DecShared sh;
  __shared__ uint32_t s_base;
  __shared__ BlobDesc s_desc[KB];
  __shared__ uint32_t s_blob[KB];
  // Small blobs (every blob of the pattern corpora and of the 10 KiB-file corpus is < 1 KiB) are parsed out of shared
  // memory, so that the serial header / bit-stream parsing costs ~30 cycles per access instead of an HBM trip.
  // One-warp teams (NT == 32, the small-blob configuration) carry no mid-size stage and no bulk-store tile: 21 KB of
  // shared memory per blob in flight instead of 43 KB, so ~10 blobs decode concurrently per SM instead of 4.
  constexpr bool kWide = NT > 32;
  __shared__ __align__(16) uint8_t s_src[kWide ? kSrcStage + 32 : 16];
  __shared__ __align__(16) uint8_t s_small[KB][kSrcSmall + 32];
  __shared__ __align__(128) uint8_t s_tile[kWide ? kTileBytes : 128];
  if (threadIdx.x == 0) sh.tile = kWide ? s_tile : nullptr;
  zs::init_luts(Team{threadIdx.x, (uint32_t)NT}, &sh);
  const Team t{threadIdx.x, (uint32_t)NT};
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  uint8_t* lit = lit_scratch + (size_t)blockIdx.x * kLitStride;
  uint32_t predef = 0;  // which of sh.ll/of/ml currently hold the predefined tables: survives frames and blobs
  for (;;) {
    if (threadIdx.x == 0) s_base = atomicAdd(work_counter, (uint32_t)KB);
    __syncthreads();
    const uint32_t base = s_base;
    ZN_TP(20);
    if (base >= n_list) break;
    for (uint32_t k = warp; k < (uint32_t)KB && base + k < n_list; k += NT / 32) {
      const uint32_t blob = list[base + k];
      const BlobDesc d = blobs[blob];
      if (lane == 0) {
        s_desc[k] = d;
        s_blob[k] = blob;
      }
      if (d.src_len <= kSrcSmall) warp_stage(s_small[k] + 16, blobs_base + d.src_off, (uint32_t)d.src_len, lane);
    }
    __syncthreads();
    ZN_TP(21);
    for (uint32_t k = 0; k < (uint32_t)KB && base + k < n_list; k++) {
      // second pass behind the device-wide pipeline (zpipe.cuh): only the rows it handed back (flag word != 0)
      if (only_if && only_if[(size_t)(base + k) * only_stride] == 0) continue;
      const uint32_t blob = s_blob[k];
      const BlobDesc d = s_desc[k];
      uint32_t st, got = 0;
      if (d.src_len >= 0xFFFFFFF0ull || d.dst_cap >= 0xFFFFFFF0ull) {
        st = S_UNSUPPORTED;
      } else {
        const uint8_t* src = blobs_base + d.src_off;
        if (d.src_len <= kSrcSmall) {
          src = s_small[k] + 16;
        } else if (kWide && d.src_len <= kSrcStage) {
          team_copy(t, s_src + 16, src, (uint32_t)d.src_len);
          __syncthreads();
          src = s_src + 16;
        }
        if (kStop) {
          zs::StopAt h;
          h.stop = stop[blob];
          st = decode_blob(t, &sh, src, (uint32_t)d.src_len, out_base + d.dst_off, (uint32_t)d.dst_cap, lit, predef, &got, h);
          if (st == S_OK && got < h.stop) st = S_SIZE_MISMATCH;
        } else if (d.flags & F_LZ4_BLOCK) {
          st = decode_lz4_block(t, &sh, src, (uint32_t)d.src_len, out_base + d.dst_off, (uint32_t)d.dst_cap, &got);
        } else {
          st = decode_blob(t, &sh, src, (uint32_t)d.src_len, out_base + d.dst_off, (uint32_t)d.dst_cap, lit, predef, &got);
        }
        if (!kStop && st == S_OK && got != (uint32_t)d.dst_cap) st = S_SIZE_MISMATCH;
      }
      ZN_TP(22);
      if (kWide && threadIdx.x < kBulkIssuers) bulk_wait_all();  // bulk stores read the tile: drain before it is reused
      __syncthreads();  // every path out of decode_blob is team-uniform; this also fences the blob's last stores
      ZN_TP(23);
      if (threadIdx.x == 0) {
        status[blob] = st;
        produced[blob] = got;
      }
    }
  }
}

// Store-as-is rows with an output buffer (decompress.rs:164-166 + the pwrite source): plain gather, one CTA per
// 64 KiB piece so that a single 200 MiB jar still spreads over the whole machine.
constexpr uint32_t kGatherPiece = 64u * 1024u;
__global__ void __launch_bounds__(256) k_gather_raw(const BlobDesc* __restrict__ blobs,
                                                    const uint32_t* __restrict__ piece_blob,
                                                    const uint32_t* __restrict__ piece_idx, uint32_t n_pieces,
                                                    const uint8_t* __restrict__ blobs_base, uint8_t* out_base) {
  for (uint32_t p = blockIdx.x; p < n_pieces; p += gridDim.x) {
    const BlobDesc d = blobs[piece_blob[p]];
    const uint64_t o = (uint64_t)piece_idx[p] * kGatherPiece;
    const uint64_t rem = d.dst_cap - o;
    const uint32_t n = rem < kGatherPiece ? (uint32_t)rem : kGatherPiece;
    const Team t{threadIdx.x, blockDim.x};
    team_copy(t, out_base + d.dst_off + o, blobs_base + d.src_off + o, n);
  }
}


// Rows whose payload is a Zstandard frame without its magic (envelope layer, compressed == 3): the four bytes in front of
// the payload become the magic, so every decoder sees an ordinary frame.
__global__ void __launch_bounds__(256) k_patch_magic(uint8_t* blobs_base, const uint64_t* __restrict__ off, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t* p = blobs_base + off[i];
  p[0] = 0x28; p[1] = 0xB5; p[2] = 0x2F; p[3] = 0xFD;
}


// Frames of a compress batch packed back to back for the way home (one warp per frame): n small device-to-host copies
// cost ~3 us each, one copy of the packed bytes costs their size.
__global__ void __launch_bounds__(256) k_pack_frames(const uint8_t* __restrict__ src, const uint64_t* __restrict__ src_off,
                                                     const uint64_t* __restrict__ len, const uint64_t* __restrict__ dst_off,
                                                     uint32_t n, uint8_t* dst) {
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const Team t{threadIdx.x & 31u, 32u, 0u};
  for (uint32_t i = warp; i < n; i += nwarps) team_copy(t, dst + dst_off[i], src + src_off[i], (uint32_t)len[i]);
}

}  // namespace zn
