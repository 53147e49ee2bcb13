// Shared device/host definitions for libznippy_cuda (sm_100a).
#pragma once
#include <cstdint>
#include <cstddef>

#if defined(__CUDACC__)
#define ZN_HD __host__ __device__ __forceinline__
#define ZN_D __device__ __forceinline__
#else
#define ZN_HD inline
#define ZN_D inline
#endif

#ifndef ZN_CNT
#define ZN_CNT(i, v) do {} while (0)  // debug counters, only live in tools/trace_decode.cu
#endif
#ifndef ZN_TP
#define ZN_TP(id) do {} while (0)  // phase trace points, only live in tools/trace_decode.cu
#endif

namespace zn {

// per-blob status values; must match include/znippy_cuda.h
enum : uint32_t {
  S_OK = 0,
  S_DECODE_ERROR = 1,
  S_DIGEST_MISMATCH = 2,
  S_DST_TOO_SMALL = 3,
  S_UNSUPPORTED = 4,
  S_SIZE_MISMATCH = 5
};

// blob flags in BlobDesc.flags
enum : uint32_t {
  F_COMPRESSED = 1u,   // run the codec; otherwise content == blob bytes (store-as-is, decompress.rs:164-166)
  F_HAS_EXPECT = 2u,   // compare digest with expect[]
  F_HASHED = 8u,       // chunk chaining values are written by the fused decode+hash kernel, k_b3_chunks skips the blob
  F_LZ4_BLOCK = 4u     // the blob is one raw LZ4 block (no frame, no magic): compressed[i] == 2 in the C ABI
};

// One row of the batch (index row: blob_offset, blob_size, uncompressed_size, compressed — index.rs:45-52).
struct BlobDesc {
  uint64_t src_off;   // offset of the blob inside the blobs buffer
  uint64_t src_len;   // blob_size
  uint64_t dst_off;   // offset of the content inside the output buffer (16-byte aligned by the planner)
  uint64_t dst_cap;   // uncompressed_size from the index = output capacity and expected length
  uint64_t cv_base;   // first slot of this blob in the chunk chaining-value array
  uint32_t n_chunks;  // max(1, ceil(dst_cap / 1024))
  uint32_t flags;
};

#if defined(__CUDACC__)
// 16-byte global -> shared copies that bypass L1 (the hash kernels stage their input through these)
ZN_D void cp_async16(void* smem_dst, const void* gmem_src) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src) : "memory");
}
ZN_D void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
ZN_D void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }
#endif

constexpr uint32_t kChunk = 1024;
constexpr uint32_t kWarp = 32;
constexpr uint32_t kZstdBlockMax = 128u * 1024u;

}  // namespace zn
