// Host-side interfaces between the translation units of libznippy_cuda.so (znippy_cuda.cu: C ABI, decode and hash
// kernels; compress_tu.cu: compression kernels; zpipe_tu.cu: the device-wide zstd decode pipeline).  Splitting the
// library keeps a change to one kernel family from recompiling the other two.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "codec_word.h"
#include "zpipe.cuh"

namespace zn {

// ---------------------------------------------------------------------------------------------- compress_tu.cu
struct CompressScratch {
  uint8_t* tmp = nullptr;
  size_t tmp_cap = 0;
  uint64_t* seqs = nullptr;
  size_t seqs_cap = 0;
  void* small = nullptr;  // slices + meta + dst_len
  size_t small_cap = 0;
  // long effort (levels >= 20): units of the batch, the round's keys (sorted in place between the two buffers; the
  // buffer the sort leaves free holds the rank array) and the sort's temporary storage
  void* lunits = nullptr;
  size_t lunits_cap = 0;
  uint64_t* lkeys0 = nullptr;
  size_t lkeys0_cap = 0;
  uint64_t* lkeys1 = nullptr;
  size_t lkeys1_cap = 0;
  void* lsort = nullptr;
  size_t lsort_cap = 0;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  float last_ms = 0.f;  // device time of the kernels of the last compress_run
  void release() {
    if (tmp) cudaFree(tmp);
    if (seqs) cudaFree(seqs);
    if (small) cudaFree(small);
    if (lunits) cudaFree(lunits);
    if (lkeys0) cudaFree(lkeys0);
    if (lkeys1) cudaFree(lkeys1);
    if (lsort) cudaFree(lsort);
    if (ev[0]) cudaEventDestroy(ev[0]);
    if (ev[1]) cudaEventDestroy(ev[1]);
    ev[0] = ev[1] = nullptr;
    tmp = nullptr; seqs = nullptr; small = nullptr;
    tmp_cap = seqs_cap = small_cap = 0;
    lunits = nullptr; lkeys0 = nullptr; lkeys1 = nullptr; lsort = nullptr;
    lunits_cap = lkeys0_cap = lkeys1_cap = lsort_cap = 0;
  }
};
void compress_init_attrs();
size_t compress_bound(size_t n, int codec);  // zn_compress_bound: raw-block fallback makes this exact
struct SliceDesc;
// What compress_prepare works out from the slice sizes alone: the effort, the grid, the device descriptors (inside the
// scratch), and for the long effort the rounds of units, each with its block range and the kernels of its key sort.
struct CompressPrep {
  bool lz4 = false;
  bool seekable = false;  // zstd only, levels <= 19: one frame per block and a seek table (cz::zstd_seek_table)
  bool checksum = false;  // ZN_CODEC_CHECKSUM: every frame ends in its content checksum
  int effort = 0;
  uint32_t n = 0, nb = 0, grid = 0, sm_count = 0;
  SliceDesc* d_sl = nullptr;   // n slice descriptors
  uint32_t* d_meta = nullptr;  // per-block results: zstd {payload offset, size} pairs, LZ4 sizes
  uint64_t* d_len = nullptr;   // n frame lengths
  uint32_t* d_raw = nullptr;   // n RAW decisions of the packed layout
  uint32_t* d_xxh = nullptr;   // seekable: nb block checksums (k_block_xxh); nullptr otherwise
  uint32_t* d_csum = nullptr;  // checksum: n slice checksums (k_slice_xxh); nullptr otherwise
  std::vector<uint32_t> round_first{0}, round_pos, round_blk0, round_nblk, round_sort_launches;
  uint32_t long_grid = 0;
  size_t sort_temp = 0;
  uint32_t launches = 0;  // kernels compress_enqueue launches
};
// Plans a batch: grows `cs` to fit, uploads the descriptors on `st` (dst_off[i]: where slice i's frame goes; nullable
// for a packed layout, which places the frames on the device).  No kernel runs.  `cw` has passed codec_split.
int compress_prepare(CompressScratch* cs, cudaStream_t st, int sm_count, const uint64_t* src_off, const uint64_t* src_len,
                     uint32_t n, int level, const CodecWord& cw, const uint64_t* dst_off, CompressPrep* P, uint32_t* status,
                     std::string* err);
// Enqueues the block kernels of a prepared batch on `st` (P.launches kernels): fills the per-block results.
int compress_enqueue(CompressScratch* cs, const CompressPrep& P, cudaStream_t st, const uint8_t* d_src, std::string* err);
// Enqueues the packed layout and the frame assembly after compress_enqueue (2 kernels; none when P.n == 0):
// d_offsets[0..n] (exclusive prefix sum of the blob sizes), ZNB1 headers when `envelope`, and every blob in place.
void compress_pack(CompressScratch* cs, const CompressPrep& P, cudaStream_t st, const uint8_t* d_src, uint8_t* d_dst,
                   uint64_t* d_offsets, bool envelope);
// Compresses n slices resident on the device into frames at d_dst + dst_off[i]; synchronises `st` before returning.
int compress_run(CompressScratch* cs, cudaStream_t st, int sm_count, const uint8_t* d_src, const uint64_t* src_off,
                 const uint64_t* src_len, uint32_t n, int level, const CodecWord& cw, uint8_t* d_dst, const uint64_t* dst_off,
                 const uint64_t* dst_cap, uint64_t* out_len, uint32_t* status, uint32_t* launches, std::string* err);

// ---------------------------------------------------------------------------------------------- zpipe_tu.cu
namespace zp {
bool pipeline_init();  // predefined tables + kernel attributes, once per context
struct PipelineLaunch {
  ZArgs a;
  uint32_t slots, seq_cap, lit_cap16, tab_cap;  // pool capacities of this batch
  uint32_t sm_count;
  uint64_t mean_bytes;  // mean decoded size of the batch's blobs: picks the exec team size
  uint8_t* d_out;
  uint32_t* produced;
  uint32_t* exec_counter;
};
// Enqueues init, walk, tables, seq (one kernel, or phase 1 + phase 2 for batches of large blobs), lit, chain, exec on
// `st` and returns the number of launches (7 or 8).  `marks` (nullable): 9 events; [0..6] are recorded before the first
// kernel and after walk / tables / seq / lit / chain / exec, [8] after seq phase 1 when ZN_ZPROF_SEQ1 is set.
uint32_t pipeline_enqueue(const PipelineLaunch& L, cudaStream_t st, cudaEvent_t* marks);
void pipeline_trace_dump();  // development builds (ZN_TRACE_BUILD=1): prints and clears the exec kernel's phase counters
}  // namespace zp

}  // namespace zn

// ---------------------------------------------------------------------------------------------- znippy_cuda.cu
// Windowed host-buffer decode behind zn_archive_read_ranges (container.cpp declares it too: it is compiled without the
// CUDA headers).  Row i (compressed[i]: 1 = frame, 2 = raw LZ4 block) decodes into device scratch of out_len[i] bytes:
//   stop[i] < out_len[i] and a frame: only up to the block that reaches stop[i] (k_decode<.., true>), no digest tree and
//                                     no content checksum; S_SIZE_MISMATCH when the frames end before stop[i];
//   otherwise:                        in full, through the plan of zn_decode_verify_batch (no expected digests).
// Then only the n_win windows come back: win_len[w] bytes at offset win_off[w] of row win_row[w], packed back to back
// into `pack` (host memory, pinned for speed).  status[i] as zn_decode_verify_batch; produced[i] = bytes decoded.
struct zn_ctx;
extern "C" int zn_decode_windows(zn_ctx* c, const uint8_t* blobs_base, const uint64_t* blob_off, const uint64_t* blob_len,
                                 const uint8_t* compressed, const uint64_t* out_len, const uint64_t* stop, uint32_t n,
                                 const uint32_t* win_row, const uint64_t* win_off, const uint64_t* win_len, uint32_t n_win,
                                 uint8_t* pack, uint32_t* status, uint64_t* produced);
// zn_decode_windows that also checks frames of seekable payloads (n_ck of them, nullable arrays when 0): bytes
// [ck_off[k], + ck_len[k]) of row ck_row[k], decoded in full, must have the low 32 bits of XXH64 ck_sum[k]
// (k_frame_xxh_check); a mismatch turns a good row's status into S_DECODE_ERROR.
extern "C" int zn_decode_windows_checked(zn_ctx* c, const uint8_t* blobs_base, const uint64_t* blob_off, const uint64_t* blob_len,
                                         const uint8_t* compressed, const uint64_t* out_len, const uint64_t* stop, uint32_t n,
                                         const uint32_t* win_row, const uint64_t* win_off, const uint64_t* win_len, uint32_t n_win,
                                         const uint32_t* ck_row, const uint64_t* ck_off, const uint64_t* ck_len,
                                         const uint32_t* ck_sum, uint32_t n_ck, uint8_t* pack, uint32_t* status, uint64_t* produced);
