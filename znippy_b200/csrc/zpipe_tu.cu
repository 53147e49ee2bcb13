// Translation unit of the device-wide zstd decode pipeline: kernels (zpipe_kernels.cuh) + their launcher.
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "host_api.h"
#include "zpipe_kernels.cuh"

namespace zn {
namespace zp {

__global__ void k_zinit(ZPools* pools, uint32_t seq_cap, uint32_t lit_cap16, uint32_t tab_cap, uint32_t comp_cap) {
  ZPools z;
  z.seq_used = 0; z.seq_cap = seq_cap;
  z.lit_used16 = 0; z.lit_cap16 = lit_cap16;
  z.tab_used = 0; z.tab_cap = tab_cap;
  z.comp_used = 0; z.comp_cap = comp_cap;
  *pools = z;
}

bool pipeline_init() {
  static FseD zset[kTabSet];
  build_predef_set(zset);
  if (cudaMemcpyToSymbol(g_zpredef, zset, sizeof zset) != cudaSuccess) return false;
  cudaFuncSetAttribute(k_zseq1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSeq1Smem);
  cudaFuncSetAttribute(k_zlit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLitSmem);
  cudaFuncSetAttribute(k_zexec2<512, 4, 16384, 2, 8192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Exec2Shared<512, 4, 16384, 8192>));
  cudaFuncSetAttribute(k_zexec2<512, 2, 16384, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Exec2Shared<512, 2, 16384, 4096>));
  return true;
}

void pipeline_trace_dump() {
#ifdef ZP_TRACE
  unsigned long long h[32];
  cudaMemcpyFromSymbol(h, g_ztrace, sizeof h);
  fprintf(stderr, "zexec2 trace (thread 0 cycles summed over CTAs): other %llu formation %llu lits+prefetch %llu setup %llu jobs %llu rounds %llu flush %llu rest %llu | rounds %llu groups %llu unknown-after-round %llu scan-rounds %llu jobs %llu\n",
          h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8], h[9], h[10], h[11], h[12]);
  unsigned long long z[32] = {0};
  cudaMemcpyToSymbol(g_ztrace, z, sizeof z);
#endif
}

uint32_t pipeline_enqueue(const PipelineLaunch& L, cudaStream_t st, cudaEvent_t* marks) {
  const ZArgs& a = L.a;
  const uint32_t sms = L.sm_count, slots = L.slots;
  int m = 0;
  auto mark = [&]() { if (marks) cudaEventRecord(marks[m++], st); };
  mark();
  k_zinit<<<1, 1, 0, st>>>(a.pools, L.seq_cap, L.lit_cap16, L.tab_cap, slots);
  k_zwalk<<<(a.nzb + 63) / 64, 64, 0, st>>>(a);
  mark();
  // (Running the literal kernel on a second stream beside tables + seq was measured and removed: 67.8 ms instead of
  // 45.4 ms per step on real text — its 48 KB-per-CTA blocks crowd the sequence decoders off the SMs.)
  const uint32_t lit_grid = std::min<uint32_t>((slots + kLitBlocks - 1) / kLitBlocks, sms * 3);
  k_ztables<<<std::min<uint32_t>((slots + kTabWarps - 1) / kTabWarps, sms * 8), kTabWarps * 32, 0, st>>>(a);
  mark();
  // Sequence stage.  The two-phase form runs its state chains ~7x faster per sequence but only kSeq1Lanes blocks per SM at
  // a time; the one-pass form has every block of the batch in flight at once.  So: two-phase when the blocks are long
  // (large blobs: ~10 000 sequences each) or when there are no more of them than two rounds of lanes; one-pass for
  // batches of very many small blobs (40 000 files of 2-48 KB: 4.2 ms against 6.3).
  const uint64_t est_blocks = L.mean_bytes * a.nzb / kZstdBlockMax + a.nzb;
  const bool large = L.mean_bytes >= (256u << 10);
  uint32_t n_launch = 7;
  if (large || est_blocks <= 2ull * sms * kSeq1Lanes) {
    k_zseq1<<<std::min<uint32_t>((slots + kSeq1Lanes - 1) / kSeq1Lanes, sms), 64, kSeq1Smem, st>>>(a);
    if (marks && getenv("ZN_ZPROF_SEQ1")) { cudaEventRecord(marks[8], st); }  // development: end of phase 1
    k_zseq2<<<std::min<uint32_t>((slots + kSeq2Warps - 1) / kSeq2Warps, sms * 16), kSeq2Warps * 32, 0, st>>>(a);
    n_launch = 8;
  } else {
    k_zseq_g<<<(slots + 31) / 32, 32, 0, st>>>(a);
  }
  mark();
  k_zlit<<<lit_grid, kLitBlocks * 4, kLitSmem, st>>>(a);
  mark();
  k_zchain<<<(a.nzb + 63) / 64, 64, 0, st>>>(a);
  mark();
  // exec: the team shape follows the mean decoded size, with the same threshold as the sequence stage
  if (large)
    k_zexec2<512, 4, 16384, 2, 8192><<<std::min<uint32_t>(a.nzb, sms * 2), 512, sizeof(Exec2Shared<512, 4, 16384, 8192>), st>>>(
        a, L.d_out, L.produced, L.exec_counter);
  else
    k_zexec2<512, 2, 16384, 3><<<std::min<uint32_t>(a.nzb, sms * 3), 512, sizeof(Exec2Shared<512, 2, 16384, 4096>), st>>>(
        a, L.d_out, L.produced, L.exec_counter);
  mark();
  return n_launch;
}

}  // namespace zp
}  // namespace zn
