// Development tool: per-phase clock trace of ONE CTA decoding ONE blob (latency budget of a zstd block).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DZN_TRACE -o tools/bin/trace_decode tools/trace_decode.cu
//   tools/bin/trace_decode blob.zst <decoded size> [n_ctas]
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
#ifndef TRACE_NT
#define TRACE_NT 256
#define TRACE_KB 1
#endif
__device__ unsigned long long g_trace[4096];
__device__ unsigned int g_trace_n;
__device__ unsigned long long g_cnt[16];
#if defined(__CUDA_ARCH__)
#define ZN_CNT(i, v) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) atomicAdd(&g_cnt[i], (unsigned long long)(v)); } while (0)
#else
#define ZN_CNT(i, v) do {} while (0)
#endif
#if defined(__CUDA_ARCH__)
#define ZN_TP(id)                                                            \
  do {                                                                       \
    if (threadIdx.x == 0 && blockIdx.x == 0) {                               \
      unsigned int i__ = g_trace_n;                                          \
      if (i__ < 4096) { g_trace[i__] = ((unsigned long long)(id) << 56) | (clock64() & 0xFFFFFFFFFFFFFFull); g_trace_n = i__ + 1; } \
    }                                                                        \
  } while (0)
#else
#define ZN_TP(id) do {} while (0)
#endif
#include "../znippy_b200/csrc/par_kernel.cuh"
using namespace zn;

int main(int argc, char** argv) {
  FILE* f = fopen(argv[1], "rb");
  std::vector<uint8_t> blob(16 << 20);
  size_t n = fread(blob.data(), 1, blob.size(), f);
  fclose(f);
  const uint64_t out_len = strtoull(argv[2], 0, 10);
  const int nb = argc > 3 ? atoi(argv[3]) : 1;
  uint8_t *d_in, *d_out, *d_lit;
  cudaMalloc(&d_in, n + 256);
  cudaMalloc(&d_out, out_len * nb + 256);
  cudaMalloc(&d_lit, (size_t)kLitStride * nb);
  cudaMemcpy(d_in, blob.data(), n, cudaMemcpyHostToDevice);
  std::vector<BlobDesc> descs(nb);
  std::vector<uint32_t> list(nb);
  for (int i = 0; i < nb; i++) {
    descs[i] = BlobDesc{0, n, out_len * i, out_len, 0, (uint32_t)(out_len / 1024), F_COMPRESSED};
    list[i] = i;
  }
  BlobDesc* d_desc; uint32_t *d_list, *d_status, *d_prod, *d_ctr;
  cudaMalloc(&d_desc, sizeof(BlobDesc) * nb); cudaMalloc(&d_list, 4 * nb); cudaMalloc(&d_status, 4 * nb); cudaMalloc(&d_prod, 4 * nb); cudaMalloc(&d_ctr, 4);
  cudaMemcpy(d_desc, descs.data(), sizeof(BlobDesc) * nb, cudaMemcpyHostToDevice);
  cudaMemcpy(d_list, list.data(), 4 * nb, cudaMemcpyHostToDevice);
  PredefTables pd;
  { zs::FseTable t; uint16_t next[64];
    zs::fse_build(&t, zs::kLLDefault, 36, 6, next); for (int i = 0; i < 64; i++) pd.ll[i] = t.e[i];
    zs::fse_build(&t, zs::kOFDefault, 29, 5, next); for (int i = 0; i < 32; i++) pd.of[i] = t.e[i];
    zs::fse_build(&t, zs::kMLDefault, 53, 6, next); for (int i = 0; i < 64; i++) pd.ml[i] = t.e[i]; }
  cudaMemcpyToSymbol(g_predef, &pd, sizeof pd);
  uint8_t* d_par = nullptr;
#ifdef TRACE_PAR
  cudaMalloc(&d_par, par::kParScratchPerCta * nb);
  cudaFuncSetAttribute(par::k_decode_par, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(par::ParShared));
#endif
  for (int rep = 0; rep < 2; rep++) {
    unsigned int zero = 0;
    cudaMemcpyToSymbol(g_trace_n, &zero, 4);
    cudaMemset(d_ctr, 0, 4);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0);
#ifdef TRACE_PAR
    par::k_decode_par<<<nb, par::kParThreads, sizeof(par::ParShared)>>>(d_desc, d_list, nb, d_in, d_out, d_par, d_status, d_prod, d_ctr);
#else
    k_decode<TRACE_NT, TRACE_KB><<<(nb + TRACE_KB - 1) / TRACE_KB, TRACE_NT>>>(d_desc, d_list, nb, d_in, d_out, d_lit, d_status, d_prod, d_ctr, nullptr, 1u, nullptr, 0u);
#endif
    cudaEventRecord(e1);
    cudaDeviceSynchronize();
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    uint32_t st; cudaMemcpy(&st, d_status, 4, cudaMemcpyDeviceToHost);
    printf("rep %d: %d CTAs, %.3f ms, status %u, %s\n", rep, nb, ms, st, cudaGetErrorString(cudaGetLastError()));
  }
  static unsigned long long tr[4096];
  unsigned int tn;
  cudaMemcpyFromSymbol(&tn, g_trace_n, 4);
  cudaMemcpyFromSymbol(tr, g_trace, sizeof tr);
  if (tn > 4096) tn = 4096;
  const int first = argc > 4 ? atoi(argv[4]) : 20;
  // print phases of blocks first..first+3 (steady state): id, delta cycles
  unsigned long long prev = 0;
  int blocks = 0;
  for (unsigned i = 0; i < tn; i++) {
    const unsigned id = (unsigned)(tr[i] >> 56);
    const unsigned long long c = tr[i] & 0xFFFFFFFFFFFFFFull;
    if (id == 1 || id == 30) blocks++;
    if (blocks >= first && blocks < first + 4) printf("  blk %d  tp %2u  +%llu cyc\n", blocks, id, prev ? c - prev : 0ull);
    prev = c;
  }
  unsigned long long cnt[16];
  cudaMemcpyFromSymbol(cnt, g_cnt, sizeof cnt);
  for (int i = 0; i < 8; i++) printf("cnt[%d] = %llu\n", i, cnt[i]);
  return 0;
}
