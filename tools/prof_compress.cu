// Development tool: where a warp of k_zstd_blocks spends its cycles (per-phase clock64 sums over all warps).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o tools/bin/prof_compress tools/prof_compress.cu
//   tools/bin/prof_compress file [bytes]
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
__device__ unsigned long long g_cprof[16];
#if defined(__CUDA_ARCH__)
#define ZN_CP_BEGIN() long long cp__ = clock64()
#define ZN_CP(i) do { long long n__ = clock64(); if (w.lane == 0) atomicAdd(&g_cprof[i], (unsigned long long)(n__ - cp__)); cp__ = clock64(); } while (0)
#else
#define ZN_CP_BEGIN() do {} while (0)
#define ZN_CP(i) do {} while (0)
#endif
#include "../znippy_b200/csrc/compress_kernels.cuh"
using namespace zn;

int main(int argc, char** argv) {
  FILE* f = fopen(argv[1], "rb");
  if (!f) return 1;
  size_t cap = argc > 2 ? strtoull(argv[2], 0, 10) : (64u << 20);
  std::vector<uint8_t> data(cap);
  size_t n = fread(data.data(), 1, cap, f);
  fclose(f);
  while (n < cap) { size_t k = n < cap - n ? n : cap - n; memcpy(data.data() + n, data.data(), k); n += k; }
  compress_init_attrs();
  uint8_t *d_src, *d_dst;
  cudaMalloc(&d_src, n + 64);
  cudaMalloc(&d_dst, compress_bound(n, 1) + 64);
  cudaMemcpy(d_src, data.data(), n, cudaMemcpyHostToDevice);
  CompressScratch cs;
  cudaDeviceProp pr; cudaGetDeviceProperties(&pr, 0);
  uint64_t so = 0, sl = n, dofs = 0, dcap = compress_bound(n, 1), olen = 0; uint32_t st = 0, launches = 0; std::string err;
  for (int rep = 0; rep < 2; rep++) {
    unsigned long long z[16] = {0};
    cudaMemcpyToSymbol(g_cprof, z, sizeof z);
    int rc = compress_run(&cs, 0, pr.multiProcessorCount, d_src, &so, &sl, 1, argc > 3 ? atoi(argv[3]) : 1, 1, d_dst, &dofs, &dcap, &olen, &st, &launches, &err);
    printf("rep %d rc %d: %zu -> %llu bytes, %.3f ms (%.2f GB/s) %s\n", rep, rc, n, (unsigned long long)olen, cs.last_ms, n / cs.last_ms / 1e6, err.c_str());
  }
  unsigned long long c[16];
  cudaMemcpyFromSymbol(c, g_cprof, sizeof c);
  const char* names[9] = {"table init+prime", "load/hash/lookup", "probe", "argmax+insert", "extend", "literal copy", "tail", "-", "huffman+sequences"};
  unsigned long long tot = 0;
  for (int i = 0; i < 9; i++) tot += c[i];
  for (int i = 0; i < 9; i++) printf("  %-18s %12llu cyc  %5.1f%%\n", names[i], c[i], 100.0 * c[i] / tot);
  return 0;
}
