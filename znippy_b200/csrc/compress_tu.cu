// Translation unit of the compression kernels (compress_kernels.cuh) + their host launcher.
#include <cub/device/device_radix_sort.cuh>

#include "host_api.h"
#include "compress_kernels.cuh"

namespace zn {

void compress_init_attrs() {
  cz::PredefCTables ct;
  cz::build_predef_ctables(&ct);
  cudaMemcpyToSymbol(cz::g_predef_c, &ct, sizeof ct);
  cudaFuncSetAttribute(k_zstd_blocks<cz::WinFast>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZstdLaunch<cz::WinFast>::kSmemBytes);
  cudaFuncSetAttribute(k_zstd_blocks<cz::WinMid>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZstdLaunch<cz::WinMid>::kSmemBytes);
  cudaFuncSetAttribute(k_zstd_blocks<cz::WinHigh>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZstdLaunch<cz::WinHigh>::kSmemBytes);
}

size_t compress_bound(size_t n, int codec) {
  if (codec == 2) return n + 4 * ((n + cz::kLz4Block - 1) / cz::kLz4Block) + 32;
  return n + 3 * ((n + cz::kZstdCBlock - 1) / cz::kZstdCBlock) + 32;
}

template <typename T>
static bool grow(T** p, size_t* cap, size_t need_bytes) {
  if (*cap >= need_bytes) return true;
  if (*p) cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  if (cudaMalloc((void**)p, need_bytes) != cudaSuccess) { cudaGetLastError(); return false; }
  *cap = need_bytes;
  return true;
}

// Radix sort of the round's keys (the bits in use only), captured into a graph so that its kernels can be counted.
static cudaError_t long_sort(CompressScratch* cs, cudaStream_t st, cub::DoubleBuffer<uint64_t>* db, uint32_t n, uint32_t* launches) {
  size_t temp = 0;
  cudaError_t e = cub::DeviceRadixSort::SortKeys(nullptr, temp, *db, n, 0, (int)cz::kLongKeyBits, st);
  if (e != cudaSuccess) return e;
  if (!grow((uint8_t**)&cs->lsort, &cs->lsort_cap, std::max<size_t>(temp, 1))) return cudaErrorMemoryAllocation;
  cudaGraph_t g = nullptr;
  cudaGraphExec_t ge = nullptr;
  e = cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed);
  if (e != cudaSuccess) return e;
  const cudaError_t es = cub::DeviceRadixSort::SortKeys(cs->lsort, temp, *db, n, 0, (int)cz::kLongKeyBits, st);
  e = cudaStreamEndCapture(st, &g);
  if (es != cudaSuccess) e = es;
  if (e == cudaSuccess) {
    size_t nn = 0;
    cudaGraphGetNodes(g, nullptr, &nn);
    std::vector<cudaGraphNode_t> nodes(nn);
    cudaGraphGetNodes(g, nodes.data(), &nn);
    for (cudaGraphNode_t node : nodes) {
      cudaGraphNodeType t;
      if (cudaGraphNodeGetType(node, &t) == cudaSuccess && t == cudaGraphNodeTypeKernel) (*launches)++;
    }
    e = cudaGraphInstantiate(&ge, g, 0);
    if (e == cudaSuccess) e = cudaGraphLaunch(ge, st);
  }
  if (ge) cudaGraphExecDestroy(ge);
  if (g) cudaGraphDestroy(g);
  return e;
}

// Long effort: units of every slice, grouped into rounds of <= kLongRound indexed positions; per round the keys, the
// sort, the ranks and the block parse.  Fills meta for every block, as k_zstd_blocks does.
static int long_blocks(CompressScratch* cs, cudaStream_t st, int sm_count, const uint8_t* d_src, const std::vector<SliceDesc>& sl,
                       uint32_t* d_meta, uint32_t* launches, std::string* err) {
  std::vector<LongUnit> units;
  std::vector<uint32_t> round_first{0};  // units [round_first[r], round_first[r + 1]) form round r
  std::vector<uint32_t> round_pos;       // indexed positions of round r
  uint32_t cur = 0, max_blk = 0, blk = 0;
  for (const SliceDesc& d : sl) {
    for (uint64_t ps = 0; ps < d.src_len; ps += cz::kLongPiece) {
      LongUnit u;
      u.src_off = d.src_off;
      u.parse_lo = (uint32_t)ps;
      u.lo = (uint32_t)(ps - std::min<uint64_t>(ps, cz::kLongReach));
      u.hi = (uint32_t)std::min<uint64_t>(ps + cz::kLongPiece, d.src_len);
      u.blk_first = d.blk_first + (uint32_t)(ps / cz::kZstdCBlock);
      const uint32_t len = u.hi - u.lo;
      if (cur + (uint64_t)len > cz::kLongRound) {
        round_pos.push_back(cur);
        round_first.push_back((uint32_t)units.size());
        max_blk = std::max(max_blk, blk);
        cur = blk = 0;
      }
      u.q0 = cur;
      cur += len;
      blk += (u.hi - u.parse_lo + cz::kZstdCBlock - 1) / cz::kZstdCBlock;
      units.push_back(u);
    }
  }
  if (units.empty()) return 0;
  round_pos.push_back(cur);
  round_first.push_back((uint32_t)units.size());
  max_blk = std::max(max_blk, blk);
  const uint32_t max_pos = *std::max_element(round_pos.begin(), round_pos.end());
  const uint32_t grid = std::max<uint32_t>(1, std::min<uint32_t>(max_blk, (uint32_t)sm_count * kLongCtasPerSm));
  if (!grow((uint8_t**)&cs->lunits, &cs->lunits_cap, units.size() * sizeof(LongUnit)) ||
      !grow(&cs->lkeys0, &cs->lkeys0_cap, (size_t)max_pos * 8) || !grow(&cs->lkeys1, &cs->lkeys1_cap, (size_t)max_pos * 8) ||
      !grow(&cs->seqs, &cs->seqs_cap, (size_t)grid * cz::kZstdMaxSeq * 8)) {
    *err = "compress scratch allocation failed";
    return -3;
  }
  LongUnit* d_units = (LongUnit*)cs->lunits;
  if (cudaMemcpyAsync(d_units, units.data(), units.size() * sizeof(LongUnit), cudaMemcpyHostToDevice, st) != cudaSuccess) {
    *err = "compress H2D failed";
    return -2;
  }
  for (size_t r = 0; r + 1 < round_first.size(); r++) {
    const uint32_t u0 = round_first[r], nu = round_first[r + 1] - u0, np = round_pos[r];
    const uint32_t pgrid = std::min<uint32_t>((np + 255) / 256, (uint32_t)sm_count * 16);
    k_long_keys<<<pgrid, 256, 0, st>>>(d_units + u0, nu, np, d_src, cs->lkeys0);
    cub::DoubleBuffer<uint64_t> db(cs->lkeys0, cs->lkeys1);
    const cudaError_t e = long_sort(cs, st, &db, np, launches);
    if (e != cudaSuccess) {
      cudaGetLastError();
      *err = std::string("long-effort key sort: ") + cudaGetErrorString(e);
      return e == cudaErrorMemoryAllocation ? -3 : -2;
    }
    uint32_t* rank = reinterpret_cast<uint32_t*>(db.Alternate());
    k_long_rank<<<pgrid, 256, 0, st>>>(db.Current(), np, rank);
    const uint32_t blk0 = units[u0].blk_first, nblk = units[u0 + nu - 1].blk_first - blk0 +
                          (units[u0 + nu - 1].hi - units[u0 + nu - 1].parse_lo + cz::kZstdCBlock - 1) / cz::kZstdCBlock;
    k_long_blocks<<<std::min(grid, nblk), 32, 0, st>>>(d_units + u0, nu, blk0, nblk, d_src, db.Current(), rank, cs->tmp, cs->seqs, d_meta);
    *launches += 3;
  }
  return 0;
}

// Compresses n slices resident on the device into frames at d_dst + dst_off[i]; synchronises `st` before returning.
int compress_run(CompressScratch* cs, cudaStream_t st, int sm_count, const uint8_t* d_src, const uint64_t* src_off,
                        const uint64_t* src_len, uint32_t n, int level, int codec, uint8_t* d_dst, const uint64_t* dst_off,
                        const uint64_t* /*dst_cap*/, uint64_t* out_len, uint32_t* status, uint32_t* launches, std::string* err) {
  // zstd: the level picks the match finder: three window geometries, then (levels >= 20) the whole-slice long effort;
  // LZ4 has one effort
  const int effort = level <= 2 ? 0 : (level <= 9 ? 1 : (level <= 19 ? 2 : 3));
  const bool lz4 = codec == 2;
  const uint64_t bsz = lz4 ? cz::kLz4Block : cz::kZstdCBlock;
  std::vector<SliceDesc> sl(n);
  uint64_t total_blocks = 0;
  for (uint32_t i = 0; i < n; i++) {
    sl[i].src_off = src_off[i];
    sl[i].src_len = src_len[i];
    sl[i].dst_off = dst_off[i];
    sl[i].blk_first = (uint32_t)total_blocks;
    sl[i].n_blocks = (uint32_t)((src_len[i] + bsz - 1) / bsz);
    total_blocks += sl[i].n_blocks;
    status[i] = src_len[i] >= 0xFFFFFFF0ull ? 4u /*UNSUPPORTED*/ : 0u;
    if (status[i]) { *err = "slice too large"; return -1; }
  }
  if (total_blocks > 0x7FFFFFFFull) { *err = "too many blocks"; return -1; }
  const uint32_t nb = (uint32_t)total_blocks;
  const size_t slot = lz4 ? cz::kLz4Slot : cz::kZstdSlot;
  const uint32_t wpc = lz4 ? kLz4WarpsPerCta : kZstdWarpsPerCta;
  const uint32_t grid = std::max<uint32_t>(1, std::min<uint32_t>((nb + wpc - 1) / wpc, (uint32_t)sm_count * (lz4 ? 6u : (effort == 0 ? ZstdLaunch<cz::WinFast>::kCtasPerSm
                                                                  : effort == 1 ? ZstdLaunch<cz::WinMid>::kCtasPerSm
                                                                                : ZstdLaunch<cz::WinHigh>::kCtasPerSm))));
  const size_t small_bytes = (size_t)n * sizeof(SliceDesc) + (size_t)nb * 8 + (size_t)n * 8 + 64;
  if (!grow(&cs->tmp, &cs->tmp_cap, std::max<size_t>(1, (size_t)nb * slot)) ||
      !grow((uint8_t**)&cs->small, &cs->small_cap, small_bytes) ||
      (!lz4 && effort < 3 && !grow(&cs->seqs, &cs->seqs_cap, (size_t)grid * wpc * cz::kZstdMaxSeq * 8))) {
    *err = "compress scratch allocation failed";
    return -3;
  }
  SliceDesc* d_sl = (SliceDesc*)cs->small;
  uint32_t* d_meta = (uint32_t*)((uint8_t*)cs->small + (size_t)n * sizeof(SliceDesc));
  uint64_t* d_len = (uint64_t*)((uint8_t*)d_meta + (size_t)nb * 8);
  d_len = (uint64_t*)(((uintptr_t)d_len + 7) & ~(uintptr_t)7);
  if (cudaMemcpyAsync(d_sl, sl.data(), (size_t)n * sizeof(SliceDesc), cudaMemcpyHostToDevice, st) != cudaSuccess) {
    *err = "compress H2D failed";
    return -2;
  }
  if (!cs->ev[0]) { cudaEventCreate(&cs->ev[0]); cudaEventCreate(&cs->ev[1]); }
  *launches = 0;
  cudaEventRecord(cs->ev[0], st);
  if (nb && !lz4 && effort == 3) {
    const int rc = long_blocks(cs, st, sm_count, d_src, sl, d_meta, launches, err);
    if (rc) return rc;
  } else if (nb) {
    if (lz4) k_lz4_blocks<<<grid, kLz4WarpsPerCta * 32, 0, st>>>(d_sl, n, nb, d_src, cs->tmp, d_meta);
    else if (effort == 0)
      k_zstd_blocks<cz::WinFast><<<grid, 32, ZstdLaunch<cz::WinFast>::kSmemBytes, st>>>(d_sl, n, nb, d_src, cs->tmp, cs->seqs, d_meta);
    else if (effort == 1)
      k_zstd_blocks<cz::WinMid><<<grid, 32, ZstdLaunch<cz::WinMid>::kSmemBytes, st>>>(d_sl, n, nb, d_src, cs->tmp, cs->seqs, d_meta);
    else
      k_zstd_blocks<cz::WinHigh><<<grid, 32, ZstdLaunch<cz::WinHigh>::kSmemBytes, st>>>(d_sl, n, nb, d_src, cs->tmp, cs->seqs, d_meta);
    (*launches)++;
  }
  if (lz4) k_lz4_assemble<<<n, 256, 0, st>>>(d_sl, d_src, cs->tmp, d_meta, d_dst, d_len);
  else k_zstd_assemble<<<n, 256, 0, st>>>(d_sl, d_src, cs->tmp, d_meta, d_dst, d_len);
  (*launches)++;
  cudaEventRecord(cs->ev[1], st);
  if (cudaMemcpyAsync(out_len, d_len, (size_t)n * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess) {
    *err = std::string("compress kernels: ") + cudaGetErrorString(cudaGetLastError());
    return -2;
  }
  cudaEventElapsedTime(&cs->last_ms, cs->ev[0], cs->ev[1]);
  return 0;
}


}  // namespace zn
