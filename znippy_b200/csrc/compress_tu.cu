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
  cudaFuncSetAttribute(k_zstd_blocks<cz::WinFast, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZstdLaunch<cz::WinFast>::kSmemBytes);
  cudaFuncSetAttribute(k_zstd_blocks<cz::WinMid, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZstdLaunch<cz::WinMid>::kSmemBytes);
  cudaFuncSetAttribute(k_zstd_blocks<cz::WinHigh, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZstdLaunch<cz::WinHigh>::kSmemBytes);
}

size_t compress_bound(size_t n, int codec) {
  const CodecWord cw = codec_parts(codec);
  const size_t nb = (n + cz::kZstdCBlock - 1) / cz::kZstdCBlock;
  if (cw.seekable)  // exact: every block stored raw in a frame of its own (cz::zstd_seekable_size)
    return n ? n + (13 + 3 + cz::kSeekEntry) * nb + cz::kSeekFixed : 9 + cz::kSeekEntry + cz::kSeekFixed;
  const size_t ck = cw.checksum ? 4 : 0;
  if (cw.base == ZN_CODEC_LZ4) return n + 4 * ((n + cz::kLz4Block - 1) / cz::kLz4Block) + 32 + ck;
  return n + 3 * nb + 32 + ck;
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

// Kernels of the radix sort of `n` keys (the bits in use only): the sort is captured into a graph, which is counted
// and dropped.  The temporary storage must already hold cs->lsort_cap >= temp bytes.
static cudaError_t long_sort_launches(CompressScratch* cs, cudaStream_t st, uint32_t n, size_t temp, uint32_t* launches) {
  cub::DoubleBuffer<uint64_t> db(cs->lkeys0, cs->lkeys1);
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed);
  if (e != cudaSuccess) return e;
  const cudaError_t es = cub::DeviceRadixSort::SortKeys(cs->lsort, temp, db, n, 0, (int)cz::kLongKeyBits, st);
  e = cudaStreamEndCapture(st, &g);
  if (es != cudaSuccess) e = es;
  *launches = 0;
  if (e == cudaSuccess) {
    size_t nn = 0;
    cudaGraphGetNodes(g, nullptr, &nn);
    std::vector<cudaGraphNode_t> nodes(nn);
    cudaGraphGetNodes(g, nodes.data(), &nn);
    for (cudaGraphNode_t node : nodes) {
      cudaGraphNodeType t;
      if (cudaGraphNodeGetType(node, &t) == cudaSuccess && t == cudaGraphNodeTypeKernel) (*launches)++;
    }
  }
  if (g) cudaGraphDestroy(g);
  return e;
}

// Long effort: units of every slice, grouped into rounds of <= kLongRound indexed positions; per round the keys, the
// sort, the ranks and the block parse (compress_enqueue).  Here: the units and rounds, the scratch, the sort's
// temporary storage and kernel count, and the units' upload.
static int long_prepare(CompressScratch* cs, cudaStream_t st, int sm_count, const std::vector<SliceDesc>& sl, CompressPrep* P,
                        std::string* err) {
  std::vector<LongUnit> units;
  std::vector<uint32_t>& round_first = P->round_first;  // units [round_first[r], round_first[r + 1]) form round r
  std::vector<uint32_t>& round_pos = P->round_pos;      // indexed positions of round r
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
  P->long_grid = std::max<uint32_t>(1, std::min<uint32_t>(max_blk, (uint32_t)sm_count * kLongCtasPerSm));
  if (!grow((uint8_t**)&cs->lunits, &cs->lunits_cap, units.size() * sizeof(LongUnit)) ||
      !grow(&cs->lkeys0, &cs->lkeys0_cap, (size_t)max_pos * 8) || !grow(&cs->lkeys1, &cs->lkeys1_cap, (size_t)max_pos * 8) ||
      !grow(&cs->seqs, &cs->seqs_cap, (size_t)P->long_grid * cz::kZstdMaxSeq * 8)) {
    *err = "compress scratch allocation failed";
    return -3;
  }
  for (size_t r = 0; r + 1 < round_first.size(); r++) {
    const uint32_t u0 = round_first[r], nu = round_first[r + 1] - u0;
    const LongUnit& ul = units[u0 + nu - 1];
    P->round_blk0.push_back(units[u0].blk_first);
    P->round_nblk.push_back(ul.blk_first - units[u0].blk_first + (ul.hi - ul.parse_lo + cz::kZstdCBlock - 1) / cz::kZstdCBlock);
    size_t temp = 0;
    cub::DoubleBuffer<uint64_t> db(cs->lkeys0, cs->lkeys1);
    const cudaError_t e = cub::DeviceRadixSort::SortKeys(nullptr, temp, db, round_pos[r], 0, (int)cz::kLongKeyBits, st);
    if (e != cudaSuccess) {
      cudaGetLastError();
      *err = std::string("long-effort key sort: ") + cudaGetErrorString(e);
      return -2;
    }
    P->sort_temp = std::max(P->sort_temp, std::max<size_t>(temp, 1));
  }
  if (!grow((uint8_t**)&cs->lsort, &cs->lsort_cap, P->sort_temp)) {
    *err = "compress scratch allocation failed";
    return -3;
  }
  for (size_t r = 0; r + 1 < round_first.size(); r++) {
    uint32_t k = 0;
    const cudaError_t e = long_sort_launches(cs, st, round_pos[r], P->sort_temp, &k);
    if (e != cudaSuccess) {
      cudaGetLastError();
      *err = std::string("long-effort key sort: ") + cudaGetErrorString(e);
      return -2;
    }
    P->round_sort_launches.push_back(k);
    P->launches += 3 + k;
  }
  if (cudaMemcpyAsync(cs->lunits, units.data(), units.size() * sizeof(LongUnit), cudaMemcpyHostToDevice, st) != cudaSuccess) {
    *err = "compress H2D failed";
    return -2;
  }
  return 0;
}

int compress_prepare(CompressScratch* cs, cudaStream_t st, int sm_count, const uint64_t* src_off, const uint64_t* src_len,
                     uint32_t n, int level, const CodecWord& cw, const uint64_t* dst_off, CompressPrep* P, uint32_t* status,
                     std::string* err) {
  // zstd: the level picks the match finder: three window geometries, then (levels >= 20) the whole-slice long effort;
  // LZ4 has one effort
  const int effort = level <= 2 ? 0 : (level <= 9 ? 1 : (level <= 19 ? 2 : 3));
  const bool seekable = cw.seekable, lz4 = cw.base == ZN_CODEC_LZ4;
  const uint64_t bsz = lz4 ? cz::kLz4Block : cz::kZstdCBlock;
  std::vector<SliceDesc> sl(n);
  uint64_t total_blocks = 0;
  for (uint32_t i = 0; i < n; i++) {
    sl[i].src_off = src_off[i];
    sl[i].src_len = src_len[i];
    sl[i].dst_off = dst_off ? dst_off[i] : 0;
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
  const size_t small_bytes = (size_t)n * sizeof(SliceDesc) + (size_t)nb * 8 + (size_t)n * 8 + (size_t)n * 4 + 64 +
                             (seekable ? (size_t)nb * 4 : 0) + (cw.checksum ? (size_t)n * 4 : 0);
  if (!grow(&cs->tmp, &cs->tmp_cap, std::max<size_t>(1, (size_t)nb * slot)) ||
      !grow((uint8_t**)&cs->small, &cs->small_cap, small_bytes) ||
      (!lz4 && effort < 3 && !grow(&cs->seqs, &cs->seqs_cap, (size_t)grid * wpc * cz::kZstdMaxSeq * 8))) {
    *err = "compress scratch allocation failed";
    return -3;
  }
  *P = CompressPrep();
  P->lz4 = lz4;
  P->seekable = seekable;
  P->checksum = cw.checksum;
  P->effort = effort;
  P->n = n;
  P->nb = nb;
  P->grid = grid;
  P->sm_count = (uint32_t)sm_count;
  P->d_sl = (SliceDesc*)cs->small;
  P->d_meta = (uint32_t*)((uint8_t*)cs->small + (size_t)n * sizeof(SliceDesc));
  uint64_t* d_len = (uint64_t*)((uint8_t*)P->d_meta + (size_t)nb * 8);
  P->d_len = (uint64_t*)(((uintptr_t)d_len + 7) & ~(uintptr_t)7);
  P->d_raw = (uint32_t*)(P->d_len + n);
  if (seekable) P->d_xxh = P->d_raw + n;
  if (cw.checksum) P->d_csum = P->d_raw + n;
  if (cudaMemcpyAsync(P->d_sl, sl.data(), (size_t)n * sizeof(SliceDesc), cudaMemcpyHostToDevice, st) != cudaSuccess) {
    *err = "compress H2D failed";
    return -2;
  }
  if (cw.checksum && n) P->launches = 1;  // k_slice_xxh
  if (nb && !lz4 && effort == 3) return long_prepare(cs, st, sm_count, sl, P, err);
  if (nb) P->launches += seekable ? 2 : 1;
  return 0;
}

int compress_enqueue(CompressScratch* cs, const CompressPrep& P, cudaStream_t st, const uint8_t* d_src, std::string* err) {
  if (P.checksum && P.n) {
    const uint32_t grid = std::min<uint32_t>((P.n + kSliceXxhWarps - 1) / kSliceXxhWarps, P.sm_count * 16u);
    if (P.lz4) k_slice_xxh<32><<<grid, kSliceXxhWarps * 32, 0, st>>>(P.d_sl, P.n, d_src, P.d_csum);
    else k_slice_xxh<64><<<grid, kSliceXxhWarps * 32, 0, st>>>(P.d_sl, P.n, d_src, P.d_csum);
  }
  if (!P.nb) return 0;
  if (!P.lz4 && P.effort == 3) {
    const LongUnit* d_units = (const LongUnit*)cs->lunits;
    for (size_t r = 0; r + 1 < P.round_first.size(); r++) {
      const uint32_t u0 = P.round_first[r], nu = P.round_first[r + 1] - u0, np = P.round_pos[r];
      const uint32_t pgrid = std::min<uint32_t>((np + 255) / 256, P.sm_count * 16);
      k_long_keys<<<pgrid, 256, 0, st>>>(d_units + u0, nu, np, d_src, cs->lkeys0);
      cub::DoubleBuffer<uint64_t> db(cs->lkeys0, cs->lkeys1);
      size_t temp = P.sort_temp;
      const cudaError_t e = cub::DeviceRadixSort::SortKeys(cs->lsort, temp, db, np, 0, (int)cz::kLongKeyBits, st);
      if (e != cudaSuccess) {
        cudaGetLastError();
        *err = std::string("long-effort key sort: ") + cudaGetErrorString(e);
        return -2;
      }
      uint32_t* rank = reinterpret_cast<uint32_t*>(db.Alternate());
      k_long_rank<<<pgrid, 256, 0, st>>>(db.Current(), np, rank);
      k_long_blocks<<<std::min(P.long_grid, P.round_nblk[r]), 32, 0, st>>>(d_units + u0, nu, P.round_blk0[r], P.round_nblk[r], d_src,
                                                                          db.Current(), rank, cs->tmp, cs->seqs, P.d_meta);
    }
    return 0;
  }
  const uint32_t n = P.n, nb = P.nb, grid = P.grid;
  if (P.seekable) {
    k_block_xxh<<<(nb + kXxhThreads - 1) / kXxhThreads, kXxhThreads, 0, st>>>(P.d_sl, n, nb, d_src, P.d_xxh);
    if (P.effort == 0)
      k_zstd_blocks<cz::WinFast, true><<<grid, 32, ZstdLaunch<cz::WinFast>::kSmemBytes, st>>>(P.d_sl, n, nb, d_src, cs->tmp, cs->seqs, P.d_meta);
    else if (P.effort == 1)
      k_zstd_blocks<cz::WinMid, true><<<grid, 32, ZstdLaunch<cz::WinMid>::kSmemBytes, st>>>(P.d_sl, n, nb, d_src, cs->tmp, cs->seqs, P.d_meta);
    else
      k_zstd_blocks<cz::WinHigh, true><<<grid, 32, ZstdLaunch<cz::WinHigh>::kSmemBytes, st>>>(P.d_sl, n, nb, d_src, cs->tmp, cs->seqs, P.d_meta);
    return 0;
  }
  if (P.lz4) k_lz4_blocks<<<grid, kLz4WarpsPerCta * 32, 0, st>>>(P.d_sl, n, nb, d_src, cs->tmp, P.d_meta);
  else if (P.effort == 0)
    k_zstd_blocks<cz::WinFast><<<grid, 32, ZstdLaunch<cz::WinFast>::kSmemBytes, st>>>(P.d_sl, n, nb, d_src, cs->tmp, cs->seqs, P.d_meta);
  else if (P.effort == 1)
    k_zstd_blocks<cz::WinMid><<<grid, 32, ZstdLaunch<cz::WinMid>::kSmemBytes, st>>>(P.d_sl, n, nb, d_src, cs->tmp, cs->seqs, P.d_meta);
  else
    k_zstd_blocks<cz::WinHigh><<<grid, 32, ZstdLaunch<cz::WinHigh>::kSmemBytes, st>>>(P.d_sl, n, nb, d_src, cs->tmp, cs->seqs, P.d_meta);
  return 0;
}

void compress_pack(CompressScratch* cs, const CompressPrep& P, cudaStream_t st, const uint8_t* d_src, uint8_t* d_dst,
                   uint64_t* d_offsets, bool envelope) {
  if (!P.n) return;
  k_pack_layout<<<1, kLayoutThreads, 0, st>>>(P.d_sl, P.n, P.d_meta, P.lz4 ? 1u : 0u, P.seekable ? 1u : 0u, P.checksum ? 1u : 0u,
                                              envelope ? 1u : 0u, d_dst, d_offsets, P.d_raw);
  if (P.lz4) k_assemble_packed<true><<<P.n, 256, 0, st>>>(P.d_sl, d_src, cs->tmp, P.d_meta, nullptr, P.d_csum, P.d_raw, d_dst, P.d_len);
  else k_assemble_packed<false><<<P.n, 256, 0, st>>>(P.d_sl, d_src, cs->tmp, P.d_meta, P.d_xxh, P.d_csum, P.d_raw, d_dst, P.d_len);
}

// Compresses n slices resident on the device into frames at d_dst + dst_off[i]; synchronises `st` before returning.
int compress_run(CompressScratch* cs, cudaStream_t st, int sm_count, const uint8_t* d_src, const uint64_t* src_off,
                        const uint64_t* src_len, uint32_t n, int level, const CodecWord& cw, uint8_t* d_dst, const uint64_t* dst_off,
                        const uint64_t* /*dst_cap*/, uint64_t* out_len, uint32_t* status, uint32_t* launches, std::string* err) {
  CompressPrep P;
  *launches = 0;
  int rc = compress_prepare(cs, st, sm_count, src_off, src_len, n, level, cw, dst_off, &P, status, err);
  if (rc) return rc;
  if (!cs->ev[0]) { cudaEventCreate(&cs->ev[0]); cudaEventCreate(&cs->ev[1]); }
  cudaEventRecord(cs->ev[0], st);
  rc = compress_enqueue(cs, P, st, d_src, err);
  if (rc) return rc;
  *launches = P.launches;
  if (P.lz4) k_lz4_assemble<<<n, 256, 0, st>>>(P.d_sl, d_src, cs->tmp, P.d_meta, P.d_csum, d_dst, P.d_len);
  else k_zstd_assemble<<<n, 256, 0, st>>>(P.d_sl, d_src, cs->tmp, P.d_meta, P.d_xxh, P.d_csum, d_dst, P.d_len);
  (*launches)++;
  cudaEventRecord(cs->ev[1], st);
  if (cudaMemcpyAsync(out_len, P.d_len, (size_t)n * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess) {
    *err = std::string("compress kernels: ") + cudaGetErrorString(cudaGetLastError());
    return -2;
  }
  cudaEventElapsedTime(&cs->last_ms, cs->ev[0], cs->ev[1]);
  return 0;
}


}  // namespace zn
