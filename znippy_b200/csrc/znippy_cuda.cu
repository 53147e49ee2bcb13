// libznippy_cuda.so — host side of the C ABI declared in include/znippy_cuda.h (sm_100a only, no CPU fallback).
//
// A zn_ctx owns one device, one stream, device staging buffers and the decode scratch; a zn_plan owns the device
// descriptor tables of one batch (the index rows blob_offset/blob_size/compressed/uncompressed_size/checksum of
// znippy-common/src/index.rs:45-52) and can be run any number of times on resident data; a compress plan also owns its
// compressor scratch, so that it runs on any stream beside other plans and the ctx's own calls.  The host-buffer entry
// points are the plan API wrapped in one H2D copy before and one D2H copy after.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <numeric>
#include <string>
#include <unordered_map>
#include <vector>

#define ZN_BACKBITS_DEPTH 1  // one-team decoders: see bitio.cuh
#include "../../include/znippy_cuda.h"
#include "blake3_kernels.cuh"
#include "host_api.h"
#include "decode_kernels.cuh"
#include "par_kernel.cuh"
#include "fused_ws.cuh"

using namespace zn;

// --------------------------------------------------------------------------------------------- ctx / plan
struct zn_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;  // hash stream of the overlapped schedule
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
  // pinned bump arena for the per-row arrays of a plan (descriptors, chunk prefix, work lists): built in place and uploaded
  // by DMA — from pageable vectors the driver staged ~10 MB per 100 000 rows through its own bounce buffer first
  uint8_t* plan_pin = nullptr;
  size_t plan_pin_cap = 0, plan_pin_used = 0;
  template <typename T>
  T* arena(size_t count) {
    plan_pin_used = (plan_pin_used + 63) & ~(size_t)63;
    T* r = reinterpret_cast<T*>(plan_pin + plan_pin_used);
    plan_pin_used += count * sizeof(T);
    return r;
  }
  uint8_t* d_lit = nullptr;  // Huffman literal scratch, one slot per decode CTA
  uint8_t* d_par = nullptr;  // scratch of the block-parallel decoder (sequence records + literals), allocated on first use
  uint32_t dec_grid = 0;
  uint32_t dec_grid_small = 0;
  uint8_t* d_in = nullptr;   // staging for the host-buffer API
  size_t d_in_cap = 0;
  uint8_t* d_out = nullptr;
  size_t d_out_cap = 0;
  CompressScratch cs;        // compressor work space (grown on demand)
  // scratch of the device-wide zstd pipeline (zpipe.cuh), grown on demand: block table, work list, fat FSE tables,
  // sequence records, regenerated literals, pool counters
  struct ZScratch {
    zp::ZBlock* blocks = nullptr; uint32_t* comp_list = nullptr; size_t slots = 0;
    zp::FseD* tabs = nullptr; size_t tab_sets = 0;
    zp::SeqRec16* recs = nullptr; size_t seqs = 0;
    zp::SeqP1* p1 = nullptr; size_t p1s = 0;
    uint8_t* lits = nullptr; size_t lit16 = 0;
    zp::ZPools* pools = nullptr;
  } zs;
  uint64_t launches = 0;
  std::string err;
};

enum PlanKind { PLAN_DECODE_VERIFY = 1, PLAN_HASH = 2, PLAN_COMPRESS = 3 };

// decode classes: every compressed row of a batch is routed by its own sizes (index columns only, no device feedback)
enum DecClass {
  DC_PIPE = 0,  // entropy-coded Zstandard frames: device-wide pipeline (zpipe.cuh)
  DC_BIGPAT,    // large and highly compressible (pattern corpora): fused decode+hash, TMA bulk stores
  DC_BIGRAW,    // large, not compressible (frames of raw blocks) or LZ4: block-parallel / team kernel
  DC_SMALL,     // decoded size <= 64 KiB: one-warp teams
  DC_MID,       // the rest: 128-thread teams
  DC_COUNT
};

struct zn_plan {
  zn_ctx* ctx = nullptr;
  int kind = 0;
  uint32_t n = 0;
  uint32_t total_chunks = 0;
  uint32_t n_dec = 0, n_small = 0, n_large = 0, n_pieces = 0;
  BlobDesc* d_blobs = nullptr;
  uint32_t* d_chunk_prefix = nullptr;
  uint32_t *d_list_dec = nullptr, *d_list_small = nullptr, *d_list_large = nullptr;
  uint32_t *d_piece_blob = nullptr, *d_piece_idx = nullptr;
  uint64_t* d_magic_off = nullptr;  // rows flagged compressed == 3: where the zstd magic is rebuilt on the device copy
  uint32_t n_magic = 0;
  uint32_t *d_cvs = nullptr, *d_digests = nullptr, *d_expect = nullptr, *d_status = nullptr, *d_produced = nullptr,
           *d_counter = nullptr, *d_wsq = nullptr, *d_cvs2 = nullptr, *d_status0 = nullptr;  // d_status0: initial statuses (rows rejected by the planner)
  // d_wsq: tile queue of the warp-specialised fused kernel (fused_ws.cuh); d_cvs2: second level buffer of the large-blob tree
  uint32_t ws_tiles = 0;
  bool ran_ws = false;             // the last run used the warp-specialised fused kernel
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaStream_t last_stream = nullptr;
  bool ran = false;
  uint32_t cls_off[DC_COUNT + 1] = {0};  // class c = d_list_dec[cls_off[c] .. cls_off[c + 1]), largest blobs first
  uint32_t n_hashed = 0;     // rows whose chunks k_b3_chunks may skip
  // device-wide pipeline (DC_PIPE rows)
  zp::ZBlob* d_zb = nullptr;
  uint32_t nzb = 0;
  size_t z_slots = 0, z_tabs = 0, z_seqs = 0, z_lit16 = 0;
  uint64_t z_mean = 0;       // mean decoded size of the pipeline rows (picks the exec team size)
  bool uploads_synced = false;  // the plan's arrays (uploaded on the ctx stream) are known to have landed
  uint32_t launches_per_run = 0;
  // compress plans: their own scratch and descriptors (compress_prepare), the hash plan of the source slices (digests),
  // ZNB1 packing, the d_dst bytes any input of these sizes may need, and the statuses the planner gave
  CompressScratch cs;
  CompressPrep cp;
  zn_plan* hp = nullptr;
  bool envelope = false;
  uint64_t capacity = 0;
  std::vector<uint32_t> h_status;
};

static const int kDecodeThreads = 128;
static const int kDecodeCtasPerSm = 4;  // resident k_decode<128> CTAs per SM (128 regs, 42 KB smem)

#define ZN_CUDA(ctx, call)                                                              \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                 \
      return ZN_E_CUDA;                                                                 \
    }                                                                                   \
  } while (0)

extern "C" int zn_abi_version(void) { return ZN_ABI_VERSION; }

extern "C" int zn_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

extern "C" const char* zn_strerror(int code) {
  switch (code) {
    case ZN_OK: return "ok";
    case ZN_E_ARG: return "invalid argument";
    case ZN_E_CUDA: return "CUDA error";
    case ZN_E_NOMEM: return "out of memory";
    case ZN_E_STATE: return "call out of order";
    default: return "unknown error";
  }
}

extern "C" const char* zn_status_name(uint32_t s) {
  switch (s) {
    case ZN_S_OK: return "OK";
    case ZN_S_DECODE_ERROR: return "DECODE_ERROR";
    case ZN_S_DIGEST_MISMATCH: return "DIGEST_MISMATCH";
    case ZN_S_DST_TOO_SMALL: return "DST_TOO_SMALL";
    case ZN_S_UNSUPPORTED: return "UNSUPPORTED";
    case ZN_S_SIZE_MISMATCH: return "SIZE_MISMATCH";
    default: return "?";
  }
}

static void build_predef(PredefTables* p) {
  static zs::FseTable t;
  uint16_t next[64];
  zs::fse_build(&t, zs::kLLDefault, 36, 6, next);
  for (int i = 0; i < 64; i++) p->ll[i] = t.e[i];
  zs::fse_build(&t, zs::kOFDefault, 29, 5, next);
  for (int i = 0; i < 32; i++) p->of[i] = t.e[i];
  zs::fse_build(&t, zs::kMLDefault, 53, 6, next);
  for (int i = 0; i < 64; i++) p->ml[i] = t.e[i];
}

extern "C" zn_ctx* zn_ctx_create(int device, size_t staging_bytes) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return nullptr;
  if (cudaSetDevice(device) != cudaSuccess) return nullptr;
  zn_ctx* c = new zn_ctx();
  c->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return nullptr; }
  c->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking) != cudaSuccess) { delete c; return nullptr; }
  c->dec_grid = (uint32_t)(c->sm_count * kDecodeCtasPerSm);
  {  // keep freed plan memory cached in the device's default pool instead of returning it to the driver
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      uint64_t thresh = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh);
    }
  }
  c->dec_grid_small = (uint32_t)(c->sm_count * 10);
  if (cudaMalloc(&c->d_lit, (size_t)std::max(c->dec_grid, c->dec_grid_small) * kLitStride) != cudaSuccess) { zn_ctx_destroy(c); return nullptr; }
  if (staging_bytes) {
    if (cudaHostAlloc(&c->pinned, staging_bytes, cudaHostAllocDefault) != cudaSuccess) { zn_ctx_destroy(c); return nullptr; }
    c->pinned_bytes = staging_bytes;
  }
  PredefTables pd;
  build_predef(&pd);
  if (cudaMemcpyToSymbol(g_predef, &pd, sizeof pd) != cudaSuccess) { zn_ctx_destroy(c); return nullptr; }
  cudaFuncSetAttribute(k_b3_chunks, cudaFuncAttributeMaxDynamicSharedMemorySize, kB3Warps * kB3SmemPerWarp);
  cudaFuncSetAttribute(k_decode_ws, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWsSmemBytes);
  cudaFuncSetAttribute(par::k_decode_par, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(par::ParShared));
  if (!zp::pipeline_init()) { zn_ctx_destroy(c); return nullptr; }
  compress_init_attrs();
  return c;
}

extern "C" void zn_ctx_destroy(zn_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->d_lit) cudaFree(c->d_lit);
  if (c->d_par) cudaFree(c->d_par);
  for (void* q : {(void*)c->zs.blocks, (void*)c->zs.comp_list, (void*)c->zs.tabs, (void*)c->zs.recs, (void*)c->zs.p1, (void*)c->zs.lits, (void*)c->zs.pools})
    if (q) cudaFree(q);
  if (c->d_in) cudaFree(c->d_in);
  if (c->d_out) cudaFree(c->d_out);
  c->cs.release();
  if (c->pinned) cudaFreeHost(c->pinned);
  if (c->plan_pin) cudaFreeHost(c->plan_pin);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->stream2) cudaStreamDestroy(c->stream2);
  delete c;
}

extern "C" const char* zn_last_error(const zn_ctx* c) { return c ? c->err.c_str() : "null ctx"; }

extern "C" void* zn_ctx_pinned(zn_ctx* c, size_t* bytes) {
  if (!c) return nullptr;
  if (bytes) *bytes = c->pinned_bytes;
  return c->pinned;
}

extern "C" uint64_t zn_ctx_kernel_launches(const zn_ctx* c) { return c ? c->launches : 0; }

// pinned host memory for the native pipelines of container.cpp (which is compiled without the CUDA runtime headers)
// cudaHostAlloc costs ~0.3 ms per MiB (page pinning), i.e. more than moving the bytes over PCIe: the staging buffers of
// the read worker and of the archive writer are therefore recycled through a small process-wide cache (the reference
// keeps its Magazine slots for the life of the process for the same reason, slotpool.rs:93-130).
namespace {
struct PinnedCache {
  std::mutex mu;
  struct Buf { void* p; size_t cap; };
  std::vector<Buf> free_list;                       // idle buffers, at most kKeep of them
  std::unordered_map<void*, size_t> live;           // capacity of every buffer handed out
  static constexpr size_t kKeep = 6;
} g_pinned;
}  // namespace

extern "C" void* zn_ctx_pinned_alloc(size_t bytes) {
  {
    std::lock_guard<std::mutex> lk(g_pinned.mu);
    size_t best = SIZE_MAX;
    for (size_t i = 0; i < g_pinned.free_list.size(); i++) {
      const size_t cap = g_pinned.free_list[i].cap;
      if (cap >= bytes && cap <= 2 * bytes + (64u << 20) && (best == SIZE_MAX || cap < g_pinned.free_list[best].cap)) best = i;
    }
    if (best != SIZE_MAX) {
      PinnedCache::Buf b = g_pinned.free_list[best];
      g_pinned.free_list.erase(g_pinned.free_list.begin() + (long)best);
      g_pinned.live[b.p] = b.cap;
      return b.p;
    }
  }
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    // memory pressure: drop the idle buffers and try once more
    std::vector<PinnedCache::Buf> drop;
    { std::lock_guard<std::mutex> lk(g_pinned.mu); drop.swap(g_pinned.free_list); }
    for (auto& b : drop) cudaFreeHost(b.p);
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  }
  std::lock_guard<std::mutex> lk(g_pinned.mu);
  g_pinned.live[p] = bytes;
  return p;
}
extern "C" void zn_ctx_pinned_free(void* p) {
  if (!p) return;
  void* evict = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_pinned.mu);
    auto it = g_pinned.live.find(p);
    if (it == g_pinned.live.end()) { evict = p; }
    else {
      g_pinned.free_list.push_back({p, it->second});
      g_pinned.live.erase(it);
      if (g_pinned.free_list.size() > PinnedCache::kKeep) {  // drop the smallest idle buffer
        size_t k = 0;
        for (size_t i = 1; i < g_pinned.free_list.size(); i++) if (g_pinned.free_list[i].cap < g_pinned.free_list[k].cap) k = i;
        evict = g_pinned.free_list[k].p;
        g_pinned.free_list.erase(g_pinned.free_list.begin() + (long)k);
      }
    }
  }
  if (evict) cudaFreeHost(evict);
}

// --------------------------------------------------------------------------------------------- plans
template <typename T>
static bool upload(zn_ctx* c, T** dptr, const T* h, size_t count) {
  *dptr = nullptr;
  // stream-ordered pool allocation: plans are built per batch by the host-buffer API, so this must be cheap
  if (cudaMallocAsync((void**)dptr, std::max<size_t>(count, 1) * sizeof(T), c->stream) != cudaSuccess) return false;
  if (count && h && cudaMemcpyAsync(*dptr, h, count * sizeof(T), cudaMemcpyHostToDevice, c->stream) != cudaSuccess)
    return false;
  return true;
}

extern "C" int zn_plan_set_overlap(zn_plan* p, int groups) {
  // Kept for ABI stability.  The stream-overlapped decode/hash schedule of round 1 measured slower than stages back to
  // back on every corpus (DESIGN.md) and was removed together with the batch-wide kernel choice: classes of rows now
  // get their own kernels, and the pattern class fuses decode and hash in one kernel.
  (void)groups;
  return p ? ZN_OK : ZN_E_ARG;
}

static zn_plan* plan_build(zn_ctx* c, int kind, uint32_t n, const uint64_t* src_off, const uint64_t* src_len,
                           const uint8_t* compressed, const uint64_t* out_off, const uint64_t* out_len,
                           const uint8_t* expect, bool gather_raw) {
  if (!c || (n && (!src_off || !src_len))) return nullptr;
  cudaSetDevice(c->device);
  zn_plan* p = new zn_plan();
  p->ctx = c;
  p->kind = kind;
  p->n = n;
  {  // the arena is free again: the previous plan_build synchronised its uploads before returning
    const size_t need = (size_t)n * (sizeof(BlobDesc) + 4 * 4) + 4096;
    if (need > c->plan_pin_cap) {
      if (c->plan_pin) cudaFreeHost(c->plan_pin);
      c->plan_pin = nullptr;
      c->plan_pin_cap = 0;
      if (cudaHostAlloc((void**)&c->plan_pin, need + need / 4, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        delete p;
        c->err = "pinned plan arena allocation failed";
        return nullptr;
      }
      c->plan_pin_cap = need + need / 4;
    }
    c->plan_pin_used = 0;
  }
  BlobDesc* descs = c->arena<BlobDesc>(n);
  uint32_t* prefix = c->arena<uint32_t>((size_t)n + 1);
  uint32_t* status0 = c->arena<uint32_t>(n);
  memset(status0, 0, (size_t)n * 4);
  uint32_t* lsmall_a = c->arena<uint32_t>(n);  // rows whose tree fits one lane (the common case: filled in place)
  uint32_t n_lsmall = 0;
  std::vector<uint32_t> llarge, pblob, pidx, cls[DC_COUNT];
  std::vector<uint64_t> magic_off;
  uint64_t chunks = 0;
  bool any_status = false;
  for (uint32_t i = 0; i < n; i++) {
    BlobDesc& d = descs[i];
    const bool comp = kind == PLAN_DECODE_VERIFY && compressed && compressed[i];
    d.src_off = src_off[i];
    d.src_len = src_len[i];
    if (comp && compressed[i] == 3) {  // magicless zstd frame: decoded as magic + payload (k_patch_magic)
      if (d.src_off < 4) { delete p; c->err = "compressed == 3 needs four bytes in front of the payload"; return nullptr; }
      d.src_off -= 4;
      d.src_len += 4;
      magic_off.push_back(d.src_off);
    }
    d.dst_off = out_off ? out_off[i] : 0;
    d.dst_cap = kind == PLAN_DECODE_VERIFY ? (out_len ? out_len[i] : 0) : src_len[i];
    bool skip = false;
    if (!comp && kind == PLAN_DECODE_VERIFY && d.dst_cap != d.src_len) {
      // store-as-is row whose index sizes disagree (blob_size != uncompressed_size): the reference would hand back
      // blob_size bytes for a file region of uncompressed_size — a corrupt index row.  Nothing is gathered or hashed.
      status0[i] = S_SIZE_MISMATCH;
      any_status = true;
      skip = true;
      d.src_len = 0;
      d.dst_cap = 0;
    }
    const uint64_t nc = std::max<uint64_t>(1, (d.dst_cap + kChunk - 1) / kChunk);
    d.n_chunks = (uint32_t)nc;
    d.cv_base = chunks;
    d.flags = (comp ? F_COMPRESSED : 0u) | (expect && !skip ? F_HAS_EXPECT : 0u) | (comp && compressed[i] == 2 ? F_LZ4_BLOCK : 0u);
    prefix[i] = (uint32_t)chunks;
    chunks += nc;
    if (chunks > 0xFFFFFFF0ull) { delete p; c->err = "batch too large (chunk count)"; return nullptr; }
    if (comp) {
      const bool big = d.dst_cap >= (512u << 10), pat = d.src_len * 64 <= d.dst_cap, lz4b = (d.flags & F_LZ4_BLOCK) != 0;
      int k;
      if (big && pat && !lz4b) k = DC_BIGPAT;
      else if (!lz4b && !pat && d.src_len < d.dst_cap && d.dst_cap >= 4096 && d.dst_cap < 0xFFFFFFF0ull) k = DC_PIPE;
      else if (big) k = DC_BIGRAW;
      else if (d.dst_cap <= (64u << 10)) k = DC_SMALL;
      else k = DC_MID;
      cls[k].push_back(i);
    } else if (gather_raw && kind == PLAN_DECODE_VERIFY && !skip)
      for (uint64_t o = 0, k = 0; o < d.dst_cap; o += kGatherPiece, k++) { pblob.push_back(i); pidx.push_back((uint32_t)k); }
    if (nc <= kTreeSmallMax) lsmall_a[n_lsmall++] = i; else llarge.push_back(i);
  }
  prefix[n] = (uint32_t)chunks;
  p->total_chunks = (uint32_t)chunks;
  // class lists back to back, largest first inside a class (dynamic work counters)
  uint32_t* ldec = c->arena<uint32_t>(n);
  uint32_t n_ldec = 0;
  for (int k = 0; k < DC_COUNT; k++) {
    auto& L = cls[k];
    bool sorted_desc = true;
    for (size_t j = 1; j < L.size() && sorted_desc; j++) sorted_desc = descs[L[j]].dst_cap <= descs[L[j - 1]].dst_cap;
    if (!sorted_desc) std::stable_sort(L.begin(), L.end(), [&](uint32_t x, uint32_t y) { return descs[x].dst_cap > descs[y].dst_cap; });
    p->cls_off[k] = n_ldec;
    if (!L.empty()) memcpy(ldec + n_ldec, L.data(), L.size() * 4);
    n_ldec += (uint32_t)L.size();
  }
  p->cls_off[DC_COUNT] = n_ldec;
  p->n_dec = n_ldec;
  // Large, highly compressible blobs go through the fused decode+hash kernel (fused_ws.cuh).
  for (uint32_t i : cls[DC_BIGPAT]) { descs[i].flags |= F_HASHED; p->ws_tiles += (descs[i].n_chunks + 31u) / 32u; p->n_hashed++; }
  // device-wide pipeline: per-blob block-table slots and pool budgets (zpipe.cuh; anything that does not fit is decoded
  // by the one-team kernel instead)
  std::vector<zp::ZBlob> zb(cls[DC_PIPE].size());
  {
    uint64_t slots = 0, seqs = 0, lit16 = 0, tabs = 0, bytes = 0;
    for (size_t j = 0; j < zb.size(); j++) {
      const uint64_t cap = descs[cls[DC_PIPE][j]].dst_cap;
      const uint32_t sc = (uint32_t)(cap / 16384 + 8);  // level >= 16 frames split their 128 KiB blocks
      memset(&zb[j], 0, sizeof zb[j]);
      zb[j].blob = cls[DC_PIPE][j];
      zb[j].slot0 = (uint32_t)slots;
      zb[j].slot_cap = sc;
      slots += sc;
      seqs += cap / 5 + 64;
      lit16 += cap / 16 + 2ull * sc + 2;
      tabs += cap / 32768 + 2;
      bytes += cap;
    }
    const uint64_t lim = 0xFFFFFFF0ull;
    p->nzb = (uint32_t)zb.size();
    p->z_slots = (size_t)std::min(slots, lim);
    p->z_seqs = (size_t)std::min(seqs, lim);
    p->z_lit16 = (size_t)std::min(lit16, lim);
    p->z_tabs = (size_t)std::min(tabs, lim);
    p->z_mean = zb.empty() ? 0 : bytes / zb.size();
    if (slots > lim) { delete p; c->err = "batch too large (zstd block slots)"; return nullptr; }
  }
  p->n_small = n_lsmall;
  p->n_large = (uint32_t)llarge.size();
  p->n_pieces = (uint32_t)pblob.size();
  p->n_magic = (uint32_t)magic_off.size();
  bool ok = upload(c, &p->d_blobs, descs, n) && upload(c, &p->d_chunk_prefix, prefix, (size_t)n + 1) &&
            upload(c, &p->d_list_dec, ldec, n_ldec) && upload(c, &p->d_list_small, lsmall_a, n_lsmall) &&
            upload(c, &p->d_list_large, llarge.data(), llarge.size()) &&
            upload(c, &p->d_piece_blob, pblob.data(), pblob.size()) && upload(c, &p->d_piece_idx, pidx.data(), pidx.size()) &&
            upload(c, &p->d_magic_off, magic_off.data(), magic_off.size()) &&
            upload(c, &p->d_expect, (const uint32_t*)expect, expect ? (size_t)n * 8 : 0) &&
            upload(c, &p->d_cvs, (const uint32_t*)nullptr, (size_t)chunks * 8) &&
            upload(c, &p->d_cvs2, (const uint32_t*)nullptr, llarge.empty() ? 0 : (size_t)chunks * 8) &&
            upload(c, &p->d_digests, (const uint32_t*)nullptr, (size_t)n * 8) &&
            upload(c, &p->d_status, (const uint32_t*)nullptr, n) && upload(c, &p->d_produced, (const uint32_t*)nullptr, n) &&
            upload(c, &p->d_counter, (const uint32_t*)nullptr, 16) &&
            upload(c, &p->d_wsq, (const uint32_t*)nullptr, cls[DC_BIGPAT].empty() ? 0 : 6 + 2 * (size_t)p->ws_tiles) &&
            upload(c, &p->d_zb, zb.data(), zb.size());
  if (ok && any_status) ok = upload(c, &p->d_status0, status0, n);
  for (int i = 0; ok && i < 4; i++) ok = cudaEventCreate(&p->ev[i]) == cudaSuccess;
  if (ok) ok = cudaStreamSynchronize(c->stream) == cudaSuccess;  // host vectors go out of scope
  if (!ok) {
    c->err = std::string("plan allocation failed: ") + cudaGetErrorString(cudaGetLastError());
    zn_plan_destroy(p);
    return nullptr;
  }
  p->uploads_synced = true;
  return p;
}

extern "C" zn_plan* zn_plan_decode_verify(zn_ctx* ctx, uint32_t n, const uint64_t* h_blob_off, const uint64_t* h_blob_len,
                                          const uint8_t* h_compressed, const uint64_t* h_out_off,
                                          const uint64_t* h_out_len, const uint8_t* h_expect_digest) {
  if (n && (!h_out_len || !h_compressed)) return nullptr;
  return plan_build(ctx, PLAN_DECODE_VERIFY, n, h_blob_off, h_blob_len, h_compressed, h_out_off, h_out_len,
                    h_expect_digest, h_out_off != nullptr);
}

extern "C" zn_plan* zn_plan_hash(zn_ctx* ctx, uint32_t n, const uint64_t* h_off, const uint64_t* h_len,
                                 const uint8_t* h_expect_digest) {
  return plan_build(ctx, PLAN_HASH, n, h_off, h_len, nullptr, nullptr, nullptr, h_expect_digest, false);
}

extern "C" int zn_plan_fused(const zn_plan* p) { return p && p->cls_off[DC_BIGPAT + 1] > p->cls_off[DC_BIGPAT] ? 1 : 0; }

extern "C" int zn_plan_class_counts(const zn_plan* p, uint32_t counts[5]) {
  if (!p || !counts) return ZN_E_ARG;
  if (p->kind == PLAN_COMPRESS) return ZN_E_STATE;
  for (int k = 0; k < DC_COUNT; k++) counts[k] = p->cls_off[k + 1] - p->cls_off[k];
  return ZN_OK;
}

extern "C" int zn_plan_pipeline_fallbacks(zn_plan* p, uint32_t* rows) {
  if (!p || !rows) return ZN_E_ARG;
  if (p->kind == PLAN_COMPRESS) return ZN_E_STATE;
  *rows = 0;
  if (!p->nzb || !p->ran) return ZN_OK;
  cudaSetDevice(p->ctx->device);
  if (cudaStreamSynchronize(p->last_stream) != cudaSuccess) { p->ctx->err = cudaGetErrorString(cudaGetLastError()); return ZN_E_CUDA; }
  std::vector<zp::ZBlob> hz(p->nzb);
  if (cudaMemcpy(hz.data(), p->d_zb, sizeof(zp::ZBlob) * p->nzb, cudaMemcpyDeviceToHost) != cudaSuccess) { p->ctx->err = cudaGetErrorString(cudaGetLastError()); return ZN_E_CUDA; }
  for (auto& b : hz) *rows += b.state != 0;
  return ZN_OK;
}

extern "C" void zn_plan_destroy(zn_plan* p) {
  if (!p) return;
  cudaSetDevice(p->ctx->device);
  if (p->ran) cudaStreamSynchronize(p->last_stream);
  void* ptrs[] = {p->d_blobs, p->d_chunk_prefix, p->d_list_dec, p->d_list_small, p->d_list_large, p->d_piece_blob,
                  p->d_piece_idx, p->d_cvs, p->d_digests, p->d_expect, p->d_status, p->d_produced, p->d_counter, p->d_wsq, p->d_cvs2,
                  p->d_zb, p->d_status0, p->d_magic_off};
  for (void* q : ptrs)
    if (q) cudaFreeAsync(q, p->ctx->stream);
  for (auto& e : p->ev)
    if (e) cudaEventDestroy(e);
  if (p->hp) zn_plan_destroy(p->hp);
  p->cs.release();
  delete p;
}

template <typename T>
static bool zgrow(T** ptr, size_t* have, size_t want, size_t bytes_per) {
  if (*have >= want) return true;
  if (*ptr) cudaFree(*ptr);
  *ptr = nullptr;
  *have = 0;
  const size_t cap = want + want / 8 + 16;
  if (cudaMalloc((void**)ptr, cap * bytes_per) != cudaSuccess) { cudaGetLastError(); return false; }
  *have = cap;
  return true;
}

// DC_PIPE rows: the device-wide pipeline, then the one-team decoder for whatever the pipeline handed back.
static int run_pipeline(zn_plan* p, const uint8_t* d_blobs, uint8_t* d_out, cudaStream_t st, uint32_t* launches) {
  zn_ctx* c = p->ctx;
  auto& z = c->zs;
  if (!z.pools && cudaMalloc((void**)&z.pools, sizeof(zp::ZPools)) != cudaSuccess) { c->err = "zstd pipeline scratch allocation failed"; cudaGetLastError(); return ZN_E_NOMEM; }
  {
    const size_t slots_before = z.slots;
    size_t dummy = slots_before;
    if (!zgrow(&z.blocks, &z.slots, p->z_slots, sizeof(zp::ZBlock)) || !zgrow(&z.comp_list, &dummy, p->z_slots, 4) ||
        !zgrow(&z.tabs, &z.tab_sets, p->z_tabs, sizeof(zp::FseD) * zp::kTabSet) || !zgrow(&z.recs, &z.seqs, p->z_seqs, sizeof(zp::SeqRec16)) || !zgrow(&z.p1, &z.p1s, p->z_seqs, sizeof(zp::SeqP1)) ||
        !zgrow(&z.lits, &z.lit16, p->z_lit16 + 4, 16)) {
      c->err = "zstd pipeline scratch allocation failed";
      return ZN_E_NOMEM;
    }
  }
  zp::ZArgs a;
  a.blobs = p->d_blobs; a.blobs_base = d_blobs; a.zb = p->d_zb; a.nzb = p->nzb; a.blocks = z.blocks; a.pools = z.pools;
  a.comp_list = z.comp_list; a.tabs = z.tabs; a.recs = z.recs; a.lits = z.lits; a.p1 = z.p1;
  // development: ZN_ZPROF=1 prints the device time of every pipeline kernel of this run on stderr (synchronises)
  const bool prof = getenv("ZN_ZPROF") != nullptr;
  cudaEvent_t pe[9];
  if (prof) for (auto& e : pe) cudaEventCreate(&e);
  uint32_t* ctr = p->d_counter + DC_COUNT;  // [0] exec, [1] legacy pass
  zp::PipelineLaunch L;
  L.a = a;
  L.slots = (uint32_t)p->z_slots; L.seq_cap = (uint32_t)p->z_seqs; L.lit_cap16 = (uint32_t)p->z_lit16; L.tab_cap = (uint32_t)p->z_tabs;
  L.sm_count = (uint32_t)c->sm_count;
  L.mean_bytes = p->z_mean;
  L.d_out = d_out; L.produced = p->d_produced; L.exec_counter = ctr;
  const uint32_t pipe_launches = zp::pipeline_enqueue(L, st, prof ? pe : nullptr);
  // rows the pipeline handed back (ZBlob.state != 0): the one-team decoder, which also produces their status
  const uint32_t* list = p->d_list_dec + p->cls_off[DC_PIPE];
  const uint32_t grid = std::min<uint32_t>(p->nzb, c->dec_grid);
  k_decode<kDecodeThreads, 1><<<grid, kDecodeThreads, 0, st>>>(p->d_blobs, list, p->nzb, d_blobs, d_out, c->d_lit, p->d_status,
                                                            p->d_produced, ctr + 1, nullptr, 1u, &p->d_zb[0].state,
                                                            (uint32_t)(sizeof(zp::ZBlob) / 4));
  if (prof) {
    cudaEventRecord(pe[7], st);
    cudaEventSynchronize(pe[7]);
    static const char* names[] = {"walk", "tables", "seq", "lit", "chain", "exec", "legacy"};
    zp::ZPools hp;
    cudaMemcpy(&hp, z.pools, sizeof hp, cudaMemcpyDeviceToHost);
    std::vector<zp::ZBlob> hz(p->nzb);
    cudaMemcpy(hz.data(), p->d_zb, sizeof(zp::ZBlob) * p->nzb, cudaMemcpyDeviceToHost);
    uint32_t handed = 0;
    for (auto& b : hz) handed += b.state != 0;
    fprintf(stderr, "zpipe: %u blobs (%u handed back), %u blocks, %u seqs, %u table sets, %u lit16 |", p->nzb, handed, hp.comp_used, hp.seq_used, hp.tab_used, hp.lit_used16);
    for (int i = 0; i < 7; i++) { float ms = 0; cudaEventElapsedTime(&ms, pe[i], pe[i + 1]); fprintf(stderr, " %s %.3f", names[i], ms); }
    if (getenv("ZN_ZPROF_SEQ1")) { float ms = 0; if (cudaEventElapsedTime(&ms, pe[2], pe[8]) == cudaSuccess) fprintf(stderr, " (seq phase 1 %.3f)", ms); else cudaGetLastError(); }
    fprintf(stderr, " ms\n");
    zp::pipeline_trace_dump();
    for (auto& e : pe) cudaEventDestroy(e);
  }
  *launches += pipe_launches + 1;
  return ZN_OK;
}

extern "C" int zn_plan_run(zn_plan* p, const uint8_t* d_blobs, uint8_t* d_out, void* stream_v) {
  if (!p) return ZN_E_ARG;
  if (p->kind == PLAN_COMPRESS) return ZN_E_STATE;
  zn_ctx* c = p->ctx;
  cudaSetDevice(c->device);
  cudaStream_t st = stream_v ? (cudaStream_t)stream_v : c->stream;
  if (p->n && !d_blobs) return ZN_E_ARG;
  if (p->n_dec && !d_out) return ZN_E_ARG;
  if (st != c->stream && !p->uploads_synced) {  // the plan was uploaded on the ctx stream: order it before this stream's kernels
    ZN_CUDA(c, cudaStreamSynchronize(c->stream));
    p->uploads_synced = true;
  }
  uint32_t launches = 0;
  ZN_CUDA(c, cudaEventRecord(p->ev[0], st));
  if (p->n) {
    if (p->d_status0) ZN_CUDA(c, cudaMemcpyAsync(p->d_status, p->d_status0, (size_t)p->n * 4, cudaMemcpyDeviceToDevice, st));
    else ZN_CUDA(c, cudaMemsetAsync(p->d_status, 0, (size_t)p->n * 4, st));
    ZN_CUDA(c, cudaMemsetAsync(p->d_counter, 0, 4 * 16, st));
  }
  if (p->n_magic) {  // only our copy of the blobs is touched when the call came through the host-buffer API
    k_patch_magic<<<(p->n_magic + 255) / 256, 256, 0, st>>>(const_cast<uint8_t*>(d_blobs), p->d_magic_off, p->n_magic);
    launches++;
  }
  if (p->n_pieces && d_out) {
    const uint32_t grid = std::min<uint32_t>(p->n_pieces, (uint32_t)c->sm_count * 16u);
    k_gather_raw<<<grid, 256, 0, st>>>(p->d_blobs, p->d_piece_blob, p->d_piece_idx, p->n_pieces, d_blobs, d_out);
    launches++;
  }
  auto cls_n = [&](int k) { return p->cls_off[k + 1] - p->cls_off[k]; };
  auto cls_list = [&](int k) { return p->d_list_dec + p->cls_off[k]; };
  if (p->nzb) {
    const int rc = run_pipeline(p, d_blobs, d_out, st, &launches);
    if (rc != ZN_OK) return rc;
  }
  if (const uint32_t nd = cls_n(DC_BIGPAT)) {  // highly compressible large blobs (few, long sequences)
    // warp-specialised fused kernel: one CTA per SM, two decode teams each; its tile queue starts empty
    ZN_CUDA(c, cudaMemsetAsync(p->d_wsq, 0, 24 + 8 * (size_t)p->ws_tiles, st));
    p->ran_ws = true;
    // tests (ZN_WS_TEST_STALL=1): announce one tile more than the producers will ever publish, so that a hash warp waits
    // for an entry that never comes and the watchdog has to end the kernel
    const uint32_t phantom = getenv("ZN_WS_TEST_STALL") ? 1u : 0u;
    WsQueue q{p->d_wsq, reinterpret_cast<unsigned long long*>(p->d_wsq + 4), p->ws_tiles + phantom};
    uint32_t wgrid = (uint32_t)c->sm_count;  // every SM hashes, whether or not one of its teams gets a blob
    // tests (ZN_WS_GRID): a smaller grid, so that every decode team takes several blobs
    if (const char* gs = getenv("ZN_WS_GRID")) wgrid = std::max(1, std::min<int>((int)wgrid, atoi(gs)));
    k_decode_ws<<<wgrid, kWsThreads, kWsSmemBytes, st>>>(p->d_blobs, cls_list(DC_BIGPAT), nd, d_blobs, d_out, c->d_lit, p->d_status,
                                                         p->d_produced, p->d_counter + DC_BIGPAT, p->d_cvs, q, 1u);
    launches++;
  }
  if (const uint32_t nd = cls_n(DC_BIGRAW)) {  // large raw-block / LZ4 blobs: one CTA per SM
    const uint32_t max_grid = (uint32_t)c->sm_count;
    if (!c->d_par && cudaMalloc(&c->d_par, (size_t)max_grid * par::kParScratchPerCta) != cudaSuccess) {
      c->err = "block-parallel decode scratch allocation failed";
      cudaGetLastError();
      return ZN_E_NOMEM;
    }
    par::k_decode_par<<<std::min<uint32_t>(nd, max_grid), par::kParThreads, sizeof(par::ParShared), st>>>(
        p->d_blobs, cls_list(DC_BIGRAW), nd, d_blobs, d_out, c->d_par, p->d_status, p->d_produced, p->d_counter + DC_BIGRAW);
    launches++;
  }
  if (const uint32_t nd = cls_n(DC_SMALL)) {  // many small blobs: one warp per blob, ~10 blobs in flight per SM
    const uint32_t grid = std::min<uint32_t>((nd + 1) / 2, c->dec_grid_small);
    k_decode<32, 2><<<grid, 32, 0, st>>>(p->d_blobs, cls_list(DC_SMALL), nd, d_blobs, d_out, c->d_lit, p->d_status, p->d_produced,
                                         p->d_counter + DC_SMALL, nullptr, 1u, nullptr, 0u);
    launches++;
  }
  if (const uint32_t nd = cls_n(DC_MID)) {
    const uint32_t grid = std::min<uint32_t>((nd + 3) / 4, c->dec_grid);
    k_decode<kDecodeThreads, 4><<<grid, kDecodeThreads, 0, st>>>(p->d_blobs, cls_list(DC_MID), nd, d_blobs, d_out, c->d_lit,
                                                              p->d_status, p->d_produced, p->d_counter + DC_MID, nullptr, 1u,
                                                              nullptr, 0u);
    launches++;
  }
  ZN_CUDA(c, cudaEventRecord(p->ev[1], st));
  if (p->total_chunks && p->n_hashed != p->n) {
    const uint32_t tiles = (p->total_chunks + 31u) / 32u;
    const uint32_t ctas = (tiles + kB3Warps - 1) / kB3Warps;
    const uint32_t grid = std::min<uint32_t>(ctas, (uint32_t)c->sm_count * 3u);  // 3 hash CTAs fill an SM's shared memory
    k_b3_chunks<<<grid, kB3Warps * 32, kB3Warps * kB3SmemPerWarp, st>>>(p->d_blobs, p->d_chunk_prefix, p->n, 0u, p->total_chunks,
                                                                       d_blobs, d_out, p->d_cvs, 1u);
    launches++;
  }
  ZN_CUDA(c, cudaEventRecord(p->ev[2], st));
  // Zstandard content checksums are checked where a row's digest is compared (xxh_verify.cuh)
  const uint8_t* xxh_out = p->n_dec ? d_out : nullptr;
  if (p->n_small) {
    k_b3_tree_small<<<(p->n_small + 127) / 128, 128, 0, st>>>(p->d_blobs, p->d_list_small, p->n_small, p->d_cvs, p->d_digests,
                                                              p->d_expect, p->d_status, 1u, d_blobs, xxh_out);
    launches++;
  }
  if (p->n_large) {
    k_b3_tree_large<<<p->n_large, 512, 0, st>>>(p->d_blobs, p->d_list_large, p->d_cvs, p->d_cvs2, p->d_digests, p->d_expect, p->d_status, 1u,
                                                d_blobs, xxh_out);
    launches++;
  }
  ZN_CUDA(c, cudaEventRecord(p->ev[3], st));
  ZN_CUDA(c, cudaGetLastError());
  p->launches_per_run = launches;
  c->launches += launches;
  p->last_stream = st;
  p->ran = true;
  return ZN_OK;
}

extern "C" int zn_plan_results(zn_plan* p, uint32_t* h_status, uint8_t* h_digests) {
  if (!p) return ZN_E_ARG;
  if (!p->ran) return ZN_E_STATE;
  zn_ctx* c = p->ctx;
  cudaSetDevice(c->device);
  if (p->kind == PLAN_COMPRESS) {
    ZN_CUDA(c, cudaStreamSynchronize(p->last_stream));
    if (h_status && p->n) memcpy(h_status, p->h_status.data(), (size_t)p->n * 4);
    return h_digests && p->hp ? zn_plan_results(p->hp, nullptr, h_digests) : ZN_OK;
  }
  if (h_status && p->n) ZN_CUDA(c, cudaMemcpyAsync(h_status, p->d_status, (size_t)p->n * 4, cudaMemcpyDeviceToHost, p->last_stream));
  if (h_digests && p->n) ZN_CUDA(c, cudaMemcpyAsync(h_digests, p->d_digests, (size_t)p->n * 32, cudaMemcpyDeviceToHost, p->last_stream));
  uint32_t stall = 0;
  if (p->d_wsq && p->ran_ws) ZN_CUDA(c, cudaMemcpyAsync(&stall, p->d_wsq + 2, 4, cudaMemcpyDeviceToHost, p->last_stream));
  ZN_CUDA(c, cudaStreamSynchronize(p->last_stream));
  if (stall) { c->err = "fused decode+hash kernel stalled (internal error): results are incomplete"; return ZN_E_CUDA; }
  return ZN_OK;
}

extern "C" uint32_t zn_plan_launches(const zn_plan* p) { return p ? p->launches_per_run : 0; }

extern "C" int zn_plan_last_ms(zn_plan* p, float ms[4]) {
  if (!p || !ms) return ZN_E_ARG;
  if (!p->ran) return ZN_E_STATE;
  zn_ctx* c = p->ctx;
  cudaSetDevice(c->device);
  ZN_CUDA(c, cudaEventSynchronize(p->ev[3]));
  ZN_CUDA(c, cudaEventElapsedTime(&ms[0], p->ev[0], p->ev[3]));
  ZN_CUDA(c, cudaEventElapsedTime(&ms[1], p->ev[0], p->ev[1]));
  ZN_CUDA(c, cudaEventElapsedTime(&ms[2], p->ev[1], p->ev[2]));
  ZN_CUDA(c, cudaEventElapsedTime(&ms[3], p->ev[2], p->ev[3]));
  return ZN_OK;
}

// --------------------------------------------------------------------------------------------- compress plans
extern "C" zn_plan* zn_plan_compress(zn_ctx* c, uint32_t n, const uint64_t* h_src_off, const uint64_t* h_src_len, int level,
                                     int codec, int digests) {
  if (!c) return nullptr;
  const int base = codec & ~ZN_CODEC_ENVELOPE;
  if (base != ZN_CODEC_ZSTD && base != ZN_CODEC_LZ4) {
    c->err = "zn_plan_compress: codec must be ZN_CODEC_ZSTD or ZN_CODEC_LZ4, optionally | ZN_CODEC_ENVELOPE";
    return nullptr;
  }
  if (n && (!h_src_off || !h_src_len)) { c->err = "zn_plan_compress: null size arrays"; return nullptr; }
  cudaSetDevice(c->device);
  zn_plan* p = new zn_plan();
  p->ctx = c;
  p->kind = PLAN_COMPRESS;
  p->n = n;
  p->envelope = (codec & ZN_CODEC_ENVELOPE) != 0;
  p->h_status.assign(n, 0);
  for (uint32_t i = 0; i < n; i++) {
    uint8_t hdr[ZN_ENVELOPE_ZNB1_MAX_HEADER];
    p->capacity += p->envelope ? zn_envelope_znb1_header(ZN_PAYLOAD_RAW, h_src_len[i], hdr, sizeof hdr) + h_src_len[i]
                               : compress_bound(h_src_len[i], base);
  }
  std::string err;
  if (compress_prepare(&p->cs, c->stream, c->sm_count, h_src_off, h_src_len, n, level, base, nullptr, &p->cp, p->h_status.data(),
                       &err) != 0) {
    c->err = "zn_plan_compress: " + err;
    zn_plan_destroy(p);
    return nullptr;
  }
  if (digests && n && !(p->hp = zn_plan_hash(c, n, h_src_off, h_src_len, nullptr))) {  // c->err says why
    zn_plan_destroy(p);
    return nullptr;
  }
  bool ok = true;
  for (int i = 0; ok && i < 4; i++) ok = cudaEventCreate(&p->ev[i]) == cudaSuccess;
  if (ok) ok = cudaStreamSynchronize(c->stream) == cudaSuccess;  // descriptors and units have landed
  if (!ok) {
    c->err = std::string("zn_plan_compress: ") + cudaGetErrorString(cudaGetLastError());
    zn_plan_destroy(p);
    return nullptr;
  }
  p->uploads_synced = true;
  return p;
}

extern "C" uint64_t zn_plan_compress_capacity(const zn_plan* p) { return p && p->kind == PLAN_COMPRESS ? p->capacity : 0; }

extern "C" int zn_plan_run_compress(zn_plan* p, const uint8_t* d_src, uint8_t* d_dst, uint64_t* d_offsets, void* stream_v) {
  if (!p) return ZN_E_ARG;
  if (p->kind != PLAN_COMPRESS) return ZN_E_STATE;
  zn_ctx* c = p->ctx;
  if (!d_offsets || ((uintptr_t)d_offsets & 7) || (p->n && (!d_src || !d_dst))) {
    c->err = "zn_plan_run_compress: null pointer or d_offsets not 8-byte aligned";
    return ZN_E_ARG;
  }
  cudaSetDevice(c->device);
  cudaStream_t st = stream_v ? (cudaStream_t)stream_v : c->stream;
  ZN_CUDA(c, cudaEventRecord(p->ev[0], st));
  if (compress_enqueue(&p->cs, p->cp, st, d_src, &c->err) != 0) return ZN_E_CUDA;
  ZN_CUDA(c, cudaEventRecord(p->ev[1], st));
  uint32_t hash_launches = 0;
  if (p->hp) {  // digests of the source slices: the hash plan's kernels, on the same stream
    const int rc = zn_plan_run(p->hp, d_src, nullptr, st);
    if (rc != ZN_OK) return rc;
    hash_launches = p->hp->launches_per_run;
  }
  ZN_CUDA(c, cudaEventRecord(p->ev[2], st));
  if (p->n) compress_pack(&p->cs, p->cp, st, d_src, d_dst, d_offsets, p->envelope);
  else ZN_CUDA(c, cudaMemsetAsync(d_offsets, 0, 8, st));
  ZN_CUDA(c, cudaEventRecord(p->ev[3], st));
  ZN_CUDA(c, cudaGetLastError());
  const uint32_t launches = p->cp.launches + (p->n ? 2u : 0u);
  c->launches += launches;  // zn_plan_run counted the hash kernels
  p->launches_per_run = launches + hash_launches;
  p->last_stream = st;
  p->ran = true;
  return ZN_OK;
}

// --------------------------------------------------------------------------------------------- host-buffer API
static int ensure(zn_ctx* c, uint8_t** buf, size_t* cap, size_t need) {
  need += 256;  // slack for the aligned-word over-reads of the byte movers
  if (*cap >= need) return ZN_OK;
  if (*buf) cudaFree(*buf);
  *buf = nullptr;
  *cap = 0;
  const size_t want = need + need / 8;
  if (cudaMalloc((void**)buf, want) != cudaSuccess) {
    c->err = "device staging allocation failed";
    cudaGetLastError();
    return ZN_E_NOMEM;
  }
  *cap = want;
  return ZN_OK;
}

// Device layout of a set of host ranges: when the ranges sit compactly inside one span (an archive's blob region,
// a Magazine slot) the device copy mirrors it and moves with ONE memcpy; otherwise ranges are packed 16-byte aligned.
struct Layout {
  bool span = false;
  bool exact = false;  // span only: no gap of 16 bytes or more between consecutive ranges
  uint64_t span_lo = 0, span_bytes = 0;  // host span [span_lo, span_lo + span_bytes)
  uint64_t total = 0;                    // device bytes
  std::vector<uint64_t> dev_off;
};

static Layout make_layout(const uint64_t* off, const uint64_t* len, uint32_t n) {
  Layout L;
  L.dev_off.resize(n);
  if (n == 0) return L;
  // one pass: extent, total, and — for the common case of rows in ascending, non-overlapping order — whether any gap
  // between consecutive ranges reaches 16 bytes
  uint64_t lo = ~0ull, hi = 0, sum = 0, prev_end = 0, max_gap = 0;
  bool ascending = true;
  for (uint32_t i = 0; i < n; i++) {
    const uint64_t o = off[i], e = o + len[i];
    lo = std::min(lo, o);
    hi = std::max(hi, e);
    sum += len[i];
    if (i) {
      if (o < prev_end) ascending = false;
      else max_gap = std::max(max_gap, o - prev_end);
    }
    prev_end = e;
  }
  bool disjoint = true;
  if ((hi - lo) <= sum + sum / 4 + 4096) {
    if (!ascending) {
      std::vector<uint32_t> ord(n);
      std::iota(ord.begin(), ord.end(), 0u);
      std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return off[a] < off[b]; });
      max_gap = 0;
      for (uint32_t k = 1; k < n && disjoint; k++) {
        const uint64_t pe = off[ord[k - 1]] + len[ord[k - 1]];
        if (off[ord[k]] < pe) disjoint = false;
        else max_gap = std::max(max_gap, off[ord[k]] - pe);
      }
    }
    if (disjoint) {
      // exact: the ranges tile the span up to alignment padding (< 16 bytes after a row) — the only gaps a D2H span
      // copy may write over (include/znippy_cuda.h)
      L.exact = max_gap < 16;
      L.span = true;
      L.span_lo = lo;
      L.span_bytes = hi - lo;
      L.total = hi - lo;
      for (uint32_t i = 0; i < n; i++) L.dev_off[i] = off[i] - lo;
      return L;
    }
  }
  uint64_t cur = 0;
  for (uint32_t i = 0; i < n; i++) {
    L.dev_off[i] = cur;
    cur += (len[i] + 15) & ~15ull;
  }
  L.total = cur;
  return L;
}

static int copy_in(zn_ctx* c, uint8_t* d, const uint8_t* base, const uint64_t* off, const uint64_t* len, uint32_t n,
                   const Layout& L) {
  if (L.span) {
    if (L.span_bytes) ZN_CUDA(c, cudaMemcpyAsync(d, base + L.span_lo, L.span_bytes, cudaMemcpyHostToDevice, c->stream));
    return ZN_OK;
  }
  for (uint32_t i = 0; i < n; i++)
    if (len[i]) ZN_CUDA(c, cudaMemcpyAsync(d + L.dev_off[i], base + off[i], len[i], cudaMemcpyHostToDevice, c->stream));
  return ZN_OK;
}

extern "C" int zn_hash_batch(zn_ctx* c, const uint8_t* base, const uint64_t* off, const uint64_t* len, uint32_t n,
                             uint8_t* digests) {
  if (!c || (n && (!base || !off || !len || !digests))) return ZN_E_ARG;
  if (n == 0) return ZN_OK;
  cudaSetDevice(c->device);
  Layout L = make_layout(off, len, n);
  int rc = ensure(c, &c->d_in, &c->d_in_cap, L.total);
  if (rc) return rc;
  rc = copy_in(c, c->d_in, base, off, len, n, L);
  if (rc) return rc;
  zn_plan* p = zn_plan_hash(c, n, L.dev_off.data(), len, nullptr);
  if (!p) return ZN_E_NOMEM;
  rc = zn_plan_run(p, c->d_in, nullptr, nullptr);
  if (rc == ZN_OK) rc = zn_plan_results(p, nullptr, digests);
  zn_plan_destroy(p);
  return rc;
}

extern "C" int zn_decode_verify_batch(zn_ctx* c, const uint8_t* blobs_base, const uint64_t* blob_off,
                                      const uint64_t* blob_len, const uint8_t* compressed, const uint64_t* out_len,
                                      const uint8_t* expect_digest, uint8_t* out_base, const uint64_t* out_off, uint32_t n,
                                      uint32_t* status, uint8_t* digest_out) {
  if (!c || (n && (!blobs_base || !blob_off || !blob_len || !compressed || !out_len || !status))) return ZN_E_ARG;
  if (out_base && n && !out_off) return ZN_E_ARG;
  if (n == 0) return ZN_OK;
  cudaSetDevice(c->device);
  const bool prof = getenv("ZN_HOST_PROF") != nullptr;  // development: host-side stage times of this call on stderr
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double tp[8] = {0};
  tp[0] = now();
  Layout Li = make_layout(blob_off, blob_len, n);
  // envelope layer (csrc/envelope.cpp): rows flagged 4 are resolved to {payload codec, payload range} here, on the
  // host, before anything is planned — the whole blob still travels (the header bytes in front of a magicless zstd
  // payload become its magic on the device copy), the plan only sees payload ranges
  std::vector<uint64_t> e_off, e_len;
  std::vector<uint8_t> e_comp;
  std::vector<uint32_t> e_status;
  const uint64_t* src_off = Li.dev_off.data();
  const uint64_t* src_len = blob_len;
  for (uint32_t i = 0; i < n; i++)
    if (compressed[i] == 4) {
      if (e_off.empty()) {
        e_off = Li.dev_off;
        e_len.assign(blob_len, blob_len + n);
        e_comp.assign(compressed, compressed + n);
        e_status.assign(n, 0);
      }
      zn_envelope e;
      const int erc = zn_envelope_parse(blobs_base + blob_off[i], (size_t)blob_len[i], &e);
      if (erc != ZN_OK || (e.out_len != ~0ull && e.out_len != out_len[i])) {
        e_status[i] = erc != ZN_OK ? ZN_S_UNSUPPORTED : ZN_S_SIZE_MISMATCH;
        e_len[i] = 0;  // an empty frame: the decoder drops the row at once, its status is replaced below
        e_comp[i] = 1;
        continue;
      }
      static const uint8_t flag_of[5] = {0, 1, 3, 1, 2};  // ZN_PAYLOAD_* -> compressed[] value of the plan
      e_off[i] += e.payload_off;
      e_len[i] = e.payload_len;
      e_comp[i] = flag_of[e.codec];
    }
  if (!e_off.empty()) { src_off = e_off.data(); src_len = e_len.data(); compressed = e_comp.data(); }
  // output layout: mirror the caller's when it is compact, so that one D2H copy returns everything
  Layout Lo;
  std::vector<uint64_t> zero_off;
  if (out_base) {
    Lo = make_layout(out_off, out_len, n);
  } else {  // verify-only: decoded rows still need device space; store-as-is rows need none
    std::vector<uint64_t> need(n);
    for (uint32_t i = 0; i < n; i++) need[i] = compressed[i] ? out_len[i] : 0;
    Lo.dev_off.resize(n);
    uint64_t cur = 0;
    for (uint32_t i = 0; i < n; i++) { Lo.dev_off[i] = cur; cur += (need[i] + 15) & ~15ull; }
    Lo.total = cur;
  }
  tp[1] = now();
  int rc = ensure(c, &c->d_in, &c->d_in_cap, Li.total);
  if (rc) return rc;
  rc = ensure(c, &c->d_out, &c->d_out_cap, Lo.total);
  if (rc) return rc;
  rc = copy_in(c, c->d_in, blobs_base, blob_off, blob_len, n, Li);
  if (rc) return rc;
  tp[2] = now();
  zn_plan* p = plan_build(c, PLAN_DECODE_VERIFY, n, src_off, src_len, compressed, Lo.dev_off.data(), out_len,
                          expect_digest, out_base != nullptr);
  if (!p) return ZN_E_NOMEM;
  tp[3] = now();
  rc = zn_plan_run(p, c->d_in, c->d_out, nullptr);
  tp[4] = now();
  if (rc == ZN_OK && out_base) {
    if (Lo.span && Lo.exact) {
      if (Lo.span_bytes)
        rc = cudaMemcpyAsync(out_base + Lo.span_lo, c->d_out, Lo.span_bytes, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess
                 ? ZN_OK : ZN_E_CUDA;
    } else {  // caller memory between the declared ranges is never written: one copy per row
      for (uint32_t i = 0; i < n && rc == ZN_OK; i++)
        if (out_len[i] &&
            cudaMemcpyAsync(out_base + out_off[i], c->d_out + Lo.dev_off[i], out_len[i], cudaMemcpyDeviceToHost, c->stream) !=
                cudaSuccess)
          rc = ZN_E_CUDA;
    }
    if (rc != ZN_OK) c->err = std::string("D2H: ") + cudaGetErrorString(cudaGetLastError());
  }
  if (rc == ZN_OK) rc = zn_plan_results(p, status, digest_out);
  if (rc == ZN_OK)
    for (uint32_t i = 0; i < (uint32_t)e_status.size(); i++)
      if (e_status[i]) status[i] = e_status[i];
  tp[5] = now();
  zn_plan_destroy(p);
  tp[6] = now();
  if (prof)
    fprintf(stderr, "zn_decode_verify_batch n=%u: layout %.3f  ensure+copy_in %.3f  plan_build %.3f  enqueue %.3f  wait+results %.3f  destroy %.3f ms\n",
            n, tp[1] - tp[0], tp[2] - tp[1], tp[3] - tp[2], tp[4] - tp[3], tp[5] - tp[4], tp[6] - tp[5]);
  return rc;
}

extern "C" int zn_frame_content_size(const uint8_t* blob, size_t len, uint64_t* size_out) {
  if (!blob || !size_out) return ZN_E_ARG;
  *size_out = 0;
  if (len >= 4 && ld32le(blob) == 0x184D2204u) {  // LZ4 frame
    if (len < 7) return ZN_E_ARG;
    const uint32_t flg = blob[4];
    if (!((flg >> 3) & 1)) return 1;
    if (len < 14) return ZN_E_ARG;
    uint64_t v = 0;
    for (int i = 0; i < 8; i++) v |= (uint64_t)blob[6 + i] << (8 * i);
    *size_out = v;
    return ZN_OK;
  }
  if (len < 5 || ld32le(blob) != 0xFD2FB528u) return ZN_E_ARG;
  const uint32_t fhd = blob[4], fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, did_flag = fhd & 3;
  size_t pos = 5 + (single ? 0 : 1) + (did_flag == 3 ? 4 : did_flag);
  const uint32_t fb = fcs_flag == 0 ? single : (fcs_flag == 1 ? 2u : (fcs_flag == 2 ? 4u : 8u));
  if (fb == 0) return 1;
  if (len < pos + fb) return ZN_E_ARG;
  uint64_t v = 0;
  for (uint32_t i = 0; i < fb; i++) v |= (uint64_t)blob[pos + i] << (8 * i);
  if (fb == 2) v += 256;
  *size_out = v;
  return ZN_OK;
}

// --------------------------------------------------------------------------------------------- compression
extern "C" size_t zn_compress_bound(size_t src_len, int codec) { return compress_bound(src_len, codec); }

extern "C" float zn_ctx_last_compress_ms(const zn_ctx* c) { return c ? c->cs.last_ms : 0.f; }

extern "C" int zn_compress_batch(zn_ctx* c, const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                                 uint32_t n, int level, int codec, uint8_t* dst_base, const uint64_t* dst_off,
                                 uint64_t* dst_len_out, uint8_t* digest_out, uint32_t* status) {
  if (!c || (n && (!src_base || !src_off || !src_len || !dst_base || !dst_off || !dst_len_out || !status))) return ZN_E_ARG;
  if (codec != ZN_CODEC_ZSTD && codec != ZN_CODEC_LZ4) return ZN_E_ARG;
  if (n == 0) return ZN_OK;
  cudaSetDevice(c->device);
  for (uint32_t i = 0; i < n; i++)
    if (dst_off[i + 1] < dst_off[i] || dst_off[i + 1] - dst_off[i] < compress_bound(src_len[i], codec)) {
      c->err = "zn_compress_batch: destination capacity below zn_compress_bound";
      return ZN_E_ARG;
    }
  Layout Li = make_layout(src_off, src_len, n);
  std::vector<uint64_t> cap(n), doff(n);
  uint64_t cur = 0;
  for (uint32_t i = 0; i < n; i++) {
    cap[i] = compress_bound(src_len[i], codec);
    doff[i] = cur;
    cur += (cap[i] + 15) & ~15ull;
  }
  int rc = ensure(c, &c->d_in, &c->d_in_cap, Li.total);
  if (rc) return rc;
  rc = ensure(c, &c->d_out, &c->d_out_cap, cur);
  if (rc) return rc;
  rc = copy_in(c, c->d_in, src_base, src_off, src_len, n, Li);
  if (rc) return rc;
  // digest of the ORIGINAL bytes (stream_packer.rs:219) — same kernels as the read side
  zn_plan* hp = nullptr;
  if (digest_out) {
    hp = zn_plan_hash(c, n, Li.dev_off.data(), src_len, nullptr);
    if (!hp) return ZN_E_NOMEM;
    rc = zn_plan_run(hp, c->d_in, nullptr, nullptr);
    if (rc) { zn_plan_destroy(hp); return rc; }
  }
  std::vector<uint64_t> out_len(n, 0);
  uint32_t launches = 0;
  rc = compress_run(&c->cs, c->stream, c->sm_count, c->d_in, Li.dev_off.data(), src_len, n, level, codec, c->d_out, doff.data(),
                    cap.data(), out_len.data(), status, &launches, &c->err);
  c->launches += launches;
  if (rc == ZN_OK) {
    uint64_t packed = 0;
    for (uint32_t i = 0; i < n; i++) { dst_len_out[i] = out_len[i]; if (status[i] == ZN_S_OK) packed += out_len[i]; }
    if (n >= 64 && packed < (1ull << 32)) {
      // many frames: pack them back to back on the device (they sit zn_compress_bound apart), ONE copy into pinned
      // scratch, scatter on the host — 25 000 ten-KiB slices were 25 000 cudaMemcpyAsync calls (~75 ms) before
      std::vector<uint64_t> h(3 * (size_t)n);
      uint64_t cur2 = 0;
      for (uint32_t i = 0; i < n; i++) {
        const uint64_t l = status[i] == ZN_S_OK ? out_len[i] : 0;
        h[i] = doff[i]; h[n + i] = l; h[2 * (size_t)n + i] = cur2;
        cur2 += l;
      }
      uint64_t* d_tab = nullptr;
      uint8_t* d_pack = nullptr;
      uint8_t* h_pack = (uint8_t*)zn_ctx_pinned_alloc(packed + 64);
      const bool ok = h_pack && cudaMallocAsync((void**)&d_tab, h.size() * 8, c->stream) == cudaSuccess &&
                      cudaMallocAsync((void**)&d_pack, packed + 64, c->stream) == cudaSuccess &&
                      cudaMemcpyAsync(d_tab, h.data(), h.size() * 8, cudaMemcpyHostToDevice, c->stream) == cudaSuccess;
      if (ok) {
        k_pack_frames<<<std::min<uint32_t>((n + 7) / 8, (uint32_t)c->sm_count * 8u), 256, 0, c->stream>>>(c->d_out, d_tab, d_tab + n, d_tab + 2 * (size_t)n, n, d_pack);
        c->launches++;
        if (packed && cudaMemcpyAsync(h_pack, d_pack, packed, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) rc = ZN_E_CUDA;
        if (rc == ZN_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) rc = ZN_E_CUDA;
        if (rc == ZN_OK)
          for (uint32_t i = 0; i < n; i++)
            if (h[n + i]) memcpy(dst_base + dst_off[i], h_pack + h[2 * (size_t)n + i], h[n + i]);
      } else rc = ZN_E_NOMEM;
      if (d_tab) cudaFreeAsync(d_tab, c->stream);
      if (d_pack) cudaFreeAsync(d_pack, c->stream);
      if (h_pack) zn_ctx_pinned_free(h_pack);
    } else {
      for (uint32_t i = 0; i < n && rc == ZN_OK; i++)
        if (status[i] == ZN_S_OK && out_len[i] &&
            cudaMemcpyAsync(dst_base + dst_off[i], c->d_out + doff[i], out_len[i], cudaMemcpyDeviceToHost, c->stream) != cudaSuccess)
          rc = ZN_E_CUDA;
      if (rc == ZN_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) rc = ZN_E_CUDA;
    }
    if (rc != ZN_OK) c->err = std::string("compress D2H: ") + cudaGetErrorString(cudaGetLastError());
  }
  if (hp) {
    if (rc == ZN_OK) rc = zn_plan_results(hp, nullptr, digest_out);
    zn_plan_destroy(hp);
  }
  return rc;
}

// --------------------------------------------------------------------------------------------- native read worker
// The shell of the reference's read pipeline (znippy-common/src/decompress.rs:105-192) in C++: the row cursor advances
// one BATCH at a time instead of one row at a time (fetch_add(B), §8b of SURVEY.md), blobs are pread into a pinned
// staging slot by a few I/O threads, ONE zn_decode_verify_batch replaces the per-row decode + blake3 + compare, the
// decoded bytes are pwritten at fdata_offset from the pinned output region, and status[] is folded into the
// counters with the reference's rules (decompress.rs:140,156-184).
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <atomic>
#include <thread>

namespace {
struct Pinned {  // staging buffer from the process-wide pinned cache
  uint8_t* p = nullptr;
  size_t cap = 0;
  bool ensure(size_t need) {
    if (cap >= need) return true;
    if (p) zn_ctx_pinned_free(p);
    p = (uint8_t*)zn_ctx_pinned_alloc(need + 4096);
    cap = p ? need + 4096 : 0;
    return p != nullptr;
  }
  ~Pinned() { if (p) zn_ctx_pinned_free(p); }
};

template <typename F>
void parallel_rows(uint32_t n, int threads, F f, uint32_t serial_below = 7) {
  std::atomic<uint32_t> cur{0};
  auto body = [&] {
    for (;;) {
      const uint32_t i = cur.fetch_add(1, std::memory_order_relaxed);
      if (i >= n) break;
      f(i);
    }
  };
  if (threads <= 1 || n <= serial_below) { body(); return; }
  std::vector<std::thread> ts;
  for (int t = 0; t < threads; t++) ts.emplace_back(body);
  for (auto& t : ts) t.join();
}
}  // namespace

// Internal (container.cpp): zn_decompress_rows plus LAZY rows — out_fd[row] == -2 means "this row is its file": the writer
// thread that holds the row opens out_root/path(row) (O_CREAT | O_TRUNC), writes, closes.  A corpus of 100 000 one-row
// files then needs no descriptor window at all, and its open / close calls run on the io threads beside the pwrites.
extern "C" int zn_decompress_rows_ex(zn_ctx* c, int archive_fd, uint64_t row_lo, uint64_t row_hi, const uint64_t* blob_offset,
                                     const uint64_t* blob_size, const uint64_t* fdata_offset, const uint8_t* compressed,
                                     const uint64_t* uncompressed_size, const uint8_t* checksums, const int* out_fd,
                                     size_t batch_bytes, int io_threads, uint64_t* corrupt_rows_out, zn_verify_stats* stats,
                                     const char* out_root, const char* paths, const uint64_t* path_off);

extern "C" int zn_decompress_rows(zn_ctx* c, int archive_fd, uint64_t row_lo, uint64_t row_hi, const uint64_t* blob_offset,
                                  const uint64_t* blob_size, const uint64_t* fdata_offset, const uint8_t* compressed,
                                  const uint64_t* uncompressed_size, const uint8_t* checksums, const int* out_fd,
                                  size_t batch_bytes, int io_threads, uint64_t* corrupt_rows_out, zn_verify_stats* stats) {
  return zn_decompress_rows_ex(c, archive_fd, row_lo, row_hi, blob_offset, blob_size, fdata_offset, compressed, uncompressed_size,
                               checksums, out_fd, batch_bytes, io_threads, corrupt_rows_out, stats, nullptr, nullptr, nullptr);
}

extern "C" int zn_decompress_rows_ex(zn_ctx* c, int archive_fd, uint64_t row_lo, uint64_t row_hi, const uint64_t* blob_offset,
                                     const uint64_t* blob_size, const uint64_t* fdata_offset, const uint8_t* compressed,
                                     const uint64_t* uncompressed_size, const uint8_t* checksums, const int* out_fd,
                                     size_t batch_bytes, int io_threads, uint64_t* corrupt_rows_out, zn_verify_stats* stats,
                                     const char* out_root, const char* paths, const uint64_t* path_off) {
  if (!c || !stats || row_hi < row_lo) return ZN_E_ARG;
  if (row_hi > row_lo && (!blob_offset || !blob_size || !compressed || !uncompressed_size || !checksums)) return ZN_E_ARG;
  if (out_fd && !fdata_offset) return ZN_E_ARG;
  memset(stats, 0, sizeof *stats);
  {
    // The index columns are untrusted input (they come out of the archive): bound every row before any size is summed.
    // Sizes below 4 GiB and fewer than 2^32 rows keep all u64 sums below exact; a blob must lie inside the archive file.
    struct stat sb;
    if (fstat(archive_fd, &sb) != 0) { c->err = "cannot stat the archive"; return ZN_E_ARG; }
    const uint64_t flen = (uint64_t)sb.st_size;
    const bool regular = S_ISREG(sb.st_mode);
    if (row_hi - row_lo > 0xFFFFFFF0ull) { c->err = "row range too large"; return ZN_E_ARG; }
    for (uint64_t r = row_lo; r < row_hi; r++) {
      if (blob_size[r] >= (1ull << 32) || uncompressed_size[r] >= (1ull << 32)) { c->err = "index row with a blob of 4 GiB or more"; return ZN_E_ARG; }
      if (regular && (blob_offset[r] > flen || blob_size[r] > flen - blob_offset[r])) { c->err = "index row points outside the archive file"; return ZN_E_ARG; }
      if (out_fd && fdata_offset[r] > (1ull << 62)) { c->err = "index row with a file offset out of range"; return ZN_E_ARG; }
    }
  }
  if (batch_bytes < (64u << 20)) batch_bytes = 64u << 20;
  if (io_threads < 1) io_threads = 1;
  // Three stages — pread into pinned memory, GPU decode+verify, pwrite from pinned memory — over two sets of staging
  // buffers: while the GPU works on batch k, helper threads read batch k+1 and write batch k-1 (the reference overlaps
  // the same three through its reader / worker / writer threads, decompress.rs:105-192).  A range that fits one
  // staging budget is still cut into a few batches so that there is something to overlap.
  {
    // ... but only where I/O is worth hiding: many rows, or hundreds of MiB of blobs to read / of cheaply decoded bytes to
    // write.  Entropy-coded data (the slow decode) keeps its rows together: its kernels need every blob they can get.
    uint64_t in_b = 0, out_b = 0;
    for (uint64_t r = row_lo; r < row_hi; r++) { in_b += blob_size[r]; out_b += uncompressed_size[r]; }
    const uint64_t rows = row_hi - row_lo;
    const bool cheap_decode = in_b <= out_b / 16 || in_b >= out_b - out_b / 10;
    const bool split = rows >= 1200 || in_b >= (256ull << 20) || (out_fd && cheap_decode && out_b >= (256ull << 20));
    if (split) {
      const uint64_t quarter = std::max<uint64_t>((in_b + out_b) / 4 + 32 * rows, 64u << 20);
      if (quarter < batch_bytes) batch_bytes = (size_t)quarter;
    }
  }
  struct Batch {
    uint64_t a = 0, b = 0;
    uint32_t n = 0;
    Pinned pin_in, pin_out;
    std::vector<uint64_t> in_off, out_off;
    std::vector<uint32_t> status;
    std::thread reader, writer;
    bool span = false;  // pin_in mirrors the archive bytes [span_lo, span_lo + span_bytes)
    uint64_t span_lo = 0, span_bytes = 0;
  } bt[2];
  std::atomic<int> io_err{0};
  auto join = [](std::thread& t) { if (t.joinable()) t.join(); };
  auto claim = [&](Batch& B, uint64_t a) -> bool {  // next row range whose blobs + outputs fit the staging budget
    uint64_t b = a, need = 0, in_bytes = 0, out_bytes = 0;
    while (b < row_hi) {
      const uint64_t r = blob_size[b] + uncompressed_size[b] + 32;
      if (b > a && need + r > batch_bytes) break;
      need += r;
      in_bytes += (blob_size[b] + 15) & ~15ull;
      out_bytes += (uncompressed_size[b] + 15) & ~15ull;
      b++;
    }
    B.a = a; B.b = b; B.n = (uint32_t)(b - a);
    // Blobs of consecutive rows normally sit back to back in the archive (the writer appends them in row order): then
    // the staging buffer mirrors that span, it is read with a few large preads instead of one per blob (100 000 small
    // files = 100 000 syscalls otherwise) and travels to the device in one copy.
    uint64_t lo = ~0ull, hi = 0, sum = 0;
    for (uint64_t r = a; r < b; r++) {
      lo = std::min(lo, blob_offset[r]);
      hi = std::max(hi, blob_offset[r] + blob_size[r]);
      sum += blob_size[r];
    }
    B.span = b > a && hi - lo <= sum + sum / 8 + 65536;
    B.span_lo = B.span ? lo : 0;
    B.span_bytes = B.span ? hi - lo : 0;
    if (B.span) in_bytes = B.span_bytes;
    if (!B.pin_in.ensure(in_bytes + 16) || (out_fd && !B.pin_out.ensure(out_bytes + 16))) return false;
    B.in_off.resize(B.n);
    B.out_off.resize(B.n);
    B.status.assign(B.n, 0);
    uint64_t ci = 0, co = 0;
    for (uint32_t i = 0; i < B.n; i++) {
      if (B.span) B.in_off[i] = blob_offset[a + i] - lo;
      else { B.in_off[i] = ci; ci += (blob_size[a + i] + 15) & ~15ull; }
      B.out_off[i] = co; co += (uncompressed_size[a + i] + 15) & ~15ull;
    }
    return true;
  };
  auto start_read = [&](Batch& B) {
    B.reader = std::thread([&B, &io_err, archive_fd, blob_size, blob_offset, io_threads]() {
      if (B.span) {
        constexpr uint64_t kPiece = 8ull << 20;
        const uint32_t pieces = (uint32_t)((B.span_bytes + kPiece - 1) / kPiece);
        parallel_rows(pieces, io_threads, [&](uint32_t k) {
          uint64_t done = (uint64_t)k * kPiece;
          const uint64_t end = std::min(B.span_bytes, done + kPiece);
          while (done < end) {
            const ssize_t r = pread(archive_fd, B.pin_in.p + done, end - done, (off_t)(B.span_lo + done));
            if (r <= 0) { io_err = 1; return; }
            done += (uint64_t)r;
          }
        }, 1);
        return;
      }
      parallel_rows(B.n, io_threads, [&](uint32_t i) {  // pread (decompress.rs:148-153)
        uint64_t done = 0, len = blob_size[B.a + i];
        while (done < len) {
          const ssize_t r = pread(archive_fd, B.pin_in.p + B.in_off[i] + done, len - done, (off_t)(blob_offset[B.a + i] + done));
          if (r <= 0) { io_err = 1; return; }
          done += (uint64_t)r;
        }
      });
    });
  };
  auto start_write = [&](Batch& B) {
    B.writer = std::thread([&B, &io_err, out_fd, uncompressed_size, fdata_offset, io_threads, out_root, paths, path_off]() {
      parallel_rows(B.n, io_threads, [&](uint32_t i) {  // pwrite at fdata_offset (decompress.rs:186-189)
        const uint32_t s = B.status[i];
        const bool ok = s == ZN_S_OK || s == ZN_S_DIGEST_MISMATCH;
        int fd = out_fd[B.a + i];
        const bool lazy = fd == -2 && out_root && paths && path_off;
        if (lazy) {  // the file exists afterwards even when its only chunk failed to decode, as with the reference's up-front creation
          std::string full(out_root);
          full += '/';
          full.append(paths + path_off[B.a + i], (size_t)(path_off[B.a + i + 1] - path_off[B.a + i]));
          fd = open(full.c_str(), O_CREAT | O_WRONLY | O_TRUNC, 0644);
          if (fd < 0) { io_err = 1; return; }
        }
        if (ok && fd >= 0) {
          uint64_t done = 0, len = uncompressed_size[B.a + i];
          while (done < len) {
            const ssize_t r = pwrite(fd, B.pin_out.p + B.out_off[i] + done, len - done, (off_t)(fdata_offset[B.a + i] + done));
            if (r <= 0) { io_err = 1; break; }
            done += (uint64_t)r;
          }
        }
        if (lazy) close(fd);
      });
    });
  };
  int rc = ZN_OK;
  uint64_t next = row_lo;
  int cur = 0;
  bool have = false;
  if (next < row_hi) {
    if (!claim(bt[0], next)) { c->err = "pinned staging allocation failed"; return ZN_E_NOMEM; }
    next = bt[0].b;
    start_read(bt[0]);
    have = true;
  }
  while (have && rc == ZN_OK) {
    Batch& B = bt[cur];
    Batch& O = bt[cur ^ 1];
    join(B.reader);
    if (io_err) { c->err = "failed to read blob from archive"; rc = ZN_E_ARG; break; }
    bool more = false;
    if (next < row_hi) {  // the other buffer set is free once its writer is done
      join(O.writer);
      if (io_err) { c->err = "pwrite to output file failed"; rc = ZN_E_ARG; break; }
      if (!claim(O, next)) { c->err = "pinned staging allocation failed"; rc = ZN_E_NOMEM; break; }
      next = O.b;
      start_read(O);
      more = true;
    }
    rc = zn_decode_verify_batch(c, B.pin_in.p, B.in_off.data(), blob_size + B.a, compressed + B.a, uncompressed_size + B.a,
                                checksums + 32 * B.a, out_fd ? B.pin_out.p : nullptr, out_fd ? B.out_off.data() : nullptr, B.n,
                                B.status.data(), nullptr);
    if (rc != ZN_OK) break;
    for (uint32_t i = 0; i < B.n; i++) {  // fold, decompress.rs:140,156-184
      stats->total_chunks++;
      const uint32_t s = B.status[i];
      if (s != ZN_S_OK && s != ZN_S_DIGEST_MISMATCH) { stats->decode_errors++; continue; }
      const uint64_t len = uncompressed_size[B.a + i];
      stats->total_written_bytes += len;
      if (s == ZN_S_OK) stats->verified_bytes += len;
      else {
        stats->corrupt_bytes += len;
        if (corrupt_rows_out) corrupt_rows_out[stats->corrupt_rows] = B.a + i;
        stats->corrupt_rows++;
      }
    }
    if (out_fd) start_write(B);
    have = more;
    cur ^= 1;
  }
  for (auto& B : bt) { join(B.reader); join(B.writer); }
  if (rc == ZN_OK && io_err) { c->err = "pwrite to output file failed"; rc = ZN_E_ARG; }
  return rc;
}

#ifdef ZN_WS_DEBUG
// development only (tools/ws_times.py): reset / read the fused kernel's phase stamps
extern "C" void zn_debug_ws_times(unsigned long long* out, int reset) {
  if (reset) {
    unsigned long long init[4] = {~0ull, 0, 0, 0};
    cudaMemcpyToSymbol(g_ws_dbg, init, sizeof init);
  } else {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_ws_dbg, 32);
  }
}
#endif
