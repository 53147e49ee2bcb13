// Kernels of the device-wide Zstandard decode pipeline (see zpipe.cuh for the phases and what they replace:
// codec::decompress_into, znippy-common/src/codec.rs:67-78, for every row of a batch at once).
//
//   k_zwalk    thread per blob      block table + pool allocation
//   k_ztables  warp per block       FSE table descriptions -> fat decoding tables (all lanes, position by position)
//   k_zseq1    LANE per block       sequence stage, phase 1: the FSE state chain alone (tables + bit stream in shared memory)
//   k_zseq2    warp per block       sequence stage, phase 2: values, positions, repeat offsets (prefix scans), 16-byte records
//   k_zseq_g   LANE per block       the one-pass sequence stage (batches of many small blobs)
//   k_zlit     LANE per stream      Huffman literals, decoding table in shared memory, word stores
//   k_zchain   thread per blob      output offsets, repeat-offset histories, size checks
//   k_zexec2   CTA per blob         sequence execution in shared memory, group by group
//
// Every kernel is latency-bound integer work; the design goal is the number of independent dependent-chains in flight
// (32 per warp in seq / lit, versus one per warp in the one-team-per-blob decoders), not bytes per instruction.
#pragma once
#include "coop.cuh"
#include "zpipe.cuh"

namespace zn {
namespace zp {

__device__ FseD g_zpredef[kTabSet];  // decoding tables of the predefined distributions (filled by zn_ctx_create)

// shared-memory accesses by 32-bit shared address (no generic-address arithmetic in the byte loops)
ZN_D uint32_t lds8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
ZN_D void sts8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
// table reads of the sequence decoder: not volatile (the lane's tables never change while it decodes), so the
// compiler may schedule them early
ZN_D uint32_t lds32_ro(uint32_t a) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }

constexpr uint32_t kTabWarps = 8;    // k_ztables: warps per CTA
constexpr uint32_t kLitBlocks = 16;  // k_zlit: blocks per CTA (4 lanes each), one 4 KiB Huffman table per block
constexpr uint32_t kLitSmem = kLitBlocks * 2048 * 2;


// ---------------------------------------------------------------------------------------------------------------- walk
__global__ void __launch_bounds__(64) k_zwalk(ZArgs a) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.nzb) return;
  ZBlob z = a.zb[i];
  const BlobDesc d = a.blobs[z.blob];
  uint32_t state = 1, nb = 0;
  if (d.src_len < 0xFFFFFFF0ull && d.dst_cap < 0xFFFFFFF0ull && !(d.flags & F_LZ4_BLOCK)) {
    WalkNeeds needs;
    ZBlock* blocks = a.blocks + z.slot0;
    nb = walk_blob(a.blobs_base + d.src_off, (uint32_t)d.src_len, z.slot_cap, blocks, &needs);
    if (nb != ~0u) {
      ZPools* p = a.pools;
      const uint32_t comp0 = atomicAdd(&p->comp_used, needs.comp);
      bool ok = comp0 + needs.comp <= p->comp_cap;
      uint32_t seq0 = 0, lit0 = 0, tab0 = 0;
      if (ok) { seq0 = atomicAdd(&p->seq_used, needs.nseq); ok = (uint64_t)seq0 + needs.nseq <= p->seq_cap; }
      if (ok) { lit0 = atomicAdd(&p->lit_used16, needs.lit16); ok = (uint64_t)lit0 + needs.lit16 <= p->lit_cap16; }
      if (ok) { tab0 = atomicAdd(&p->tab_used, needs.tabs); ok = (uint64_t)tab0 + needs.tabs <= p->tab_cap; }
      uint32_t c = 0;
      for (uint32_t j = 0; j < nb; j++) {
        ZBlock* b = &blocks[j];
        b->seq_base += seq0;
        b->lit_base16 += lit0;
        if (b->tab_slot != kNoSlot) b->tab_slot += tab0;
        b->pad[0] = i;  // owning pipeline blob
        if ((b->flags & ZB_TYPE_MASK) == 2) {
          if (comp0 + c < p->comp_cap) a.comp_list[comp0 + c] = ok ? z.slot0 + j : kNoSlot;
          c++;
        }
      }
      if (ok) state = 0;
    } else nb = 0;
  }
  a.zb[i].n_blocks = nb;
  a.zb[i].state = state;
}

// -------------------------------------------------------------------------------------------------------------- tables
// One table built by the whole warp, position by position (zpipe.cuh: fat_symbol_at; build_fat_table_by_position is the
// host mirror).  cum / lowsym / run: 64 uint16 each of shared memory.  Lane l takes positions l, l + 32, ...: the symbol
// at a position comes out of the closed form, its number within the symbol is a running count per symbol that the
// warp advances 32 positions at a time (match.any groups the lanes that hold the same symbol).
ZN_D bool build_fat_table_warp(FseD* t, int k, const int16_t* norm, int nsym, int log, uint16_t* cum, uint16_t* lowsym, uint16_t* run,
                               uint32_t lane) {
  const uint32_t size = 1u << log, inv = fat_step_inv(size), FULL = 0xFFFFFFFFu, lt = (1u << lane) - 1u;
  uint32_t acc = 0, n_low = 0;
#pragma unroll
  for (uint32_t sb = 0; sb < 64; sb += 32) {
    const uint32_t s = sb + lane;
    const int c = (int)s < nsym ? (int)norm[s] : 0;
    uint32_t v = c > 0 ? (uint32_t)c : 0u;
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) {
      const uint32_t n = __shfl_up_sync(FULL, v, d);
      if (lane >= d) v += n;
    }
    cum[s] = (int)s < nsym ? (uint16_t)(acc + v) : (uint16_t)0xFFFF;
    run[s] = 0;
    const uint32_t lowb = __ballot_sync(FULL, c == -1);
    if (c == -1) lowsym[n_low + __popc(lowb & lt)] = (uint16_t)s;
    acc += __shfl_sync(FULL, v, 31);
    n_low += __popc(lowb);
  }
  __syncwarp();
  bool ok = true;
  for (uint32_t p0 = 0; p0 < size; p0 += 32) {
    const uint32_t p = p0 + lane;
    const uint32_t sym = fat_symbol_at(p, size, n_low, inv, cum, lowsym);
    const bool valid = sym < (uint32_t)nsym;
    const uint32_t key = valid ? sym : 63u;
    const uint32_t peers = __match_any_sync(FULL, key);
    const uint32_t rank = (uint32_t)run[key] + __popc(peers & lt);
    __syncwarp();
    if ((peers & lt) == 0) run[key] = (uint16_t)(run[key] + __popc(peers));  // the group's lowest lane
    __syncwarp();
    FseD e = 0;
    bool good = valid;
    if (valid) {
      const int cs = (int)norm[sym];
      good = fat_entry(k, sym, (cs == -1 ? 1u : (uint32_t)cs) + rank, log, &e);
    }
    if (good) t[p] = e;
    ok = ok && good;
  }
  return __all_sync(FULL, ok);
}

__global__ void __launch_bounds__(kTabWarps * 32) k_ztables(ZArgs a) {
  __shared__ int16_t s_norm[kTabWarps][3][64];
  __shared__ uint16_t s_aux[kTabWarps][3][64];  // cum / lowsym / run of the table being built
  __shared__ int s_nsym[kTabWarps][3], s_log[kTabWarps][3];
  __shared__ uint32_t s_bits[kTabWarps], s_ok[kTabWarps];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const uint32_t n_comp = min(a.pools->comp_used, a.pools->comp_cap);
  for (uint32_t it = blockIdx.x * kTabWarps + warp; it < n_comp; it += gridDim.x * kTabWarps) {
    const uint32_t slot = a.comp_list[it];
    if (slot == kNoSlot) continue;
    ZBlock* b = &a.blocks[slot];
    if (b->nseq == 0) continue;
    const BlobDesc d = a.blobs[a.zb[b->pad[0]].blob];
    const uint8_t* src = a.blobs_base + d.src_off;
    FseD* set = b->tab_slot != kNoSlot ? a.tabs + (size_t)b->tab_slot * kTabSet : nullptr;
    if (lane == 0) {
      uint32_t bits_off = 0;
      s_ok[warp] = parse_table_descs(src, b, set, s_norm[warp], s_nsym[warp], s_log[warp], &bits_off) ? 1u : 0u;
      s_bits[warp] = bits_off;
    }
    __syncwarp();
    bool ok = s_ok[warp] != 0;
    if (ok) {
#pragma unroll
      for (int k = 0; k < 3; k++) {
        if (s_log[warp][k] < 5) continue;  // predefined, RLE (written by the parser) or repeated: nothing to build
        const uint32_t offs = k == 0 ? kTabOffLL : (k == 1 ? kTabOffOF : kTabOffML);
        ok = build_fat_table_warp(set + offs, k, s_norm[warp][k], s_nsym[warp][k], s_log[warp][k], s_aux[warp][0], s_aux[warp][1],
                                  s_aux[warp][2], lane) && ok;
        __syncwarp();
      }
    }
    if (lane == 0 && ok) {
      uint32_t tl = 0;
      for (int k = 0; k < 3; k++)
        if (s_log[warp][k] >= 0) tl |= (uint32_t)s_log[warp][k] << (8 * k);
      b->tlogs = tl;
      b->bits_off = s_bits[warp];
    }
    __syncwarp();
  }
}

// ----------------------------------------------------------------------------------------------------------------- seq
// Where a block's three tables come from (own set, an earlier block's, predefined) and their logs; false = undefined.
ZN_D bool seq_table_sources(const ZArgs& a, const ZBlock* b, const ZBlob& z, const FseD** t, uint32_t* logs) {
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const uint32_t offs = k == 0 ? kTabOffLL : (k == 1 ? kTabOffOF : kTabOffML);
    const uint32_t def = b->seq_def[k];
    t[k] = g_zpredef + offs;
    logs[k] = k == 1 ? 5u : 6u;
    if (def == kDefNone) ok = false;
    else if (def != kDefPredef) {
      const ZBlock* db = &a.blocks[z.slot0 + def];
      if (db->bits_off == ~0u || db->tab_slot == kNoSlot) ok = false;
      else {
        t[k] = a.tabs + (size_t)db->tab_slot * kTabSet + offs;
        logs[k] = (db->tlogs >> (8 * k)) & 0xFFu;
      }
    }
  }
  return ok;
}

// One-pass form: one lane per block, every block of the batch at once.  The tables stay in global memory (4-byte
// entries: all table sets of a 2 GiB batch are 84 MB and stay L2-resident when the record stores stream past them).
struct GlobalTabs {
  const FseD* t[3];
  uint32_t lut_s;
  // .cg: the table sets of the lanes of one SM (3.5 warps x 32 lanes x 5 KiB) are several times its L1; left to allocate
  // there they evict the lanes' bitstream lines, and the refill then waits for L2 as well
  ZN_D uint32_t ld(int k, uint32_t i) const { return __ldcg(t[k] + i); }
  ZN_D uint32_t base(int k, uint32_t sym) const { return lds32_ro(lut_s + 4u * ((k == 0 ? 0u : 36u) + sym)); }
};

__global__ void __launch_bounds__(32) k_zseq_g(ZArgs a) {
  __shared__ uint32_t s_lut[36 + 53];
  const uint32_t tid = threadIdx.x;
  for (uint32_t i = tid; i < 36; i += 32) s_lut[i] = zs::kLLBase[i];
  for (uint32_t i = tid; i < 53; i += 32) s_lut[36 + i] = zs::kMLBase[i];
  __syncwarp();
  GlobalTabs st;
  st.lut_s = (uint32_t)__cvta_generic_to_shared(s_lut);
  const uint32_t n_comp = min(a.pools->comp_used, a.pools->comp_cap);
  for (uint32_t it = blockIdx.x * 32 + tid; it < n_comp; it += gridDim.x * 32) {
    const uint32_t slot = a.comp_list[it];
    if (slot == kNoSlot) continue;
    ZBlock* b = &a.blocks[slot];
    if (b->nseq == 0 || b->bits_off == ~0u) continue;
    const ZBlob z = a.zb[b->pad[0]];
    const BlobDesc d = a.blobs[z.blob];
    const uint8_t* src = a.blobs_base + d.src_off;
    uint32_t logs[3];
    if (!seq_table_sources(a, b, z, st.t, logs)) continue;
    uint32_t matched, lit_used, rep[3];
    if (decode_sequences(src, b, st, logs, a.recs + b->seq_base, &matched, &lit_used, rep)) {
      b->matched = matched;
      b->lit_used = lit_used;
      b->rep_fin[0] = rep[0]; b->rep_fin[1] = rep[1]; b->rep_fin[2] = rep[2];
      b->st_seq = 0;
    }
  }
}

// ------------------------------------------------------------------------------------------------- seq, two-phase form
// (zpipe.cuh, "seq, two-phase form").  Phase 1 is the state chain alone, one lane per block; phase 2 decodes the values
// of every sequence independently, a thread per run of consecutive sequences, and writes the final records.

// phase 1, tables in shared memory in the 3-byte phase-1 format (converted while they are copied in): per lane kTabSet
// u16 {base | state bits << 10}, then kTabSet u8 {state bits + extra bits}
ZN_D uint32_t lds16_ro(uint32_t a) { uint32_t v; asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
ZN_D uint32_t lds8_ro(uint32_t a) { uint32_t v; asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
struct SmemTabs1 {
  uint32_t tab_s;
  ZN_D void ld1(int k, uint32_t i, uint32_t* nb, uint32_t* tot) const {
    const uint32_t e = (k == 0 ? kTabOffLL : (k == 1 ? kTabOffOF : kTabOffML)) + i;
    *nb = lds16_ro(tab_s + 2u * e);
    *tot = lds8_ro(tab_s + 2u * kTabSet + e);
  }
};
constexpr uint32_t kSeq1Lanes = 56;
constexpr uint32_t kSeq1Set = kTabSet * 3;  // bytes of one lane's tables
constexpr uint32_t kSeq1Smem = kSeq1Lanes * (kSeq1Set + RingBits::kRingBytes);  // tables + one stream ring per lane

__global__ void __launch_bounds__(64, 1) k_zseq1(ZArgs a) {
  extern __shared__ __align__(16) uint8_t seq_smem[];
  const uint32_t tid = threadIdx.x;
  if (tid >= kSeq1Lanes) return;
  SmemTabs1 st;
  st.tab_s = (uint32_t)__cvta_generic_to_shared(seq_smem) + tid * kSeq1Set;
  RingBits sb;
  sb.ring_s = (uint32_t)__cvta_generic_to_shared(seq_smem) + kSeq1Lanes * kSeq1Set + tid * RingBits::kRingBytes;
  const uint32_t n_comp = min(a.pools->comp_used, a.pools->comp_cap);
  for (uint32_t it = blockIdx.x * kSeq1Lanes + tid; it < n_comp; it += gridDim.x * kSeq1Lanes) {
    const uint32_t slot = a.comp_list[it];
    if (slot == kNoSlot) continue;
    ZBlock* b = &a.blocks[slot];
    if (b->nseq == 0 || b->bits_off == ~0u) continue;
    const ZBlob z = a.zb[b->pad[0]];
    const BlobDesc d = a.blobs[z.blob];
    const FseD* t[3];
    uint32_t logs[3];
    if (!seq_table_sources(a, b, z, t, logs)) continue;
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const uint32_t n = 1u << logs[k], e0 = k == 0 ? kTabOffLL : (k == 1 ? kTabOffOF : kTabOffML);
#pragma unroll 8
      for (uint32_t i = 0; i < n; i++) {
        const FseD e = t[k][i];
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(st.tab_s + 2u * (e0 + i)), "r"(e & 0x3FFFu) : "memory");
        sts8(st.tab_s + 2u * kTabSet + e0 + i, fd_nbits(e) + fd_extra(e));
      }
    }
    if (seq_phase1(sb, a.blobs_base + d.src_off, b, st, logs, a.p1 + b->seq_base)) b->st_seq = 2;
  }
}

// phase 2: one warp per block, 128 consecutive sequences per step, four per lane (zpipe.cuh: seq_phase2_host is the same
// arithmetic with the lanes as arrays)
struct GlobalTabs2 {
  const FseD* t[3];
  uint32_t lut_s;
  ZN_D uint32_t ld(int k, uint32_t i) const { return __ldg(t[k] + i); }
  ZN_D uint32_t base(int k, uint32_t sym) const { return lds32_ro(lut_s + 4u * ((k == 0 ? 0u : 36u) + sym)); }
};
constexpr uint32_t kSeq2Warps = 4;

__global__ void __launch_bounds__(kSeq2Warps * 32) k_zseq2(ZArgs a) {
  __shared__ uint32_t s_lut[36 + 53];
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  for (uint32_t i = tid; i < 36; i += kSeq2Warps * 32) s_lut[i] = zs::kLLBase[i];
  for (uint32_t i = tid; i < 53; i += kSeq2Warps * 32) s_lut[36 + i] = zs::kMLBase[i];
  __syncthreads();
  GlobalTabs2 st;
  st.lut_s = (uint32_t)__cvta_generic_to_shared(s_lut);
  const uint32_t n_comp = min(a.pools->comp_used, a.pools->comp_cap);
  const uint32_t FULL = 0xFFFFFFFFu;
  for (uint32_t it = blockIdx.x * kSeq2Warps + warp; it < n_comp; it += gridDim.x * kSeq2Warps) {
    const uint32_t slot = a.comp_list[it];
    if (slot == kNoSlot) continue;
    ZBlock* b = &a.blocks[slot];
    const uint32_t nseq = b->nseq;
    if (nseq == 0 || b->st_seq != 2) continue;  // phase 1 did not get through: the blob goes to the legacy decoder
    const ZBlob z = a.zb[b->pad[0]];
    const BlobDesc d = a.blobs[z.blob];
    const uint8_t* src = a.blobs_base + d.src_off;
    uint32_t logs[3];
    seq_table_sources(a, b, z, st.t, logs);
    SeqBits sb;
    sb.init(src + b->bits_off, b->src_off + b->len - b->bits_off);
    SeqRec16* rec = a.recs + b->seq_base;
    const SeqP1* p1 = a.p1 + b->seq_base;
    const uint32_t lit_len = b->lit_regen;
    uint32_t c_lit = 0, c_out = 0, c0 = sym_make(0), c1 = sym_make(1), c2 = sym_make(2);  // state carried from step to step
    uint32_t bad = 0;
    for (uint32_t base = 0; base < nseq; base += 32 * kSeqPerLane) {
      const uint32_t i0 = base + lane * kSeqPerLane;
      uint32_t ll[kSeqPerLane], ml[kSeqPerLane], offx[kSeqPerLane], pl[kSeqPerLane], po[kSeqPerLane];
      uint32_t m0 = sym_make(0), m1 = sym_make(1), m2 = sym_make(2), sl = 0, so = 0;
#pragma unroll
      for (uint32_t j = 0; j < kSeqPerLane; j++) {  // the lane's own sequences: values, effect on an unknown history, local positions
        ll[j] = 0; ml[j] = 0; offx[j] = 0;
        if (i0 + j < nseq) {
          uint32_t ov, zf = 0;
          seq_values(sb, st, p1 + i0 + j, &ll[j], &ml[j], &ov);
          offx[j] = rep_step(ov, ll[j], m0, m1, m2, &zf);
        }
        pl[j] = sl; po[j] = so;
        sl += ll[j]; so += ll[j] + ml[j];
      }
      const uint32_t tot_l = sl, tot_o = so;
#pragma unroll
      for (uint32_t dd = 1; dd < 32; dd <<= 1) {  // inclusive scans over the lanes: the two sums, the history maps
        const uint32_t tl = __shfl_up_sync(FULL, sl, dd), to = __shfl_up_sync(FULL, so, dd);
        const uint32_t t0 = __shfl_up_sync(FULL, m0, dd), t1 = __shfl_up_sync(FULL, m1, dd), t2 = __shfl_up_sync(FULL, m2, dd);
        if (lane >= dd) {
          sl += tl; so += to;
          const uint32_t n0 = sym_compose(m0, t0, t1, t2), n1 = sym_compose(m1, t0, t1, t2), n2 = sym_compose(m2, t0, t1, t2);
          m0 = n0; m1 = n1; m2 = n2;
        }
      }
      uint32_t e0 = __shfl_up_sync(FULL, m0, 1), e1 = __shfl_up_sync(FULL, m1, 1), e2 = __shfl_up_sync(FULL, m2, 1);
      if (lane == 0) { e0 = sym_make(0); e1 = sym_make(1); e2 = sym_make(2); }
      const uint32_t lit_base = c_lit + (sl - tot_l), out_base = c_out + (so - tot_o);
#pragma unroll
      for (uint32_t j = 0; j < kSeqPerLane; j++)
        if (i0 + j < nseq) {
          const uint32_t offset = sym_compose(sym_compose(offx[j], e0, e1, e2), c0, c1, c2);
          const uint32_t lit_pos = lit_base + pl[j], out_pos = out_base + po[j];
          bad |= (offset == 0) | (lit_pos + ll[j] > lit_len) | (out_pos + ll[j] + ml[j] > kZstdBlockMax);
          rec_store(rec + i0 + j, rec_pack(out_pos & 0x3FFFFu, lit_pos & 0x3FFFFu, ll[j] & 0x3FFFFu, ml[j] & 0x3FFFFu, offset));
        }
      const uint32_t T0 = __shfl_sync(FULL, m0, 31), T1 = __shfl_sync(FULL, m1, 31), T2 = __shfl_sync(FULL, m2, 31);
      const uint32_t n0 = sym_compose(T0, c0, c1, c2), n1 = sym_compose(T1, c0, c1, c2), n2 = sym_compose(T2, c0, c1, c2);
      c0 = n0; c1 = n1; c2 = n2;
      c_lit = sat_add(c_lit, __shfl_sync(FULL, sl, 31));
      c_out = sat_add(c_out, __shfl_sync(FULL, so, 31));
    }
    bad = __any_sync(FULL, bad != 0);
    if (lane == 0 && !bad) {
      b->matched = c_out;
      b->lit_used = c_lit;
      b->rep_fin[0] = c0; b->rep_fin[1] = c1; b->rep_fin[2] = c2;
      b->st_seq = 0;
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------- lit
__global__ void __launch_bounds__(kLitBlocks * 4) k_zlit(ZArgs a) {
  extern __shared__ __align__(16) uint8_t lit_smem[];
  __shared__ uint32_t s_mb[kLitBlocks];
  uint16_t* tables = reinterpret_cast<uint16_t*>(lit_smem);
  const uint32_t q = threadIdx.x >> 2, k = threadIdx.x & 3u;
  const uint32_t n_comp = min(a.pools->comp_used, a.pools->comp_cap);
  for (uint32_t base = blockIdx.x * kLitBlocks; base < n_comp; base += gridDim.x * kLitBlocks) {
    const uint32_t it = base + q;
    ZBlock* b = nullptr;
    const uint8_t* src = nullptr;
    uint32_t slot0 = 0;
    if (it < n_comp) {
      const uint32_t slot = a.comp_list[it];
      if (slot != kNoSlot) {
        b = &a.blocks[slot];
        if (((b->flags >> ZB_LIT_SHIFT) & 3u) < 2) b = nullptr;
      }
    }
    if (b) {
      const ZBlob z = a.zb[b->pad[0]];
      src = a.blobs_base + a.blobs[z.blob].src_off;
      slot0 = z.slot0;
    }
    uint16_t* h = tables + q * 2048;
    if (k == 0) {
      uint32_t mb = 0;
      if (b) {
        const ZBlock* db = &a.blocks[slot0 + b->huf_def];
        mb = huf_build(h, src + db->huf_desc, db->huf_dlen);
      }
      s_mb[q] = mb;
    }
    __syncthreads();
    const uint32_t mb = s_mb[q];
    if (b && mb && k < ((b->flags & ZB_STREAMS4) ? 4u : 1u)) {
      uint32_t so, sl, oo, ol;
      if (huf_stream_ranges(src, b, k, &so, &sl, &oo, &ol) &&
          huf_decode_stream_w(h, mb, src + b->lit_off + so, sl, a.lits + (size_t)b->lit_base16 * 16 + oo, ol))
        atomicSub(&b->st_lit, 1u);
    }
    __syncthreads();
  }
}

// --------------------------------------------------------------------------------------------------------------- chain
__global__ void __launch_bounds__(64) k_zchain(ZArgs a) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.nzb) return;
  const ZBlob z = a.zb[i];
  if (z.state) return;
  const BlobDesc d = a.blobs[z.blob];
  if (!chain_blob(a.blocks + z.slot0, z.n_blocks, (uint32_t)d.dst_cap)) a.zb[i].state = 1;
}

// ---------------------------------------------------------------------------------------------------------------- exec
// One CTA per blob, blocks in order.  A block's sequences are executed in GROUPS: the next <= K * NT sequences whose
// output spans <= GB bytes, assembled in a shared-memory buffer and flushed with one coalesced copy.  A sequence longer
// than the buffer, raw / RLE blocks and a block's trailing literals are written straight to global memory by the whole
// team.
//
// LZ77 execution is only serial where a match reads bytes that an earlier match of the same neighbourhood produces.
// Measured on python sources (zstd level 3): the TRUE dependence depth of a 128 KiB block is ~70 matches, while it
// holds ~10 000 of them.  So the matches that read bytes of their own group are resolved by POINTER JUMPING over bytes:
//
//   setup   every output byte of the group is either KNOWN — a literal, or a match byte whose source lies before the group
//           (final, in global memory): stored into the buffer at once — or it gets a PARENT: the group-relative position it
//           copies from (par[], 16 bits per byte; a match with distance < length points every byte into the window before
//           the match, so it adds one level, not length / distance levels);
//   rounds  the first round scans par[] (8 entries per 16-byte load) and lists the bytes that are still unknown after it;
//           later rounds walk that list densely, one lane per unknown byte, compacting it as they go.  An unknown byte
//           looks at its parent: known -> copy the byte and become known; unknown -> adopt the parent's parent.  Chains
//           halve every round, so a group whose dependence depth is ~20 matches is done in ~5 rounds of plain loads and
//           stores: no atomics, no fences — one barrier per round.  "Known" must mean "known before this round's
//           barrier": a byte resolved in round r is marked with r's parity (kFresh); a reader in a round of the same
//           parity waits one round (the marker may be this round's), a reader of the other parity copies — so nobody
//           ever reads a byte that was stored in the same round, and no marker ever needs a second visit;
//   flush   one coalesced copy of the group to global memory, par[] reset to kKnown.
//
// Everything is sized by instruction issue, not bytes: a lone lane that copies costs its warp as much as 32, so the
// common cases are straight-line predicated code and longer runs become jobs that a whole warp copies.
constexpr uint32_t kLitLane = 8;     // literal runs up to this length: straight-line code in the owning lane
constexpr uint32_t kMatchLane = 16;  // matches up to this length likewise; longer ones become warp jobs

// development (build with ZN_TRACE_BUILD=1): cycle counters of the exec kernel's phases, summed over the grid
#ifdef ZP_TRACE
__device__ unsigned long long g_ztrace[32];
#define ZT_DECL long long zt_t = clock64(); long long zt_acc[16] = {0}
#define ZT(i) do { const long long n__ = clock64(); zt_acc[i] += n__ - zt_t; zt_t = n__; } while (0)
#define ZT_CNT(i, v) zt_acc[i] += (v)
#define ZT_FLUSH(base, n) do { for (int i__ = 0; i__ < (n); i__++) atomicAdd(&g_ztrace[(base) + i__], (unsigned long long)zt_acc[i__]); } while (0)
#else
#define ZT_DECL
#define ZT(i)
#define ZT_CNT(i, v)
#define ZT_FLUSH(base, n)
#endif

// bytes per group (template parameter GB) <= 16384: parents are < 2^14, which leaves two flag bits in 16
constexpr uint32_t kKnown = 0xFFFFu;  // par[] value of a byte whose value is in the buffer (since an earlier round)
constexpr uint32_t kFresh = 0x8000u;  // | parity << 14: resolved in the round of that parity

ZN_D uint32_t lds16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
ZN_D void sts16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
ZN_D uint4 lds128(uint32_t a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v; }
ZN_D void sts128(uint32_t a, uint4 v) { asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory"); }

template <int NT, int K, uint32_t GB, uint32_t LC>
struct Exec2Shared {
  static_assert(GB <= 16384, "parents are 14-bit");
  // LC = entries per list of unknown bytes.  GB / 4: the two lists alias the literal staging area (dead once the jobs are
  // done); larger: they get their own array (a scan round costs ~17 k cycles, and with GB / 4 entries 70 % of the groups of
  // python sources needed a second one)
  static constexpr bool kOwnLists = LC > GB / 4;
  alignas(16) uint16_t lists[kOwnLists ? 2 * LC : 8];
  static constexpr uint32_t kSeqs = K * NT;
  alignas(16) uint8_t buf[GB + 16];
  alignas(16) uint16_t par[GB + 8];
  alignas(16) uint8_t lits[GB + 32];
  uint16_t jobs[kSeqs * 2];  // warp jobs of the setup: sequence (offset from the group's first) | kind << 15 (1 = literal run, 0 = match)
  uint32_t n_jobs;
  uint32_t lcnt[3];          // unknown bytes left after a round, rotating: round r appends to [(r + 1) % 3], clears [(r + 2) % 3]
  uint32_t pat[kPatWords];
  SeqRec16 first;
  uint32_t cnt, gend, lit_hi;
  uint32_t err, item;
};

template <int NT, int K, uint32_t GB, int MINB, uint32_t LC = GB / 4>
__global__ void __launch_bounds__(NT, MINB) k_zexec2(ZArgs a, uint8_t* out_base, uint32_t* produced, uint32_t* work_counter) {
  extern __shared__ __align__(16) uint8_t exec_smem[];
  using Sh = Exec2Shared<NT, K, GB, LC>;
  Sh* sh = reinterpret_cast<Sh*>(exec_smem);
  const Team t{threadIdx.x, (uint32_t)NT};
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t buf_s = (uint32_t)__cvta_generic_to_shared(sh->buf), lits_s = (uint32_t)__cvta_generic_to_shared(sh->lits),
                 par_s = (uint32_t)__cvta_generic_to_shared(sh->par);
  const uint4 known4 = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
  for (uint32_t i = tid * 8; i < GB + 8; i += NT * 8) sts128(par_s + 2 * i, known4);
  for (;;) {
    if (tid == 0) sh->item = atomicAdd(work_counter, 1u);
    __syncthreads();
    const uint32_t item = sh->item;
    if (tid == 0) { sh->err = 0; sh->cnt = 0; sh->gend = 0; sh->lit_hi = 0; sh->n_jobs = 0; }
    __syncthreads();
    if (item >= a.nzb) break;
    const ZBlob z = a.zb[item];
    if (z.state) continue;
    const BlobDesc d = a.blobs[z.blob];
    const uint8_t* src = a.blobs_base + d.src_off;
    uint8_t* out = out_base + d.dst_off;
    bool bad = false;
    ZT_DECL;
    for (uint32_t j = 0; j < z.n_blocks && !bad; j++) {
      const ZBlock* b = &a.blocks[z.slot0 + j];
      const uint32_t flags = b->flags, type = flags & ZB_TYPE_MASK;
      const uint32_t blk0 = b->out_base;
      if (type == 0) { team_copy(t, out + blk0, src + b->src_off, b->len); __syncthreads(); continue; }
      if (type == 1) { team_fill(t, out + blk0, src[b->src_off], b->len); __syncthreads(); continue; }
      const uint32_t lt = (flags >> ZB_LIT_SHIFT) & 3u;
      const uint8_t* lit = lt == 0 ? src + b->lit_off : a.lits + (size_t)b->lit_base16 * 16;
      const int rle = lt == 1 ? (int)b->lit_off : -1;
      const SeqRec16* seqs = a.recs + b->seq_base;
      const uint32_t nseq = b->nseq, frame_start = b->frame_start;
      const uint32_t r0 = b->rep_in[0], r1 = b->rep_in[1], r2 = b->rep_in[2];
      uint32_t s0 = 0, gpos = blk0;  // gpos: blob-absolute output position where the next group starts
      uint32_t lit_next = 0;         // literal position where the next group starts
      SeqRec16 rn[K];                // prefetched records of sequences s0 + k * NT + tid
#pragma unroll
      for (int k = 0; k < K; k++) {
        rn[k].w0 = rn[k].w1 = rn[k].w2 = rn[k].w3 = 0;
        if (k * NT + tid < nseq) rn[k] = seqs[k * NT + tid];
      }
      while (s0 < nseq) {
        ZT(0);
        // ---- the group: the leading sequences that fit the buffer (end positions are monotonic, so "fits" is a prefix)
        uint32_t inm = 0, my_gend = 0, my_lit_hi = 0;
        SeqRec16 r[K];
#pragma unroll
        for (int k = 0; k < K; k++) {
          r[k] = rn[k];
          const bool have = s0 + k * NT + tid < nseq;
          const uint32_t endp = blk0 + rec_out(r[k]) + rec_ll(r[k]) + rec_ml(r[k]);
          if (have && endp - gpos <= GB && rec_lit(r[k]) + rec_ll(r[k]) - lit_next <= GB) {
            inm |= 1u << k;
            my_gend = endp;  // k ascending = sequence index ascending
            my_lit_hi = rec_lit(r[k]) + rec_ll(r[k]);
          }
        }
        {
          const uint32_t c = __reduce_add_sync(0xFFFFFFFFu, (uint32_t)__popc(inm));
          const uint32_t ge = __reduce_max_sync(0xFFFFFFFFu, my_gend), lh = __reduce_max_sync(0xFFFFFFFFu, my_lit_hi);
          if (lane == 0 && c) { atomicAdd(&sh->cnt, c); atomicMax(&sh->gend, ge); atomicMax(&sh->lit_hi, lh); }
          if (tid == 0) sh->first = r[0];
        }
        __syncthreads();
        const uint32_t count = sh->cnt, gend = sh->gend, lit_hi = sh->lit_hi;
        const SeqRec16 q = sh->first;
        if (count == 0) {
          // ---- a sequence longer than the buffer: alone, in global memory, by the whole team
          const uint32_t qo = blk0 + rec_out(q), qll = rec_ll(q), qlr = rec_lit(q), qml = rec_ml(q);
          if (qll) {
            if (rle >= 0) team_fill(t, out + qo, (uint32_t)rle, qll);
            else team_copy(t, out + qo, lit + qlr, qll);
          }
          const uint32_t o = sym_resolve(rec_off(q), r0, r1, r2);
          const uint32_t da = qo + qll;
          if (qml && (o == 0 || o > da - frame_start)) { bad = true; break; }
          __syncthreads();
          if (qml) team_match(t, out + da, o, qml, sh->pat, nullptr);
          __syncthreads();
          gpos = da + qml;
          lit_next = qlr + qll;
          s0 += 1;
#pragma unroll
          for (int k = 0; k < K; k++) {
            rn[k].w0 = rn[k].w1 = rn[k].w2 = rn[k].w3 = 0;
            if (s0 + k * NT + tid < nseq) rn[k] = seqs[s0 + k * NT + tid];
          }
          continue;
        }
        // prefetch the next group's records: their latency hides behind this group's rounds
#pragma unroll
        for (int k = 0; k < K; k++) {
          rn[k].w0 = rn[k].w1 = rn[k].w2 = rn[k].w3 = 0;
          if (s0 + count + k * NT + tid < nseq) rn[k] = seqs[s0 + count + k * NT + tid];
        }
        ZT(1);
        const uint32_t lit_lo = rec_lit(q);
        if (rle < 0 && lit_hi > lit_lo) team_copy(t, sh->lits, lit + lit_lo, lit_hi - lit_lo);
        // far sources into L1 while the literals arrive
#pragma unroll
        for (int k = 0; k < K; k++) {
          if ((inm >> k) & 1u) {
            const uint32_t ml = rec_ml(r[k]), off = sym_resolve(r[k].w0, r0, r1, r2);
            const uint32_t dabs = blk0 + rec_out(r[k]) + rec_ll(r[k]);
            if (ml && off && off <= dabs && dabs - off < gpos) {
              const uint8_t* sp = out + (dabs - off);
              asm volatile("prefetch.global.L1 [%0];" ::"l"(sp));
              if (ml > 1) asm volatile("prefetch.global.L1 [%0];" ::"l"(sp + (ml <= kMatchLane ? ml : kMatchLane) - 1));
            }
          }
        }
        __syncthreads();
        if (tid == 0) { sh->cnt = 0; sh->gend = 0; sh->lit_hi = 0; }  // (used again only after more barriers)
        ZT(2);
        // ---- setup: known bytes into the buffer, parents for the rest
#pragma unroll
        for (int k = 0; k < K; k++) {
          const bool mine = (inm >> k) & 1u;
          const uint32_t orl = rec_out(r[k]), ll = mine ? rec_ll(r[k]) : 0u, lr = rec_lit(r[k]);
          const uint32_t ml = mine ? rec_ml(r[k]) : 0u;
          const uint32_t oabs = blk0 + orl, dabs = oabs + ll;
          if (ll && ll <= kLitLane) {
            const uint32_t o = buf_s + (oabs - gpos), ls = lits_s + (lr - lit_lo);
            uint32_t v[kLitLane];
#pragma unroll
            for (int i = 0; i < (int)kLitLane; i++) v[i] = rle >= 0 ? (uint32_t)rle : ((uint32_t)i < ll ? lds8(ls + i) : 0u);
#pragma unroll
            for (int i = 0; i < (int)kLitLane; i++) if ((uint32_t)i < ll) sts8(o + i, v[i]);
          }
          const bool job_lit = ll > kLitLane;
          bool job_m = false;
          if (ml) {
            const uint32_t off = sym_resolve(r[k].w0, r0, r1, r2);
            if (off == 0 || off > dabs - frame_start) sh->err = 1;
            else if (ml > kMatchLane) job_m = true;
            else {
              const uint32_t drel = dabs - gpos;
              const uint32_t sabs = dabs - off;
              if (off >= ml && sabs + ml <= gpos) {  // wholly before the group: plain gather from global memory
                const uint8_t* sp = out + sabs;
                uint32_t v[kMatchLane];
#pragma unroll
                for (int i = 0; i < (int)kMatchLane; i++) if ((uint32_t)i < ml) v[i] = sp[i];
#pragma unroll
                for (int i = 0; i < (int)kMatchLane; i++) if ((uint32_t)i < ml) sts8(buf_s + drel + i, v[i]);
              } else if (off >= ml && sabs >= gpos) {  // wholly inside the group: parents only
                const uint32_t srel = sabs - gpos;
#pragma unroll
                for (int i = 0; i < (int)kMatchLane; i++) if ((uint32_t)i < ml) sts16(par_s + 2 * (drel + i), srel + i);
              } else {  // straddles the group start and / or feeds itself: byte by byte, phase = i mod off
                uint32_t ph = 0;
#pragma unroll
                for (int i = 0; i < (int)kMatchLane; i++) {
                  if ((uint32_t)i < ml) {
                    const uint32_t sp = sabs + ph;
                    if (sp < gpos) sts8(buf_s + drel + i, (uint32_t)out[sp]);
                    else sts16(par_s + 2 * (drel + i), sp - gpos);
                    ph = ph + 1 == off ? 0u : ph + 1;
                  }
                }
              }
            }
          }
          // jobs: long literal runs and long matches, one warp each
          const uint32_t nj = (job_lit ? 1u : 0u) + (job_m ? 1u : 0u);
          const uint32_t bj = __ballot_sync(0xFFFFFFFFu, nj != 0);
          if (bj) {
            uint32_t pre = nj;  // inclusive prefix sum of nj over the lanes
#pragma unroll
            for (int sft = 1; sft < 32; sft <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, pre, sft); if ((int)lane >= sft) pre += v; }
            uint32_t base = 0;
            if (lane == 31) base = atomicAdd(&sh->n_jobs, pre);
            base = __shfl_sync(0xFFFFFFFFu, base, 31);
            uint32_t slot = base + pre - nj;
            const uint32_t idx = (uint32_t)k * NT + tid;
            if (job_lit) sh->jobs[slot++] = (uint16_t)(idx | 0x8000u);
            if (job_m) sh->jobs[slot] = (uint16_t)idx;
          }
        }
        __syncthreads();
        ZT(3);
        if (sh->err) { bad = true; break; }
        {
          ZT_CNT(12, tid == 0 ? sh->n_jobs : 0);
          const uint32_t nj = sh->n_jobs;
          for (uint32_t i = warp; i < nj; i += NT / 32) {
            const uint32_t jb = sh->jobs[i], idx = jb & 0x7FFFu;
            const SeqRec16 rr = seqs[s0 + idx];  // idx = k * NT + tid of the owner = offset from s0 (broadcast load)
            const uint32_t oabs = blk0 + rec_out(rr), ll = rec_ll(rr);
            if (jb & 0x8000u) {
              const uint32_t dd = buf_s + (oabs - gpos), l2 = lits_s + (rec_lit(rr) - lit_lo);
              for (uint32_t x = lane; x < ll; x += 32) sts8(dd + x, rle >= 0 ? (uint32_t)rle : lds8(l2 + x));
            } else {
              const uint32_t dabs = oabs + ll, l = rec_ml(rr), oo = sym_resolve(rr.w0, r0, r1, r2);
              const uint32_t drel = dabs - gpos, sabs = dabs - oo;
              // byte x copies window[x mod oo]; the phase advances by 32 mod oo per step instead of a division per byte
              uint32_t ph = oo >= l ? lane : lane % oo;
              const uint32_t step = oo >= l ? 32u : 32u % oo;
              for (uint32_t x = lane; x < l; x += 32) {
                const uint32_t sp = sabs + ph;
                if (sp < gpos) sts8(buf_s + drel + x, (uint32_t)out[sp]);
                else sts16(par_s + 2 * (drel + x), sp - gpos);
                ph += step;
                if (oo < l && ph >= oo) ph -= oo;
              }
            }
          }
        }
        __syncthreads();
        if (tid == 0) { sh->n_jobs = 0; sh->lcnt[0] = sh->lcnt[1] = sh->lcnt[2] = 0; }
        __syncthreads();
        ZT(4);
        // ---- rounds.  The first one SCANS par[] (8 entries per 16-byte load) and writes the bytes that are still unknown
        // after it into a list; later rounds walk that list densely (one lane per unknown byte) and compact it as
        // they go, so a late round that resolves three bytes costs three bytes' worth of work, not a pass over the group.
        // The two lists alias the literal staging area (dead once the jobs are done); a group with more unknown bytes than
        // a list holds is scanned again.
        const uint32_t glen = gend - gpos;
        constexpr uint32_t kListCap = LC;
        const uint32_t lists_s = Sh::kOwnLists ? (uint32_t)__cvta_generic_to_shared(sh->lists) : lits_s;
        uint32_t nlist = ~0u;  // ~0u: scan round; else entries of list[round & 1]
        for (uint32_t round = 0;; round++) {
          const uint32_t cur = kFresh | ((round & 1u) << 14);
          const uint32_t cw = (round + 1u) % 3u;  // counter appended to this round (cleared a round ago)
          const uint32_t lst_r = lists_s + (round & 1u) * 2u * kListCap, lst_w = lists_s + ((round & 1u) ^ 1u) * 2u * kListCap;
          if (tid == 0) sh->lcnt[(round + 2u) % 3u] = 0;
          if (nlist == ~0u) {
            for (uint32_t b0 = warp * 256u; b0 < glen; b0 += NT * 8) {
              const uint32_t base = b0 + lane * 8u;
              uint32_t km = 0;  // entries of this chunk that stay unknown
              if (base < glen) {
                const uint4 pv = lds128(par_s + 2 * base);
                // bit 15 of an entry = its byte is in the buffer (kKnown, or kFresh of this or an earlier round)
                if ((pv.x & pv.y & pv.z & pv.w & 0x80008000u) != 0x80008000u) {
                  const uint32_t w4[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
                  for (int e = 0; e < 8; e++) {
                    const uint32_t me = (w4[e >> 1] >> (16 * (e & 1))) & 0xFFFFu;
                    if (me & 0x8000u) continue;
                    const uint32_t i = base + e;
                    const uint32_t pp = lds16(par_s + 2 * me);
                    if (pp == kKnown || ((pp & 0x8000u) && pp != cur)) {  // the parent's byte was stored before this round's barrier
                      sts8(buf_s + i, lds8(buf_s + me));
                      sts16(par_s + 2 * i, cur);
                    } else {
                      // a parent resolved this very round (or carrying a stale marker of this parity): look again next
                      // round; otherwise adopt the parent's parent
                      if (!(pp & 0x8000u)) sts16(par_s + 2 * i, pp);
                      km |= 1u << e;
                    }
                  }
                }
              }
              const uint32_t c = (uint32_t)__popc(km);
              if (__any_sync(0xFFFFFFFFu, c != 0)) {
                uint32_t pre = c;  // inclusive prefix sum over the lanes
#pragma unroll
                for (int sft = 1; sft < 32; sft <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, pre, sft); if ((int)lane >= sft) pre += v; }
                uint32_t slot = 0;
                if (lane == 31) slot = atomicAdd(&sh->lcnt[cw], pre);
                slot = __shfl_sync(0xFFFFFFFFu, slot, 31) + pre - c;
                while (km) {
                  const uint32_t e = (uint32_t)__ffs(km) - 1u;
                  km &= km - 1u;
                  if (slot < kListCap) sts16(lst_w + 2 * slot, base + e);
                  slot++;
                }
              }
            }
          } else {
            for (uint32_t j0 = warp * 32u; j0 < nlist; j0 += NT) {
              const uint32_t j = j0 + lane;
              bool keep = false;
              uint32_t i = 0;
              if (j < nlist) {
                i = lds16(lst_r + 2 * j);
                const uint32_t me = lds16(par_s + 2 * i);
                const uint32_t pp = lds16(par_s + 2 * me);
                if (pp == kKnown || ((pp & 0x8000u) && pp != cur)) {
                  sts8(buf_s + i, lds8(buf_s + me));
                  sts16(par_s + 2 * i, cur);
                } else {
                  if (!(pp & 0x8000u)) sts16(par_s + 2 * i, pp);
                  keep = true;
                }
              }
              const uint32_t kb = __ballot_sync(0xFFFFFFFFu, keep);
              if (kb) {
                uint32_t b1 = 0;
                if (lane == 0) b1 = atomicAdd(&sh->lcnt[cw], (uint32_t)__popc(kb));
                b1 = __shfl_sync(0xFFFFFFFFu, b1, 0);
                if (keep) sts16(lst_w + 2 * (b1 + __popc(kb & ((1u << lane) - 1u))), i);
              }
            }
          }
          if (round > 96) { if (tid == 0) sh->err = 2; break; }  // cannot happen (chains halve every round): never hang
          __syncthreads();
          const uint32_t left = sh->lcnt[cw];
          ZT_CNT(8, tid == 0 ? 1 : 0);
          ZT_CNT(10, tid == 0 ? left : 0);
          ZT_CNT(11, tid == 0 && nlist == ~0u ? 1 : 0);
          if (left == 0) break;
          nlist = left <= kListCap ? left : ~0u;
        }
        __syncthreads();
        ZT(5);
        if (sh->err) { bad = true; break; }
        // ---- flush, and every parent back to "known" for the next group
        team_copy(t, out + gpos, sh->buf, glen);
        for (uint32_t i = tid * 8; i < glen + 8; i += NT * 8) sts128(par_s + 2 * i, known4);
        __syncthreads();
        ZT(6);
        ZT_CNT(9, tid == 0 ? 1 : 0);
        gpos = gend;
        lit_next = lit_hi;
        s0 += count;
      }
      if (bad) break;
      const uint32_t rest = b->lit_regen - b->lit_used;
      if (rest) {
        if (rle >= 0) team_fill(t, out + blk0 + b->matched, (uint32_t)rle, rest);
        else team_copy(t, out + blk0 + b->matched, lit + b->lit_used, rest);
      }
      __syncthreads();
    }
    if (bad) {  // leave the shared state clean for the next blob
      __syncthreads();
      for (uint32_t i = tid * 8; i < GB + 8; i += NT * 8) sts128(par_s + 2 * i, known4);
    }
    if (tid == 0) {
      if (bad) a.zb[item].state = 1;
      else produced[z.blob] = (uint32_t)d.dst_cap;
      ZT(7);
      ZT_FLUSH(0, 16);
    }
  }
}

}  // namespace zp
}  // namespace zn
