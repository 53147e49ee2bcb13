// TEST INFRASTRUCTURE ONLY — the packed layout of device-resident compress plans, compiled for the host: the per-block
// results of every effort emulated with a "warp" of one lane (as host_compress.cpp / host_compress_long.cpp do), then the
// blob size the device computes from them (cz::zstd_frame_size / cz::lz4_frame_size, znippy_b200/csrc/compress.cuh) and
// the ZNB1 header the device writes (cz::znb1_header).
#include <algorithm>
#include <vector>

#include "../../znippy_b200/csrc/compress.cuh"

using namespace zn;

// codec 2: LZ4; 1 / 11 / 12: the zstd window efforts of levels <= 2, 3..9, 10..19; 20: the long effort (levels >= 20)
extern "C" long zn_hostemu_frame_size(int codec, const uint8_t* src, uint64_t n) {
  cz::Warp w{0, 1};
  if (codec == 2) {
    std::vector<uint16_t> tab(1u << cz::kLz4HashLog);
    std::vector<uint8_t> tmp(cz::kLz4Slot);
    std::vector<uint32_t> csize;
    for (uint64_t o = 0; o < n; o += cz::kLz4Block)
      csize.push_back(cz::lz4_compress_block(w, src + o, (uint32_t)std::min<uint64_t>(n - o, cz::kLz4Block), tmp.data(), tab.data()));
    return (long)cz::lz4_frame_size(n, csize.data());
  }
  std::vector<uint32_t> meta(2 * ((n + cz::kZstdCBlock - 1) / cz::kZstdCBlock) + 2);
  std::vector<uint8_t> stage(cz::kZstdSlot + 64);
  std::vector<uint64_t> seqs(cz::kZstdMaxSeq);
  if (codec == 20) {
    std::vector<uint64_t> keys;
    std::vector<uint32_t> rank, scratch(cz::kPayloadScratch / 4), bl(cz::kLongBatch), bo(cz::kLongBatch);
    for (uint64_t ps = 0; ps < n; ps += cz::kLongPiece) {
      const uint32_t lo = (uint32_t)(ps - std::min<uint64_t>(ps, cz::kLongReach));
      const uint32_t hi = (uint32_t)std::min<uint64_t>(ps + cz::kLongPiece, n);
      keys.resize(hi - lo);
      rank.resize(hi - lo);
      for (uint32_t q = 0; q < hi - lo; q++) keys[q] = cz::long_key(src, lo + q, hi, q);
      std::sort(keys.begin(), keys.end());
      for (uint32_t i = 0; i < hi - lo; i++) rank[(uint32_t)keys[i] & (cz::kLongRound - 1u)] = i;
      const cz::LongIndex ix{keys.data(), rank.data(), 0, lo};
      for (uint32_t o = (uint32_t)ps; o < hi; o += cz::kZstdCBlock) {
        uint32_t poff = 0;
        meta[2 * (o / cz::kZstdCBlock) + 1] = cz::zstd_long_block(w, src, ix, o, std::min<uint32_t>(hi - o, cz::kZstdCBlock), stage.data(),
                                                                  seqs.data(), bl.data(), bo.data(), scratch.data(), &poff);
      }
    }
  } else {
    std::vector<uint16_t> tab(1u << 14);
    std::vector<cz::V16> win(cz::WinHigh::kSmem / 16 + 2);
    for (uint64_t o = 0; o < n; o += cz::kZstdCBlock) {
      uint32_t poff = 0;
      meta[2 * (o / cz::kZstdCBlock) + 1] =
          (codec == 12 ? cz::zstd_compress_block<cz::WinHigh> : codec == 11 ? cz::zstd_compress_block<cz::WinMid> : cz::zstd_compress_block<cz::WinFast>)(
              w, src, (uint32_t)o, (uint32_t)std::min<uint64_t>(n - o, cz::kZstdCBlock), stage.data(), seqs.data(),
              reinterpret_cast<uint8_t*>(win.data()), tab.data(), &poff);
    }
  }
  return (long)cz::zstd_frame_size(n, meta.data());
}

// the ZNB1 header the device writes for a payload of `codec` decoding to n bytes; *len_out = cz::znb1_header_len(n)
extern "C" uint32_t zn_hostemu_znb1_header(uint32_t codec, uint64_t n, uint8_t* dst, uint32_t* len_out) {
  *len_out = cz::znb1_header_len(n);
  return cz::znb1_header(dst, codec, n);
}
