// TEST INFRASTRUCTURE ONLY — the long effort of the zstd compressor (levels >= 20, znippy_b200/csrc/compress.cuh)
// compiled for the host with a "warp" of one lane.  The candidate index is built with std::sort over the same keys
// the device sorts with CUB, one unit at a time (a unit's candidates never leave it, so its place in a round does not
// matter), and the frame assembly of compress_kernels.cuh is restated in plain C++: the bytes equal the GPU's.
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../znippy_b200/csrc/compress.cuh"

using namespace zn;

extern "C" long zn_hostemu_compress_long(const uint8_t* src, uint64_t n, uint8_t* dst) {
  if (n == 0) {
    const uint8_t e[9] = {0x28, 0xB5, 0x2F, 0xFD, 0x20, 0x00, 0x01, 0x00, 0x00};
    memcpy(dst, e, 9);
    return 9;
  }
  cz::Warp w{0, 1};
  std::vector<uint8_t> stage(cz::kZstdSlot + 64);
  std::vector<uint64_t> seqs(cz::kZstdMaxSeq), keys;
  std::vector<uint32_t> rank, scratch(cz::kPayloadScratch / 4), bl(cz::kLongBatch), bo(cz::kLongBatch);
  uint64_t op = cz::zstd_frame_header(dst, n);
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
      const uint32_t bn = std::min<uint32_t>(hi - o, cz::kZstdCBlock);
      uint32_t poff = 0;
      const uint32_t c = cz::zstd_long_block(w, src, ix, o, bn, stage.data(), seqs.data(), bl.data(), bo.data(), scratch.data(), &poff);
      const uint32_t last = o + bn == n;
      if (c == 0) {
        cz::zstd_block_header(dst + op, last, 0, bn);
        memcpy(dst + op + 3, src + o, bn);
        op += 3 + bn;
      } else {
        cz::zstd_block_header(dst + op, last, 2, c);
        memcpy(dst + op + 3, stage.data() + poff, c);
        op += 3 + c;
      }
    }
  }
  return (long)op;
}
