// TEST INFRASTRUCTURE ONLY — the seekable layout (ZN_CODEC_SEEKABLE) compiled for the host: every block compressed by
// the window efforts of znippy_b200/csrc/compress.cuh with a "warp" of one lane and no history (as k_zstd_blocks<WN, true>
// calls it), the checksums of xxh64_1 (xxh_verify.cuh), the frame-per-block assembly of zstd_seekable_assemble
// (compress_kernels.cuh) restated in plain C++, and the seek table and size the device computes (cz::zstd_seek_table,
// cz::zstd_seekable_size).
#include <cstring>
#include <vector>

#include "../../znippy_b200/csrc/compress.cuh"
#include "../../znippy_b200/csrc/xxh_verify.cuh"

using namespace zn;

// codec 1 / 11 / 12: the window efforts of levels <= 2, 3..9, 10..19.  Writes the blob at dst, returns its length;
// *size_out = cz::zstd_seekable_size from the block results alone.
extern "C" long zn_hostemu_compress_seekable(int codec, const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t* size_out) {
  cz::Warp w{0, 1};
  const uint64_t nb = (n + cz::kZstdCBlock - 1) / cz::kZstdCBlock;
  std::vector<uint32_t> meta(2 * nb + 2), xxh(nb + 1);
  std::vector<uint16_t> tab(1u << 14);
  std::vector<cz::V16> win(cz::WinHigh::kSmem / 16 + 2);
  std::vector<uint8_t> stage(cz::kZstdSlot + 64);
  std::vector<uint64_t> seqs(cz::kZstdMaxSeq);
  uint64_t op = n ? 0 : cz::zstd_empty_frame(dst);
  for (uint64_t o = 0, j = 0; o < n; o += cz::kZstdCBlock, j++) {
    const uint32_t bn = (uint32_t)(n - o < cz::kZstdCBlock ? n - o : cz::kZstdCBlock);
    uint32_t poff = 0;
    const uint32_t c = (codec == 12 ? cz::zstd_compress_block<cz::WinHigh> : codec == 11 ? cz::zstd_compress_block<cz::WinMid> : cz::zstd_compress_block<cz::WinFast>)(
        w, src + o, 0, bn, stage.data(), seqs.data(), reinterpret_cast<uint8_t*>(win.data()), tab.data(), &poff);
    meta[2 * j] = poff;
    meta[2 * j + 1] = c;
    xxh[j] = (uint32_t)xxh64_1(src + o, bn);
    cz::zstd_frame_header(dst + op, bn);
    cz::zstd_block_header(dst + op + 13, 1, c ? 2 : 0, c ? c : bn);
    memcpy(dst + op + 16, c ? stage.data() + poff : src + o, c ? c : bn);
    op += 16 + (c ? c : bn);
  }
  op += cz::zstd_seek_table(dst + op, n, meta.data(), xxh.data());
  *size_out = cz::zstd_seekable_size(n, meta.data());
  return (long)op;
}
