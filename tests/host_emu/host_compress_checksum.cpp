// TEST INFRASTRUCTURE ONLY — frames with content checksums (ZN_CODEC_CHECKSUM) compiled for the host: the frame
// assembly of zstd_assemble / lz4_assemble (compress_kernels.cuh) restated in plain C++ around the blocks of
// tests/host_emu/host_compress.cpp's compressor, the checksum of xxh64_1 / xxh32_1 (xxh_verify.cuh, the scalar forms of
// the staged hash), and the sizes the packed layout computes (cz::zstd_frame_size / cz::lz4_frame_size).  Also the
// read-side row check (xxh_row_bad) over a host buffer.
#include <cstring>
#include <vector>

#include "../../znippy_b200/csrc/compress.cuh"
#include "../../znippy_b200/csrc/xxh_verify.cuh"

using namespace zn;

// codec 2 = LZ4, 1 / 11 / 12 = the zstd window efforts.  Writes the frame at dst, returns its length; *size_out = the
// packed layout's size from the block results alone.
extern "C" long zn_hostemu_compress_checksum(int codec, const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t* size_out) {
  cz::Warp w{0, 1};
  uint64_t op = 0;
  if (codec == 2) {
    std::vector<uint16_t> tab(1u << cz::kLz4HashLog);
    std::vector<uint8_t> tmp(cz::kLz4Slot);
    std::vector<uint32_t> csize(n / cz::kLz4Block + 1);
    op = cz::lz4_frame_header(dst, n, true);
    for (uint64_t o = 0, j = 0; o < n; o += cz::kLz4Block, j++) {
      const uint32_t bn = (uint32_t)(n - o < cz::kLz4Block ? n - o : cz::kLz4Block);
      const uint32_t c = cz::lz4_compress_block(w, src + o, bn, tmp.data(), tab.data());
      csize[j] = c;
      const bool raw = c >= bn;
      const uint32_t sz = raw ? bn : c, word = sz | (raw ? 0x80000000u : 0u);
      memcpy(dst + op, &word, 4);
      memcpy(dst + op + 4, raw ? src + o : tmp.data(), sz);
      op += 4 + sz;
    }
    memset(dst + op, 0, 4);
    cz::put_le32(dst + op + 4, xxh32_1(src, n));
    *size_out = cz::lz4_frame_size(n, csize.data(), true);
    return (long)(op + 8);
  }
  if (n == 0) {
    *size_out = cz::zstd_frame_size(0, nullptr, true);
    return (long)cz::zstd_empty_frame(dst, true);
  }
  std::vector<uint16_t> tab(1u << 14);
  std::vector<cz::V16> win(cz::WinHigh::kSmem / 16 + 2);
  std::vector<uint8_t> stage(cz::kZstdSlot + 64);
  std::vector<uint64_t> seqs(cz::kZstdMaxSeq);
  std::vector<uint32_t> meta(2 * (n / cz::kZstdCBlock + 1));
  op = cz::zstd_frame_header(dst, n, true);
  for (uint64_t o = 0, j = 0; o < n; o += cz::kZstdCBlock, j++) {
    const uint32_t bn = (uint32_t)(n - o < cz::kZstdCBlock ? n - o : cz::kZstdCBlock);
    uint32_t poff = 0;
    const uint32_t c = (codec == 12 ? cz::zstd_compress_block<cz::WinHigh> : codec == 11 ? cz::zstd_compress_block<cz::WinMid> : cz::zstd_compress_block<cz::WinFast>)(
        w, src, (uint32_t)o, bn, stage.data(), seqs.data(), reinterpret_cast<uint8_t*>(win.data()), tab.data(), &poff);
    meta[2 * j] = poff;
    meta[2 * j + 1] = c;
    cz::zstd_block_header(dst + op, o + bn == n, c ? 2 : 0, c ? c : bn);
    memcpy(dst + op + 3, c ? stage.data() + poff : src + o, c ? c : bn);
    op += 3 + (c ? c : bn);
  }
  cz::put_le32(dst + op, (uint32_t)xxh64_1(src, n));
  *size_out = cz::zstd_frame_size(n, meta.data(), true);
  return (long)(op + 4);
}

// xxh_row_bad over one decoded row: `blob` as stored, `content` what it decoded to.  1 = a checksum disagrees.
extern "C" int zn_hostemu_row_bad(const uint8_t* blob, uint64_t blob_len, const uint8_t* content, uint64_t content_len) {
  BlobDesc d{};
  d.src_len = blob_len;
  d.dst_cap = content_len;
  d.flags = F_COMPRESSED;
  return xxh_row_bad(d, blob, content) ? 1 : 0;
}

// The two hashes alone: bits 64 = XXH64, 32 = XXH32 (seed 0), scalar forms.
extern "C" uint64_t zn_hostemu_xxh(int bits, const uint8_t* p, uint64_t n) { return bits == 64 ? xxh64_1(p, n) : xxh32_1(p, n); }
