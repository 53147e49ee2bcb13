// The envelope layer (SURVEY.md §8c, row f4): everything between "a blob as the index row describes it" and "a codec
// payload a kernel can decode".  The reference hands every blob to OpenZL (znippy-common/src/codec.rs:67-78:
// zl_get_decompressed_size, then zl_decompress), whose frame wraps a zstd / LZ4 payload in its own header.  That
// header's layout is unpinned in this environment (no OpenZL sources, no archive written by the reference), so no
// kernel knows about envelopes at all: the host asks zn_envelope_parse for {codec, payload range, decoded size} and
// hands the payload range to the batch calls.  Three things plug in here:
//   * bare frames (what the batch calls always accepted): Zstandard and LZ4 frame magic;
//   * ZNB1, this library's own envelope ("ZNB1", codec id, LEB128 decoded size, payload) — the format it can emit, and
//     the carrier of the on-device store-if-incompressible decision (codec id RAW);
//   * one registered foreign parser (zn_envelope_register): where a host that links OpenZL plugs its frame-header
//     reader in, without touching a kernel.
// Host code only; no CUDA.
#include <atomic>
#include <cstring>

#include "../../include/znippy_cuda.h"

namespace {
std::atomic<zn_envelope_parser> g_foreign{nullptr};
inline uint32_t le32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

// Decoded size of a zstd blob that ends in a seek table of the Zstandard seekable format (ZN_CODEC_SEEKABLE writes
// them): the sum of its entries' decompressed sizes.  False unless the footer magic, the descriptor's reserved bits,
// the skippable frame's magic and size, and the entries' compressed sizes all agree with a blob of len bytes.
bool seekable_content_size(const uint8_t* blob, size_t len, uint64_t* out) {
  if (len < 17 || le32(blob + len - 4) != 0x8F92EAB1u) return false;
  const uint64_t n = le32(blob + len - 9);
  const uint8_t desc = blob[len - 5];
  if (desc & 0x7C) return false;
  const uint64_t esz = desc & 0x80 ? 12 : 8, tl = 8 + esz * n + 9;
  if (tl > len) return false;
  const uint8_t* t = blob + len - tl;
  if (le32(t) != 0x184D2A5Eu || le32(t + 4) != esz * n + 9) return false;
  uint64_t c = 0, d = 0;
  for (uint64_t k = 0; k < n; k++) {
    c += le32(t + 8 + esz * k);
    d += le32(t + 8 + esz * k + 4);
  }
  if (c + tl != len) return false;
  *out = d;
  return true;
}
}  // namespace

extern "C" void zn_envelope_register(zn_envelope_parser fn) { g_foreign.store(fn); }

// zn_envelope_parse over the first `head` bytes of a blob of `len` bytes (the archive reader preads only a blob's head):
// ZNB1 headers and frame headers are read from the head; a bare zstd blob is sized from its seek table, and a foreign
// parser runs, only when the whole blob is given (head == len).
extern "C" int zn_envelope_parse_head(const uint8_t* blob, size_t head, size_t len, zn_envelope* e) {
  if (!e || (head && !blob) || head > len) return ZN_E_ARG;
  memset(e, 0, sizeof *e);
  e->out_len = ~0ull;
  e->payload_len = len;
  if (head >= 4) {
    const uint32_t magic = le32(blob);
    if (magic == 0xFD2FB528u || (magic & 0xFFFFFFF0u) == 0x184D2A50u) {  // Zstandard frame (or a skippable frame before one)
      e->kind = ZN_ENV_BARE;
      e->codec = ZN_PAYLOAD_ZSTD;
      uint64_t sz = 0;
      if (zn_frame_content_size(blob, head, &sz) == ZN_OK) e->out_len = sz;
      // concatenated frames with a seek table: the first frame holds only 128 KiB of the content
      if (magic == 0xFD2FB528u && head == len && seekable_content_size(blob, len, &sz)) e->out_len = sz;
      return ZN_OK;
    }
    if (magic == 0x184D2204u) {
      e->kind = ZN_ENV_BARE;
      e->codec = ZN_PAYLOAD_LZ4_FRAME;
      uint64_t sz = 0;
      if (zn_frame_content_size(blob, head, &sz) == ZN_OK) e->out_len = sz;
      return ZN_OK;
    }
    if (memcmp(blob, "ZNB1", 4) == 0) {
      e->kind = ZN_ENV_ZNB1;
      if (head < 6) return 1;
      const uint32_t codec = blob[4];
      if (codec > ZN_PAYLOAD_LZ4_BLOCK) return 1;
      uint64_t v = 0;
      size_t p = 5;
      for (uint32_t shift = 0;; shift += 7) {  // LEB128, at most 5 bytes: decoded sizes stay below 4 GiB
        if (p >= head || shift > 28) return 1;
        const uint8_t b = blob[p++];
        v |= (uint64_t)(b & 0x7F) << shift;
        if (!(b & 0x80)) break;
      }
      if (v >= (1ull << 32)) return 1;
      e->codec = codec;
      e->out_len = v;
      e->payload_off = p;
      e->payload_len = len - p;
      if (codec == ZN_PAYLOAD_RAW && e->payload_len != v) return 1;
      return ZN_OK;
    }
  }
  zn_envelope_parser f = g_foreign.load();
  if (f && head == len) {
    const int rc = f(blob, len, e);
    if (rc == ZN_OK) {
      if (e->payload_off > len || e->payload_len > len - e->payload_off || e->codec > ZN_PAYLOAD_LZ4_BLOCK) return 1;
      // a magicless zstd payload is decoded as "magic + payload": the four bytes in front of it are overwritten on
      // the device copy, so they must belong to the blob
      if (e->codec == ZN_PAYLOAD_ZSTD_MAGICLESS && e->payload_off < 4) return 1;
      e->kind = ZN_ENV_FOREIGN;
    }
    return rc;
  }
  e->kind = ZN_ENV_UNKNOWN;
  return 1;
}

extern "C" int zn_envelope_parse(const uint8_t* blob, size_t len, zn_envelope* e) { return zn_envelope_parse_head(blob, len, len, e); }

extern "C" size_t zn_envelope_znb1_header(uint32_t codec, uint64_t out_len, uint8_t* hdr, size_t cap) {
  if (!hdr || cap < ZN_ENVELOPE_ZNB1_MAX_HEADER || codec > ZN_PAYLOAD_LZ4_BLOCK || out_len >= (1ull << 32)) return 0;
  memcpy(hdr, "ZNB1", 4);
  hdr[4] = (uint8_t)codec;
  size_t p = 5;
  do {
    uint8_t b = out_len & 0x7F;
    out_len >>= 7;
    if (out_len) b |= 0x80;
    hdr[p++] = b;
  } while (out_len);
  return p;
}
