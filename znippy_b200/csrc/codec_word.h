// The codec word of the compress entry points (zn_compress_batch, zn_plan_compress, zn_archive_writer_create,
// zn_archive_compress_dir): a base codec with flag bits OR-ed in.  Every entry point splits and validates it here, so
// which combinations are refused is decided in one place.
#pragma once
#include "../../include/znippy_cuda.h"

namespace zn {

struct CodecWord {
  int base = 0;  // ZN_CODEC_ZSTD or ZN_CODEC_LZ4
  bool envelope = false, seekable = false, checksum = false;
};

// The word's parts, without validation (zn_compress_bound sizes any word it is given).
inline CodecWord codec_parts(int codec) {
  CodecWord w;
  w.envelope = (codec & ZN_CODEC_ENVELOPE) != 0;
  w.seekable = (codec & ZN_CODEC_SEEKABLE) != 0;
  w.checksum = (codec & ZN_CODEC_CHECKSUM) != 0;
  w.base = codec & ~(ZN_CODEC_ENVELOPE | ZN_CODEC_SEEKABLE | ZN_CODEC_CHECKSUM);
  return w;
}

// Splits `codec` into *out and returns nullptr, or returns why the word is refused.  `envelope_ok`: the entry point
// writes ZNB1 envelopes (compress plans and the archive writer; zn_compress_batch emits bare frames).
inline const char* codec_split(int codec, int level, bool envelope_ok, CodecWord* out) {
  const CodecWord w = codec_parts(codec);
  if (w.base != ZN_CODEC_ZSTD && w.base != ZN_CODEC_LZ4) return "unknown codec";
  if (w.envelope && !envelope_ok) return "ZN_CODEC_ENVELOPE is not accepted here";
  // the long effort reaches up to 8 MiB back, which a one-block frame rules out
  if (w.seekable && (w.base != ZN_CODEC_ZSTD || level >= 20)) return "seekable frames need the zstd codec at a level <= 19";
  // the seek table already carries one XXH64 per frame
  if (w.seekable && w.checksum) return "ZN_CODEC_CHECKSUM cannot be combined with ZN_CODEC_SEEKABLE";
  *out = w;
  return nullptr;
}

}  // namespace zn
