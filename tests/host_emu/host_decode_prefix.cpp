// TEST INFRASTRUCTURE ONLY — the decoders with a stop point (range reads: zs::StopAt), compiled for the host with a team
// of one, exactly as host_decode.cpp compiles them without one.  Never linked into libznippy_cuda.so.
#include <cstdlib>
#include <cstring>

#include "../../znippy_b200/csrc/lz4_decode.cuh"

// What k_decode<.., true> does with one blob: decode_blob with zs::StopAt{stop}; a raw LZ4 block (lz4_block != 0) is one
// block and decodes whole; stop 0xFFFFFFFF decodes in full.  The output buffer is the caller's (canary bytes past `produced` must survive).
extern "C" int zn_hostemu_decode_prefix(const uint8_t* src, uint32_t src_len, int lz4_block, uint32_t stop, uint8_t* out,
                                        uint32_t cap, uint32_t* produced) {
  zn::DecShared* sh = (zn::DecShared*)calloc(1, sizeof(zn::DecShared));
  uint8_t* lit = (uint8_t*)malloc(zn::kZstdBlockMax + 64);
  zn::Team t{0, 1};
  uint32_t predef = 0;
  zn::zs::init_luts(t, sh);
  // the device code may read the aligned 32-bit word around any valid byte: give the input 4-byte alignment + slack
  uint8_t* in = (uint8_t*)calloc(1, (size_t)src_len + 16);
  memcpy(in + 4, src, src_len);
  uint32_t st;
  if (lz4_block) {
    st = zn::decode_lz4_block(t, sh, in + 4, src_len, out, cap, produced);
  } else if (stop == 0xFFFFFFFFu) {  // no stop: the full decode of k_decode, for comparison
    st = zn::decode_blob(t, sh, in + 4, src_len, out, cap, lit, predef, produced);
    if (st == zn::S_OK && *produced != cap) st = zn::S_SIZE_MISMATCH;
  } else {
    zn::zs::StopAt h;
    h.stop = stop;
    st = zn::decode_blob(t, sh, in + 4, src_len, out, cap, lit, predef, produced, h);
    if (st == zn::S_OK && *produced < stop) st = zn::S_SIZE_MISMATCH;
  }
  free(in);
  free(lit);
  free(sh);
  return (int)st;
}
