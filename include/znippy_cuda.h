/*
 * znippy_cuda.h — C ABI of libznippy_cuda.so, the B200 (sm_100a) back-end for znippy's per-chunk codec +
 * integrity hot path.  Plain pointers and sizes only; no CUDA/torch types in any signature (streams are
 * passed as opaque `void*` = cudaStream_t).
 *
 * What each entry point replaces in the reference (paths relative to the znippy repository root):
 *
 *   zn_decode_verify_batch / zn_plan_*      the body of the read worker loop, znippy-common/src/decompress.rs:148-184
 *                                           (codec::decompress_into, codec.rs:67-78, then blake3::hash + 32-byte
 *                                           compare, decompress.rs:172-184), and the per-chunk decode of
 *                                           ZnippyArchive::extract_file, znippy-common/src/archive.rs:154-165
 *   zn_hash_batch                           blake3::hash(&[u8]) at decompress.rs:172, stream_packer.rs:219,
 *                                           slot_packer.rs:553 (store-as-is rows: decompress.rs:164-166)
 *   zn_compress_batch                       CompressCtx::compress_into (codec.rs:43-55) + blake3::hash of the source
 *                                           slice, i.e. the barrel body stream_packer.rs:217-232 and the worker body
 *                                           slot_packer.rs:551-572
 *   zn_compress_bound                       openzl zl_compress_bound as used at codec.rs:32,45
 *   zn_frame_content_size                   zl_get_decompressed_size as used at codec.rs:69
 *   zn_ctx_create / zn_ctx_destroy          CompressCtx::new (codec.rs:16-28) — one long-lived context per worker,
 *                                           Send but not Sync (codec.rs:13): a zn_ctx is likewise single-threaded
 *   zn_ctx_pinned                           a Magazine slot (znippy-common/src/slotpool.rs:93-130) as a pinned
 *                                           host staging buffer
 *
 * Error model (SURVEY.md §8b): the int return value reports whole-call failures (bad arguments, CUDA errors);
 * data errors are reported per blob in status[] so that one corrupt blob never fails the batch — the
 * reference's read loop logs and `continue`s on a codec error (decompress.rs:159-162) and counts a digest
 * mismatch (decompress.rs:175-184).  Nothing aborts or throws across this boundary.  There is no CPU fallback:
 * every entry point that computes runs CUDA kernels, and fails with ZN_E_CUDA when no device is usable.
 *
 * Blob wire formats accepted by the decoder (self-identifying by magic): Zstandard frames (RFC 8878, magic
 * 28 B5 2F FD; several concatenated frames and skippable frames allowed; no dictionaries) and LZ4 frames (magic
 * 04 22 4D 18, independent or linked blocks).  A Zstandard frame's optional content checksum (XXH64) IS verified, as
 * libzstd does: a mismatch is ZN_S_DECODE_ERROR.  The optional XXH32 content / block checksums of LZ4 frames are
 * skipped, not verified: integrity on this path is the blake3 digest.  Envelopes around those payloads go through
 * the envelope layer below (zn_envelope_parse): this library's own ZNB1 is built in; the OpenZL envelope the reference
 * writes is NOT (its layout is unpinned in this environment, see DESIGN.md) — until a parser for it is registered with
 * zn_envelope_register such blobs get ZN_S_UNSUPPORTED.
 */
#ifndef ZNIPPY_CUDA_H
#define ZNIPPY_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZN_ABI_VERSION 1

/* ---- whole-call return codes ---- */
enum {
  ZN_OK = 0,
  ZN_E_ARG = -1,     /* null pointer / inconsistent sizes */
  ZN_E_CUDA = -2,    /* CUDA runtime error; see zn_last_error() */
  ZN_E_NOMEM = -3,   /* device or pinned allocation failed */
  ZN_E_STATE = -4    /* call out of order (e.g. results before run) */
};

/* ---- per-blob status[] values ---- */
enum {
  ZN_S_OK = 0,
  ZN_S_DECODE_ERROR = 1,     /* corrupt / truncated compressed data (reference: codec Err -> row skipped) */
  ZN_S_DIGEST_MISMATCH = 2,  /* decoded fine, blake3 != expected (reference: corrupt_bytes / corrupt_rows) */
  ZN_S_DST_TOO_SMALL = 3,    /* decoded size exceeds the capacity given in out_len[] */
  ZN_S_UNSUPPORTED = 4,      /* unknown magic, dictionary id, reserved bits, blob >= 4 GiB */
  ZN_S_SIZE_MISMATCH = 5     /* decoded size != out_len[] (index uncompressed_size) or != frame content size */
};

/* ---- codecs for zn_compress_batch ---- */
enum {
  ZN_CODEC_ZSTD = 1, /* one Zstandard frame per slice */
  ZN_CODEC_LZ4 = 2,  /* one LZ4 frame (independent 64 KiB blocks, content size in header) per slice */
  /* archive writer and compress plans, OR-ed into `codec`: every compressed row's blob is a ZNB1 envelope (see the
   * envelope layer below) around the frame, or around the raw bytes when the frame did not shrink them
   * (store-if-incompressible); the index metadata gets znippy_envelope = "ZNB1" and readers resolve such rows through
   * zn_envelope_parse.  A compress plan makes the same decision on the device and emits the same blob bytes. */
  ZN_CODEC_ENVELOPE = 0x100,
  /* OR-ed into ZN_CODEC_ZSTD at levels <= 19 (zn_compress_batch, compress plans, archive writer): the Zstandard seekable
   * format.  Every 128 KiB block of a slice is an independent frame (13-byte header, one last block, no history from
   * the block before), followed by a skippable frame holding the seek table {compressed size, decompressed size, low 32
   * bits of XXH64(content)} per frame and the footer {N, 0x80, 0x8F92EAB1}.  Every zstd decoder reads such a blob as the
   * concatenated frames and skips the table; archive range reads use the table to decode only the frames a range
   * touches.  An empty slice is the 9-byte empty frame and a one-entry table.  The archive writer records
   * znippy_seekable = "zstd" in the index metadata.  LZ4 and levels >= 20 (whose matches reach up to 8 MiB back) are
   * refused. */
  ZN_CODEC_SEEKABLE = 0x400, /* 0x200 | ZN_CODEC_ZSTD stays an unknown codec */
  /* OR-ed into ZN_CODEC_ZSTD (levels 1-22) or ZN_CODEC_LZ4, optionally with ZN_CODEC_ENVELOPE (zn_compress_batch,
   * compress plans, archive writer): every frame carries a content checksum, as the zstd and lz4 command-line tools
   * write by default.  Zstandard: frame-header descriptor bit 2 set (0xE4) and the low 32 bits of XXH64(slice, 0) after
   * the last block; the empty slice is the 13-byte frame 28 B5 2F FD 24 00 01 00 00 99 E9 D8 51.  LZ4: FLG bit 2 set
   * (header checksum byte recomputed) and XXH32(slice, 0) after the EndMark; no block checksums.  A frame is 4 bytes
   * longer than without the flag, and so is zn_compress_bound.  Refused with ZN_CODEC_SEEKABLE (ZN_E_ARG): the seek
   * table already carries one XXH64 per frame. */
  ZN_CODEC_CHECKSUM = 0x800
};

typedef struct zn_ctx zn_ctx;   /* one CUDA device + streams + scratch + pinned staging; not thread-safe */
typedef struct zn_plan zn_plan; /* device-resident descriptors of one decode/verify, hash or compress batch, reusable */

/* ---- library / context ---- */
int zn_abi_version(void);
int zn_device_count(void);
const char* zn_strerror(int code);            /* whole-call codes */
const char* zn_status_name(uint32_t status);  /* per-blob codes */
zn_ctx* zn_ctx_create(int device, size_t staging_bytes); /* NULL on failure */
void zn_ctx_destroy(zn_ctx* ctx);
const char* zn_last_error(const zn_ctx* ctx);
/* pinned host staging buffer owned by the ctx (the Magazine-slot analogue); *bytes receives its size */
void* zn_ctx_pinned(zn_ctx* ctx, size_t* bytes);
/* number of kernels this ctx has launched since creation (bench.py reports it as gpu_launches) */
uint64_t zn_ctx_kernel_launches(const zn_ctx* ctx);

/* ---- host-buffer API: H2D, kernels, D2H all inside the call; synchronous on return ---- */

/* digests[i] = BLAKE3(base[off[i] .. off[i]+len[i]))  */
int zn_hash_batch(zn_ctx* ctx, const uint8_t* base, const uint64_t* off, const uint64_t* len, uint32_t n,
                  uint8_t* digests /* n*32 */);

/*
 * For each blob i: if compressed[i], decode blobs_base[blob_off[i] .. +blob_len[i]) (capacity out_len[i]);
 * else the blob bytes are the content.  compressed[i] == 1: the codec is identified by the frame magic (Zstandard
 * or LZ4 frame); 2: the blob is one raw LZ4 block (no header; both sizes come from the index); 3: a Zstandard frame
 * without its 4-byte magic (the 4 bytes in front of it must belong to the caller's buffer; only the device copy is
 * touched); 4: enveloped — zn_envelope_parse decides per blob (ZNB1, bare frame, registered foreign parser; a RAW
 * payload is treated like a store-as-is row, an envelope whose decoded size disagrees with out_len[i] gets
 * ZN_S_SIZE_MISMATCH, an unknown one ZN_S_UNSUPPORTED).  Then BLAKE3 the content, compare with expect_digest[i] when given,
 * and copy the content to out_base[out_off[i] ..] when out_base is given.
 *   expect_digest  nullable (n*32)  -> no compare (extract_file semantics, archive.rs:144-168)
 *   out_base       nullable         -> verify-only (decompress_archive with save_data=false)
 *   digest_out     nullable (n*32)
 *   status         required (n)
 * Writes to out_base touch the declared ranges only, with one exception: when consecutive ranges are separated by
 * alignment padding of fewer than 16 bytes each, the whole span returns in one copy and the padding bytes are
 * unspecified.  Ranges further apart are copied row by row and the memory between them is left alone.
 */
int zn_decode_verify_batch(zn_ctx* ctx, const uint8_t* blobs_base, const uint64_t* blob_off,
                           const uint64_t* blob_len, const uint8_t* compressed, const uint64_t* out_len,
                           const uint8_t* expect_digest, uint8_t* out_base, const uint64_t* out_off, uint32_t n,
                           uint32_t* status, uint8_t* digest_out);

/*
 * For each slice i: digest_out[i] = BLAKE3(src), dst_base[dst_off[i] ..] = one frame of `codec` holding src.
 * dst_off has n+1 entries; capacity of slice i is dst_off[i+1]-dst_off[i] and must be >= zn_compress_bound().
 * `level` keeps the meaning of CompressCtx::new(level) (codec.rs:16): higher = more effort.  The zstd match finder
 * has four efforts: levels <= 2, 3..9, 10..19 search a window of 20 / 40 / 62 KiB; levels >= 20 (the long effort) find
 * matches anywhere in the slice up to 8 MiB back, through a candidate index sorted on the device, and take several
 * times longer.  A match never reaches into another slice, and a frame depends only on its slice's bytes.  LZ4 has
 * one effort.  The frame is always decodable by stock libzstd / liblz4.
 * codec ZN_CODEC_ZSTD | ZN_CODEC_SEEKABLE (levels <= 19): the blob is the seekable layout described at the codec enum;
 * ZN_E_ARG for LZ4 or a level >= 20 with the flag.  | ZN_CODEC_CHECKSUM (zstd or LZ4, not seekable): every frame ends
 * in its content checksum.
 */
int zn_compress_batch(zn_ctx* ctx, const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                      uint32_t n, int level, int codec, uint8_t* dst_base, const uint64_t* dst_off,
                      uint64_t* dst_len_out, uint8_t* digest_out /* nullable */, uint32_t* status);

/* ZN_CODEC_ZSTD | ZN_CODEC_SEEKABLE: exact, per 128 KiB block 13 + 3 + the block's bytes + 12, plus 17 for the seek
 * table; 38 for an empty slice.  ZN_CODEC_CHECKSUM adds 4 bytes. */
size_t zn_compress_bound(size_t src_len, int codec);
/* device time (ms, CUDA events) of the compression kernels of the most recent zn_compress_batch on this ctx */
float zn_ctx_last_compress_ms(const zn_ctx* ctx);

/* decoded size announced by the frame header. returns ZN_OK, 1 when the frame carries no size, <0 on error.  Only the
 * first frame is read: the decoded size of a blob of concatenated frames with a seek table (ZN_CODEC_SEEKABLE) is what
 * zn_envelope_parse reports. */
int zn_frame_content_size(const uint8_t* blob, size_t len, uint64_t* size_out);

/* ---- envelope layer (csrc/envelope.cpp): what the reference's zl_get_decompressed_size / zl_decompress pair does
 * before any codec runs (znippy-common/src/codec.rs:67-78) — find the codec payload inside the blob and its decoded
 * size.  Kernels never see an envelope; the host-buffer calls resolve rows flagged compressed == 4 through
 * zn_envelope_parse and pass the payload range on.  Recognised: bare Zstandard / LZ4 frames (by magic); ZNB1, this
 * library's own envelope: "ZNB1", one byte payload codec, LEB128 decoded size (< 4 GiB), payload; and whatever the one
 * registered foreign parser accepts — the seam where a host that links OpenZL plugs in its frame-header reader (the
 * OpenZL layout itself is unpinned here, DESIGN.md §1). ---- */
enum { ZN_PAYLOAD_RAW = 0, ZN_PAYLOAD_ZSTD = 1, ZN_PAYLOAD_ZSTD_MAGICLESS = 2, ZN_PAYLOAD_LZ4_FRAME = 3, ZN_PAYLOAD_LZ4_BLOCK = 4 };
enum { ZN_ENV_UNKNOWN = 0, ZN_ENV_BARE = 1, ZN_ENV_ZNB1 = 2, ZN_ENV_FOREIGN = 3 };
#define ZN_ENVELOPE_ZNB1_MAX_HEADER 10
typedef struct {
  uint32_t kind;        /* ZN_ENV_* */
  uint32_t codec;       /* ZN_PAYLOAD_* */
  uint64_t payload_off; /* payload = blob[payload_off .. payload_off + payload_len) */
  uint64_t payload_len;
  uint64_t out_len;     /* decoded size the envelope announces; UINT64_MAX when it carries none */
} zn_envelope;
/* ZN_OK; 1 = not a recognised / well-formed envelope (the row gets ZN_S_UNSUPPORTED); < 0 bad arguments.  A bare zstd
 * blob that ends in a valid seek table (ZN_CODEC_SEEKABLE) announces the sum of the table's decompressed sizes. */
int zn_envelope_parse(const uint8_t* blob, size_t len, zn_envelope* out);
/* Writes the ZNB1 header for a payload of `codec` decoding to out_len bytes; returns its length (0 on bad arguments). */
size_t zn_envelope_znb1_header(uint32_t codec, uint64_t out_len, uint8_t* hdr, size_t cap);
/* Foreign envelope parser, consulted for blobs that are neither bare frames nor ZNB1 (NULL unregisters).  It fills
 * codec / payload_off / payload_len / out_len and returns ZN_OK, or 1 to decline.  A ZN_PAYLOAD_ZSTD_MAGICLESS payload
 * needs payload_off >= 4 (the decoder rebuilds the magic in front of it on the device copy). */
typedef int (*zn_envelope_parser)(const uint8_t* blob, size_t len, zn_envelope* out);
void zn_envelope_register(zn_envelope_parser fn);

/* ---- native read worker: the loop shell of decompress_archive (znippy-common/src/decompress.rs:105-192) over rows
 * [row_lo, row_hi) of the merged index.  Per batch of rows: pread blobs into pinned staging (io_threads threads),
 * one zn_decode_verify_batch, pwrite of the decoded bytes at fdata_offset to out_fd[row] (out_fd NULL = verify only,
 * out_fd[row] < 0 = skip), and the reference's counter rules.  corrupt_rows_out (nullable) receives the indices of
 * digest-mismatch rows (capacity row_hi - row_lo). ---- */
typedef struct {
  uint64_t total_chunks, total_written_bytes, verified_bytes, corrupt_bytes, corrupt_rows, decode_errors;
} zn_verify_stats;
int zn_decompress_rows(zn_ctx* ctx, int archive_fd, uint64_t row_lo, uint64_t row_hi, const uint64_t* blob_offset,
                       const uint64_t* blob_size, const uint64_t* fdata_offset, const uint8_t* compressed,
                       const uint64_t* uncompressed_size, const uint8_t* checksums, const int* out_fd, size_t batch_bytes,
                       int io_threads, uint64_t* corrupt_rows_out, zn_verify_stats* stats);

/* ---- `.znippy` v0.7 container, natively (csrc/container.cpp; no Arrow library): footer -> manifest -> sub-indexes
 * (znippy-common/src/index.rs:245-441), rows of all sub-indexes concatenated, columns looked up by name. ---- */
typedef struct zn_index zn_index;
zn_index* zn_index_open(const char* path, char* err, size_t errcap); /* NULL on failure, message in err */
void zn_index_close(zn_index* index);
uint64_t zn_index_rows(const zn_index* index);
/* col: 0 blob_offset, 1 blob_size, 2 fdata_offset, 3 uncompressed_size */
const uint64_t* zn_index_u64(const zn_index* index, int col);
const uint32_t* zn_index_chunk_seq(const zn_index* index);
const uint8_t* zn_index_compressed(const zn_index* index); /* one byte per row, 0/1 */
const uint8_t* zn_index_checksums(const zn_index* index);  /* rows * 32 */
const char* zn_index_path(const zn_index* index, uint64_t row, uint32_t* len); /* not NUL terminated */
uint64_t zn_index_groups(const zn_index* index);            /* manifest entries */
int zn_index_group(const zn_index* index, uint64_t g, int8_t* pkg_type, const char** repo, uint64_t* index_offset,
                   uint64_t* index_len, uint64_t* row_count);
const char* zn_index_metadata(const zn_index* index, const char* key); /* schema key/value of the first sub-index */
uint32_t zn_index_field_count(const zn_index* index);
const char* zn_index_field_name(const zn_index* index, uint32_t i);

/* writer tail (meta_sink.rs:71-118): sub-index per (pkg_type, repo) group -> manifest -> "ZNPYMIDX" + offset, fsync */
typedef struct zn_index_writer zn_index_writer;
zn_index_writer* zn_index_writer_create(int fd, uint64_t blob_end);
int zn_index_writer_metadata(zn_index_writer* w, const char* key, const char* value); /* before the first group */
int zn_index_writer_push_group(zn_index_writer* w, int8_t pkg_type, const char* repo, uint64_t n, const char* const* paths,
                               const uint32_t* chunk_seq, const uint64_t* fdata_offset, const uint8_t* compressed,
                               const uint64_t* uncompressed_size, const uint64_t* blob_offset, const uint64_t* blob_size,
                               const uint8_t* checksums);
int zn_index_writer_finish(zn_index_writer* w); /* also destroys w */

/* decompress_archive (decompress.rs:39-222) end to end without Python: index -> output files -> zn_decompress_rows ->
 * VerifyReport (index.rs:490-499).  Rows [row_lo, row_hi) (clamped): one call per GPU shard. */
typedef struct {
  uint64_t total_files, verified_files, corrupt_files, total_bytes, verified_bytes, corrupt_bytes, chunks;
} zn_verify_report;
int zn_archive_decompress(zn_ctx* ctx, const char* index_path, int save_data, const char* out_dir, uint64_t row_lo,
                          uint64_t row_hi, size_t batch_bytes, int io_threads, zn_verify_report* report, char* err,
                          size_t errcap);

/* ---- native random access: ZnippyArchive (znippy-common/src/archive.rs:20-168).  extract_files = every chunk of every
 * requested file in one batch (no digest compare, as archive.rs:144-168), chunks concatenated in fdata_offset order at
 * out_base + out_off[i] (capacity = zn_archive_file_size).  file_status[i]: 0 ok, 1 not in the archive,
 * 2 | (blob status << 16) a chunk failed to decode. */
typedef struct zn_archive zn_archive;
zn_archive* zn_archive_open(const char* path, char* err, size_t errcap);
void zn_archive_close(zn_archive* a);
uint64_t zn_archive_file_count(const zn_archive* a);
const char* zn_archive_file_name(const zn_archive* a, uint64_t i, uint64_t* size);
int zn_archive_file_size(const zn_archive* a, const char* path, uint64_t* size); /* 1 = present */
int zn_archive_extract_files(zn_ctx* ctx, zn_archive* a, const char* const* paths, uint32_t n, uint8_t* out_base,
                             const uint64_t* out_off, uint32_t* file_status);
/* Byte ranges of files (HTTP Range requests, the zip central directory at the end of a jar or wheel).  Request i asks
 * for bytes [offset[i], offset[i] + length[i]) of file paths[i], clamped at the file's end as pread clamps: an offset at
 * or past the end, or a zero length, gives got[i] = 0 with status 0.  The bytes go to out_base + out_off[i] ..; got[i] =
 * bytes written, and out_base is written only inside [out_off[i], out_off[i] + got[i]).  file_status[i] as
 * zn_archive_extract_files (2 | (blob status << 16) for the first failing chunk of the request, which then gets got = 0).
 * All requests of a call are one batch:
 *   - only the chunks a range touches are read; a chunk several requests touch is decoded once;
 *   - a chunk covered in full is decoded and checked exactly as extract_files decodes it (no digest compare);
 *   - a chunk covered in part is decoded only up to the end of the block that holds the furthest byte any request of the
 *     call needs from it (at most one 128 KiB zstd block or one LZ4 frame block more).  Only that prefix is checked:
 *     damage past the block where decoding stopped goes unseen, and the content checksum is not checked.  A frame that
 *     ends before that point gives ZN_S_SIZE_MISMATCH.  A raw LZ4 block chunk is one block and decodes whole;
 *   - in seekable archives (index metadata znippy_seekable = "zstd", ZN_CODEC_SEEKABLE), a zstd chunk covered in part
 *     is served from its seek table instead: only the 128 KiB frames the requests touch are read, each run of adjacent
 *     ones is decoded whole, and every decoded frame is checked against the table's XXH64 (a mismatch is
 *     ZN_S_DECODE_ERROR).  A table that is missing or inconsistent with the chunk sends it down the prefix path above.
 *     The counters then count the frames' output and the table + frame bytes read;
 *   - store-as-is chunks and ZNB1 chunks with a RAW payload never reach the GPU: only the requested bytes are pread,
 *     straight into out_base.  A call whose ranges lie only in such chunks launches no kernel;
 *   - with the LRU on, cached chunks are copied from it, chunks decoded in full are inserted, partial chunks never.
 * stats (nullable) counts what the call did. */
typedef struct {
  uint64_t rows_decoded;    /* distinct index rows run through a decoder in this call */
  uint64_t bytes_decoded;   /* bytes those decoders produced (whole rows + edge-row prefixes) */
  uint64_t blob_bytes_read; /* bytes pread from the archive */
  uint64_t rows_from_cache; /* rows answered by the LRU of decoded slices */
} zn_range_stats;
int zn_archive_read_ranges(zn_ctx* ctx, zn_archive* a, const char* const* paths, const uint64_t* offset,
                           const uint64_t* length, uint32_t n, uint8_t* out_base, const uint64_t* out_off, uint64_t* got,
                           uint32_t* file_status, zn_range_stats* stats /* nullable */);
/* LRU of decoded slices for a serving process (SURVEY §8f-2): with a non-zero budget, every slice extract_files decodes is
 * kept in host memory (keyed by index row, evicted least-recently-used first) and later requests for it skip pread, H2D
 * and the decode.  0 (the default) turns it off and drops what is cached.  stats: hits, misses, evictions, bytes, slices. */
int zn_archive_set_cache(zn_archive* a, uint64_t budget_bytes);
int zn_archive_cache_stats(zn_archive* a, uint64_t stats[5]);

/* ---- native write pipeline: compress_stream (znippy-compress/src/stream_packer.rs:58-372).  Entries are cut into
 * <= 8 MiB rounds into a pinned slot; each full slot is one zn_compress_batch (+ zn_hash_batch for store-as-is rounds),
 * payloads are pwritten at a running cursor, finish() writes sub-indexes per (pkg_type, repo), manifest and footer. */
typedef struct zn_archive_writer zn_archive_writer;
typedef struct {
  uint64_t total_files, compressed_files, uncompressed_files, chunks, total_bytes_in, total_bytes_out, compressed_bytes,
      uncompressed_bytes;
} zn_compression_report; /* CompressionReport, znippy-common/src/lib.rs:39-51 */
zn_archive_writer* zn_archive_writer_create(zn_ctx* ctx, const char* output_path, int no_skip, int level, int codec,
                                            size_t slot_bytes);
int zn_archive_writer_add(zn_archive_writer* w, const char* relative_path, const uint8_t* data, uint64_t len, int has_pkg_type,
                          int8_t pkg_type, const char* repo); /* data is consumed (copied into the slot) before returning */
int zn_archive_writer_finish(zn_archive_writer* w, zn_compression_report* report); /* also destroys w */
const char* zn_archive_writer_error(const zn_archive_writer* w);
/* The writer is a three-stage pipeline over three pinned slots (the Magazine, slotpool.rs:93-227): filling slot k+2,
 * compressing slot k+1 on the GPU and pwriting slot k overlap; `ctx` belongs to the writer until finish().
 * compress_dir (slot_packer.rs:329-609): walks input_dir (sorted), cuts every file into rounds placed in the slots and
 * lets io_threads readers pread the bytes into place — the whole directory in one call.
 * codec ZN_CODEC_ZSTD | ZN_CODEC_SEEKABLE (levels <= 19) writes seekable blobs and the index metadata
 * znippy_seekable = "zstd"; with LZ4 or a level >= 20 zn_archive_writer_create returns NULL and zn_archive_compress_dir
 * returns ZN_E_ARG with a message.  codec | ZN_CODEC_CHECKSUM (zstd or LZ4, not seekable) writes a content checksum
 * into every compressed row's frame. */
int zn_archive_compress_dir(zn_ctx* ctx, const char* input_dir, const char* output_path, int no_skip, int level, int codec,
                            size_t slot_bytes, int io_threads, zn_compression_report* report, char* err, size_t errcap);
/* pinned host memory (cudaHostAlloc) for callers that stage their own buffers */
void* zn_ctx_pinned_alloc(size_t bytes);
void zn_ctx_pinned_free(void* p);

/* ---- device-resident API (inputs and outputs already in HBM; used for the device GB/s metric and by
 *      callers that keep a batch resident).  d_* are device pointers; h_* host pointers. ---- */

/* Builds the device-side descriptor tables for a decode+verify batch (uploads them, sizes scratch). */
zn_plan* zn_plan_decode_verify(zn_ctx* ctx, uint32_t n, const uint64_t* h_blob_off, const uint64_t* h_blob_len,
                               const uint8_t* h_compressed, const uint64_t* h_out_off, const uint64_t* h_out_len,
                               const uint8_t* h_expect_digest /* nullable */);
/* Hash-only plan over resident bytes (store-as-is verify / write-side hashing). */
zn_plan* zn_plan_hash(zn_ctx* ctx, uint32_t n, const uint64_t* h_off, const uint64_t* h_len,
                      const uint8_t* h_expect_digest /* nullable */);
void zn_plan_destroy(zn_plan* plan);
/* Enqueues the batch on `stream` (cudaStream_t; NULL = the ctx's own stream). Asynchronous.
 * d_out may be NULL only for hash-only plans. */
int zn_plan_run(zn_plan* plan, const uint8_t* d_blobs, uint8_t* d_out, void* stream);
/* Waits for the last run and copies results back. status / digests nullable.  Compress plans: per-slice statuses, and
 * the BLAKE3 digests of the source slices when the plan was created with `digests` (otherwise h_digests is untouched). */
int zn_plan_results(zn_plan* plan, uint32_t* h_status, uint8_t* h_digests);
/* Kept for ABI stability; has no effect.  (Round 1 offered a stream-overlapped decode/hash schedule here; it measured
 * slower than the stages back to back on every corpus and was replaced by per-row kernel classes.) */
int zn_plan_set_overlap(zn_plan* plan, int groups);
/* Rows of a decode+verify plan per decode class, chosen per row from the index columns alone (the reference's worker
 * treats every row alike, decompress.rs:156-166; here the row's sizes pick its kernel):
 *   [0] entropy-coded Zstandard frames      -> device-wide pipeline (csrc/zpipe.cuh)
 *   [1] large, highly compressible frames   -> fused decode+hash kernel (csrc/fused_ws.cuh)
 *   [2] large raw-block / LZ4 blobs         -> block-parallel team kernel
 *   [3] decoded size <= 64 KiB              -> one-warp teams
 *   [4] the rest                            -> 128-thread teams */
int zn_plan_class_counts(const zn_plan* plan, uint32_t counts[5]); /* ZN_E_STATE on a compress plan */
/* Rows of class [0] that the device-wide pipeline handed back to the one-team decoder in the last zn_plan_run (anything
 * malformed or beyond the pipeline's budgets; the result is the same, only slower).  Synchronises with the run's
 * stream.  A well-formed batch reports 0 — tests and bench.py check exactly that. */
int zn_plan_pipeline_fallbacks(zn_plan* plan, uint32_t* rows); /* ZN_E_STATE on a compress plan */
/* kernels launched by one zn_plan_run of this plan */
uint32_t zn_plan_launches(const zn_plan* plan);
/* 1 when the plan decodes and hashes in ONE kernel (batches of large, highly compressible blobs: decode warps feed
 * hash warps through a device-wide tile queue, fused_ws.cuh); the decode stage of zn_plan_last_ms then covers both
 * and the hash stage is empty. */
int zn_plan_fused(const zn_plan* plan);
/* device time of the most recent completed run, per stage, in ms (CUDA events on the run's stream):
 * [0] total, [1] decode stage, [2] hash stage (chunks), [3] tree+compare stage.  Synchronises.
 * Compress plans: [0] total, [1] compress kernels, [2] hash, [3] sizing and packing. */
int zn_plan_last_ms(zn_plan* plan, float ms[4]);

/* ---- device-resident compression: the write side of the plan API.  zn_compress_batch copies host slices in, waits for
 * the frame sizes and copies the frames out; a compress plan takes slices already in HBM (a torch tensor, the output of
 * a decode plan) and leaves packed blobs in HBM, without waiting.  The frame sizes are only known on the device, so the
 * layout is made there too: every blob's size from the per-block results, an exclusive scan into offsets, the frames
 * assembled straight into place.  Blob i is byte for byte the frame zn_compress_batch writes for the same slice, level
 * and codec when the slice sits at the same 16-byte phase in device memory: the zstd efforts of levels <= 19 stage a
 * block's window from the 16-byte boundary below it, so their frames depend on that phase (zn_compress_batch keeps a
 * compact host span's layout from its first byte, and places other batches 16-byte aligned).  With ZN_CODEC_ENVELOPE it is what the archive writer stores for a compressed row: a ZNB1 header and the
 * frame, or, when the frame is not smaller than the slice, a RAW-payload header and the slice's bytes.
 * A plan owns its scratch: two plans may run at once on different streams, and zn_compress_batch calls on the same ctx
 * do not disturb it.  zn_plan_results / zn_plan_launches / zn_plan_last_ms / zn_plan_destroy apply; zn_plan_run on a
 * compress plan, and zn_plan_run_compress on any other plan, return ZN_E_STATE. ---- */

/* Compress plan over slices that will be resident in HBM: sizes fixed at creation, data supplied per run.  Slice i is
 * d_src[h_src_off[i] .. + h_src_len[i]) of every run.  `level` and `codec` as for zn_compress_batch; `digests` != 0 also
 * hashes the source slices (the zn_hash_batch kernels, on the run's stream).  All planning, uploads and allocation
 * happen here.  NULL, with zn_last_error set, for a slice of 4 GiB or more, a codec other than ZN_CODEC_ZSTD
 * (optionally | ZN_CODEC_SEEKABLE or | ZN_CODEC_CHECKSUM) / ZN_CODEC_LZ4 (optionally | ZN_CODEC_CHECKSUM), optionally
 * | ZN_CODEC_ENVELOPE, or ZN_CODEC_SEEKABLE at a level >= 20.  Seekable plans also run the frame checksum kernel, and
 * checksummed plans the slice checksum kernel, counted in stage [1] of zn_plan_last_ms.  n = 0 is a valid plan. */
zn_plan* zn_plan_compress(zn_ctx* ctx, uint32_t n, const uint64_t* h_src_off, const uint64_t* h_src_len, int level,
                          int codec /* ZN_CODEC_ZSTD [| ZN_CODEC_SEEKABLE] | ZN_CODEC_LZ4, optionally | ZN_CODEC_CHECKSUM, | ZN_CODEC_ENVELOPE */,
                          int digests);
/* bytes d_dst must hold for any input of these sizes */
uint64_t zn_plan_compress_capacity(const zn_plan* plan);
/* Enqueues the batch on `stream` (NULL = ctx stream) and returns without waiting. Blob i lands at
 * d_dst[d_offsets[i] .. d_offsets[i+1]), back to back with no padding; d_offsets has n+1 entries, written on the
 * device; d_offsets[n] = total bytes.  d_src offsets and d_dst may have any alignment; d_offsets must be 8-byte aligned
 * (ZN_E_ARG otherwise).  The call only enqueues kernels: no allocation, no synchronisation. */
int zn_plan_run_compress(zn_plan* plan, const uint8_t* d_src, uint8_t* d_dst, uint64_t* d_offsets, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ZNIPPY_CUDA_H */
