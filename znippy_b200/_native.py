"""ctypes binding of libznippy_cuda.so (include/znippy_cuda.h).  This is the same binding a Rust `-sys` crate would
declare; see INTEGRATION.md.  There is no CPU fallback: if the library is missing or no CUDA device is usable, every
compute entry point raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

ZN_OK, ZN_E_ARG, ZN_E_CUDA, ZN_E_NOMEM, ZN_E_STATE = 0, -1, -2, -3, -4
S_OK, S_DECODE_ERROR, S_DIGEST_MISMATCH, S_DST_TOO_SMALL, S_UNSUPPORTED, S_SIZE_MISMATCH = range(6)
CODEC_ZSTD, CODEC_LZ4 = 1, 2
CODEC_ENVELOPE = 0x100  # archive writer and compress plans: wrap compressed rows in ZNB1 (include/znippy_cuda.h)

EXPORTS = [
    "zn_abi_version", "zn_device_count", "zn_strerror", "zn_status_name", "zn_ctx_create", "zn_ctx_destroy",
    "zn_last_error", "zn_ctx_pinned", "zn_ctx_kernel_launches", "zn_hash_batch", "zn_decode_verify_batch",
    "zn_compress_batch", "zn_compress_bound", "zn_frame_content_size", "zn_plan_decode_verify", "zn_plan_hash",
    "zn_plan_destroy", "zn_plan_run", "zn_plan_results", "zn_plan_launches", "zn_plan_fused", "zn_plan_last_ms", "zn_plan_set_overlap", "zn_plan_class_counts", "zn_plan_pipeline_fallbacks", "zn_ctx_last_compress_ms", "zn_decompress_rows",
    "zn_index_open", "zn_index_close", "zn_index_rows", "zn_index_u64", "zn_index_chunk_seq", "zn_index_compressed",
    "zn_index_checksums", "zn_index_path", "zn_index_groups", "zn_index_group", "zn_index_metadata", "zn_index_field_count",
    "zn_index_field_name", "zn_index_writer_create", "zn_index_writer_metadata", "zn_index_writer_push_group",
    "zn_index_writer_finish", "zn_archive_decompress", "zn_archive_writer_create", "zn_archive_writer_add",
    "zn_archive_writer_finish", "zn_archive_writer_error", "zn_ctx_pinned_alloc", "zn_ctx_pinned_free",
    "zn_archive_open", "zn_archive_close", "zn_archive_file_count", "zn_archive_file_name", "zn_archive_file_size",
    "zn_archive_extract_files", "zn_archive_set_cache", "zn_archive_cache_stats", "zn_archive_compress_dir", "zn_envelope_parse", "zn_envelope_znb1_header", "zn_envelope_register",
    "zn_plan_compress", "zn_plan_compress_capacity", "zn_plan_run_compress",
]


class NativeError(RuntimeError):
    pass


_lib = None


def lib_path() -> str:
    return _build.SO


def lib() -> C.CDLL:
    """Loads (building first if the .so is absent and nvcc is present) the CUDA library.  Raises when impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.SO):
        _build.build()
    L = C.CDLL(_build.SO)
    vp, u32, u64, sz = C.c_void_p, C.c_uint32, C.c_uint64, C.c_size_t
    L.zn_abi_version.restype = C.c_int
    L.zn_device_count.restype = C.c_int
    L.zn_strerror.argtypes = [C.c_int]
    L.zn_strerror.restype = C.c_char_p
    L.zn_status_name.argtypes = [u32]
    L.zn_status_name.restype = C.c_char_p
    L.zn_ctx_create.argtypes = [C.c_int, sz]
    L.zn_ctx_create.restype = vp
    L.zn_ctx_destroy.argtypes = [vp]
    L.zn_ctx_destroy.restype = None
    L.zn_last_error.argtypes = [vp]
    L.zn_last_error.restype = C.c_char_p
    L.zn_ctx_pinned.argtypes = [vp, C.POINTER(sz)]
    L.zn_ctx_pinned.restype = vp
    L.zn_ctx_kernel_launches.argtypes = [vp]
    L.zn_ctx_kernel_launches.restype = u64
    L.zn_hash_batch.argtypes = [vp, vp, vp, vp, u32, vp]
    L.zn_decode_verify_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, u32, vp, vp]
    L.zn_compress_batch.argtypes = [vp, vp, vp, vp, u32, C.c_int, C.c_int, vp, vp, vp, vp, vp]
    L.zn_compress_bound.argtypes = [sz, C.c_int]
    L.zn_compress_bound.restype = sz
    L.zn_frame_content_size.argtypes = [vp, sz, C.POINTER(u64)]
    L.zn_plan_decode_verify.argtypes = [vp, u32, vp, vp, vp, vp, vp, vp]
    L.zn_plan_decode_verify.restype = vp
    L.zn_plan_hash.argtypes = [vp, u32, vp, vp, vp]
    L.zn_plan_hash.restype = vp
    L.zn_plan_destroy.argtypes = [vp]
    L.zn_plan_destroy.restype = None
    L.zn_plan_run.argtypes = [vp, vp, vp, vp]
    L.zn_plan_compress.argtypes = [vp, u32, vp, vp, C.c_int, C.c_int, C.c_int]
    L.zn_plan_compress.restype = vp
    L.zn_plan_compress_capacity.argtypes = [vp]
    L.zn_plan_compress_capacity.restype = u64
    L.zn_plan_run_compress.argtypes = [vp, vp, vp, vp, vp]
    L.zn_plan_results.argtypes = [vp, vp, vp]
    L.zn_plan_launches.argtypes = [vp]
    L.zn_plan_launches.restype = u32
    L.zn_plan_fused.argtypes = [vp]
    L.zn_plan_fused.restype = C.c_int
    L.zn_plan_last_ms.argtypes = [vp, C.POINTER(C.c_float * 4)]
    L.zn_plan_set_overlap.argtypes = [vp, C.c_int]
    L.zn_plan_class_counts.argtypes = [vp, C.POINTER(C.c_uint32)]
    L.zn_plan_pipeline_fallbacks.argtypes = [vp, C.POINTER(C.c_uint32)]
    L.zn_decompress_rows.argtypes = [vp, C.c_int, u64, u64, vp, vp, vp, vp, vp, vp, vp, sz, C.c_int, vp, vp]
    L.zn_index_open.argtypes = [C.c_char_p, C.c_char_p, sz]
    L.zn_index_open.restype = vp
    L.zn_index_close.argtypes = [vp]
    L.zn_index_close.restype = None
    L.zn_index_rows.argtypes = [vp]
    L.zn_index_rows.restype = u64
    L.zn_index_u64.argtypes = [vp, C.c_int]
    L.zn_index_u64.restype = C.POINTER(C.c_uint64)
    L.zn_index_chunk_seq.argtypes = [vp]
    L.zn_index_chunk_seq.restype = C.POINTER(C.c_uint32)
    L.zn_index_compressed.argtypes = [vp]
    L.zn_index_compressed.restype = C.POINTER(C.c_uint8)
    L.zn_index_checksums.argtypes = [vp]
    L.zn_index_checksums.restype = C.POINTER(C.c_uint8)
    L.zn_index_path.argtypes = [vp, u64, C.POINTER(u32)]
    L.zn_index_path.restype = C.POINTER(C.c_char)
    L.zn_index_groups.argtypes = [vp]
    L.zn_index_groups.restype = u64
    L.zn_index_group.argtypes = [vp, u64, C.POINTER(C.c_int8), C.POINTER(C.c_char_p), C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
    L.zn_index_metadata.argtypes = [vp, C.c_char_p]
    L.zn_index_metadata.restype = C.c_char_p
    L.zn_index_field_count.argtypes = [vp]
    L.zn_index_field_count.restype = u32
    L.zn_index_field_name.argtypes = [vp, u32]
    L.zn_index_field_name.restype = C.c_char_p
    L.zn_index_writer_create.argtypes = [C.c_int, u64]
    L.zn_index_writer_create.restype = vp
    L.zn_index_writer_metadata.argtypes = [vp, C.c_char_p, C.c_char_p]
    L.zn_index_writer_push_group.argtypes = [vp, C.c_int8, C.c_char_p, u64, vp, vp, vp, vp, vp, vp, vp, vp]
    L.zn_index_writer_finish.argtypes = [vp]
    L.zn_archive_decompress.argtypes = [vp, C.c_char_p, C.c_int, C.c_char_p, u64, u64, sz, C.c_int, vp, C.c_char_p, sz]
    L.zn_archive_open.argtypes = [C.c_char_p, C.c_char_p, sz]
    L.zn_archive_open.restype = vp
    L.zn_archive_close.argtypes = [vp]
    L.zn_archive_close.restype = None
    L.zn_archive_file_count.argtypes = [vp]
    L.zn_archive_file_count.restype = u64
    L.zn_archive_file_name.argtypes = [vp, u64, C.POINTER(u64)]
    L.zn_archive_file_name.restype = C.c_char_p
    L.zn_archive_file_size.argtypes = [vp, C.c_char_p, C.POINTER(u64)]
    L.zn_archive_extract_files.argtypes = [vp, vp, vp, u32, vp, vp, vp]
    L.zn_archive_writer_create.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.c_int, sz]
    L.zn_archive_writer_create.restype = vp
    L.zn_archive_writer_add.argtypes = [vp, C.c_char_p, vp, u64, C.c_int, C.c_int8, C.c_char_p]
    L.zn_archive_writer_finish.argtypes = [vp, vp]
    L.zn_archive_writer_error.argtypes = [vp]
    L.zn_archive_writer_error.restype = C.c_char_p
    L.zn_ctx_pinned_alloc.argtypes = [sz]
    L.zn_ctx_pinned_alloc.restype = vp
    L.zn_ctx_pinned_free.argtypes = [vp]
    L.zn_ctx_pinned_free.restype = None
    L.zn_archive_set_cache.argtypes = [vp, u64]
    L.zn_archive_cache_stats.argtypes = [vp, vp]
    L.zn_archive_compress_dir.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, sz, C.c_int, vp, C.c_char_p, sz]
    L.zn_envelope_parse.argtypes = [vp, sz, vp]
    L.zn_envelope_znb1_header.argtypes = [u32, u64, vp, sz]
    L.zn_envelope_znb1_header.restype = sz
    L.zn_envelope_register.argtypes = [vp]
    L.zn_envelope_register.restype = None
    L.zn_ctx_last_compress_ms.argtypes = [vp]
    L.zn_ctx_last_compress_ms.restype = C.c_float
    if L.zn_abi_version() != 1:
        raise NativeError("libznippy_cuda.so ABI version mismatch")
    _lib = L
    return L


def u8(a) -> np.ndarray:
    """Contiguous uint8 view of bytes / bytearray / memoryview / ndarray (no copy when already contiguous)."""
    if isinstance(a, np.ndarray):
        return np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    return np.frombuffer(a, dtype=np.uint8)


def u64(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint64))


def ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class Ctx:
    """One CUDA device + stream + staging (zn_ctx).  Mirrors the lifetime of the reference's per-worker
    `CompressCtx` (codec.rs:8-28): long-lived, single-threaded."""

    def __init__(self, device: int = 0, staging_bytes: int = 0):
        L = lib()
        if L.zn_device_count() <= 0:
            raise NativeError("no CUDA device: znippy_b200 has no CPU fallback")
        self._h = L.zn_ctx_create(device, staging_bytes)
        if not self._h:
            raise NativeError(f"zn_ctx_create(device={device}) failed")
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            lib().zn_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def check(self, rc: int, what: str):
        if rc != ZN_OK:
            raise NativeError(f"{what}: {lib().zn_strerror(rc).decode()} ({lib().zn_last_error(self._h).decode()})")

    def launches(self) -> int:
        return int(lib().zn_ctx_kernel_launches(self._h))

    def last_compress_ms(self) -> float:
        return float(lib().zn_ctx_last_compress_ms(self._h))

    def pinned(self) -> np.ndarray:
        n = C.c_size_t(0)
        p = lib().zn_ctx_pinned(self._h, C.byref(n))
        if not p or n.value == 0:
            raise NativeError("context was created without a staging buffer")
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n.value,))


_default: dict[int, Ctx] = {}


def default_ctx(device: int = 0) -> Ctx:
    if device not in _default:
        _default[device] = Ctx(device)
    return _default[device]


class Plan:
    """Device-resident batch (zn_plan)."""

    def __init__(self, ctx: Ctx, handle, n: int):
        if not handle:
            raise NativeError("plan creation failed: " + lib().zn_last_error(ctx.handle).decode())
        self.ctx, self._h, self.n = ctx, handle, n

    @classmethod
    def decode_verify(cls, ctx: Ctx, blob_off, blob_len, compressed, out_off, out_len, expect=None) -> "Plan":
        bo, bl, oo, ol = u64(blob_off), u64(blob_len), u64(out_off), u64(out_len)
        cf = np.ascontiguousarray(np.asarray(compressed, dtype=np.uint8))
        ex = None if expect is None else u8(expect)
        n = bo.size
        assert bl.size == n and oo.size == n and ol.size == n and cf.size == n and (ex is None or ex.size == 32 * n)
        h = lib().zn_plan_decode_verify(ctx.handle, n, ptr(bo), ptr(bl), ptr(cf), ptr(oo), ptr(ol), ptr(ex))
        return cls(ctx, h, n)

    @classmethod
    def hash(cls, ctx: Ctx, off, length, expect=None) -> "Plan":
        o, l = u64(off), u64(length)
        ex = None if expect is None else u8(expect)
        h = lib().zn_plan_hash(ctx.handle, o.size, ptr(o), ptr(l), ptr(ex))
        return cls(ctx, h, o.size)

    @classmethod
    def compress(cls, ctx: Ctx, src_off, src_len, level: int = 1, codec: int = CODEC_ZSTD, envelope: bool = False,
                 digests: bool = True) -> "Plan":
        """Compress plan over slices resident on the device (zn_plan_compress): slice i = d_src[src_off[i] : + src_len[i]]
        of every run_compress.  envelope=True: ZNB1 blobs, RAW when the frame does not shrink the slice."""
        o, l = u64(src_off), u64(src_len)
        assert l.size == o.size
        h = lib().zn_plan_compress(ctx.handle, o.size, ptr(o), ptr(l), level, codec | (CODEC_ENVELOPE if envelope else 0),
                                   1 if digests else 0)
        return cls(ctx, h, o.size)

    def capacity(self) -> int:
        """bytes the d_dst of run_compress must hold (zn_plan_compress_capacity)"""
        return int(lib().zn_plan_compress_capacity(self._h))

    def run_compress(self, d_src_ptr: int, d_dst_ptr: int, d_offsets_ptr: int, stream: int = 0):
        """Enqueues the compress plan on `stream` (zn_plan_run_compress) and returns at once: blob i lands at
        d_dst[d_offsets[i] : d_offsets[i + 1]] (n + 1 uint64 offsets, 8-byte aligned)."""
        self.ctx.check(lib().zn_plan_run_compress(self._h, C.c_void_p(d_src_ptr), C.c_void_p(d_dst_ptr),
                                                  C.c_void_p(d_offsets_ptr), C.c_void_p(stream)), "zn_plan_run_compress")

    def run(self, d_blobs_ptr: int, d_out_ptr: int = 0, stream: int = 0):
        self.ctx.check(lib().zn_plan_run(self._h, C.c_void_p(d_blobs_ptr), C.c_void_p(d_out_ptr), C.c_void_p(stream)),
                       "zn_plan_run")

    def results(self):
        st = np.zeros(self.n, np.uint32)
        dg = np.zeros((self.n, 32), np.uint8)
        self.ctx.check(lib().zn_plan_results(self._h, ptr(st), ptr(dg)), "zn_plan_results")
        return st, dg

    def class_counts(self):
        """rows per decode class: [pipeline, fused pattern, big raw, small, mid] (zn_plan_class_counts)"""
        out = (C.c_uint32 * 5)()
        self.ctx.check(lib().zn_plan_class_counts(self._h, out), "zn_plan_class_counts")
        return list(out)

    def pipeline_fallbacks(self) -> int:
        """rows the device-wide pipeline handed back to the one-team decoder in the last run (zn_plan_pipeline_fallbacks)"""
        n = C.c_uint32(0)
        self.ctx.check(lib().zn_plan_pipeline_fallbacks(self._h, C.byref(n)), "zn_plan_pipeline_fallbacks")
        return int(n.value)

    def set_overlap(self, groups: int):
        self.ctx.check(lib().zn_plan_set_overlap(self._h, groups), "zn_plan_set_overlap")

    def launches(self) -> int:
        return int(lib().zn_plan_launches(self._h))

    def fused(self) -> bool:
        return bool(lib().zn_plan_fused(self._h))

    def last_ms(self):
        ms = (C.c_float * 4)()
        self.ctx.check(lib().zn_plan_last_ms(self._h, C.byref(ms)), "zn_plan_last_ms")
        return [float(x) for x in ms]

    def close(self):
        if getattr(self, "_h", None):
            lib().zn_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
