"""Host-side mirror of the reference's codec boundary, backed by libznippy_cuda.so.

Same names, argument meaning and error behaviour as `znippy-common/src/codec.rs`:

    CompressCtx.new(level) / .compress / .compress_into      codec.rs:16-55
    decompress_frame / decompress_into                       codec.rs:58-78
    blake3_hash                                              blake3::hash at decompress.rs:172,
                                                             stream_packer.rs:219, slot_packer.rs:553

plus the batch-first forms the worker loops call (one call per batch of index rows instead of one per row).
The wire format of a compressed blob is a standard Zstandard frame or LZ4 frame, bare or inside this library's own ZNB1
envelope; the envelope layer (`envelope_parse`, csrc/envelope.cpp) is also where a parser for the reference's OpenZL
envelope plugs in (its layout is unpinned in this environment, see DESIGN.md).  Everything computes on the GPU; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from ._native import (CODEC_LZ4, CODEC_ZSTD, S_DECODE_ERROR, S_DIGEST_MISMATCH, S_DST_TOO_SMALL, S_OK,  # noqa: F401
                      S_SIZE_MISMATCH, S_UNSUPPORTED, Ctx, NativeError, default_ctx)


class CodecError(RuntimeError):
    """The `anyhow::Error` of codec.rs: raised by the single-blob calls when the blob's status is not OK."""

    def __init__(self, status: int, what: str):
        self.status = int(status)
        super().__init__(f"{what}: {N.lib().zn_status_name(int(status)).decode()}")


# ----------------------------------------------------------------------------------------------- batch forms

def hash_batch(base, off, length, ctx: Ctx | None = None) -> np.ndarray:
    """digests[i] = BLAKE3(base[off[i] : off[i]+length[i]]) -> (n, 32) uint8."""
    ctx = ctx or default_ctx()
    b, o, l = N.u8(base), N.u64(off), N.u64(length)
    n = o.size
    if n and int((o + l).max()) > b.size:
        raise ValueError("range outside base")
    out = np.zeros((n, 32), np.uint8)
    if b.size == 0:
        b = np.zeros(1, np.uint8)
    ctx.check(N.lib().zn_hash_batch(ctx.handle, N.ptr(b), N.ptr(o), N.ptr(l), n, N.ptr(out)), "zn_hash_batch")
    return out


def decode_verify_batch(blobs, blob_off, blob_len, compressed, out_len, expect=None, out=None, out_off=None,
                        ctx: Ctx | None = None):
    """Body of the reference read loop (decompress.rs:148-184) for a batch of rows.

    Returns (status[n] uint32, digests[n,32] uint8).  `out` (uint8 array) receives the content of row i at
    out_off[i] when given; `expect` (n*32 bytes) enables the digest compare."""
    ctx = ctx or default_ctx()
    b, bo, bl, ol = N.u8(blobs), N.u64(blob_off), N.u64(blob_len), N.u64(out_len)
    cf = np.ascontiguousarray(np.asarray(compressed, dtype=np.uint8))
    n = bo.size
    if not (bl.size == n and ol.size == n and cf.size == n):
        raise ValueError("descriptor arrays differ in length")
    if n and int((bo + bl).max()) > b.size:
        raise ValueError("blob range outside blobs buffer")
    ex = None if expect is None else N.u8(expect)
    if ex is not None and ex.size != 32 * n:
        raise ValueError("expect must hold n*32 bytes")
    oo = None
    if out is not None:
        oo = N.u64(out_off)
        if n and int((oo + ol).max()) > out.size:
            raise ValueError("output range outside out buffer")
    if b.size == 0:
        b = np.zeros(1, np.uint8)
    st = np.empty(n, np.uint32)  # both fully written by the call
    dg = np.empty((n, 32), np.uint8)
    ctx.check(N.lib().zn_decode_verify_batch(ctx.handle, N.ptr(b), N.ptr(bo), N.ptr(bl), N.ptr(cf), N.ptr(ol), N.ptr(ex),
                                             N.ptr(out), N.ptr(oo), n, N.ptr(st), N.ptr(dg)), "zn_decode_verify_batch")
    return st, dg


def compress_bound(n: int, codec: int = CODEC_ZSTD) -> int:
    return int(N.lib().zn_compress_bound(n, codec))


def compress_batch(src, src_off, src_len, level: int = 1, codec: int = CODEC_ZSTD, ctx: Ctx | None = None):
    """Barrel body of the write side (stream_packer.rs:217-232) for a batch of slices.

    Returns (blobs: list[bytes], digests[n,32], status[n])."""
    ctx = ctx or default_ctx()
    s, so, sl = N.u8(src), N.u64(src_off), N.u64(src_len)
    n = so.size
    caps = np.array([compress_bound(int(x), codec) for x in sl], dtype=np.uint64)
    doff = np.zeros(n + 1, np.uint64)
    np.cumsum(caps, out=doff[1:])
    dst = np.empty(int(doff[-1]) + 1, np.uint8)  # every byte that is read back below was written by the call
    dlen = np.zeros(n, np.uint64)
    dg = np.zeros((n, 32), np.uint8)
    st = np.zeros(n, np.uint32)
    if s.size == 0:
        s = np.zeros(1, np.uint8)
    ctx.check(N.lib().zn_compress_batch(ctx.handle, N.ptr(s), N.ptr(so), N.ptr(sl), n, level, codec, N.ptr(dst), N.ptr(doff),
                                        N.ptr(dlen), N.ptr(dg), N.ptr(st)), "zn_compress_batch")
    blobs = [dst[int(doff[i]): int(doff[i]) + int(dlen[i])].tobytes() for i in range(n)]
    return blobs, dg, st


def frame_content_size(blob) -> int | None:
    """zl_get_decompressed_size (codec.rs:69): decoded size announced by the frame header, None when absent."""
    b = N.u8(blob)
    v = C.c_uint64(0)
    rc = N.lib().zn_frame_content_size(N.ptr(b) if b.size else None, b.size, C.byref(v))
    if rc < 0:
        raise CodecError(S_UNSUPPORTED, "frame header")
    return None if rc == 1 else int(v.value)


# ----------------------------------------------------------------------------------------------- envelope layer
PAYLOAD_RAW, PAYLOAD_ZSTD, PAYLOAD_ZSTD_MAGICLESS, PAYLOAD_LZ4_FRAME, PAYLOAD_LZ4_BLOCK = range(5)
ENV_UNKNOWN, ENV_BARE, ENV_ZNB1, ENV_FOREIGN = range(4)
COMPRESSED_ENVELOPED = 4  # compressed[] value: zn_envelope_parse decides per blob (include/znippy_cuda.h)


class _Envelope(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("codec", C.c_uint32), ("payload_off", C.c_uint64), ("payload_len", C.c_uint64),
                ("out_len", C.c_uint64)]


def envelope_parse(blob):
    """zn_envelope_parse: (kind, payload codec, payload_off, payload_len, out_len | None), or None when the blob is not a
    recognised envelope (the batch calls give such a row S_UNSUPPORTED).  What OpenZL's frame-header read does in the
    reference (codec.rs:69) happens here; kernels only ever see payload ranges."""
    b = N.u8(blob)
    e = _Envelope()
    rc = N.lib().zn_envelope_parse(N.ptr(b) if b.size else None, b.size, C.byref(e))
    if rc < 0:
        raise ValueError("zn_envelope_parse: bad arguments")
    if rc != 0:
        return None
    return e.kind, e.codec, int(e.payload_off), int(e.payload_len), None if e.out_len == 2**64 - 1 else int(e.out_len)


def envelope_wrap(payload_codec: int, out_len: int, payload) -> bytes:
    """One ZNB1 blob: "ZNB1", payload codec, LEB128 decoded size, payload."""
    hdr = (C.c_uint8 * 10)()
    n = N.lib().zn_envelope_znb1_header(payload_codec, out_len, hdr, 10)
    if n == 0:
        raise ValueError("zn_envelope_znb1_header: bad codec or size")
    return bytes(hdr[:n]) + bytes(payload)


# ----------------------------------------------------------------------------------------------- codec.rs mirror

def blake3_hash(data, ctx: Ctx | None = None) -> bytes:
    b = N.u8(data)
    return hash_batch(b, [0], [b.size], ctx)[0].tobytes()


class CompressCtx:
    """codec.rs:8-55.  `level` follows the reference's meaning (higher = more effort); the GPU match finder has
    four efforts: three window geometries for levels <= 2, 3..9 and 10..19, and for levels >= 20 (zstd only) the long
    effort, whose matches reach back anywhere in the slice up to 8 MiB (DESIGN.md §4.3)."""

    def __init__(self, compression_level: int, codec: int = CODEC_ZSTD, ctx: Ctx | None = None, envelope: bool = False):
        self.level = int(compression_level)
        self.codec = codec
        self.ctx = ctx or default_ctx()
        self.envelope = envelope  # wrap every frame in ZNB1; incompressible input is then stored RAW (size + 6..10 bytes)

    @classmethod
    def new(cls, compression_level: int) -> "CompressCtx":
        return cls(compression_level)

    def compress(self, data) -> bytes:
        b = N.u8(data)
        blobs, _, st = compress_batch(b, [0], [b.size], self.level, self.codec, self.ctx)
        if st[0] != S_OK:
            raise CodecError(st[0], "compress")
        if self.envelope:
            if len(blobs[0]) >= b.size:
                return envelope_wrap(PAYLOAD_RAW, b.size, b.tobytes())
            return envelope_wrap(PAYLOAD_ZSTD if self.codec == CODEC_ZSTD else PAYLOAD_LZ4_FRAME, b.size, blobs[0])
        return blobs[0]

    def compress_into(self, data, out: bytearray) -> int:
        blob = self.compress(data)
        out[:] = blob  # resize-to-bound then truncate-to-written, codec.rs:45-54
        return len(blob)


def decompress_into(compressed, out: bytearray) -> int:
    """codec.rs:67-78: size from the frame header, grow `out`, decode, truncate to bytes written."""
    env = envelope_parse(compressed)  # zl_get_decompressed_size: the size comes out of the frame / envelope header
    if env is None or env[4] is None:
        raise CodecError(S_UNSUPPORTED, "getDecompressedSize")
    size = env[4]
    b = N.u8(compressed)
    buf = np.zeros(max(size, 1), np.uint8)
    st, _ = decode_verify_batch(b, [0], [b.size], [COMPRESSED_ENVELOPED], [size], None, buf, [0])
    if st[0] != S_OK:
        raise CodecError(st[0], "decompress")
    out[:] = buf[:size].tobytes()
    return size


def decompress_frame(compressed) -> bytes:
    out = bytearray()
    decompress_into(compressed, out)
    return bytes(out)
