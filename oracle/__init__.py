"""znippy-b200 CPU ORACLE — test infrastructure only.

ctypes front-end of ``oracle/liboracle.so`` (plain-C restatements, see ``oracle.h``) plus thin bindings to the
*independent* truth libraries present in this image: ``libzstd.so.1`` 1.5.5, ``liblz4.so.1`` 1.9.4 (runtime
libraries only; prototypes declared by hand) and the official ``blake3`` Python bindings.

Only ``tests/``, ``bench.py``'s cpu_baseline / ``--impl reference`` leg and ``__graft_entry__.smoke()`` may
import this package.  Nothing under ``znippy_b200/`` does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")

OK = 0
ERR_SRC_TRUNCATED, ERR_BAD_MAGIC, ERR_DST_TOO_SMALL, ERR_CORRUPT, ERR_UNSUPPORTED, ERR_CHECKSUM, ERR_SIZE_MISMATCH = (
    -1, -2, -3, -4, -5, -6, -7)


def build(force: bool = False) -> str:
    """Compile liboracle.so with gcc (make) if it is missing or stale."""
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".c", ".h"))]
    stale = (not os.path.exists(_SO)) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-B", "liboracle.so"], check=True, capture_output=True)
    return _SO


class ZstdStats(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in (
        "frames", "skippable_frames", "blocks_raw", "blocks_rle", "blocks_compressed",
        "lit_raw", "lit_rle", "lit_huf_1stream", "lit_huf_4stream", "lit_treeless",
        "huf_weights_direct", "huf_weights_fse",
        "mode_predefined", "mode_rle", "mode_fse", "mode_repeat",
        "repcode_uses", "overlap_matches")] + [
        ("sequences", C.c_uint64), ("literal_bytes", C.c_uint64), ("match_bytes", C.c_uint64),
        ("checksums_verified", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class VerifyStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "total_chunks", "total_written_bytes", "verified_bytes", "corrupt_bytes", "corrupt_rows", "decode_errors")]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        u8p = C.c_void_p
        L.zn_ref_blake3.argtypes = [u8p, C.c_size_t, u8p]
        L.zn_ref_blake3_fast.argtypes = [u8p, C.c_size_t, u8p]
        L.zn_ref_xxh64.argtypes = [u8p, C.c_size_t, C.c_uint64]
        L.zn_ref_xxh64.restype = C.c_uint64
        L.zn_ref_xxh32.argtypes = [u8p, C.c_size_t, C.c_uint32]
        L.zn_ref_xxh32.restype = C.c_uint32
        L.zn_ref_zstd_decompress.argtypes = [u8p, C.c_size_t, u8p, C.c_size_t, C.POINTER(C.c_size_t), C.c_void_p]
        L.zn_ref_zstd_frame_content_size.argtypes = [u8p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.zn_ref_lz4_block_decompress.argtypes = [u8p, C.c_size_t, u8p, C.c_size_t]
        L.zn_ref_lz4_block_decompress.restype = C.c_long
        L.zn_ref_lz4_frame_decompress.argtypes = [u8p, C.c_size_t, u8p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.zn_ref_lz4_frame_content_size.argtypes = [u8p, C.c_size_t, C.POINTER(C.c_uint64)]
        for n in ("zn_ref_gen_text", "zn_ref_gen_binary"):
            getattr(L, n).argtypes = [u8p, C.c_size_t, C.c_size_t]
            getattr(L, n).restype = None
        L.zn_ref_gen_random.argtypes = [u8p, C.c_size_t]
        L.zn_ref_gen_random.restype = None
        L.zn_ref_gen_incompressible.argtypes = [u8p, C.c_size_t, C.c_uint64]
        L.zn_ref_gen_incompressible.restype = None
        L.zn_ref_decompress_rows.argtypes = [u8p] * 7 + [C.c_uint64, C.c_int, u8p, u8p, C.c_void_p, C.c_void_p,
                                                        C.c_int, C.POINTER(VerifyStats)]
        L.zn_ref_compress_slices.argtypes = [u8p, u8p, u8p, C.c_uint64, C.c_int, C.c_int, u8p, u8p, u8p, u8p,
                                             C.c_void_p, C.c_void_p, C.c_int]
        _lib = L
    return _lib


def _buf(b) -> np.ndarray:
    a = np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else b
    return np.ascontiguousarray(a.view(np.uint8).reshape(-1))


def _ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


# ----------------------------------------------------------------------------- restatements

def blake3(data, fast: bool = False) -> bytes:
    a = _buf(data)
    out = np.zeros(32, np.uint8)
    (lib().zn_ref_blake3_fast if fast else lib().zn_ref_blake3)(_ptr(a), a.size, _ptr(out))
    return out.tobytes()


def xxh64(data, seed: int = 0) -> int:
    a = _buf(data)
    return int(lib().zn_ref_xxh64(_ptr(a), a.size, seed))


def xxh32(data, seed: int = 0) -> int:
    a = _buf(data)
    return int(lib().zn_ref_xxh32(_ptr(a), a.size, seed))


def zstd_decompress(blob, cap: int, want_stats: bool = False):
    """Returns (rc, bytes[, stats dict]) — rc is one of the ERR_* codes."""
    a = _buf(blob)
    out = np.zeros(max(cap, 1), np.uint8)
    n = C.c_size_t(0)
    st = ZstdStats()
    rc = lib().zn_ref_zstd_decompress(_ptr(a), a.size, _ptr(out), cap, C.byref(n), C.byref(st))
    res = out[: n.value].tobytes()
    return (rc, res, st.as_dict()) if want_stats else (rc, res)


def zstd_frame_content_size(blob):
    a = _buf(blob)
    v = C.c_uint64(0)
    rc = lib().zn_ref_zstd_frame_content_size(_ptr(a), a.size, C.byref(v))
    return rc, v.value


def lz4_block_decompress(blob, cap: int):
    a = _buf(blob)
    out = np.zeros(max(cap, 1), np.uint8)
    r = lib().zn_ref_lz4_block_decompress(_ptr(a), a.size, _ptr(out), cap)
    return (r, b"") if r < 0 else (0, out[:r].tobytes())


def lz4_frame_decompress(blob, cap: int):
    a = _buf(blob)
    out = np.zeros(max(cap, 1), np.uint8)
    n = C.c_size_t(0)
    rc = lib().zn_ref_lz4_frame_decompress(_ptr(a), a.size, _ptr(out), cap, C.byref(n))
    return rc, out[: n.value].tobytes()


def lz4_frame_content_size(blob):
    a = _buf(blob)
    v = C.c_uint64(0)
    rc = lib().zn_ref_lz4_frame_content_size(_ptr(a), a.size, C.byref(v))
    return rc, v.value


# ----------------------------------------------------------------------------- corpora (perf_bench.rs:74-92)

def gen_text(n: int, phase: int = 0) -> np.ndarray:
    out = np.empty(n, np.uint8)
    lib().zn_ref_gen_text(_ptr(out), n, phase)
    return out


def gen_binary(n: int, start: int = 0) -> np.ndarray:
    out = np.empty(n, np.uint8)
    lib().zn_ref_gen_binary(_ptr(out), n, start)
    return out


def gen_random(n: int) -> np.ndarray:
    out = np.empty(n, np.uint8)
    lib().zn_ref_gen_random(_ptr(out), n)
    return out


def gen_incompressible(n: int, seed: int) -> np.ndarray:
    out = np.empty(n, np.uint8)
    lib().zn_ref_gen_incompressible(_ptr(out), n, seed)
    return out


def real_text(n: int) -> np.ndarray:
    """Entropy-coded test corpus from files guaranteed in the image (python stdlib sources), SURVEY §8(c)."""
    import sysconfig
    root = sysconfig.get_paths()["stdlib"]
    chunks, total = [], 0
    for name in sorted(os.listdir(root)):
        if not name.endswith(".py"):
            continue
        with open(os.path.join(root, name), "rb") as f:
            b = f.read()
        chunks.append(b)
        total += len(b)
        if total >= n:
            break
    data = b"".join(chunks)
    while len(data) < n:
        data += data
    return np.frombuffer(data[:n], np.uint8).copy()


def gen_small_alphabet(n: int, nsym: int = 9, seed: int = 3) -> np.ndarray:
    """Skewed symbols 0..nsym-1: libzstd emits Huffman literals whose tree uses DIRECT 4-bit weights."""
    rng = np.random.default_rng(seed)
    p = np.array([2.0 ** -(i + 1) for i in range(nsym - 1)] + [2.0 ** -(nsym - 1)])
    return rng.choice(np.arange(nsym), n, p=p).astype(np.uint8)


def gen_periodic_noise(n: int, dist: int, period: int, seed: int = 1) -> np.ndarray:
    """out[i] = out[i-dist] except every `period`-th byte is fresh noise: many near-identical sequences, which makes
    libzstd choose RLE mode for a sequence table (dist=200, period=12, n=2000 at level 3)."""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 256, n, dtype=np.uint8)
    for i in range(dist, n):
        if i % period:
            d[i] = d[i - dist]
    return d


def gen_rle_literals(n_matches: int = 3000, seed: int = 0) -> np.ndarray:
    """128 KiB of noise followed by (run of 'a', slice copied from the noise) pairs: at zstd level 19 the second
    and later blocks carry RLE literals sections plus repeat-mode tables (a path the README corpora never hit)."""
    rng = np.random.default_rng(seed)
    noise = rng.integers(0, 256, 131072, dtype=np.uint8)
    parts = [noise]
    for _ in range(n_matches):
        s = int(rng.integers(0, 131072 - 40))
        parts.append(np.full(int(rng.integers(1, 6)), 97, np.uint8))
        parts.append(noise[s: s + int(rng.integers(8, 40))])
    return np.concatenate(parts)


# ----------------------------------------------------------------------------- independent truth: libzstd / liblz4

class _Zstd:
    def __init__(self):
        z = C.CDLL("libzstd.so.1")
        z.ZSTD_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]
        z.ZSTD_compress.restype = C.c_size_t
        z.ZSTD_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        z.ZSTD_decompress.restype = C.c_size_t
        z.ZSTD_compressBound.argtypes = [C.c_size_t]
        z.ZSTD_compressBound.restype = C.c_size_t
        z.ZSTD_isError.argtypes = [C.c_size_t]
        z.ZSTD_isError.restype = C.c_uint
        z.ZSTD_getErrorName.argtypes = [C.c_size_t]
        z.ZSTD_getErrorName.restype = C.c_char_p
        z.ZSTD_createCCtx.restype = C.c_void_p
        z.ZSTD_freeCCtx.argtypes = [C.c_void_p]
        z.ZSTD_CCtx_setParameter.argtypes = [C.c_void_p, C.c_int, C.c_int]
        z.ZSTD_CCtx_setParameter.restype = C.c_size_t
        z.ZSTD_compress2.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        z.ZSTD_compress2.restype = C.c_size_t
        z.ZSTD_compressSequences.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                             C.c_size_t]
        z.ZSTD_compressSequences.restype = C.c_size_t
        z.ZSTD_CCtx_refPrefix.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        z.ZSTD_CCtx_refPrefix.restype = C.c_size_t
        z.ZSTD_writeSkippableFrame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint]
        z.ZSTD_writeSkippableFrame.restype = C.c_size_t
        self.z = z

    # Experimental parameter ids of zstd.h 1.5.5 (ZSTD_c_experimentalParam5 / 11 / 12 / 19); the ids move between releases.
    C_LITERAL_COMPRESSION_MODE = 1002    # ZSTD_ps_enable = 1 (Huffman), ZSTD_ps_disable = 2 (raw literals)
    C_BLOCK_DELIMITERS = 1008            # ZSTD_sf_explicitBlockDelimiters = 1
    C_VALIDATE_SEQUENCES = 1009          # checks offsets against the content only: a frame with a prefix needs it off
    C_SEARCH_EXTERNAL_REPCODES = 1016    # below level 10 libzstd would otherwise never turn a given offset into a repeat code

    class _Seq(C.Structure):  # ZSTD_Sequence
        _fields_ = [("offset", C.c_uint), ("litLength", C.c_uint), ("matchLength", C.c_uint), ("rep", C.c_uint)]

    def _check(self, r):
        if self.z.ZSTD_isError(r):
            raise RuntimeError(self.z.ZSTD_getErrorName(r).decode())
        return r

    def compress_sequences(self, blocks, literals, level: int = 3, params: dict | None = None, prefix=None):
        """One frame whose blocks carry exactly the given LZ77 parse (ZSTD_compressSequences; libzstd chooses the entropy
        coding, repeat codes included).  `blocks`: one list of (ll, ml, off) per block; a last tuple with ml == 0 holds
        the block's trailing literals.  Literal bytes are taken from `literals` in order.  `prefix`: content the frame
        may reference before its start (ZSTD_CCtx_refPrefix); a decoder needs the same prefix.
        Returns (content, frame); content excludes the prefix."""
        lit = bytes(_buf(literals))
        pre = bytes(_buf(prefix)) if prefix is not None else b""
        out, li, arr = bytearray(pre), 0, []
        for block in blocks:
            for k, (ll, ml, off) in enumerate(block):
                if li + ll > len(lit):
                    raise ValueError("literal source too short")
                out += lit[li:li + ll]
                li += ll
                if ml == 0:
                    if k != len(block) - 1:
                        raise ValueError("only a block's last tuple may have no match")
                    break
                s = len(out) - off
                if off <= 0 or s < 0:
                    raise ValueError(f"offset {off} reaches before the content")
                out += out[s:s + ml] if off >= ml else (out[s:] * (ml // off + 1))[:ml]
                arr.append((off, ll, ml, 0))
            last = block[-1] if block else (0, 0, 0)
            arr.append((0, last[0] if last[1] == 0 else 0, 0, 0))  # block delimiter carrying the trailing literals
        content = bytes(out[len(pre):])
        seqs = (self._Seq * len(arr))(*[self._Seq(*a) for a in arr])
        cap = self.z.ZSTD_compressBound(len(content)) + 64 * len(blocks)
        dst = np.empty(cap, np.uint8)
        src = np.frombuffer(content, np.uint8) if content else np.zeros(1, np.uint8)
        cctx = self.z.ZSTD_createCCtx()
        try:
            settings = {100: level, self.C_BLOCK_DELIMITERS: 1, self.C_VALIDATE_SEQUENCES: 1,  # 100: compressionLevel
                        self.C_SEARCH_EXTERNAL_REPCODES: 1}
            settings.update(params or {})
            for k, v in settings.items():
                self._check(self.z.ZSTD_CCtx_setParameter(cctx, int(k), int(v)))
            pbuf = np.frombuffer(pre, np.uint8) if pre else None
            if pre:
                self._check(self.z.ZSTD_CCtx_refPrefix(cctx, _ptr(pbuf), len(pre)))
            r = self._check(self.z.ZSTD_compressSequences(cctx, _ptr(dst), cap, seqs, len(arr), _ptr(src), len(content)))
        finally:
            self.z.ZSTD_freeCCtx(cctx)
        return content, dst[:r].tobytes()

    def skippable_frame(self, payload: bytes, variant: int = 0) -> bytes:
        """ZSTD_writeSkippableFrame: magic 0x184D2A50 + variant, size, payload."""
        src = np.frombuffer(payload, np.uint8) if payload else np.zeros(1, np.uint8)
        dst = np.empty(len(payload) + 8, np.uint8)
        r = self._check(self.z.ZSTD_writeSkippableFrame(_ptr(dst), dst.size, _ptr(src), len(payload), variant))
        return dst[:r].tobytes()

    def version(self) -> int:
        return int(self.z.ZSTD_versionNumber())

    def compress(self, data, level: int = 3, checksum: bool = False, params: dict | None = None) -> bytes:
        a = _buf(data)
        cap = self.z.ZSTD_compressBound(a.size)
        out = np.empty(cap, np.uint8)
        if not checksum and not params:
            r = self.z.ZSTD_compress(_ptr(out), cap, _ptr(a), a.size, level)
        else:
            cctx = self.z.ZSTD_createCCtx()
            self.z.ZSTD_CCtx_setParameter(cctx, 100, level)  # ZSTD_c_compressionLevel
            if checksum:
                self.z.ZSTD_CCtx_setParameter(cctx, 201, 1)  # ZSTD_c_checksumFlag
            for k, v in (params or {}).items():
                rr = self.z.ZSTD_CCtx_setParameter(cctx, int(k), int(v))
                if self.z.ZSTD_isError(rr):
                    raise RuntimeError(self.z.ZSTD_getErrorName(rr).decode())
            r = self.z.ZSTD_compress2(cctx, _ptr(out), cap, _ptr(a), a.size)
            self.z.ZSTD_freeCCtx(cctx)
        if self.z.ZSTD_isError(r):
            raise RuntimeError(self.z.ZSTD_getErrorName(r).decode())
        return out[:r].tobytes()

    def decompress(self, blob, cap: int) -> bytes:
        a = _buf(blob)
        out = np.empty(max(cap, 1), np.uint8)
        r = self.z.ZSTD_decompress(_ptr(out), cap, _ptr(a), a.size)
        if self.z.ZSTD_isError(r):
            raise RuntimeError(self.z.ZSTD_getErrorName(r).decode())
        return out[:r].tobytes()

    def fn_ptrs(self):
        """(decompress, isError, compress) raw addresses for the C pipeline restatement."""
        cast = lambda f: C.cast(f, C.c_void_p)
        return cast(self.z.ZSTD_decompress), cast(self.z.ZSTD_isError), cast(self.z.ZSTD_compress)


class _Lz4:
    def __init__(self):
        l = C.CDLL("liblz4.so.1")
        l.LZ4_compressBound.argtypes = [C.c_int]
        l.LZ4_compress_default.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        l.LZ4_compress_HC.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        l.LZ4_decompress_safe.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        l.LZ4F_compressFrameBound.argtypes = [C.c_size_t, C.c_void_p]
        l.LZ4F_compressFrameBound.restype = C.c_size_t
        l.LZ4F_compressFrame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
        l.LZ4F_compressFrame.restype = C.c_size_t
        l.LZ4F_isError.argtypes = [C.c_size_t]
        l.LZ4F_getErrorName.argtypes = [C.c_size_t]
        l.LZ4F_getErrorName.restype = C.c_char_p
        l.LZ4F_createDecompressionContext.argtypes = [C.POINTER(C.c_void_p), C.c_uint]
        l.LZ4F_createDecompressionContext.restype = C.c_size_t
        l.LZ4F_freeDecompressionContext.argtypes = [C.c_void_p]
        l.LZ4F_decompress.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t), C.c_void_p,
                                      C.POINTER(C.c_size_t), C.c_void_p]
        l.LZ4F_decompress.restype = C.c_size_t
        self.l = l

    def compress_block(self, data, hc_level: int | None = None) -> bytes:
        a = _buf(data)
        cap = self.l.LZ4_compressBound(a.size)
        out = np.empty(cap, np.uint8)
        if hc_level is None:
            r = self.l.LZ4_compress_default(_ptr(a), _ptr(out), a.size, cap)
        else:
            r = self.l.LZ4_compress_HC(_ptr(a), _ptr(out), a.size, cap, hc_level)
        if r <= 0:
            raise RuntimeError("LZ4 compress failed")
        return out[:r].tobytes()

    def decompress_block(self, blob, cap: int) -> bytes:
        a = _buf(blob)
        out = np.empty(max(cap, 1), np.uint8)
        r = self.l.LZ4_decompress_safe(_ptr(a), _ptr(out), a.size, cap)
        if r < 0:
            raise RuntimeError(f"LZ4_decompress_safe -> {r}")
        return out[:r].tobytes()

    class _Prefs(C.Structure):  # LZ4F_preferences_t (1.9.x layout)
        _fields_ = [("blockSizeID", C.c_int), ("blockMode", C.c_int), ("contentChecksumFlag", C.c_int),
                    ("frameType", C.c_int), ("contentSize", C.c_ulonglong), ("dictID", C.c_uint),
                    ("blockChecksumFlag", C.c_int), ("compressionLevel", C.c_int), ("autoFlush", C.c_uint),
                    ("favorDecSpeed", C.c_uint), ("reserved", C.c_uint * 3)]

    def compress_frame(self, data, block_size_id: int = 4, independent: bool = True, content_size: bool = True,
                       content_checksum: bool = False, block_checksum: bool = False, level: int = 0) -> bytes:
        a = _buf(data)
        p = self._Prefs()
        p.blockSizeID = block_size_id
        p.blockMode = 1 if independent else 0
        p.contentChecksumFlag = int(content_checksum)
        p.contentSize = a.size if content_size else 0
        p.blockChecksumFlag = int(block_checksum)
        p.compressionLevel = level
        cap = self.l.LZ4F_compressFrameBound(a.size, C.byref(p))
        out = np.empty(cap, np.uint8)
        r = self.l.LZ4F_compressFrame(_ptr(out), cap, _ptr(a), a.size, C.byref(p))
        if self.l.LZ4F_isError(r):
            raise RuntimeError(self.l.LZ4F_getErrorName(r).decode())
        return out[:r].tobytes()

    def decompress_frame(self, blob, cap: int) -> bytes:
        a = _buf(blob)
        ctx = C.c_void_p()
        r = self.l.LZ4F_createDecompressionContext(C.byref(ctx), 100)
        if self.l.LZ4F_isError(r):
            raise RuntimeError("LZ4F ctx")
        out = np.empty(max(cap, 1), np.uint8)
        ip = op = 0
        try:
            while ip < a.size:
                dn = C.c_size_t(cap - op)
                sn = C.c_size_t(a.size - ip)
                r = self.l.LZ4F_decompress(ctx, C.c_void_p(out.ctypes.data + op), C.byref(dn),
                                           C.c_void_p(a.ctypes.data + ip), C.byref(sn), None)
                if self.l.LZ4F_isError(r):
                    raise RuntimeError(self.l.LZ4F_getErrorName(r).decode())
                ip += sn.value
                op += dn.value
                if r == 0:
                    break
                if sn.value == 0 and dn.value == 0:
                    raise RuntimeError("LZ4F_decompress made no progress (dst too small?)")
        finally:
            self.l.LZ4F_freeDecompressionContext(ctx)
        return out[:op].tobytes()


_z = _l = None


def libzstd() -> _Zstd:
    global _z
    if _z is None:
        _z = _Zstd()
    return _z


def liblz4() -> _Lz4:
    global _l
    if _l is None:
        _l = _Lz4()
    return _l


def blake3_official(data) -> bytes:
    import blake3 as _b3
    return _b3.blake3(bytes(data) if not isinstance(data, (bytes, bytearray, memoryview)) else data).digest()


# ----------------------------------------------------------------------------- reference worker loops on CPU

@dataclass
class CpuVerify:
    total_chunks: int
    total_written_bytes: int
    verified_bytes: int
    corrupt_bytes: int
    corrupt_rows: int
    decode_errors: int


def decompress_rows(archive: np.ndarray, blob_offset, blob_size, fdata_offset, compressed, uncompressed_size,
                    checksums: np.ndarray, n_threads: int, use_libzstd: bool = True, fast_hash: bool = True,
                    out: np.ndarray | None = None, out_off=None) -> CpuVerify:
    """decompress.rs:105-192 restated (see cpu_pipeline.c)."""
    u64 = lambda x: np.ascontiguousarray(np.asarray(x, np.uint64))
    bo, bs, fo, us = u64(blob_offset), u64(blob_size), u64(fdata_offset), u64(uncompressed_size)
    cf = np.ascontiguousarray(np.asarray(compressed, np.uint8))
    ck = np.ascontiguousarray(checksums.reshape(-1).view(np.uint8))
    oo = u64(out_off) if out_off is not None else None
    st = VerifyStats()
    d, e, _ = libzstd().fn_ptrs() if use_libzstd else (None, None, None)
    lib().zn_ref_decompress_rows(_ptr(archive), _ptr(bo), _ptr(bs), _ptr(fo), _ptr(cf), _ptr(us), _ptr(ck),
                                 len(bo), n_threads, _ptr(out) if out is not None else None,
                                 _ptr(oo) if oo is not None else None, d, e, int(fast_hash), C.byref(st))
    return CpuVerify(*(getattr(st, n) for n, _ in VerifyStats._fields_))


def compress_slices(src: np.ndarray, src_off, src_len, level: int, n_threads: int, fast_hash: bool = True):
    """stream_packer.rs:215-247 restated: blake3 + ZSTD_compress(level) per slice. Returns (blobs, digests)."""
    u64 = lambda x: np.ascontiguousarray(np.asarray(x, np.uint64))
    so, sl = u64(src_off), u64(src_len)
    z = libzstd()
    caps = np.array([z.z.ZSTD_compressBound(int(x)) for x in sl], np.uint64)
    doff = np.zeros(len(sl) + 1, np.uint64)
    np.cumsum(caps, out=doff[1:])
    dst = np.empty(int(doff[-1]), np.uint8)
    dlen = np.zeros(len(sl), np.uint64)
    dig = np.zeros((len(sl), 32), np.uint8)
    _, e, c = z.fn_ptrs()
    rc = lib().zn_ref_compress_slices(_ptr(src), _ptr(so), _ptr(sl), len(sl), level, n_threads, _ptr(dst), _ptr(doff),
                                      _ptr(dlen), _ptr(dig), c, e, int(fast_hash))
    if rc != 0:
        raise RuntimeError("zn_ref_compress_slices failed")
    blobs = [dst[int(doff[i]): int(doff[i]) + int(dlen[i])].tobytes() for i in range(len(sl))]
    return blobs, dig


# ---------------------------------------------------------------------------------------------- envelope layer
# Restatement of the ZNB1 envelope of csrc/envelope.cpp (this build's own blob wrapper, SURVEY §8c): "ZNB1", one byte
# payload codec, LEB128 decoded size (< 4 GiB), payload.  The reference's counterpart is OpenZL's frame header
# (codec.rs:67-78), whose layout is unpinned here — so this pins OUR format only.
PAYLOAD_RAW, PAYLOAD_ZSTD, PAYLOAD_ZSTD_MAGICLESS, PAYLOAD_LZ4_FRAME, PAYLOAD_LZ4_BLOCK = range(5)


def znb1_wrap(codec: int, out_len: int, payload: bytes) -> bytes:
    v, leb = out_len, bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        leb.append(b | (0x80 if v else 0))
        if not v:
            break
    return b"ZNB1" + bytes([codec]) + bytes(leb) + bytes(payload)


def znb1_parse(blob: bytes):
    """(codec, payload_off, payload_len, out_len) or None when malformed."""
    if len(blob) < 6 or blob[:4] != b"ZNB1" or blob[4] > PAYLOAD_LZ4_BLOCK:
        return None
    v, p, shift = 0, 5, 0
    while True:
        if p >= len(blob) or shift > 28:
            return None
        b = blob[p]
        p += 1
        v |= (b & 0x7F) << shift
        shift += 7
        if not b & 0x80:
            break
    if v >= 1 << 32 or (blob[4] == PAYLOAD_RAW and len(blob) - p != v):
        return None
    return blob[4], p, len(blob) - p, v


def envelope_decode(blob: bytes):
    """Decoded content of one enveloped blob through the CPU decoders of this oracle (None when unsupported)."""
    e = znb1_parse(blob)
    if e is None:
        return None
    codec, off, n, out_len = e
    payload = blob[off:off + n]
    if codec == PAYLOAD_RAW:
        return payload
    if codec == PAYLOAD_ZSTD:
        rc, out = zstd_decompress(payload, out_len)
    elif codec == PAYLOAD_ZSTD_MAGICLESS:
        rc, out = zstd_decompress(b"\x28\xb5\x2f\xfd" + payload, out_len)
    elif codec == PAYLOAD_LZ4_FRAME:
        rc, out = lz4_frame_decompress(payload, out_len)
    else:
        rc, out = lz4_block_decompress(payload, out_len)
    return out if rc == 0 and len(out) == out_len else None
