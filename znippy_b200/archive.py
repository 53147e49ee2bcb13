"""`.znippy` v0.7 container (unchanged) and the three host loops that sit on the GPU codec boundary.

Mirrors, with the same names and semantics:

    read_znippy_index / interpret_footer / manifest      znippy-common/src/index.rs:245-468
    ArrowIpcSink.push_subindex / finish                  znippy-common/src/meta_sink.rs:71-118
    decompress_archive -> VerifyReport                   znippy-common/src/decompress.rs:39-222
    ZnippyArchive.open / extract_file / extract_files    znippy-common/src/archive.rs:20-168
    compress_stream -> StreamCompressor                  znippy-compress/src/stream_packer.rs:58-372
    should_skip_compression                              znippy-common/src/index.rs:470-488

The loop shells (row cursor, pread, pwrite, counters) stay on the host; the loop BODIES (decode / blake3 / compare /
compress) are one `zn_*_batch` call per batch of rows.  Index I/O uses pyarrow (the container is metadata, not the
hot path).  Archives written here hold standard Zstandard / LZ4 frames as blobs (DESIGN.md: OpenZL envelope unpinned).
"""
from __future__ import annotations

import io
import os
import struct
from dataclasses import dataclass, field

import numpy as np
import pyarrow as pa

from . import codec
from ._native import Ctx, default_ctx

MULTI_INDEX_MAGIC = b"ZNPYMIDX"  # index.rs:245
SLICE_SIZE = 8 * 1024 * 1024     # stream_packer.rs:31
COMPRESSION_LEVEL = 19           # common_config.rs:37 (echoed into the schema metadata)

_SKIP_EXT = {  # index.rs:470-484
    "zip", "gz", "bz2", "xz", "lz", "lzma", "7z", "rar", "cab", "jar", "war", "ear", "zst", "sz", "lz4", "tgz", "txz",
    "tbz", "apk", "dmg", "deb", "rpm", "arrow", "mpeg", "mpg", "jpeg", "jpg", "gif", "bmp", "png", "crate", "znippy",
    "zdata", "parquet", "webp", "webm"}


def should_skip_compression(path: str) -> bool:
    """Case-insensitive test of the LAST extension only (`deps.tar.gz` -> `gz`)."""
    base = os.path.basename(path)
    if "." not in base:
        return False
    return base.rsplit(".", 1)[1].lower() in _SKIP_EXT


INDEX_SCHEMA = pa.schema([  # index.rs:43-54, all non-nullable
    pa.field("relative_path", pa.utf8(), False), pa.field("chunk_seq", pa.uint32(), False),
    pa.field("fdata_offset", pa.uint64(), False), pa.field("compressed", pa.bool_(), False),
    pa.field("uncompressed_size", pa.uint64(), False), pa.field("blob_offset", pa.uint64(), False),
    pa.field("blob_size", pa.uint64(), False), pa.field("checksum", pa.binary(32), False)])

MANIFEST_SCHEMA = pa.schema([  # index.rs:279-288
    pa.field("pkg_type", pa.int8(), False), pa.field("repo", pa.utf8(), False),
    pa.field("module_name", pa.utf8(), False), pa.field("index_offset", pa.uint64(), False),
    pa.field("index_len", pa.uint64(), False), pa.field("row_count", pa.uint64(), False)])


def config_metadata(level: int = COMPRESSION_LEVEL) -> dict:
    """index.rs:73-85: config echoed as decimal strings into the schema metadata."""
    cores = os.cpu_count() or 1
    return {"znippy_format_version": "3", "max_core_in_flight": str(max(1, -(-cores * 9 // 10))),
            "max_core_in_compress": str(cores), "max_mem_allowed": "0", "min_free_memory_ratio": "0.1",
            "file_split_block_size": str(10 * 1024 * 1024), "max_chunks": "128", "compression_level": str(level),
            "zstd_output_buffer_size": str(1 << 20)}


@dataclass
class VerifyReport:  # index.rs:490-499
    total_files: int = 0
    verified_files: int = 0
    corrupt_files: int = 0
    total_bytes: int = 0
    verified_bytes: int = 0
    corrupt_bytes: int = 0
    chunks: int = 0


@dataclass
class CompressionReport:  # znippy-common/src/lib.rs:39-51
    total_files: int = 0
    compressed_files: int = 0
    uncompressed_files: int = 0
    chunks: int = 0
    total_bytes_in: int = 0
    total_bytes_out: int = 0
    compressed_bytes: int = 0
    uncompressed_bytes: int = 0


# --------------------------------------------------------------------------------------------- container

def interpret_footer(tail: bytes):
    """index.rs:269-277 -> ("multi", manifest_offset) | ("single", index_offset)."""
    off = struct.unpack("<Q", tail[-8:])[0]
    if len(tail) >= 16 and tail[-16:-8] == MULTI_INDEX_MAGIC:
        return "multi", off
    return "single", off


def write_manifest_bytes(entries) -> bytes:
    cols = list(zip(*entries)) if entries else [[] for _ in range(6)]
    batch = pa.record_batch([pa.array(cols[i], type=MANIFEST_SCHEMA.field(i).type) for i in range(6)],
                            schema=MANIFEST_SCHEMA)
    sink = io.BytesIO()
    with pa.ipc.new_stream(sink, MANIFEST_SCHEMA) as w:
        w.write_batch(batch)
    return sink.getvalue()


def read_manifest_bytes(b: bytes):
    t = pa.ipc.open_stream(b).read_all()
    return [tuple(t.column(i)[r].as_py() for i in range(6)) for r in range(t.num_rows)]


def read_znippy_manifest(path: str):
    with open(path, "rb") as f:
        f.seek(0, 2)
        flen = f.tell()
        if flen < 16:
            raise ValueError("not a znippy archive (too small)")
        f.seek(flen - 16)
        kind, off = interpret_footer(f.read(16))
        if kind != "multi":
            raise ValueError("v0.6 archives are not supported")  # index.rs:387-389
        f.seek(off)
        return read_manifest_bytes(f.read(flen - 16 - off))


def read_znippy_index(path: str) -> pa.Table:
    """index.rs:374-441: footer -> manifest -> every sub-index, concatenated with the first sub-index's schema."""
    entries = read_znippy_manifest(path)
    tables = []
    with open(path, "rb") as f:
        for (_pt, _repo, _mod, ioff, ilen, _rows) in entries:
            f.seek(ioff)
            tables.append(pa.ipc.open_stream(f.read(ilen)).read_all())
    if not tables:
        return INDEX_SCHEMA.empty_table()
    first = tables[0].schema
    return pa.concat_tables([t.cast(first) if t.schema != first else t for t in tables])


class ArrowIpcSink:
    """meta_sink.rs:52-118: sub-index(es) -> manifest -> magic + LE offset, appended after the blob region."""

    def __init__(self, f, cursor: int):
        self.f, self.cursor, self.entries = f, cursor, []

    def push_subindex(self, key, schema: pa.Schema, batches):
        sink = io.BytesIO()
        with pa.ipc.new_stream(sink, schema) as w:
            for b in batches:
                w.write_batch(b)
        data = sink.getvalue()
        self.f.seek(self.cursor)
        self.f.write(data)
        pkg_type, repo = key
        self.entries.append((pkg_type, repo, "", self.cursor, len(data), sum(b.num_rows for b in batches)))
        self.cursor += len(data)

    def finish(self):
        m = write_manifest_bytes(self.entries)
        self.f.seek(self.cursor)
        self.f.write(m)
        self.f.write(MULTI_INDEX_MAGIC + struct.pack("<Q", self.cursor))
        self.f.flush()
        os.fsync(self.f.fileno())


def build_metadata_batch(rows, schema: pa.Schema) -> pa.RecordBatch:
    """index.rs:131-191.  rows: (path, chunk_seq, fdata_offset, compressed, uncompressed_size, blob_offset, blob_size, checksum)."""
    cols = list(zip(*rows)) if rows else [[] for _ in range(8)]
    arrays = [pa.array(cols[i], type=INDEX_SCHEMA.field(i).type) for i in range(8)]
    return pa.record_batch(arrays, schema=schema)


# --------------------------------------------------------------------------------------------- read side

def _columns(table: pa.Table):
    g = lambda name, dt: np.asarray(table.column(name).combine_chunks().to_numpy(zero_copy_only=False), dtype=dt)
    checks = table.column("checksum").combine_chunks()
    n = table.num_rows
    ck = (np.frombuffer(checks.buffers()[1], np.uint8, count=32 * n, offset=32 * checks.offset).reshape(n, 32)
          if n else np.zeros((0, 32), np.uint8))
    comp = g("compressed", np.uint8)
    md = table.schema.metadata or {}
    if md.get(b"znippy_envelope") == b"ZNB1":  # compressed rows carry ZNB1 envelopes: resolved by zn_envelope_parse
        comp = (comp * np.uint8(4)).astype(np.uint8)
    return (g("blob_offset", np.uint64), g("blob_size", np.uint64), g("fdata_offset", np.uint64),
            comp, g("uncompressed_size", np.uint64), ck)


def plan_row_batches(blob_size, uncompressed_size, lo: int, hi: int, budget: int):
    """Cuts the row range [lo, hi) into consecutive batches whose blobs + outputs fit `budget` bytes: the GPU
    analogue of `cursor.fetch_add(1)` (decompress.rs:136) is `cursor.fetch_add(B)` over these ranges."""
    out, start, acc = [], lo, 0
    for r in range(lo, hi):
        need = int(blob_size[r]) + int(uncompressed_size[r])
        if r > start and acc + need > budget:
            out.append((start, r))
            start, acc = r, 0
        acc += need
    if hi > start:
        out.append((start, hi))
    return out


def shard_rows(uncompressed_size, world: int):
    """SURVEY §8(e): contiguous row ranges balanced on the prefix sum of uncompressed_size; no exchange."""
    n = len(uncompressed_size)
    pre = np.concatenate([[0], np.cumsum(np.asarray(uncompressed_size, dtype=np.float64) + 1.0)])
    cuts = [int(np.searchsorted(pre, pre[-1] * k / world, side="left")) for k in range(world + 1)]
    cuts[0], cuts[-1] = 0, n
    for k in range(1, world + 1):
        cuts[k] = max(cuts[k], cuts[k - 1])
    return [(cuts[k], cuts[k + 1]) for k in range(world)]


def decompress_rows(archive_fd: int, cols, lo: int, hi: int, save_files=None, ctx: Ctx | None = None,
                    budget: int = 1 << 30, io_threads: int = 8):
    """The worker of decompress.rs:113-192 over rows [lo, hi): returns WorkerStats as a dict.

    The loop itself is native (zn_decompress_rows in libznippy_cuda.so): per batch pread blobs into pinned staging ->
    zn_decode_verify_batch -> fold status[] with the reference's rules (decompress.rs:140,156-184) -> pwrite at
    fdata_offset.  Python only hands over the Arrow columns and the per-row output descriptors."""
    import ctypes as C

    from . import _native as N
    ctx = ctx or default_ctx()
    blob_off, blob_size, fdata_off, compressed, usize, checks = (np.ascontiguousarray(c) for c in cols)
    n = len(blob_off)
    fds = None
    if save_files is not None:
        fds = np.array([-1 if f is None else int(f) for f in save_files], dtype=np.int32)
    st = np.zeros(6, np.uint64)
    corrupt = np.zeros(max(hi - lo, 1), np.uint64)
    rc = N.lib().zn_decompress_rows(ctx.handle, archive_fd, lo, hi, N.ptr(blob_off), N.ptr(blob_size), N.ptr(fdata_off),
                                    N.ptr(compressed), N.ptr(usize), N.ptr(checks.reshape(-1)) if n else None,
                                    None if fds is None else N.ptr(fds), budget, io_threads, N.ptr(corrupt), N.ptr(st))
    ctx.check(rc, "zn_decompress_rows")
    return dict(total_chunks=int(st[0]), total_written_bytes=int(st[1]), verified_bytes=int(st[2]), corrupt_bytes=int(st[3]),
                corrupt_rows=[int(x) for x in corrupt[: int(st[4])]], decode_errors=int(st[5]))


def decompress_archive(index_path: str, save_data: bool, out_dir: str, ctx: Ctx | None = None,
                       row_range=None, native: bool = True) -> VerifyReport:
    """decompress.rs:39-222.  `row_range` restricts the call to one shard (multi-GPU: one process per GPU).

    native=True (default): the whole function runs in libznippy_cuda.so (`zn_archive_decompress`: C++ container
    reader, output-file creation, threaded pread/pwrite worker, batched GPU decode+verify) — no pyarrow, no Python
    loop.  native=False keeps the pyarrow index reader in front of the same native worker (used by the tests to
    cross-check the two readers)."""
    if native:
        import ctypes as C

        from . import _native as N
        ctx = ctx or default_ctx()
        rep = (C.c_uint64 * 7)()
        err = C.create_string_buffer(512)
        lo, hi = row_range if row_range is not None else (0, (1 << 64) - 1)
        rc = N.lib().zn_archive_decompress(ctx.handle, index_path.encode(), int(bool(save_data)), (out_dir or ".").encode(), lo, hi,
                                           1 << 30, 8, C.byref(rep), err, 512)
        if rc != 0:
            raise N.NativeError(f"zn_archive_decompress: {err.value.decode(errors='replace')}")
        return VerifyReport(*[int(x) for x in rep])
    table = read_znippy_index(index_path)
    cols = _columns(table)
    paths = table.column("relative_path").to_pylist()
    total_rows = table.num_rows
    lo, hi = row_range if row_range is not None else (0, total_rows)
    total_files = len(set(paths[lo:hi]))
    files, opened = None, {}
    if save_data:
        files = [None] * total_rows
        # A file whose rows straddle this row range is also written by the neighbouring shard (another process / GPU):
        # truncating it here could destroy chunks that shard has already written.  Such files are opened without
        # O_TRUNC and sized to their full length from the index instead (idempotent, never cuts live data).
        shared = set()
        if lo < hi and lo > 0 and paths[lo - 1] == paths[lo]:
            shared.add(paths[lo])
        if lo < hi and hi < total_rows and paths[hi] == paths[hi - 1]:
            shared.add(paths[hi - 1])
        fo, us = cols[2], cols[4]
        for r in range(lo, hi):
            p = paths[r]
            if p not in opened:
                full = os.path.join(out_dir, p)
                os.makedirs(os.path.dirname(full) or ".", exist_ok=True)
                if p in shared:
                    a = b = r
                    while a > 0 and paths[a - 1] == p:
                        a -= 1
                    while b + 1 < total_rows and paths[b + 1] == p:
                        b += 1
                    opened[p] = os.open(full, os.O_CREAT | os.O_WRONLY, 0o644)
                    os.ftruncate(opened[p], max(int(fo[k]) + int(us[k]) for k in range(a, b + 1)))
                else:
                    opened[p] = os.open(full, os.O_CREAT | os.O_WRONLY | os.O_TRUNC, 0o644)
            files[r] = opened[p]
    fd = os.open(index_path, os.O_RDONLY)
    try:
        st = decompress_rows(fd, cols, lo, hi, files, ctx)
    finally:
        os.close(fd)
        for f in opened.values():
            os.close(f)
    corrupt_files = len(set(st["corrupt_rows"]))  # the reference counts corrupt ROWS here (decompress.rs:210)
    return VerifyReport(total_files=total_files, verified_files=max(0, total_files - corrupt_files),
                        corrupt_files=corrupt_files, total_bytes=st["total_written_bytes"],
                        verified_bytes=st["verified_bytes"], corrupt_bytes=st["corrupt_bytes"],
                        chunks=st["total_chunks"])


def verify_archive_integrity(path: str, ctx: Ctx | None = None) -> VerifyReport:
    return decompress_archive(path, False, "/dev/null", ctx)  # index.rs:550-553


class ZnippyArchive:
    """archive.rs:46-168: random-access reader; `extract_files` is one GPU batch over all requested chunks.  Backed by
    the native `zn_archive_*` (container.cpp): index, per-file chunk lists, pread, batch decode — no pyarrow."""

    def __init__(self, path: str, ctx: Ctx | None = None):
        import ctypes as C

        from . import _native as N
        self.path, self.ctx = path, ctx
        err = C.create_string_buffer(512)
        self._h = N.lib().zn_archive_open(path.encode(), err, 512)
        if not self._h:
            raise IOError(f"cannot open {path}: {err.value.decode(errors='replace')}")

    @classmethod
    def open(cls, path: str, ctx: Ctx | None = None, cache_bytes: int = 0) -> "ZnippyArchive":
        ar = cls(path, ctx)
        if cache_bytes:
            ar.set_cache(cache_bytes)
        return ar

    def set_cache(self, budget_bytes: int):
        """LRU of decoded slices (zn_archive_set_cache): hot files are answered from host memory after their first decode."""
        from . import _native as N
        N.lib().zn_archive_set_cache(self._h, int(budget_bytes))

    def cache_stats(self) -> dict:
        from . import _native as N
        st = np.zeros(5, np.uint64)
        N.lib().zn_archive_cache_stats(self._h, N.ptr(st))
        return dict(zip(("hits", "misses", "evictions", "bytes", "slices"), (int(x) for x in st)))

    def close(self):
        from . import _native as N
        if getattr(self, "_h", None):
            N.lib().zn_archive_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def list_files(self):
        import ctypes as C

        from . import _native as N
        L = N.lib()
        return [L.zn_archive_file_name(self._h, i, None).decode() for i in range(L.zn_archive_file_count(self._h))]

    def contains(self, relative_path: str) -> bool:
        from . import _native as N
        return bool(N.lib().zn_archive_file_size(self._h, relative_path.encode(), None))

    def file_size(self, relative_path: str):
        import ctypes as C

        from . import _native as N
        sz = C.c_uint64(0)
        return int(sz.value) if N.lib().zn_archive_file_size(self._h, relative_path.encode(), C.byref(sz)) else None

    def extract_file(self, relative_path: str) -> bytes:
        r = self.extract_files([relative_path])[0]
        if isinstance(r, Exception):
            raise r
        return r

    def extract_files(self, paths):
        """archive.rs:27-29, batched: every chunk of every requested file in one zn_decode_verify_batch
        (expect_digest = NULL: extract_file does not verify, archive.rs:144-168)."""
        import ctypes as C

        from . import _native as N
        ctx = self.ctx or default_ctx()
        n = len(paths)
        sizes = [self.file_size(p) for p in paths]
        offs = np.zeros(max(n, 1), np.uint64)
        cur = 0
        for i, sz in enumerate(sizes):
            offs[i] = cur
            cur += (sz or 0)
        out = np.zeros(max(cur, 1), np.uint8)
        st = np.zeros(max(n, 1), np.uint32)
        arr = (C.c_char_p * max(n, 1))(*[p.encode() for p in paths])
        ctx.check(N.lib().zn_archive_extract_files(ctx.handle, self._h, arr, n, N.ptr(out), N.ptr(offs), N.ptr(st)),
                  "zn_archive_extract_files")
        res = []
        for i, p in enumerate(paths):
            if st[i] == 1:
                res.append(KeyError(f"file not found in archive: {p}"))
            elif st[i] != 0:
                res.append(codec.CodecError(int(st[i]) >> 16, f"decompress chunk of {p}"))
            else:
                res.append(out[int(offs[i]): int(offs[i]) + sizes[i]].tobytes())
        return res


# --------------------------------------------------------------------------------------------- write side

@dataclass
class ArchiveEntry:  # stream_packer.rs:34-43
    relative_path: str
    data: bytes
    pkg_type: int | None = None
    repo: str | None = None


@dataclass
class _Round:  # slotpool.rs:39-63
    file_index: int
    chunk_seq: int
    fdata_offset: int
    start: int
    length: int
    skip: bool


class StreamCompressor:
    """stream_packer.rs:58-372.  `send()` queues entries; `finish()` runs reader -> GPU barrels -> writer -> sink.
    One `zn_compress_batch` (blake3 + frame per slice) per batch of rounds replaces the N barrel threads; skip
    rounds go through `zn_hash_batch` only (stream_packer.rs:222-227)."""

    def __init__(self, output: str, no_skip: bool, level: int = 19, codec_id: int = codec.CODEC_ZSTD,
                 ctx: Ctx | None = None, batch_bytes: int = 256 << 20, native_index: bool = True, native: bool = True,
                 envelope: bool = False):
        """level defaults to the reference's compression_level = 19 (common_config.rs:37); levels 20-22 select the
        long effort of the zstd match finder (smaller frames, slower writes; codec.CompressCtx).  envelope=True (native
        writer only): blobs of compressed rows are ZNB1 envelopes, incompressible slices are stored raw inside them."""
        if envelope and not native:
            raise ValueError("the ZNB1 envelope is written by the native pipeline only")
        self.envelope = envelope
        self.native_index = native_index
        self.native = native
        self._w = None
        self.output = os.path.splitext(output)[0] + ".znippy"  # stream_packer.rs:132
        self.no_skip, self.level, self.codec_id, self.ctx, self.batch_bytes = no_skip, level, codec_id, ctx, batch_bytes
        self.entries: list[ArchiveEntry] = []

    def _native_writer(self):
        from . import _native as N
        if self._w is None:
            self._ctx = self.ctx or default_ctx()
            self._w = N.lib().zn_archive_writer_create(self._ctx.handle, self.output.encode(), int(self.no_skip), self.level,
                                                       self.codec_id | (N.CODEC_ENVELOPE if self.envelope else 0), self.batch_bytes)
            if not self._w:
                raise IOError(f"cannot create {self.output}")
        return self._w

    def send(self, entry: ArchiveEntry):
        """native=True: the entry is consumed immediately by the C++ pipeline (zn_archive_writer_add copies it into the
        pinned slot and flushes full slots through the GPU), so nothing is retained on the Python side."""
        if not self.native:
            self.entries.append(entry)
            return
        from . import _native as N
        w = self._native_writer()
        d = N.u8(entry.data) if len(entry.data) else None
        rc = N.lib().zn_archive_writer_add(w, entry.relative_path.encode(), None if d is None else N.ptr(d), len(entry.data),
                                           int(entry.pkg_type is not None), entry.pkg_type or 0, (entry.repo or "").encode())
        if rc != 0:
            raise codec.NativeError("zn_archive_writer_add: " + N.lib().zn_archive_writer_error(w).decode())

    def sender(self):
        return self

    def _rounds(self):
        for fi, e in enumerate(self.entries):
            skip = (not self.no_skip) and should_skip_compression(e.relative_path)
            n = len(e.data)
            if n <= SLICE_SIZE:  # whole entry (also the empty entry: one len-0 round), stream_packer.rs:169-183
                yield _Round(fi, 0, 0, 0, n, skip)
            else:
                for seq, start in enumerate(range(0, n, SLICE_SIZE)):
                    yield _Round(fi, seq, start, start, min(SLICE_SIZE, n - start), skip)

    def finish(self) -> CompressionReport:
        if self.native:
            import ctypes as C

            from . import _native as N
            w = self._native_writer()
            rep8 = (C.c_uint64 * 8)()
            rc = N.lib().zn_archive_writer_finish(w, C.byref(rep8))
            self._w = None
            if rc != 0:
                raise codec.NativeError(f"zn_archive_writer_finish failed ({rc})")
            return CompressionReport(*[int(x) for x in rep8])
        rep = CompressionReport(total_files=len(self.entries))
        blobs_meta = []  # (file_index, chunk_seq, fdata_offset, compressed, usize, blob_offset, blob_size, checksum)
        out_cursor = 0
        with open(self.output, "wb") as f:
            batch, acc = [], 0

            def flush():
                nonlocal out_cursor, batch, acc
                if not batch:
                    return
                parts, offs, lens, cur = [], [], [], 0
                for r in batch:
                    d = self.entries[r.file_index].data
                    parts.append(np.frombuffer(d, np.uint8, r.length, r.start) if r.length else np.zeros(0, np.uint8))
                    offs.append(cur); lens.append(r.length)
                    cur += (r.length + 15) & ~15
                src = np.zeros(max(cur, 1), np.uint8)
                for p, o in zip(parts, offs):
                    src[o: o + p.size] = p
                ci = [i for i, r in enumerate(batch) if not r.skip]
                si = [i for i, r in enumerate(batch) if r.skip]
                payload, digest = [None] * len(batch), [None] * len(batch)
                if ci:
                    bl, dg, st = codec.compress_batch(src, [offs[i] for i in ci], [lens[i] for i in ci], self.level,
                                                      self.codec_id, self.ctx)
                    for k, i in enumerate(ci):
                        if st[k] != codec.S_OK:
                            raise codec.CodecError(int(st[k]), "compress")  # `?` propagates, stream_packer.rs:230
                        payload[i], digest[i] = bl[k], dg[k].tobytes()
                if si:
                    dg = codec.hash_batch(src, [offs[i] for i in si], [lens[i] for i in si], self.ctx)
                    for k, i in enumerate(si):
                        payload[i] = src[offs[i]: offs[i] + lens[i]].tobytes()
                        digest[i] = dg[k].tobytes()
                for i, r in enumerate(batch):  # writer, stream_packer.rs:252-285
                    f.seek(out_cursor)
                    f.write(payload[i])
                    blobs_meta.append((r.file_index, r.chunk_seq, r.fdata_offset, not r.skip, r.length, out_cursor,
                                       len(payload[i]), digest[i]))
                    out_cursor += len(payload[i])
                    rep.chunks += 1
                    rep.total_bytes_in += r.length
                    rep.total_bytes_out += len(payload[i])
                    if r.skip:
                        rep.uncompressed_bytes += r.length
                    else:
                        rep.compressed_bytes += r.length
                batch, acc = [], 0

            for r in self._rounds():
                if batch and acc + r.length > self.batch_bytes:
                    flush()
                batch.append(r)
                acc += r.length
            flush()
            for fi, e in enumerate(self.entries):
                if (not self.no_skip) and should_skip_compression(e.relative_path):
                    rep.uncompressed_files += 1
                else:
                    rep.compressed_files += 1
            # finalizer, stream_packer.rs:293-346: sort by (file_index, chunk_seq), group by (pkg_type, repo)
            blobs_meta.sort(key=lambda b: (b[0], b[1]))
            groups: dict = {}
            for b in blobs_meta:
                e = self.entries[b[0]]
                key = (e.pkg_type if e.pkg_type is not None else 0, e.repo or "")
                groups.setdefault(key, []).append((e.relative_path,) + b[1:])
            if not groups:
                groups[(0, "")] = []
            if self.native_index:  # container.cpp writer: sub-index per group -> manifest -> footer, no pyarrow
                import ctypes as C

                from . import _native as N
                f.flush()
                L = N.lib()
                w = L.zn_index_writer_create(f.fileno(), out_cursor)
                for k, v in config_metadata().items():
                    L.zn_index_writer_metadata(w, k.encode(), v.encode())
                for key in sorted(groups):
                    rows = groups[key]
                    n = len(rows)
                    paths = (C.c_char_p * max(n, 1))(*[r[0].encode() for r in rows])
                    seq = np.array([r[1] for r in rows], np.uint32)
                    fo = np.array([r[2] for r in rows], np.uint64)
                    cp = np.array([int(r[3]) for r in rows], np.uint8)
                    us = np.array([r[4] for r in rows], np.uint64)
                    bo = np.array([r[5] for r in rows], np.uint64)
                    bs = np.array([r[6] for r in rows], np.uint64)
                    ck = np.frombuffer(b"".join(r[7] for r in rows), np.uint8) if n else np.zeros(1, np.uint8)
                    if L.zn_index_writer_push_group(w, key[0], key[1].encode(), n, paths, N.ptr(seq), N.ptr(fo), N.ptr(cp), N.ptr(us),
                                                    N.ptr(bo), N.ptr(bs), N.ptr(ck)) != 0:
                        raise IOError("zn_index_writer_push_group failed")
                if L.zn_index_writer_finish(w) != 0:
                    raise IOError("zn_index_writer_finish failed")
            else:
                schema = INDEX_SCHEMA.with_metadata(config_metadata())
                sink = ArrowIpcSink(f, out_cursor)
                for key in sorted(groups):
                    sink.push_subindex(key, schema, [build_metadata_batch(groups[key], schema)])
                sink.finish()
        return rep


def compress_stream(output: str, no_skip: bool, **kw) -> StreamCompressor:
    return StreamCompressor(output, no_skip, **kw)


def compress_dir(input_dir: str, output: str, no_skip: bool = False, level: int = 19, codec_id: int = codec.CODEC_ZSTD,
                 ctx: Ctx | None = None, envelope: bool = False, io_threads: int = 8, slot_bytes: int = 256 << 20) -> CompressionReport:
    """znippy-compress `compress_dir` (walk -> readers -> Magazine slots -> workers -> writer, slot_packer.rs:329-609) in
    one native call: `zn_archive_compress_dir` walks the directory, places every round in a pinned slot, lets
    `io_threads` readers pread the bytes into place, and runs the same three-stage slot pipeline as compress_stream.
    `level` as in compress_stream: 19 by default, 20-22 for the long effort."""
    import ctypes as C

    from . import _native as N
    ctx = ctx or default_ctx()
    out = os.path.splitext(output)[0] + ".znippy"
    rep8 = (C.c_uint64 * 8)()
    err = C.create_string_buffer(512)
    rc = N.lib().zn_archive_compress_dir(ctx.handle, input_dir.encode(), out.encode(), int(no_skip), level,
                                         codec_id | (N.CODEC_ENVELOPE if envelope else 0), slot_bytes, io_threads, C.byref(rep8), err, 512)
    if rc != 0:
        raise N.NativeError(f"zn_archive_compress_dir: {err.value.decode(errors='replace')}")
    return CompressionReport(*[int(x) for x in rep8])
