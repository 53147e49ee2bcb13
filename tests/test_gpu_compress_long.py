"""The long effort of the zstd compressor on the GPU (levels >= 20, DESIGN.md §4.3): frames equal the host emulation's
bytes, do not depend on the batch, the run or the level within 20..22, decode everywhere, and read back through the
device-wide pipeline without a hand-back to the legacy decoder."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(__file__))
from test_hostemu_compress_long import MiB, corpora, emu, stdlib_text  # noqa: E402,F401  (emu: the host emulation fixture)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def codec():
    from znippy_b200 import codec as c
    c.default_ctx()
    return c


def _batch(datas, start=5, gap=3):
    """the slices back to back at misaligned source offsets"""
    offs, cur = [], start
    for d in datas:
        offs.append(cur)
        cur += len(d) + gap
    src = np.zeros(cur + 1, np.uint8)
    for o, d in zip(offs, datas):
        src[o:o + len(d)] = d
    return src, offs, [len(d) for d in datas]


def test_gpu_long_frames_equal_host_emulation(codec, oracle, emu):
    O = oracle
    cs = corpora(O)
    names = list(cs)
    datas = [cs[k] for k in names]
    src, offs, lens = _batch(datas)
    blobs, dg, st = codec.compress_batch(src, offs, lens, level=22)
    assert not st.any()
    z = O.libzstd()
    for name, d, b, g in zip(names, datas, blobs, dg):
        assert b == emu.compress(d), name  # the one-lane warp emits the 32-lane warp's bytes
        assert g.tobytes() == O.blake3(d.tobytes()), name
        assert len(b) <= codec.compress_bound(len(d)), name
        assert z.decompress(b, len(d)) == d.tobytes(), name
    for level in (20, 21):
        assert codec.compress_batch(src, offs, lens, level=level)[0] == blobs, level
    assert codec.compress_batch(src, offs, lens, level=22)[0] == blobs  # a second run
    # a slice alone equals the same slice in the mixed batch, wherever it sits
    for name in ("real", "stdlib8m", "len5", "len8m+17"):
        d = cs[name]
        alone, _, st1 = codec.compress_batch(d, [0], [len(d)], level=22)
        assert not st1.any() and alone[0] == blobs[names.index(name)], name
    # back through the GPU decoder, digests verified
    buf = np.frombuffer(b"".join(blobs), np.uint8)
    boffs = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])[:-1]
    ooff = np.concatenate([[0], np.cumsum(lens)])[:-1]
    out = np.zeros(sum(lens) + 1, np.uint8)
    st2, _ = codec.decode_verify_batch(buf, boffs, [len(b) for b in blobs], [1] * len(blobs), lens, dg.tobytes(), out, ooff)
    assert not st2.any()
    for i, d in enumerate(datas):
        assert out[ooff[i]:ooff[i] + len(d)].tobytes() == d.tobytes(), names[i]


def test_gpu_long_32_real_text_slices_through_plan(codec, oracle):
    """32 different 8 MiB rotations of the standard library's sources at level 22, read through Plan: every status
    OK, digests match, and the device-wide pipeline takes every frame (no legacy hand-back)."""
    import torch
    from znippy_b200 import Plan
    O = oracle
    contents = [stdlib_text(8 * MiB, k * 65_537) for k in range(32)]
    src, offs, lens = _batch(contents, 0, 0)
    blobs, dg, st = codec.compress_batch(src, offs, lens, level=22)
    assert not st.any()
    boff = np.concatenate([[0], np.cumsum([len(b) for b in blobs])])[:-1]
    buf = np.frombuffer(b"".join(blobs), np.uint8)
    out_len = np.array(lens, np.uint64)
    out_off = np.concatenate([[0], np.cumsum(out_len)])[:-1].astype(np.uint64)
    d_in = torch.from_numpy(buf.copy()).cuda()
    d_out = torch.zeros(int(out_len.sum()) + 256, dtype=torch.uint8, device="cuda")
    plan = Plan.decode_verify(codec.default_ctx(), boff, [len(b) for b in blobs], [1] * 32, out_off, out_len, dg.tobytes())
    plan.run(d_in.data_ptr(), d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    st2, dg2 = plan.results()
    assert st2.tolist() == [0] * 32
    assert plan.pipeline_fallbacks() == 0
    out = d_out.cpu().numpy()
    for i in (0, 7, 31):
        assert out[int(out_off[i]):int(out_off[i]) + lens[i]].tobytes() == contents[i].tobytes(), i
        assert dg2[i].tobytes() == O.blake3(contents[i].tobytes())


def test_gpu_long_500mib_binary(codec, oracle):
    """BASELINE configs[3] at full size and level 22: the degenerate-bucket case (a 251-byte period over 500 MiB)"""
    O = oracle
    total, sl = 500 << 20, 8 << 20
    src = O.gen_binary(total)
    offs = list(range(0, total, sl))
    lens = [min(sl, total - o) for o in offs]
    blobs, dg, st = codec.compress_batch(src, offs, lens, level=22)
    assert not st.any()
    for i in (0, 1, 31, len(offs) - 1):
        assert O.libzstd().decompress(blobs[i], lens[i]) == src[offs[i]:offs[i] + lens[i]].tobytes()
    assert total / sum(len(b) for b in blobs) > 1000


def test_gpu_long_archives_end_to_end(codec, oracle, tmp_path):
    from znippy_b200 import archive as A
    O = oracle
    files = {"a/real.py": stdlib_text(9 * MiB, 4242).tobytes(), "a/small.txt": b"level twenty-two " * 300,
             "b/empty.txt": b"", "b/noise.bin": O.gen_incompressible(1_000_000, 9).tobytes()}
    sc = A.compress_stream(str(tmp_path / "s.znippy"), False, level=22)
    for p, d in files.items():
        sc.sender().send(A.ArchiveEntry(p, d))
    sc.finish()
    vr = A.decompress_archive(sc.output, True, str(tmp_path / "xs"))
    assert vr.total_files == len(files) and vr.corrupt_files == 0
    for p, d in files.items():
        assert (tmp_path / "xs" / p).read_bytes() == d, p
    assert A.ZnippyArchive.open(sc.output).extract_files(list(files)) == list(files.values())
    # compress_dir over the same tree
    src_dir = tmp_path / "tree"
    for p, d in files.items():
        (src_dir / p).parent.mkdir(parents=True, exist_ok=True)
        (src_dir / p).write_bytes(d)
    A.compress_dir(str(src_dir), str(tmp_path / "d.znippy"), level=22)
    vr = A.decompress_archive(str(tmp_path / "d.znippy"), True, str(tmp_path / "xd"))
    assert vr.total_files == len(files) and vr.corrupt_files == 0
    assert A.ZnippyArchive.open(str(tmp_path / "d.znippy")).extract_files(list(files)) == list(files.values())
    # envelope: incompressible rows still stored RAW inside the envelope (size + 8 bytes of header)
    se = A.compress_stream(str(tmp_path / "e.znippy"), False, envelope=True, level=22)
    for p, d in files.items():
        se.sender().send(A.ArchiveEntry(p, d))
    se.finish()
    t = A.read_znippy_index(se.output)
    rows = dict(zip(t.column("relative_path").to_pylist(), t.column("blob_size").to_pylist()))
    assert rows["b/noise.bin"] == 1_000_000 + 4 + 1 + 3
    assert rows["a/small.txt"] < len(files["a/small.txt"]) // 10
    vr = A.decompress_archive(se.output, True, str(tmp_path / "xe"))
    assert vr.corrupt_files == 0
    for p, d in files.items():
        assert (tmp_path / "xe" / p).read_bytes() == d, p
