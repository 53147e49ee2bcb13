"""The long effort of the zstd compressor (levels >= 20: whole-slice match finding, DESIGN.md §4.3) on the CPU: the
warp-uniform code of znippy_b200/csrc/compress.cuh with a warp of one lane (tests/host_emu/host_compress_long.cpp),
which emits the same bytes as the GPU.  Frames must decode with stock libzstd, the oracle and the device-wide decode
pipeline's logic, and the ratio must approach libzstd level 19's."""
import ctypes as C
import os
import subprocess
import sys
import sysconfig

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(os.path.dirname(__file__), "host_emu")
MiB = 1 << 20


def stdlib_text(n: int, rotate: int = 0) -> np.ndarray:
    """n bytes of the standard library's .py sources (recursive, in a fixed order), rotated by `rotate` bytes.  The
    sources hold about 10 MiB, so an 8 MiB slice never repeats inside itself (a cycled corpus would let the long window
    find the cycle and overstate the ratio)."""
    root = sysconfig.get_paths()["stdlib"]
    parts = []
    for dirpath, dirs, files in os.walk(root):
        dirs.sort()
        parts += [open(os.path.join(dirpath, f), "rb").read() for f in sorted(files) if f.endswith(".py")]
    data = b"".join(parts)
    assert len(data) > n, (len(data), n)
    r = rotate % len(data)
    return np.frombuffer((data[r:] + data[:r])[:n], np.uint8).copy()


def long_repeat() -> np.ndarray:
    """1 MiB random R, 3 MiB random, R again: the second R sits 4 MiB back, an offset above 2^20"""
    rng = np.random.default_rng(11)
    r = rng.integers(0, 256, MiB, dtype=np.uint8)
    return np.concatenate([r, rng.integers(0, 256, 3 * MiB, dtype=np.uint8), r])


def corpora(O) -> dict:
    """The corpora of test_gpu_compress plus the shapes the long effort has to get right"""
    sys.path.insert(0, os.path.dirname(__file__))
    from test_gpu_compress import _cases
    c = dict(_cases(O))
    c["stdlib8m"] = stdlib_text(8 * MiB)
    c["zeros8m"] = np.zeros(8 * MiB, np.uint8)
    for p in (1, 2, 3, 4):
        c[f"period{p}"] = np.resize(np.arange(1, p + 1, dtype=np.uint8) * 37, 2 * MiB)
    c["longrep"] = long_repeat()
    for n in (0, 1, 3, 4, 5, 128 * 1024 - 1, 128 * 1024 + 1):
        c[f"len{n}"] = stdlib_text(n, 12345)
    c["len8m+17"] = stdlib_text(8 * MiB + 17, 777)
    return c


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu_long") / "libhostemu_long.so")
    srcs = [os.path.join(EMU, f) for f in ("host_compress_long.cpp", "host_compress.cpp", "host_decode.cpp")]
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-x", "c++", *srcs, "-o", so, "-Wno-unknown-pragmas"],
                   check=True, capture_output=True)
    L = C.CDLL(so)
    L.zn_hostemu_compress_long.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    L.zn_hostemu_compress_long.restype = C.c_long
    L.zn_hostemu_compress.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]
    L.zn_hostemu_compress.restype = C.c_long
    L.zn_hostemu_decode_pipe.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]

    class E:
        @staticmethod
        def compress(d, codec=None):
            """codec None: the long effort; 12: the level-10..19 effort"""
            src = np.zeros(d.size + 64, np.uint8)
            src[:d.size] = d
            out = np.zeros(d.size + d.size // 64 + 4096, np.uint8)
            if codec is None:
                r = L.zn_hostemu_compress_long(src.ctypes.data, d.size, out.ctypes.data)
            else:
                r = L.zn_hostemu_compress(codec, src.ctypes.data, d.size, out.ctypes.data)
            return out[:r].tobytes()

        @staticmethod
        def decode_pipe(blob, cap):
            """0 = the device-wide pipeline's logic decodes the blob, 1 = it would hand the blob to the legacy decoder"""
            a = np.frombuffer(blob, np.uint8)
            out = np.zeros(max(cap, 1) + 64, np.uint8)
            stats = np.zeros(4, np.uint64)
            rc = L.zn_hostemu_decode_pipe(a.ctypes.data, a.size, out.ctypes.data, cap, stats.ctypes.data)
            return rc, out[:cap].tobytes()
    return E


@pytest.fixture(scope="module")
def frames(emu, oracle):
    cs = corpora(oracle)
    return cs, {k: emu.compress(d) for k, d in cs.items()}


def test_long_frames_decode_everywhere(emu, oracle, frames):
    O = oracle
    cs, fr = frames
    z = O.libzstd()
    for name, d in cs.items():
        b = fr[name]
        assert z.decompress(b, len(d)) == d.tobytes(), name
        rc, o = O.zstd_decompress(b, len(d))
        assert rc == 0 and o == d.tobytes(), name
    assert fr["len0"].hex() == "28b52ffd2000010000"  # same bytes as libzstd
    for name in ("stdlib8m", "real", "longrep", "len8m+17", "zeros8m"):  # whole 8 MiB slices read through the pipeline
        rc, o = emu.decode_pipe(fr[name], len(cs[name]))
        assert rc == 0 and o == cs[name].tobytes(), name


def test_long_ratio_against_libzstd_19(emu, oracle, frames):
    """Real text: <= 1.20 x libzstd-19 (the level-10..19 effort gives 1.47 x); pattern corpora <= 1.10 x; every corpus
    at most 1 % (+ 64 bytes) above the level-19 effort; the 4 MiB-back repeat costs nothing beyond the random bytes."""
    O = oracle
    cs, fr = frames
    z = O.libzstd()
    real = O.real_text(2_000_000)
    ours, ref = len(emu.compress(real)), len(z.compress(real, 19))
    print(f"real text 2 MB: long effort {ours} B = {ours / ref:.3f} x libzstd-19 ({ref} B)")
    assert ours <= 1.20 * ref, (ours, ref, ours / ref)
    for name, d in [("text", O.gen_text(8 * MiB)), ("binary", O.gen_binary(8 * MiB))]:
        ours, ref = len(emu.compress(d)), len(z.compress(d, 19))
        assert ours <= 1.10 * ref + 16, (name, ours, ref)
    for name, d in cs.items():
        assert len(fr[name]) <= 1.01 * len(emu.compress(d, 12)) + 64, (name, len(fr[name]), len(emu.compress(d, 12)))
    assert len(fr["longrep"]) <= 4 * MiB + 64 * 1024, len(fr["longrep"])
