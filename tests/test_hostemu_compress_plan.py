"""The packed layout of device-resident compress plans (zn_plan_compress) on the CPU: the blob size the device computes
from the per-block results (cz::zstd_frame_size / cz::lz4_frame_size) and the ZNB1 header it writes (cz::znb1_header),
compiled for the host next to the emulated compressor (tests/host_emu/host_compress_plan.cpp).  The size must equal the
length of the frame the assemble step emits, at every effort and for LZ4, and the header must equal the one the archive
writer stores (zn_envelope_znb1_header)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

EMU = os.path.join(os.path.dirname(__file__), "host_emu")
sys.path.insert(0, os.path.dirname(__file__))
from test_hostemu_compress_long import corpora  # noqa: E402

# emulator codec ids: LZ4, the three zstd window efforts (levels <= 2, 3..9, 10..19), the long effort (levels >= 20)
EFFORTS = {"lz4": 2, "zstd-fast": 1, "zstd-mid": 11, "zstd-high": 12, "zstd-long": 20}


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu_plan") / "libhostemu_plan.so")
    srcs = [os.path.join(EMU, f) for f in ("host_compress_plan.cpp", "host_compress_long.cpp", "host_compress.cpp")]
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-x", "c++", *srcs, "-o", so, "-Wno-unknown-pragmas"],
                   check=True, capture_output=True)
    L = C.CDLL(so)
    L.zn_hostemu_frame_size.argtypes = [C.c_int, C.c_void_p, C.c_uint64]
    L.zn_hostemu_frame_size.restype = C.c_long
    L.zn_hostemu_compress.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]
    L.zn_hostemu_compress.restype = C.c_long
    L.zn_hostemu_compress_long.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    L.zn_hostemu_compress_long.restype = C.c_long
    L.zn_hostemu_znb1_header.argtypes = [C.c_uint32, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint32)]
    L.zn_hostemu_znb1_header.restype = C.c_uint32
    return L


@pytest.mark.parametrize("effort", list(EFFORTS))
def test_blob_size_from_block_results_equals_frame_length(emu, oracle, effort):
    codec = EFFORTS[effort]
    for name, d in corpora(oracle).items():
        src = np.zeros(d.size + 64, np.uint8)
        src[:d.size] = d
        out = np.zeros(d.size + d.size // 64 + 4096, np.uint8)
        if codec == 20:
            frame = emu.zn_hostemu_compress_long(src.ctypes.data, d.size, out.ctypes.data)
        else:
            frame = emu.zn_hostemu_compress(codec, src.ctypes.data, d.size, out.ctypes.data)
        assert frame > 0, name
        assert emu.zn_hostemu_frame_size(codec, src.ctypes.data, d.size) == frame, (effort, name)


@pytest.mark.parametrize("size", [0, 1, 127, 128, 16383, 16384, 1 << 21, 8 << 20, (1 << 32) - 1])
def test_device_znb1_header_equals_envelope_writer(emu, size):
    from znippy_b200 import codec
    for pc in (codec.PAYLOAD_RAW, codec.PAYLOAD_ZSTD, codec.PAYLOAD_LZ4_FRAME):
        want = codec.envelope_wrap(pc, size, b"")  # zn_envelope_znb1_header, as the archive writer calls it
        hdr = np.zeros(16, np.uint8)
        hl = C.c_uint32(0)
        n = emu.zn_hostemu_znb1_header(pc, size, hdr.ctypes.data, C.byref(hl))
        assert hdr[:n].tobytes() == want and hl.value == n == len(want), (pc, size)
