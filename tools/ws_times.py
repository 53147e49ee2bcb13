"""Development: phase stamps of the warp-specialised fused kernel on the bench workload.  Needs a library built with
-DZN_WS_DEBUG copied over znippy_b200/libznippy_cuda.so (tools/bin/variants/lib_wsdebug.so)."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from znippy_b200 import Ctx, Plan, _native as N

blobs, lens, digs, comp, _ = bench.build_workload("text2g", 2.0, 0)
in_buf, in_off = bench.pack(blobs, 16)
in_len = np.array([len(b) for b in blobs], np.uint64)
out_len = np.array(lens, np.uint64)
out_off = np.concatenate([[0], np.cumsum((out_len + np.uint64(15)) & ~np.uint64(15))])[:-1].astype(np.uint64)
ctx = Ctx(0, staging_bytes=1 << 20)
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)
d_in = torch.from_numpy(in_buf).cuda()
d_out = torch.empty(int(out_off[-1] + out_len[-1]) + 256, dtype=torch.uint8, device="cuda")
plan = Plan.decode_verify(ctx, in_off, in_len, comp, out_off, out_len, digs)
L = N.lib()
L.zn_debug_ws_times.argtypes = [C.POINTER(C.c_ulonglong), C.c_int]
out = (C.c_ulonglong * 4)()
for rep in range(4):
    L.zn_debug_ws_times(out, 1)
    plan.run(d_in.data_ptr(), d_out.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    L.zn_debug_ws_times(out, 0)
    t0, td, th, tiles = out[0], out[1], out[2], out[3]
    print(f"rep {rep}: decode phase {1e-6 * (td - t0):.3f} ms, kernel {1e-6 * (th - t0):.3f} ms, tiles taken by the end of decode {tiles} of {sum((l + 32767) // 32768 for l in lens)}, stages {plan.last_ms()}")
st, _ = plan.results()
print("status any:", bool(st.any()))
