"""e2e lfr_solve() from pinned caller buffers (the zero-copy path), plus the host-side timeline of the
call (lfr_debug_last_host_marks).   python tools/gpu_e2e_timeline.py [cfg] [debug_flags]"""
import ctypes as C
import hashlib
import os
import sys
import time

import numpy as np

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)


def main(cfg, flags):
    import torch
    from lfr_b200 import build_problem, synth
    from lfr_b200.capi import load_b200
    import bench
    lib = load_b200()
    p = build_problem(synth.generate(cfg))
    s2, keep, pos_pinned, h2d = bench.pinned_problem(lib, p)
    opts = lib.default_options(debug_flags=flags)
    stt, bufs = lib.make_stats(p.n_components)
    marks = np.zeros(6)
    fm = lib.lib.lfr_debug_last_host_marks
    fm.argtypes = [C.c_void_p]
    ts, ks, hs, ms = [], [], [], []
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    n_it = 8 if cfg == "cfg5" else 34
    for it in range(n_it):
        pos_pinned.zero_()
        flush.fill_(it & 1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc = lib.lib.lfr_solve(C.byref(s2), C.byref(opts), pos_pinned.data_ptr(), C.byref(stt))
        t1 = time.perf_counter()
        lib.check(rc, "lfr_solve")
        if it >= 4:
            ts.append((t1 - t0) * 1e3); ks.append(stt.kernel_ms); hs.append(stt.h2d_ms)
            fm(marks.ctypes.data); ms.append(marks.copy())
    m = np.median(np.array(ms), axis=0)
    h = hashlib.sha1(pos_pinned.numpy().tobytes()).hexdigest()[:12]
    print("flags %d  e2e ms p50 %.4f min %.4f  kernels %.4f  h2d+schedule %.4f  host marks us %s  sha %s" % (
        flags, np.median(ts), np.min(ts), np.median(ks), np.median(hs), " ".join("%.0f" % v for v in m), h), flush=True)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "cfg2", int(sys.argv[2], 0) if len(sys.argv) > 2 else 0)
