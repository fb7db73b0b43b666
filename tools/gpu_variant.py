"""A/B of two or more builds of the product library: per library and workload, the median
device-resident solve time (lfr_plan_solve on a plan in HBM, CUDA events, L2 overwritten before each
solve) and a SHA-1 of the positions and iteration counts the solve returns.  Libraries take turns
round by round, so drift of the card or of other work on the host affects them alike.

    python tools/gpu_variant.py <a.so> <b.so> [...] [--workloads cfg2,cfg3,cfg4] [--rounds 15] [--per-round 3]

Relative library paths are taken from the current directory."""
import argparse
import hashlib
import os
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from lfr_b200 import build_problem, synth  # noqa: E402
from lfr_b200 import capi  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="+")
    ap.add_argument("--workloads", default="cfg2,cfg3,cfg4")
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--per-round", type=int, default=3)
    args = ap.parse_args()
    libs = [capi.Library(os.path.abspath(path)) for path in args.libs]
    names = args.workloads.split(",")
    s = torch.cuda.current_stream().cuda_stream
    plans = {}
    for name in names:
        p = build_problem(synth.generate(name))
        for li, lib in enumerate(libs):
            plan = capi.Plan(lib, p)
            for _ in range(3):
                plan.solve(s)
            plans[li, name] = plan
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    times = {k: [] for k in plans}
    for r in range(args.rounds):
        for name in names:
            for j in range(len(libs)):
                li = (r + j) % len(libs)
                for _ in range(args.per_round):
                    flush.fill_(r & 1)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    plans[li, name].solve(s)
                    b.record()
                    torch.cuda.synchronize()
                    times[li, name].append(a.elapsed_time(b))
    for name in names:
        for li, path in enumerate(args.libs):
            pos, st = plans[li, name].download(s)
            sha = hashlib.sha1(pos.tobytes() + np.ascontiguousarray(st["iterations"]).tobytes()).hexdigest()[:16]
            ts = np.array(times[li, name])
            print("%-10s %-28s median %9.4f ms  min %9.4f  p10 %9.4f  p90 %9.4f  n %3d  sha1 %s" % (
                name, os.path.basename(path), np.median(ts), ts.min(), np.percentile(ts, 10), np.percentile(ts, 90),
                ts.size, sha), flush=True)
    for plan in plans.values():
        plan.close()


if __name__ == "__main__":
    main()
