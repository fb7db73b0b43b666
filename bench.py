#!/usr/bin/env python3
"""bench.py — tracks-refined/s of the multi-view refinement solve on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl reference] [--dump-outputs DIR]

A step = one complete solve of the workload's match graph (every component,
LM to termination).  At N=1 the workload is BASELINE.json configs[1]
(Fountain-scale synthetic: 11 images x 3000 keypoints, exhaustive pairs).  For
N>1 (torchrun, one rank per GPU) every rank solves its own Fountain-scale scene
(weak scaling: independent components, no data-path collective — SURVEY 8e);
`value` = tracks of all ranks / max-over-ranks time.

  value     device-resident plan (inputs already in HBM), CUDA events per step on
            the launching stream, L2 flushed between steps (untimed)
  e2e       the same solve through the C-ABI call lfr_solve() with pinned HOST
            buffers: host->device copies, kernels and device->host results inside
            the timed region
  roofline  algorithmic bytes (sum_c iters_c (80 E_c + 36 N_c), SURVEY 8d) / kernel time
            against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the CPU oracle (oracle/lfr_oracle.cc, the specialised restatement) on the host
            cores: all cores, the reference's default 8 threads (solve.cc:384) and 1 thread
  total_scope   host graph stage (tracks, roots, cut, dispatch: solve.cc:487-606) + solve = the
            reference's "Total time" scope (solve.cc:487-641), for the B200 path and for the CPU

--impl reference times the reference's OWN solve: oracle/_ref/solve_O2 = multi-view-refinement/
solve.cc + cost.cc + graph.cc compiled unmodified (-O2) against the shim headers of oracle/ref_shims/
(Ceres' minimizer restated, see oracle/build_ref.py), on all host cores, "Solver time" scope
(thread pool creation -> Wait(), solve.cc:615-638, measured in microseconds by the pool shim).
Falls back to the oracle port when that binary was not built.

--dump-outputs DIR writes what the last timed step computed, the arrays lfr_plan_download() hands the
caller, as DIR/<name>.npy in float64: positions [N, 2] and, per component slot, iterations,
termination, initial_cost and final_cost (at N>1 with a _rank<r> suffix per rank).  The workload is
generated from a fixed seed, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "tracks_refined_per_s"
UNIT = "tracks/s"
WORKLOADS = {
    "cfg1": "cfg1 synthetic 3 images x 200 kpts, exhaustive pairs",
    "cfg2": "cfg2 Fountain-scale synthetic: 11 images x 3000 kpts, exhaustive pairs",
    "cfg3": "cfg3 Herzjesu-scale synthetic: 8 images x 8000 kpts, exhaustive pairs",
    "cfg4": "cfg4 ETH3D-courtyard-scale synthetic: 38 images x 4000 kpts, sequential+loop pairs",
    "cfg5": "cfg5 Madrid-Metropolis-scale synthetic: 1000 images x 2000 kpts, ring+random pairs",
}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(workload):
    """DRAM bytes per step of the solve kernels from the committed ncu capture of this
    workload (profiles/traffic.json), or None when none was taken."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get("dram_bytes_per_step", {}).get(workload)
    except Exception:
        return None


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays, suffix=""):
    """Writes each array as out_dir/<name><suffix>.npy in float64.  Above DUMP_LIMIT bytes in all, every
    array keeps a fixed, seeded sample of its rows (ascending), and <name><suffix>_rows.npy says which."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT:
            # half the limit for the sampled rows, at most as much again for their indices
            k = int(a.shape[0] * (DUMP_LIMIT // 2) / total)
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], size=k, replace=False))
            np.save(os.path.join(out_dir, name + suffix + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def build_workload(name, seed=None):
    from lfr_b200 import build_problem, refined_track_count, synth
    ms = synth.generate(name, seed=seed)
    p = build_problem(ms)
    return p, refined_track_count(p)


def workload_config(name, p, n_tracks, n_gpus=1):
    """The same keys and values from both arms (the driver compares the two configs)."""
    sizes = np.diff(p.comp_ptr.astype(np.int64))
    return {"workload": WORKLOADS.get(name, name), "nodes": int(p.graph.n_nodes),
            "directed_edges": int(p.graph.n_edges), "tracks": int(p.info.get("n_tracks", 0)),
            "tracks_refined": int(n_tracks), "components_solved": int((sizes > 1).sum()),
            "max_component_nodes": int(sizes.max()) if sizes.size else 0,
            "per_gpu": "one scene per GPU" if n_gpus > 1 else "single scene",
            "l2": "flushed between timed steps (256 MiB write, untimed)"}


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region.  The region is tens of
    milliseconds, so the primary sampler is an NVML thread (pynvml, back-to-back queries);
    `nvidia-smi -lms` is the fallback when NVML cannot be opened."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        import threading
        self.sm, self.ts, self.reasons, self.smax = [], [], set(), None
        self.t0 = self.t1 = None   # timed region (perf_counter), set by mark_begin / mark_end
        self.p = self.f = self.thread = None
        self.source = "none"
        self._stop = threading.Event()
        try:
            import pynvml as nv
            nv.nvmlInit()
            # CUDA_VISIBLE_DEVICES remaps cuda indices; resolve through the PCI bus id
            import torch
            bus = torch.cuda.get_device_properties(device).pci_bus_id if hasattr(
                torch.cuda.get_device_properties(device), "pci_bus_id") else None
            h = None
            if bus is not None:
                for i in range(nv.nvmlDeviceGetCount()):
                    hh = nv.nvmlDeviceGetHandleByIndex(i)
                    if nv.nvmlDeviceGetPciInfo(hh).bus == bus:
                        h = hh
                        break
            if h is None:
                h = nv.nvmlDeviceGetHandleByIndex(device)
            self.smax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                     ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                     ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap))

            def run():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                        self.ts.append(time.perf_counter())
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                        for nm, bit in names:
                            if r & bit:
                                self.reasons.add(nm)
                    except Exception:
                        pass
                    time.sleep(0.0002)   # the NVML queries themselves take a few ms

            self.thread = threading.Thread(target=run, daemon=True)
            self.source = "nvml thread, back-to-back queries"
        except Exception:
            self.thread = None
            try:
                self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q,
                                           "--format=csv,noheader,nounits", "-lms", "20"],
                                          stdout=self.f, stderr=subprocess.DEVNULL)
                self.source = "nvidia-smi -lms 20"
                time.sleep(0.5)   # nvidia-smi needs a few hundred ms before its first line
            except Exception:
                self.p = None

    def start(self):
        """Call before the warm-up: the GPU runs the same steps there as in the timed region, and a
        region of ~10 ms alone may see only one or two NVML answers."""
        if self.thread is not None:
            self.thread.start()

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.thread is not None:
            self._stop.set()
            self.thread.join(timeout=2)
            sm, smax = self.sm, ([self.smax] if self.smax else [])
        elif self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
            self.f.flush()
            self.f.seek(0)
            sm, smax = [], []
            for line in self.f.read().splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1]))
                    smax.append(float(c[2]))
                except ValueError:
                    continue
                for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 c[5:9]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            os.unlink(self.f.name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"], "samples": 0}
        in_timed = sum(1 for t in self.ts if self.t0 is not None and self.t1 is not None and self.t0 <= t <= self.t1)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None, "reasons": sorted(self.reasons),
                "samples": len(sm), "samples_in_timed_region": in_timed,
                "window": "warm-up + device-timed region", "source": self.source}


def pinned_problem(lib, p):
    """Marshal the problem into pinned host buffers (what a host application
    hands to lfr_solve)."""
    import ctypes as C
    import torch
    from lfr_b200.capi import LfrProblem
    s, arrays = lib.marshal(p)
    pinned = {}
    for k, a in arrays.items():
        raw = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        t = torch.empty(max(raw.size, 1), dtype=torch.uint8).pin_memory()
        t.numpy()[:raw.size] = raw
        pinned[k] = t
    s2 = LfrProblem(n_nodes=s.n_nodes, n_components=s.n_components, n_edges=s.n_edges,
                    **{k: t.data_ptr() for k, t in pinned.items()})
    N = p.graph.n_nodes
    pos = torch.zeros(max(2 * N, 1), dtype=torch.float64).pin_memory()
    h2d = sum(int(np.ascontiguousarray(a).nbytes) for a in arrays.values()) + 16 * N
    return s2, pinned, pos, h2d


def reference_binary():
    """oracle/_ref/solve_O2 (built by oracle/build_ref.py where /root/reference exists; shipped to the
    GPU box as a file), or None."""
    path = os.path.join(ROOT, "oracle", "_ref", "solve_O2")
    return path if os.path.exists(path) and os.access(path, os.X_OK) else None


def time_reference_binary(exe, matches_path, n_threads, repeats, tmpdir):
    """Runs the reference's main() `repeats` times; returns (solver_ms list, total_ms list, graph_cut_ms
    list, iterations-independent): "Solver time" scope from the pool shim's microsecond timer,
    "Total time" / "Graph-cut time" from the program's own stdout (whole milliseconds)."""
    solver, total, cut = [], [], []
    timing = os.path.join(tmpdir, "pool_timing.txt")
    for _ in range(repeats):
        if os.path.exists(timing):
            os.unlink(timing)
        env = dict(os.environ, LFR_POOL_TIMING_FILE=timing)
        r = subprocess.run([exe, "--matches_file", matches_path, "--output_file", os.path.join(tmpdir, "ref_solution.pb"),
                            "--n_threads", str(n_threads)], capture_output=True, text=True, env=env)
        if r.returncode != 0:
            raise RuntimeError("reference binary failed: %s" % r.stderr[-300:])
        with open(timing) as fh:
            solver.append(float(fh.read().split()[0]))
        for line in r.stdout.splitlines():
            if line.startswith("Total time:"):
                total.append(float(line.split()[2].rstrip("ms")))
            if line.startswith("Graph-cut time:"):
                cut.append(float(line.split()[2].rstrip("ms")))
    return solver, total, cut


def run_reference(args):
    """Reference arm: the reference's own CPU solve on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    # the B200 arm at --gpus N solves N scenes (one per GPU, weak scaling): same work here
    from lfr_b200 import build_problem, refined_track_count, synth, wire
    base_seed = synth.CONFIGS[synth.ALIASES.get(args.workload, args.workload)].seed
    tmpdir = tempfile.mkdtemp(prefix="lfr_ref_")
    scenes = []
    for r in range(max(1, args.gpus)):
        ms = synth.generate(args.workload, seed=(base_seed + 7919 * r) if args.gpus > 1 else None)
        p = build_problem(ms)                       # host utilities only (csrc/liblfr_host.so): no CUDA library is mapped
        path = os.path.join(tmpdir, "matches_%d.pb" % r)
        with open(path, "wb") as fh:
            fh.write(wire.encode_matching_file(ms))
        scenes.append((p, refined_track_count(p), path))
    p0 = scenes[0][0]
    n_tracks = sum(t for _, t, _ in scenes)
    exe = reference_binary()
    warm = max(args.warmup, 3)
    extra = {}
    if exe is not None:
        kind = "reference"
        for _, _, path in scenes:
            time_reference_binary(exe, path, cores, warm, tmpdir)
        per_scene = [time_reference_binary(exe, path, cores, args.steps, tmpdir) for _, _, path in scenes]
        t = [sum(ps[0][k] for ps in per_scene) / 1e3 for k in range(args.steps)]          # seconds per step
        tot = [sum(ps[1][k] for ps in per_scene) for k in range(args.steps)]
        eight = time_reference_binary(exe, scenes[0][2], 8, min(args.steps, 5), tmpdir)
        one = time_reference_binary(exe, scenes[0][2], 1, 1, tmpdir)
        extra = {"total_scope_ms_per_step": float(np.median(tot)),
                 "graph_cut_ms": float(np.median(per_scene[0][2])) if per_scene[0][2] else None,
                 "eight_thread_ms_per_scene": float(np.median(eight[0])), "single_thread_ms_per_scene": float(one[0][0])}
        sample = ("whole workload x %d steps: oracle/_ref/solve_O2 = the reference's solve.cc + cost.cc + graph.cc "
                  "compiled unmodified (-O2; the reference's own build sets no -O flag) against shim headers, "
                  "Ceres' minimizer restated (oracle/ref_shims/mini_ceres.cc); 'Solver time' scope" % args.steps)
        from_oracle = None
    else:
        kind = "port"
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from oracle_util import load_oracle
        orc = load_oracle()
        o = orc.default_options(n_threads=cores)
        for _ in range(warm):
            for q, _, _ in scenes:
                orc.solve(q, o)
        t = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            for q, _, _ in scenes:
                orc.solve(q, o)
            t.append(time.perf_counter() - t0)
        sample = ("whole workload x %d steps: Ceres-1.14-semantics CPU oracle (oracle/lfr_oracle.cc, -O2); "
                  "oracle/_ref/solve_O2 was not built" % args.steps)
    # median of the K steps: the host-side pool is sensitive to other tenants of the box; the median
    # is the conservative (faster) reading of the reference
    ms = 1e3 * float(np.median(t))
    value = n_tracks / (ms / 1e3)
    cpu = {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
    cpu.update(extra)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms, "ms_per_step_mean": 1e3 * float(np.mean(t)),
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, p0, scenes[0][1], args.gpus),
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    import shutil
    shutil.rmtree(tmpdir, ignore_errors=True)
    return 0


def sharded_record(lib, world, args):
    """BASELINE.json configs[3] (cfg4, N <= 4) / configs[4] (cfg5, N = 8): ONE scene whose components
    are LPT-packed over the N GPUs by lfr_solve_multi() (include/lfr.h) — one C-ABI call from one
    process, page-locked host arrays, every device pulling only its own components' edge records and
    writing its results straight back: no data-path collective, nothing to gather.  Timed against the
    same call on one device (strong scaling)."""
    import ctypes as C
    import torch
    from lfr_b200 import build_problem, refined_track_count, synth
    from lfr_b200.capi import LfrMultiInfo
    name = os.environ.get("LFR_BENCH_SHARDED_WORKLOAD") or ("cfg4" if world <= 4 else "cfg5")
    t0 = time.perf_counter()
    p = build_problem(synth.generate(name))
    t_build = time.perf_counter() - t0
    n_tracks = refined_track_count(p)
    s2, keep, pos_pinned, h2d = pinned_problem(lib, p)
    opts = lib.default_options()
    stt, bufs = lib.make_stats(p.n_components)

    def run(devices, reps):
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        info = LfrMultiInfo()
        wall, kern = [], []
        for i in range(2 + reps):
            pos_pinned.zero_()
            for d in devices:
                torch.cuda.synchronize(d)
            t1 = time.perf_counter()
            rc = lib.lib.lfr_solve_multi(C.byref(s2), C.byref(opts), dev.ctypes.data, len(devices),
                                         pos_pinned.data_ptr(), C.byref(stt), C.byref(info))
            dt = time.perf_counter() - t1
            lib.check(rc, "lfr_solve_multi")
            if i >= 2:
                wall.append(dt)
                kern.append(list(info.kernel_ms)[:len(devices)])
        pos = pos_pinned.numpy()[:2 * p.graph.n_nodes].copy()
        return 1e3 * float(np.median(wall)), np.median(np.array(kern), axis=0), pos, info, bufs["iterations"].copy()

    reps = 5
    ms1, k1, pos1, _, it1 = run([0], reps)
    msN, kN, posN, info, itN = run(list(range(world)), reps)
    sizes = np.diff(p.comp_ptr.astype(np.int64))
    return {
        "workload": WORKLOADS.get(name, name), "n_gpus": world, "api": "lfr_solve_multi() (include/lfr.h), page-locked host arrays",
        "nodes": int(p.graph.n_nodes), "directed_edges": int(p.graph.n_edges), "components_solved": int((sizes > 1).sum()),
        "max_component_nodes": int(sizes.max()), "tracks_refined": int(n_tracks),
        "one_gpu": {"ms_per_solve": ms1, "kernel_ms": float(k1[0]), "tracks_per_s": n_tracks / (ms1 / 1e3)},
        "n_gpu": {"ms_per_solve": msN, "kernel_ms_max": float(np.max(kN)), "kernel_ms_per_device": [float(x) for x in kN],
                  "tracks_per_s": n_tracks / (msN / 1e3), "components_per_device": list(info.n_slots)[:world],
                  "edges_per_device": list(info.n_edges)[:world], "zero_copy": int(info.zero_copy)},
        "strong_scaling_efficiency": ms1 / (world * msN),
        "strong_scaling_efficiency_kernels": float(k1[0]) / (world * float(np.max(kN))),
        "gather_ms": 0.0, "collective": "none: components never span devices; results are written straight into the caller's page-locked array",
        "bitwise_identical_to_one_gpu": bool(np.array_equal(pos1, posN) and np.array_equal(it1, itN)),
        "timing": "host wall clock around the call, median of %d (2 warm-up calls)" % reps,
        "scene_build_s": t_build, "h2d_bytes_if_copied": int(h2d),
    }


def run_b200(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from lfr_b200.capi import Plan, load_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the solve has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = load_b200()
    opts = lib.default_options(device=local, debug_flags=args.debug_flags)
    # weak scaling: rank r solves its own scene (seed offset), same shape
    from lfr_b200 import synth
    base_seed = synth.CONFIGS[synth.ALIASES.get(args.workload, args.workload)].seed
    p, n_tracks = build_workload(args.workload, seed=base_seed + 7919 * rank if world > 1 else None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    plan = Plan(lib, p, opts)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        plan.solve(stream)
    torch.cuda.synchronize()
    # ---- value: device-resident, CUDA events per step ---------------------------------
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    if sampler:
        sampler.mark_begin()
    for a, b in ev:
        flush.zero_()
        a.record()
        plan.solve(stream)
        b.record()
    barrier()
    if sampler:
        sampler.mark_end()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    ms_per_step = float(np.mean(step_ms))
    ms_per_step_median = float(np.median(step_ms))
    pos, st = plan.download(stream)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(positions=pos, **{k: st[k] for k in ("iterations", "termination",
                                                                                  "initial_cost", "final_cost")}),
                     suffix="_rank%d" % rank if world > 1 else "")
    alg_bytes, one_pass = plan.traffic(stream)
    launches = plan.num_launches()
    # clocks are sampled over warm-up + the device-timed region; the sampler stops before the
    # host-timed e2e leg so that its polling cannot perturb it
    clocks = sampler.stop() if sampler else None
    # ---- e2e: C-ABI call with pinned host buffers ------------------------------------------
    s2, keep, pos_pinned, h2d = pinned_problem(lib, p)
    stt, bufs = lib.make_stats(p.n_components)
    d2h = 16 * p.graph.n_nodes + 8 * p.n_components
    e2e_t = []
    e2e_parts = []
    for i in range(args.warmup + args.steps):
        pos_pinned.zero_()
        flush.zero_()
        barrier()
        t0 = time.perf_counter()
        rc = lib.lib.lfr_solve(C.byref(s2), C.byref(opts), pos_pinned.data_ptr(), C.byref(stt))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        lib.check(rc, "lfr_solve")
        if i >= args.warmup:
            e2e_t.append(dt)
            e2e_parts.append((stt.h2d_ms, stt.kernel_ms, stt.d2h_ms))
    e2e_ms = 1e3 * float(np.median(e2e_t))   # host wall clock: median over the K steps (robust to host jitter)
    e2e_ms_mean = 1e3 * float(np.mean(e2e_t))
    if os.environ.get("LFR_BENCH_DEBUG"):
        sys.stderr.write("e2e steps ms: %s\nparts: %s\n" % ([round(1e3 * x, 3) for x in e2e_t], [[round(y, 3) for y in x] for x in e2e_parts]))
    e2e_break = [float(x) for x in np.median(np.array(e2e_parts), axis=0)]   # medians, like e2e_ms
    # ---- reduce over ranks --------------------------------------------------------------------
    tot_tracks, tot_iters, tot_alg = n_tracks, int(st["total_iterations"]), alg_bytes
    if world > 1:
        t = torch.tensor([ms_per_step, e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step, e2e_ms = float(t[0]), float(t[1])
        c = torch.tensor([n_tracks, tot_iters, alg_bytes], dtype=torch.float64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        tot_tracks, tot_iters, tot_alg = int(c[0]), int(c[1]), int(c[2])
    # ---- N > 1: the PARTITION path (north star: components of ONE scene partitioned across the GPUs) --
    sharded = None
    if world > 1 and os.environ.get("LFR_BENCH_SHARDED", "1") != "0":
        # the other ranks idle while rank 0 drives all N devices through one C-ABI call.  They must wait on
        # the HOST (rendezvous store), not in dist.barrier(): an NCCL barrier is a kernel spinning on every
        # waiting rank's GPU, which measurably slows the solve running there (4.6 vs 2.1 ms on cfg4 / 2 GPUs)
        import datetime
        store = dist.distributed_c10d._get_default_store()
        torch.cuda.synchronize()
        dist.barrier()               # every rank is done with its own timed work
        torch.cuda.synchronize()
        if rank == 0:
            try:
                sharded = sharded_record(lib, world, args)
            except Exception as e:   # never lose the main line over the extra record
                sharded = {"error": repr(e)[:300]}
            store.set("lfr_sharded_done", "1")
        else:
            store.wait(["lfr_sharded_done"], datetime.timedelta(minutes=30))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    value = tot_tracks / (ms_per_step / 1e3)
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (ms_per_step / 1e3) / 1e9     # per GPU (rank 0's solve kernels)
    # ---- cpu baseline: oracle on the host cores, bounded sample -------------------------------
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_util import load_oracle
    orc = load_oracle()
    cores = os.cpu_count() or 1
    oo = orc.default_options(n_threads=cores)
    cpu_t = []
    t0 = time.perf_counter()
    while len(cpu_t) < 5 or (time.perf_counter() - t0 < 6.0 and len(cpu_t) < 300):
        t1 = time.perf_counter()
        orc.solve(p, oo)
        cpu_t.append(time.perf_counter() - t1)
    reps = len(cpu_t)
    cpu_ms = 1e3 * float(np.median(cpu_t))   # median: robust to host-side noise at start-up
    t1 = time.perf_counter()
    orc.solve(p, orc.default_options(n_threads=1))   # per-core figure (SURVEY 8d)
    cpu_1t_ms = 1e3 * (time.perf_counter() - t1)
    o8 = orc.default_options(n_threads=8)            # the reference's default --n_threads (solve.cc:384)
    c8 = []
    for _ in range(7):
        t1 = time.perf_counter()
        orc.solve(p, o8)
        c8.append(time.perf_counter() - t1)
    cpu_8t_ms = 1e3 * float(np.median(c8))
    # "Total time" scope (solve.cc:487-641): tracks + roots + graph cut + dispatch + solve.  Host stage =
    # csrc/lfr_host.cc (single-threaded C++), timed by its own phase clocks over 5 runs.
    from lfr_b200 import build_problem, synth
    ms_scene = synth.generate(args.workload, seed=base_seed + 7919 * rank if world > 1 else None)
    hs = []
    for _ in range(5):
        q = build_problem(ms_scene)
        hs.append(q.info["tracks_ms"] + q.info["graph_cut_ms"] + q.info["dispatch_ms"])
    host_stage_ms = float(np.median(hs))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, p, n_tracks, world),
        "lm_iterations_per_step": int(st["total_iterations"]),
        "lm_iters_per_s": tot_iters / (ms_per_step / 1e3),
        "ms_per_step_median": ms_per_step_median,
        "e2e": {"value": tot_tracks / (e2e_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_ms,
                "ms_per_step_mean": e2e_ms_mean, "timing": "host wall clock around the call, median of K steps",
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "api": "lfr_solve() (include/lfr.h) with pinned host buffers",
                "stages_ms": {"h2d_and_schedule": e2e_break[0], "kernels": e2e_break[1], "d2h": e2e_break[2]}},
        "gpu_launches": int(launches * args.steps),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": ncu_traffic(args.workload),
                     "peak_source": "%s HBM copy bandwidth (burst)" % peak_src,
                     "algorithmic_bytes_per_step": int(alg_bytes), "one_pass_bytes": int(one_pass),
                     "kernel": "solve_warp2_kernel / solve_tile_kernel / solve_cta_kernel (all size buckets of one step)"},
        "cpu_baseline": {"value": n_tracks / (cpu_ms / 1e3), "unit": UNIT, "cores": cores, "kind": "port",
                         "ms_per_step": cpu_ms, "single_thread_value": n_tracks / (cpu_1t_ms / 1e3),
                         "single_thread_ms_per_step": cpu_1t_ms,
                         "eight_thread_value": n_tracks / (cpu_8t_ms / 1e3), "eight_thread_ms_per_step": cpu_8t_ms,
                         "sample": "whole workload x %d repetitions (Ceres-1.14-semantics CPU oracle, "
                                   "oracle/lfr_oracle.cc); the reference's own solve.cc is timed by --impl reference" % reps},
        "total_scope": {"definition": "solve.cc:487-641 'Total time': tracks + roots + graph cut + dispatch + solve",
                        "host_stage_ms": host_stage_ms, "b200_ms": host_stage_ms + e2e_ms,
                        "cpu_oracle_ms_all_cores": host_stage_ms + cpu_ms, "cpu_oracle_ms_8_threads": host_stage_ms + cpu_8t_ms,
                        "host_stage": "csrc/lfr_host.cc, single-threaded C++ (same stage feeds both)"},
        "clocks": clocks,
    }
    if sharded is not None:
        line["sharded"] = sharded
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--debug-flags", type=int, default=0,
                    help="lfr_options.debug_flags for A/B experiments (LFR_DBG_*; 0 = the product path)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs is only for the b200 solve (--impl b200)")
    args.workload = {"fountain": "cfg2", "herzjesu": "cfg3"}.get(args.workload, args.workload)
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    raise SystemExit(main())
