"""The whole pipeline against the REFERENCE'S OWN main().

oracle/_ref/solve is multi-view-refinement/solve.cc (+ cost.cc, graph.cc) compiled unmodified against
the shim headers of oracle/ref_shims/ (oracle/build_ref.py).  What runs is the reference author's
code for: protobuf reading incl. `.part.N` (solve.cc:412-481), node interning and edge lists (:53-65,
:474-478), constrained Kruskal (:487-549), root selection (:551-582), separate_meta_graph /
recursive_graph_cut / bfs (:162-373), create_and_solve_problem (:79-160: which residual blocks,
which loss, constant roots, bounds, solver options), the thread-pool dispatch (:599-635), the
output assembly (:643-679), the command line (:379-403) and every stdout line.  Behind the shims:
Ceres' minimizer is the mini-Ceres restatement, the Graclus cut is csrc/lfr_cut.h (the two pieces no
build in this image can pin), protobuf / Boost.PO / ThreadPool are functional equivalents.

Rows pinned here (SURVEY 8a): A4, A5, A7, A8, H1-H5 and the drop-in boundary (b).

What the binary produced on each test input is recorded in tests/golden/reference_runs.json, so these
tests run where it cannot be built; where it can, it is run as well and checked against the record.
"""
import functools
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from lfr_b200 import build_problem, synth, wire
from lfr_b200.solver import assemble_solution
from reference_runs import recorded, sha256

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
LAUNCHER = os.path.join(ROOT, "multi-view-refinement", "build", "solve")


@functools.lru_cache(maxsize=None)
def find_ref_exe():
    """oracle/_ref/solve, or None when it is neither built nor buildable here."""
    spec = importlib.util.spec_from_file_location("lfr_build_ref", os.path.join(ROOT, "oracle", "build_ref.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    try:
        return mod.build_solve()
    except Exception:
        return None


def ref_exe():
    exe = find_ref_exe()
    if exe is None:
        pytest.skip("oracle/_ref/solve is not built and the reference sources are not available here")
    return exe


def live(fn, *args):
    """fn(*args) deferred for reference_runs.recorded(), or None where the reference binary cannot run."""
    return (lambda: fn(*args)) if find_ref_exe() is not None else None


def run_ref(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([ref_exe()] + args, capture_output=True, text=True, env=e)


def oracle_pipeline(oracle, data, banned=()):
    """host stage (native) + oracle solve + output assembly -> (SolutionFile bytes, problem, stats, log lines)"""
    lines = []
    p = build_problem(wire.decode_matching_file(data), banned_images=banned, log=lines.append)
    pos, st = oracle.solve(p, oracle.default_options(n_threads=4))
    sol = assemble_solution(p, pos)
    out = wire.encode_solution(sol.image_names, sol.fact, sol.img_ptr, sol.feature_idx, sol.di, sol.dj)
    lines.append("# points with at least one coordinate > 0.5: %d" % sol.n_outside)
    return out, p, st, lines


def untimed(stdout):
    return [l for l in stdout.splitlines() if " time:" not in l]


def reference_run(tmp_path, matches, extra=(), summaries=False):
    """The reference binary on one MatchingFile: its SolutionFile's sha256, its stdout without the timing
    lines and, with summaries=True, from the ceres::Solve summaries recorded by the shim: the total of
    line-search steps and, per problem in the order of its lowest parameter-block address (= lowest
    node index of the component), the LM iterations and the initial cost without the fixed cost of the
    all-constant (root-root) blocks, which the C ABI reports without it."""
    opath, rpath = tmp_path / "ref_solution.pb", tmp_path / "ref_summaries.txt"
    r = run_ref(["--matches_file", str(matches), "--output_file", str(opath)] + list(extra),
                env={"LFR_CERES_RECORD_FILE": str(rpath)} if summaries else None)
    assert r.returncode == 0, r.stderr
    out = {"solution_sha256": sha256(opath.read_bytes()), "stdout": untimed(r.stdout)}
    if summaries:
        # address iterations termination line-search-steps initial-cost final-cost blocks residuals fixed-cost
        rows = sorted((l.split() for l in rpath.read_text().splitlines()), key=lambda c: int(c[0]))
        out["iterations"] = [int(c[1]) for c in rows]
        out["line_search_steps"] = sum(int(c[3]) for c in rows)
        out["initial_cost"] = [float(c[4]) - float(c[8]) for c in rows]
    return out


def reference_command_line(argv):
    r = run_ref(argv)
    return {"returncode": r.returncode, "stdout": r.stdout, "stderr": r.stderr}


def scene_key(name, scale, seed):
    return "%s scale=%g seed=%s" % (name, scale, seed)


def write_scene(tmp_path, name, scale, seed):
    data = wire.encode_matching_file(synth.generate(name, scale=scale, seed=seed))
    (tmp_path / "m.pb").write_bytes(data)
    return data, tmp_path / "m.pb"


def write_banned_case(tmp_path):
    """cfg2 at 8 % with two banned images, as one file (m.pb) and as two .part.N files (split.pb)."""
    ms = synth.generate("cfg2", scale=0.08, seed=21)
    data = wire.encode_matching_file(ms)
    (tmp_path / "m.pb").write_bytes(data)
    # matches split over .part.N files (compute_match_graph.py:189-205, solve.cc:416-424)
    half = ms.n_pairs // 2
    for k, part in enumerate([ms.select_pairs(np.arange(0, half)), ms.select_pairs(np.arange(half, ms.n_pairs))]):
        (tmp_path / ("split.pb.part.%d" % k)).write_bytes(wire.encode_matching_file(part))
    return data, [ms.image_names[2], ms.image_names[5]]


def write_unparsable(tmp_path):
    bad = tmp_path / "bad.pb"
    bad.write_bytes(b"\x0a\xff\xff\xff\xff\x0f not a protobuf")
    return ["--matches_file", str(bad), "--output_file", str(tmp_path / "o.pb")]


SCENES = [("cfg1", 1.0, None), ("cfg2", 0.1, 3), ("cfg2", 0.25, 11), ("cfg3", 0.05, 5), ("cfg4", 0.05, 7),
          ("ring60", 0.5, 2)]


@pytest.mark.parametrize("name,scale,seed", SCENES)
def test_solution_file_is_byte_identical_to_the_reference_binary(oracle, tmp_path, name, scale, seed):
    data, mpath = write_scene(tmp_path, name, scale, seed)
    ref = recorded("solve", scene_key(name, scale, seed),
                   live(reference_run, tmp_path, mpath, ["--n_threads", "4"], True))
    mine, p, st, lines = oracle_pipeline(oracle, data)
    assert sha256(mine) == ref["solution_sha256"]
    # every stdout line except the three timings (solve.cc:484-485,534,549,591,606,670)
    assert ref["stdout"] == [l for l in lines if " time:" not in l]
    # per-problem LM iteration counts: ceres::Solve summaries recorded by the shim, matched to the
    # dispatch slots through the lowest parameter-block address (= lowest node index of the component)
    sizes = np.diff(p.comp_ptr.astype(np.int64))
    solved = np.nonzero(sizes > 1)[0]
    assert len(ref["iterations"]) == solved.shape[0]
    min_node = np.array([p.comp_nodes[p.comp_ptr[c]] for c in solved])       # nodes ascending inside a component
    order_mine = solved[np.argsort(min_node)]
    assert np.array_equal(np.array(ref["iterations"], np.int64), st["iterations"][order_mine])
    assert ref["line_search_steps"] == int(st["total_line_search_steps"])
    np.testing.assert_allclose(ref["initial_cost"], st["initial_cost"][order_mine], rtol=1e-11, atol=1e-14)


@pytest.mark.parametrize("name", ["tiny", "linesearch", "fountain_2pct"])
def test_committed_goldens_are_the_reference_binarys_output(tmp_path, name):
    opath = tmp_path / "s.pb"
    r = run_ref(["--matches_file", os.path.join(GOLD, name + "_matches.pb"), "--output_file", str(opath)])
    assert r.returncode == 0
    assert opath.read_bytes() == open(os.path.join(GOLD, name + "_solution.pb"), "rb").read()
    assert untimed(r.stdout) == open(os.path.join(GOLD, name + "_stdout.txt")).read().splitlines()


def test_banned_images_and_part_files(oracle, tmp_path):
    data, banned = write_banned_case(tmp_path)
    ref = recorded("solve", "banned images", live(reference_run, tmp_path, tmp_path / "m.pb",
                                                  ["--banned_images", banned[0], "--banned_images=" + banned[1]]))
    mine, _, _, lines = oracle_pipeline(oracle, data, banned=banned)
    assert sha256(mine) == ref["solution_sha256"] and ref["stdout"] == [l for l in lines if " time:" not in l]
    ref2 = recorded("solve", "part files", live(reference_run, tmp_path, tmp_path / "split.pb"))
    mine2, _, _, _ = oracle_pipeline(oracle, data)
    assert sha256(mine2) == ref2["solution_sha256"]


BAD_COMMAND_LINES = [["--help"], ["--matches_file", "x"], ["--foo", "1"], ["pos"], ["--matches_file"],
                     ["--matches_file", "a", "--matches_file", "b", "--output_file", "c"],
                     ["--n_threads", "abc", "--matches_file", "a", "--output_file", "b"],
                     ["--mat", "x", "--out", "y", "-x"], ["--output_file=y"]]


@pytest.mark.parametrize("argv", BAD_COMMAND_LINES)
def test_command_line_errors_match_the_reference_binary(argv):
    """solve.cc:379-403 (Boost.Program_options): same exit code, stdout and stderr from the drop-in
    launcher (argument handling needs no GPU)."""
    a = recorded("command_line", json.dumps(argv), live(reference_command_line, argv))
    b = subprocess.run([sys.executable, LAUNCHER] + argv, capture_output=True, text=True)
    assert (a["returncode"], a["stdout"], a["stderr"]) == (b.returncode, b.stdout, b.stderr)


def test_parse_failure_exit_code(tmp_path):
    argv = write_unparsable(tmp_path)
    a = recorded("command_line", "unparsable input", live(reference_command_line, argv))
    assert a["returncode"] == 255 and "Failed to parse proto object." in a["stderr"]      # return -1, solve.cc:433-436
    b = subprocess.run([sys.executable, LAUNCHER] + argv, capture_output=True, text=True)
    assert (a["returncode"], a["stderr"]) == (b.returncode, b.stderr)


@pytest.mark.gpu
@pytest.mark.parametrize("host", ["native", "python"])
@pytest.mark.parametrize("name", ["tiny", "linesearch", "fountain_2pct"])
def test_gpu_launcher_reproduces_the_reference_binarys_solution_file(tmp_path, name, host):
    """The drop-in executable on the GPU against the reference's own main(): same stdout lines, and
    the SolutionFile equal float for float (fp32 on the wire) — byte-identical unless a displacement
    sits within 1e-16 of a float32 rounding boundary."""
    m = os.path.join(GOLD, name + "_matches.pb")
    o = tmp_path / "gpu.pb"
    env = dict(os.environ)
    if host == "python":
        env["LFR_SOLVE_PYTHON"] = "1"     # the launcher hands over to solve_native otherwise
    r = subprocess.run([sys.executable, LAUNCHER, "--matches_file", m, "--output_file", str(o)],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    want = open(os.path.join(GOLD, name + "_solution.pb"), "rb").read()
    assert untimed(r.stdout) == open(os.path.join(GOLD, name + "_stdout.txt")).read().splitlines()
    got = o.read_bytes()
    if got != want:
        a, b = wire.decode_solution(got), wire.decode_solution(want)    # lists of (name, fact, feature_idx, di, dj)
        assert [x[0] for x in a] == [x[0] for x in b]
        n_diff = 0
        for (_, fa, ia, dia, dja), (_, fb, ib, dib, djb) in zip(a, b):
            assert fa == fb and np.array_equal(ia, ib)
            assert np.abs(dia - dib).max() <= 1e-4 / 16 and np.abs(dja - djb).max() <= 1e-4 / 16
            n_diff += int((dia != dib).sum() + (dja != djb).sum())
        assert n_diff <= 2
