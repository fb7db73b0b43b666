"""The native drop-in executable (csrc/lfr_solve_main.cc -> multi-view-refinement/build/solve_native).

Everything above the C ABI — command line, `.part.N` files, banned images, decoding, the host graph
stage, output assembly, stdout lines, exit codes — is checked on the CPU by linking the SAME source
against the checker library (oracle/liblfr_ref.so exports the C ABI of include/lfr.h; test
infrastructure only, built into a temporary directory) and comparing with the reference's own main()
(oracle/_ref/solve, the committed goldens).  The product binary links csrc/liblfr_b200.so and has no
other route: without a CUDA device it stops with an error (no CPU fallback); on a GPU it is compared
with the same goldens."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from lfr_b200 import synth, wire
from reference_runs import recorded
from test_ref_solve import BAD_COMMAND_LINES, GOLD, LAUNCHER, live, oracle_pipeline, reference_command_line, untimed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRODUCT = os.path.join(ROOT, "multi-view-refinement", "build", "solve_native")


def _csrc_build():
    spec = importlib.util.spec_from_file_location("lfr_csrc_build", os.path.join(ROOT, "local-feature-refinement_b200", "csrc", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def checker_exe(tmp_path_factory, oracle):
    """lfr_solve_main.cc linked against the CPU checker instead of the CUDA library."""
    out = str(tmp_path_factory.mktemp("native") / "solve_native_checker")
    b = _csrc_build()
    b.build_host()
    return b.build_exe(force=True, out=out, solve_lib_dir=os.path.join(ROOT, "oracle"), solve_lib="lfr_ref")


@pytest.fixture(scope="module")
def product_exe():
    b = _csrc_build()
    b.build()
    return PRODUCT


def run(exe, args):
    return subprocess.run([exe] + args, capture_output=True, text=True)


@pytest.mark.parametrize("name", ["tiny", "linesearch", "fountain_2pct"])
def test_checker_build_reproduces_the_reference_binarys_goldens(checker_exe, tmp_path, name):
    o = tmp_path / "s.pb"
    r = run(checker_exe, ["--matches_file", os.path.join(GOLD, name + "_matches.pb"), "--output_file", str(o), "--n_threads", "4"])
    assert r.returncode == 0, r.stderr
    assert o.read_bytes() == open(os.path.join(GOLD, name + "_solution.pb"), "rb").read()
    assert untimed(r.stdout) == open(os.path.join(GOLD, name + "_stdout.txt")).read().splitlines()
    timed = [l for l in r.stdout.splitlines() if " time:" in l]
    assert [l.split(":")[0] for l in timed] == ["Graph-cut time", "Solver time", "Total time"]   # solve.cc:589,638,641


def test_banned_images_part_files_and_empty_input(checker_exe, oracle, tmp_path):
    ms = synth.generate("cfg2", scale=0.08, seed=21)
    data = wire.encode_matching_file(ms)
    banned = [ms.image_names[2], ms.image_names[5]]
    m, o = tmp_path / "m.pb", tmp_path / "o.pb"
    m.write_bytes(data)
    r = run(checker_exe, ["--matches_file", str(m), "--output_file", str(o), "--banned_images", banned[0], "--banned_images=" + banned[1]])
    assert r.returncode == 0, r.stderr
    mine, _, _, lines = oracle_pipeline(oracle, data, banned=banned)
    assert o.read_bytes() == mine and untimed(r.stdout) == [l for l in lines if " time:" not in l]
    # .part.N pieces (compute_match_graph.py:189-205, solve.cc:416-424)
    half = ms.n_pairs // 2
    for k, part in enumerate([ms.select_pairs(np.arange(0, half)), ms.select_pairs(np.arange(half, ms.n_pairs))]):
        (tmp_path / ("split.pb.part.%d" % k)).write_bytes(wire.encode_matching_file(part))
    o2 = tmp_path / "o2.pb"
    r = run(checker_exe, ["--matches_file", str(tmp_path / "split.pb"), "--output_file", str(o2)])
    assert r.returncode == 0, r.stderr
    mine2, _, _, lines2 = oracle_pipeline(oracle, data)
    assert o2.read_bytes() == mine2 and untimed(r.stdout) == [l for l in lines2 if " time:" not in l]
    # no file at all: an empty SolutionFile, like the Python launcher (the reference's own binary dereferences an
    # empty container after "# tracks: 0" and dies with SIGSEGV on this input)
    o3 = tmp_path / "o3.pb"
    r = run(checker_exe, ["--matches_file", str(tmp_path / "absent.pb"), "--output_file", str(o3)])
    assert r.returncode == 0 and o3.read_bytes() == b""
    assert untimed(r.stdout) == ["# graph nodes: 0", "# graph edges: 0", "# points with at least one coordinate > 0.5: 0"]


COMMAND_LINES = BAD_COMMAND_LINES + [["--matches_file=a", "--output_file", "b", "--help=1"]]


@pytest.mark.parametrize("argv", COMMAND_LINES)
def test_command_line_errors_match_the_python_launcher_and_the_reference(product_exe, argv):
    """Argument handling needs neither a GPU nor the checker: the PRODUCT binary against the Python
    launcher and against the reference binary's recorded answer."""
    a = run(product_exe, argv)
    b = subprocess.run([sys.executable, LAUNCHER] + argv, capture_output=True, text=True)
    assert (a.returncode, a.stdout, a.stderr) == (b.returncode, b.stdout, b.stderr)
    c = recorded("command_line", json.dumps(argv), live(reference_command_line, argv))
    assert (a.returncode, a.stdout, a.stderr) == (c["returncode"], c["stdout"], c["stderr"])


def test_unparsable_and_unwritable(product_exe, checker_exe, tmp_path):
    bad = tmp_path / "bad.pb"
    bad.write_bytes(b"\x0a\xff\xff\xff\xff\x0f not a protobuf")
    r = run(product_exe, ["--matches_file", str(bad), "--output_file", str(tmp_path / "o.pb")])
    assert r.returncode == 255 and r.stderr == "Failed to parse proto object.\n"             # solve.cc:433-436
    r = run(checker_exe, ["--matches_file", os.path.join(GOLD, "tiny_matches.pb"), "--output_file", str(tmp_path / "no" / "dir" / "o.pb")])
    assert r.returncode == 255 and r.stderr == "Failed to write proto object.\n"             # solve.cc:674-677


def test_product_binary_has_no_cpu_fallback(product_exe, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = run(product_exe, ["--matches_file", os.path.join(GOLD, "tiny_matches.pb"), "--output_file", str(tmp_path / "o.pb")])
    assert r.returncode == 2 and "the solve failed" in r.stderr and not (tmp_path / "o.pb").exists()
    out = subprocess.run(["ldd", product_exe], capture_output=True, text=True).stdout
    assert "liblfr_b200.so" in out and "liblfr_ref" not in out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny", "linesearch", "fountain_2pct"])
def test_gpu_native_executable_reproduces_the_reference_binarys_solution_file(product_exe, tmp_path, name):
    m = os.path.join(GOLD, name + "_matches.pb")
    o = tmp_path / "gpu.pb"
    r = run(product_exe, ["--matches_file", m, "--output_file", str(o)])
    assert r.returncode == 0, r.stderr
    want = open(os.path.join(GOLD, name + "_solution.pb"), "rb").read()
    assert untimed(r.stdout) == open(os.path.join(GOLD, name + "_stdout.txt")).read().splitlines()
    got = o.read_bytes()
    if got != want:
        a, b = wire.decode_solution(got), wire.decode_solution(want)
        assert [x[0] for x in a] == [x[0] for x in b]
        for (na, fa, ia, dia, dja), (nb, fb, ib, dib, djb) in zip(a, b):
            assert fa == fb and np.array_equal(ia, ib)
            assert np.abs(dia - dib).max() <= 1e-4 / 16 and np.abs(dja - djb).max() <= 1e-4 / 16


def test_image_names_are_bytes_to_both_hosts(checker_exe, oracle, tmp_path):
    """Names with spaces, non-ASCII characters and invalid UTF-8 travel through unchanged (the reference
    treats them as std::string); banned images are matched on the same bytes."""
    ms = synth.generate("cfg1", seed=5)
    odd = ["im age 0.png", "bild-äöü.jpg", b"raw-\xff\xfe.png".decode("utf-8", errors="surrogateescape")]
    ms.image_names = odd[:len(ms.image_names)] + ms.image_names[len(odd):]
    data = wire.encode_matching_file(ms)
    m, o = tmp_path / "m.pb", tmp_path / "o.pb"
    m.write_bytes(data)
    r = subprocess.run([checker_exe, "--matches_file", str(m), "--output_file", str(o)], capture_output=True)
    assert r.returncode == 0, r.stderr
    mine, _, _, _ = oracle_pipeline(oracle, data)
    assert o.read_bytes() == mine
    # ban the non-ASCII one (argv carries the same bytes)
    o2 = tmp_path / "o2.pb"
    r = subprocess.run([checker_exe, "--matches_file", str(m), "--output_file", str(o2), "--banned_images", odd[1]], capture_output=True)
    assert r.returncode == 0, r.stderr
    mine2, _, _, _ = oracle_pipeline(oracle, data, banned=[odd[1]])
    assert o2.read_bytes() == mine2 and mine2 != mine
