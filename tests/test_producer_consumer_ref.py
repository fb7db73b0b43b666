"""SURVEY 8f rows 3-4 against the reference's OWN scripts:

  consumer.import_features   vs  reconstruction-scripts/colmap_utils.py::import_features
  producer.MatchGraphWriter  vs  the proto-building block of two-view-refinement/compute_match_graph.py:163-205

What the scripts produced on each test input is recorded in tests/golden/reference_runs.json; where
the reference sources are present the scripts are also run and checked against that record.

The reference scripts need `types_pb2` (protoc output, not in the reference tree or this image): the
runtime-built descriptor classes of tests/proto_runtime.py are injected under that module name.  Two
things the scripts themselves cannot do in this image are patched in the TEST, not in the product:
`ndarray.tostring()` (removed in numpy 2) -> `tobytes()`, and the `colmap matches_importer` subprocess.
"""
import importlib.util
import os
import sqlite3
import sys
import textwrap
import types

import numpy as np
import pytest

from lfr_b200 import consumer, producer, synth, wire
from lfr_b200.solver import assemble_solution
from reference_runs import as_json, recorded, sha256

REF = os.environ.get("LFR_REFERENCE_DIR", "/root/reference")
HAVE_REF = os.path.exists(os.path.join(REF, "reconstruction-scripts", "colmap_utils.py"))


def live(fn, *args):
    """fn(*args) deferred for reference_runs.recorded(), or None where the reference scripts are absent."""
    return (lambda: fn(*args)) if HAVE_REF else None


def _types_pb2():
    import proto_runtime
    mf, sf = proto_runtime.build()
    mod = types.ModuleType("types_pb2")
    mod.MatchingFile, mod.SolutionFile = mf, sf
    return mod


def _load_reference_colmap_utils():
    sys.modules["types_pb2"] = _types_pb2()
    spec = importlib.util.spec_from_file_location("ref_colmap_utils", os.path.join(REF, "reconstruction-scripts", "colmap_utils.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.array_to_blob = lambda a: a.tobytes()                    # numpy 2 removed ndarray.tostring()
    mod.subprocess = types.SimpleNamespace(call=lambda *a, **k: 0)   # no COLMAP binary here
    return mod


def _make_database(path, image_names):
    con = sqlite3.connect(path)
    cur = con.cursor()
    cur.execute("CREATE TABLE images (image_id INTEGER PRIMARY KEY, name TEXT)")
    for t in ("keypoints", "descriptors"):
        cur.execute("CREATE TABLE %s (image_id INTEGER, rows INTEGER, cols INTEGER, data BLOB)" % t)
    cur.execute("CREATE TABLE matches (pair_id INTEGER, rows INTEGER, cols INTEGER, data BLOB)")
    cur.execute("CREATE TABLE two_view_geometries (pair_id INTEGER, rows INTEGER, cols INTEGER, data BLOB, config INTEGER)")
    # image ids deliberately not in name order, so some pairs have image_id1 > image_id2 (column swap)
    ids = list(range(1, len(image_names) + 1))
    ids = ids[::2] + ids[1::2][::-1]
    for n, i in zip(image_names, ids):
        cur.execute("INSERT INTO images(image_id, name) VALUES(?, ?)", (i, n))
    cur.execute("INSERT INTO keypoints VALUES(1, 0, 4, x'')")         # stale rows must be deleted
    con.commit()
    con.close()


def _dump(path):
    """The tables import_features writes, rows sorted, blobs by their sha256."""
    con = sqlite3.connect(path)
    out = {t: [[sha256(x) if isinstance(x, bytes) else x for x in row]
               for row in sorted(con.execute("SELECT * FROM %s" % t).fetchall())]
           for t in ("keypoints", "matches", "descriptors")}
    con.close()
    return out


def write_import_features_case(tmp_path, oracle, with_solution):
    """Feature files, a two-part matches file and (with_solution) a SolutionFile; returns the arguments
    import_features needs besides the database."""
    ms = synth.generate("cfg2", scale=0.03, seed=17)
    # a duplicated pair exercises "first pair id wins"; an image without any match exercises the no-entry path
    ms = ms.select_pairs(np.concatenate([np.arange(ms.n_pairs), [3]]))
    names = list(ms.image_names) + ["lonely.png"]
    img_dir = tmp_path / "images"
    img_dir.mkdir()
    rng = np.random.default_rng(3)
    n_kp = int(max(ms.feat1.max(), ms.feat2.max())) + 5
    for k, n in enumerate(names):
        cols = (2, 3, 4)[k % 3]
        kp = rng.uniform(0, 2000, size=(n_kp if n != "lonely.png" else 0, cols))
        with open(img_dir / ("%s.%s" % (n, "sift")), "wb") as fh:
            np.savez(fh, keypoints=kp, descriptors=np.zeros((kp.shape[0], 1)))
    mfile = tmp_path / "matches.pb"
    half = ms.n_pairs // 2                                                  # two .part files
    for k, part in enumerate((ms.select_pairs(np.arange(half)), ms.select_pairs(np.arange(half, ms.n_pairs)))):
        (tmp_path / ("matches.pb.part.%d" % k)).write_bytes(wire.encode_matching_file(part))
    sfile = None
    if with_solution:
        from lfr_b200 import build_problem
        p = build_problem(ms)
        pos, _ = oracle.solve(p, oracle.default_options(n_threads=2))
        sol = assemble_solution(p, pos)
        sfile = str(tmp_path / "solution.pb")
        fact = sol.fact.copy()
        fact[0] = 1.5
        with open(sfile, "wb") as fh:
            fh.write(wire.encode_solution(sol.image_names, fact, sol.img_ptr, sol.feature_idx, sol.di, sol.dj))
    return names, img_dir, mfile, sfile


def reference_import_features(tmp_path, names, img_dir, mfile, sfile):
    ref = _load_reference_colmap_utils()
    db = str(tmp_path / "ref.db")
    _make_database(db, names)
    r = ref.import_features("/nonexistent", "sift", db, str(img_dir), "unused", str(mfile), sfile)
    return {"return": r, "tables": _dump(db)}


@pytest.mark.parametrize("with_solution", [True, False])
def test_import_features_equals_the_reference_script(tmp_path, oracle, with_solution):
    names, img_dir, mfile, sfile = case = write_import_features_case(tmp_path, oracle, with_solution)
    ref = recorded("import_features", "with_solution=%s" % with_solution,
                   live(reference_import_features, tmp_path, *case))
    db_mine = str(tmp_path / "mine.db")
    _make_database(db_mine, names)
    m = consumer.import_features("/nonexistent", "sift", db_mine, str(img_dir), "unused", str(mfile), sfile, run_colmap=False)
    assert ref["return"] == as_json(m)
    a, b = ref["tables"], _dump(db_mine)
    assert a["keypoints"] == b["keypoints"] and len(a["keypoints"]) == len(names)
    assert a["matches"] == b["matches"] and len(a["matches"]) > 0
    assert a["descriptors"] == b["descriptors"] == []


def _reference_emit(pairs, output_file, dump_interval):
    """Executes the reference's own proto-building and dumping statements, read from its source file
    at test time (two-view-refinement/compute_match_graph.py, from '# Build the proto object.' to the
    end of main), around a loop that supplies the variables those statements use."""
    src = open(os.path.join(REF, "two-view-refinement", "compute_match_graph.py")).read().split("\n")
    start = next(i for i, l in enumerate(src) if "# Build the proto object." in l)
    tail = next(i for i, l in enumerate(src) if "# Save the proto object to disk." in l)
    end = len(src)                                              # the script's main body runs to the end of the file
    body = textwrap.dedent("\n".join(src[start:tail]))          # per-pair statements (indent 8 in the file)
    final = textwrap.dedent("\n".join(src[tail:end]))           # after the loop (indent 4)
    harness = ("def run(pairs, args, MatchingFile, dump_interval):\n"
               "    matching_file_proto = MatchingFile()\n    part_idx = -1\n"
               "    for pair_idx, (image_name1, fact1, image_name2, fact2, matches, sim, grid_displacements12, "
               "grid_displacements21) in enumerate(pairs):\n"
               + textwrap.indent(body, "        ") + "\n" + textwrap.indent(final, "    ") + "\n")
    ns = {}
    exec(compile(harness, "reference_emit", "exec"), ns)
    mf, _ = __import__("proto_runtime").build()
    ns["run"](pairs, types.SimpleNamespace(output_file=output_file), mf, dump_interval)


def writer_pairs(dump_interval, n_pairs):
    rng = np.random.default_rng(dump_interval * 100 + n_pairs)
    pairs = []
    for k in range(n_pairs):
        m = int(rng.integers(0, 6)) if k != 2 else 0               # an empty pair too
        matches = np.stack([rng.permutation(50)[:m], rng.permutation(50)[:m]], axis=1).astype(np.int64) if m else np.zeros((0, 2))
        if m:
            matches[0, 0] = 0                                        # feature_idx 0: proto3 omits the field
        sim = rng.uniform(0.5, 1.0, size=m).astype(np.float32)
        g12 = rng.normal(size=(m, 3, 3, 2))
        g21 = rng.normal(size=(m, 3, 3, 2))
        if m > 1:
            g12[1] = 0.0                                             # SKIP_REFINEMENT-style zero grids (:150-152)
        pairs.append(("img%d.png" % (k % 3), float(1 + 0.25 * (k % 3)), "img%d.png" % (k % 3 + 1), 1.0,
                      matches, sim, g12, g21))
    return pairs


def reference_writer_files(tmp_path, pairs, dump_interval):
    """The files the reference's loop writes, as {name: hex bytes}."""
    ref_dir = tmp_path / "ref"
    ref_dir.mkdir()
    # the reference's loop hard-codes dump_interval = 5000 (:77-78); the harness passes it in
    _reference_emit(pairs, str(ref_dir / "m.pb"), dump_interval)
    return {f: (ref_dir / f).read_bytes().hex() for f in sorted(os.listdir(ref_dir))}


@pytest.mark.parametrize("dump_interval,n_pairs", [(5000, 7), (3, 7), (3, 6), (2, 1)])
def test_match_graph_writer_equals_the_reference_loop(tmp_path, dump_interval, n_pairs):
    pairs = writer_pairs(dump_interval, n_pairs)
    ref = recorded("match_graph_writer", "dump_interval=%d n_pairs=%d" % (dump_interval, n_pairs),
                   live(reference_writer_files, tmp_path, pairs, dump_interval))
    my_dir = tmp_path / "mine"
    my_dir.mkdir()
    w = producer.MatchGraphWriter(str(my_dir / "m.pb"), dump_interval=dump_interval, packed=True)
    for pr in pairs:
        w.add_pair(*pr)
    w.close()
    mine = sorted(f for f in os.listdir(my_dir) if not f.endswith(".npz"))
    assert sorted(ref) == mine and len(mine) >= 1
    for f in mine:
        assert ref[f] == (my_dir / f).read_bytes().hex(), f
    # the packed form holds the same matches as the protobuf parts
    from lfr_b200.matchset import MatchSet
    back = MatchSet.load_npz(str(my_dir / "m.pb.npz"))
    whole = wire.read_matching_file(str(my_dir / "m.pb"))
    assert wire.encode_matching_file(back) == wire.encode_matching_file(whole)
