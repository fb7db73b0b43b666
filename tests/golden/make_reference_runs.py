"""Record what the reference's own programs produce on the tests' inputs: tests/golden/reference_runs.json.

Needs the reference sources (LFR_REFERENCE_DIR) and oracle/_ref/ built from them (oracle/build_ref.py,
run by `python __graft_entry__.py build`).  The inputs and the way each program is run are the test
modules' own helpers, so a record always matches what its test compares against.

    python tests/golden/make_reference_runs.py
"""
import json
import os
import pathlib
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import test_native_exe as tn  # noqa: E402
import test_producer_consumer_ref as tp  # noqa: E402
import test_ref_cost as tc  # noqa: E402
import test_ref_solve as ts  # noqa: E402
from oracle_util import load_oracle  # noqa: E402
from reference_runs import PATH, as_json  # noqa: E402


TMP = tempfile.mkdtemp(prefix="lfr_golden_")


def tmp():
    return pathlib.Path(tempfile.mkdtemp(dir=TMP))


def main():
    assert ts.find_ref_exe() is not None and tp.HAVE_REF, "the reference is not available here"
    L = tc.load_refsrc()
    assert L is not None
    out = {"solve": {}, "command_line": {}, "import_features": {}, "match_graph_writer": {}, "cost": {}}
    for name, scale, seed in ts.SCENES:
        d = tmp()
        _, mpath = ts.write_scene(d, name, scale, seed)
        out["solve"][ts.scene_key(name, scale, seed)] = ts.reference_run(d, mpath, ["--n_threads", "4"], True)
    d = tmp()
    _, banned = ts.write_banned_case(d)
    out["solve"]["banned images"] = ts.reference_run(d, d / "m.pb", ["--banned_images", banned[0],
                                                                    "--banned_images=" + banned[1]])
    out["solve"]["part files"] = ts.reference_run(d, d / "split.pb")
    for argv in tn.COMMAND_LINES:
        out["command_line"][json.dumps(argv)] = ts.reference_command_line(argv)
    out["command_line"]["unparsable input"] = ts.reference_command_line(ts.write_unparsable(tmp()))
    orc = load_oracle()
    for with_solution in (True, False):
        d = tmp()
        case = tp.write_import_features_case(d, orc, with_solution)
        out["import_features"]["with_solution=%s" % with_solution] = tp.reference_import_features(d, *case)
    for dump_interval, n_pairs in ((5000, 7), (3, 7), (3, 6), (2, 1)):
        key = "dump_interval=%d n_pairs=%d" % (dump_interval, n_pairs)
        out["match_graph_writer"][key] = tp.reference_writer_files(tmp(), tp.writer_pairs(dump_interval, n_pairs),
                                                                   dump_interval)
    out["cost"]["200k inputs seed=7"] = tc.reference_200k_digests(L)
    shutil.rmtree(TMP)
    # one line per record
    with open(PATH, "w") as fh:
        fh.write("{\n" + ",\n".join(
            "%s: {\n" % json.dumps(section) + ",\n".join(
                " %s: %s" % (json.dumps(k), json.dumps(v, sort_keys=True, separators=(",", ":")))
                for k, v in sorted(as_json(records).items())) + "\n}"
            for section, records in sorted(out.items())) + "\n}\n")
    print("wrote", PATH, os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()
