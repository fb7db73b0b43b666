"""Recorded results of the reference's own programs, for the tests that compare against them.

The reference's sources exist only where the project is developed, so what its programs produced on
each test input is kept in tests/golden/reference_runs.json (written by
tests/golden/make_reference_runs.py).  A test takes its expected result from there; where the
reference can be run as well, the test also runs it and checks that it still produces the record."""
import hashlib
import json
import os

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.json")
_records = None


def as_json(value):
    """The form a result takes after a JSON round trip (tuples become lists)."""
    return json.loads(json.dumps(value))


def sha256(data: bytes) -> str:
    return hashlib.sha256(data).hexdigest()


def recorded(section, key, live=None):
    """The stored result for `key`; `live` (a callable running the reference, or None where it cannot
    run) is checked against it."""
    global _records
    if _records is None:
        with open(PATH) as fh:
            _records = json.load(fh)
    want = _records[section][key]
    if live is not None:
        assert as_json(live()) == want, "the reference no longer produces the record %s[%s]" % (section, key)
    return want
