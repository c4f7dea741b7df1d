"""The library's environment variables are exactly the documented ones (CPU only: reads the sources).

Every knob selects between code paths that the library otherwise chooses from shapes, so an undocumented one is
a path nobody knows how to reach or test.  DESIGN.md lists them at the end of section 5."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "trajnetplusplusbaselines_b200", "csrc")

KNOBS = {"TB2_DISABLE_TC", "TB2_SPARSE", "TB2_PDL", "TB2_KALMAN_THREADS"}


def _knobs_read_by_library():
    names = set()
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".h", ".cpp")):
            names |= set(re.findall(r'getenv\(\s*"(TB2_\w+)"', open(os.path.join(CSRC, f)).read()))
    return names


def test_library_reads_exactly_the_known_knobs():
    assert _knobs_read_by_library() == KNOBS


def test_every_knob_is_documented():
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    missing = sorted(k for k in _knobs_read_by_library() if k not in design)
    assert not missing, "not in DESIGN.md: " + ", ".join(missing)
