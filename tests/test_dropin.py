"""The drop-in files (integration/bioseqdb/bwa.h, bwa.cpp + integration/include/bwa/*.h) keep the reference adapter's surface: they
compile and link against the reference's UNCHANGED sequence.h / sequence.cpp and against bwa_index_from_query cut out of the
reference's extension.cpp at test time (BwaIndex returned by value, `bwa.options->field` writes, const align_sequence).  Without a GPU
the program must fail loudly with the library's "no CUDA device" error (no CPU fallback); with a GPU it aligns one read.
The reference is not redistributed here: BIOSEQDB_SRC names a checkout of unneon/bioseqdb (as in integration/CMakeLists.txt), and
that test skips without one.  The same program also runs on every machine against tests/dropin_src, a stand-in for the three
reference pieces written in this repository."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(os.environ.get("BIOSEQDB_SRC", ""), "bioseqdb")
STAND_IN = os.path.join(ROOT, "tests", "dropin_src")
BUILD = os.path.join(ROOT, "tests", "_build")


def _build(name, src_dirs, sources):
    from bioseqdb_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build_library()
    exe = os.path.join(BUILD, name)
    inc = ["-I" + os.path.join(ROOT, "integration", "bioseqdb")] + ["-I" + d for d in src_dirs] + [
        "-I" + os.path.join(ROOT, "integration", "include"), "-I" + os.path.join(ROOT, "tests", "pg_stub"), "-I" + os.path.join(ROOT, "include")]
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-Wno-unused-function", "-o", exe] + inc +
                          [os.path.join(ROOT, "tests", "dropin_check.cpp"), os.path.join(ROOT, "integration", "bioseqdb", "bwa.cpp")] + sources +
                          ["-L" + os.path.dirname(_lib.LIB_PATH), "-lbioseqdb_gpu", "-Wl,-rpath," + os.path.dirname(_lib.LIB_PATH)])
    return exe


def _run(exe):
    p = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    from bioseqdb_b200 import _lib
    if _lib.lib().bsq_device_count() > 0:
        assert p.returncode == 0 and "dropin ok" in p.stdout, p.stdout + p.stderr
    else:
        assert p.returncode == 3 and "no CUDA device" in p.stdout, p.stdout + p.stderr


def test_dropin_compiles_against_reference_sources():
    if not os.environ.get("BIOSEQDB_SRC") or not os.path.exists(os.path.join(REF, "extension.cpp")):
        pytest.skip("needs a checkout of unneon/bioseqdb named by BIOSEQDB_SRC")
    os.makedirs(BUILD, exist_ok=True)
    lines = open(os.path.join(REF, "extension.cpp")).read().split("\n")
    start = next(i for i, l in enumerate(lines) if l.startswith("BwaIndex bwa_index_from_query("))
    end = next(i for i in range(start, len(lines)) if lines[i] == "}")
    with open(os.path.join(BUILD, "dropin_excerpt.inc"), "w") as f:
        f.write("\n".join(lines[start:end + 1]) + "\n")
    _run(_build("dropin_check", [REF, BUILD], [os.path.join(REF, "sequence.cpp")]))


def test_dropin_runs_against_stand_in_sources():
    os.makedirs(BUILD, exist_ok=True)
    _run(_build("dropin_check_stand_in", [STAND_IN],
                [os.path.join(STAND_IN, "sequence.cpp"), os.path.join(ROOT, "bioseqdb_b200", "host", "sequence.cpp")]))
