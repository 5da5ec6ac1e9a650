"""Drop-in check at the C level: a caller written against the reference's turtle.h is
compiled, unchanged, against (a) the reference library with the REFERENCE's header and
(b) libturtle_b200.so with THIS repository's include/turtle.h. Both binaries must print
the same bits (host scalar path = set-up calls + the example-stepper ray loop)."""
import os
import subprocess

import pytest

from oracle import harness as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "c", "dropin_stepper.c")


def build(tmp, name, include, libdir, lib):
    exe = os.path.join(tmp, name)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I" + include, SRC, "-o", exe,
                           "-L" + libdir, "-l" + lib, "-Wl,-rpath," + libdir, "-lm"])
    return exe


def test_c_caller_compiles_and_runs_against_our_abi(tmp_path):
    exe = build(str(tmp_path), "ours", os.path.join(ROOT, "include"),
                os.path.join(ROOT, "turtle_b200"), "turtle_b200")
    out = subprocess.check_output([exe, "12"], text=True)
    lines = out.strip().splitlines()
    assert len(lines) == 13 and lines[-1].startswith("map 101 101")
    assert all(int(l.split()[1]) > 5 for l in lines[:-1])


@pytest.mark.skipif(not (os.path.exists(H.REF) and
                         os.path.isdir(os.path.join(H.REF_SOURCES, "include"))),
                    reason="needs the reference's sources (TURTLE_REF) and oracle/_ref built from them")
def test_same_bits_as_the_reference(tmp_path):
    ours = build(str(tmp_path), "ours", os.path.join(ROOT, "include"),
                 os.path.join(ROOT, "turtle_b200"), "turtle_b200")
    ref = build(str(tmp_path), "ref", os.path.join(H.REF_SOURCES, "include"),
                os.path.dirname(H.REF), "turtle_ref")
    a = subprocess.check_output([ours, "24"], text=True)
    b = subprocess.check_output([ref, "24"], text=True)
    assert a == b
