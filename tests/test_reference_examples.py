"""The reference's own example programs, UNMODIFIED (compiled from where they lie, in the
examples/ of the reference's sources: oracle.harness.REF_SOURCES), linked once against the
unmodified reference library and once against libturtle_b200.so + include/turtle.h: same
files written, same text printed. This is the drop-in claim of INTEGRATION.md section 1
taken literally -- example-projection
(stack -> Lambert 93 map -> PNG), example-demo (map meta data, projections, ECEF,
horizontal angles), example-stepper (the hot path: geoid + flat / stack / map layer, local
approximation on and off, a ray marched to 2 km of altitude) and example-pthread (clients of
a locked stack on four threads).

Runs on the host only (scalar calls). Needs the reference sources, gcc and Pillow's bundled
libpng for the REFERENCE side (it dlopen()s libpng; the product parses PNG itself): skipped
where any is missing, e.g. on the GPU box."""
import glob
import os
import shutil
import subprocess

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXAMPLES = os.path.join(H.REF_SOURCES, "examples")
REF_LIB = H.REF

pytestmark = pytest.mark.skipif(
    not os.path.isdir(EXAMPLES) or not os.path.exists(REF_LIB) or
    shutil.which("gcc") is None,
    reason="needs the reference's sources (TURTLE_REF), oracle/_ref built from them and gcc")


def _shim(tmp):
    """libpng.so for the reference's dlopen: the copy Pillow ships."""
    PIL = pytest.importorskip("PIL")
    libs = os.path.join(os.path.dirname(os.path.dirname(PIL.__file__)), "pillow.libs")
    found = glob.glob(os.path.join(libs, "libpng16-*.so*"))
    if not found:
        pytest.skip("no libpng for the reference")
    os.makedirs(os.path.join(tmp, "shim"), exist_ok=True)
    os.symlink(found[0], os.path.join(tmp, "shim", "libpng.so"))
    return os.path.join(tmp, "shim") + ":" + libs


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    """share/topography (four SRTM3-sized tiles cut from one smooth field with 25 degree
    slopes), share/data/ww15mgh.grd (a 10 degree geoid, 8 values per line like EGM96's file),
    and the four examples built against each library."""
    tmp = str(tmp_path_factory.mktemp("examples"))
    tiles = os.path.join(tmp, "tiles")
    os.makedirs(tiles)
    n = 1201
    for lat in (45, 46):
        for lon in (2, 3):
            la = lat + 1. - np.arange(n)[:, None] / (n - 1.)  # north row first
            lo = lon + np.arange(n)[None, :] / (n - 1.)
            z = (1000. + 200. * np.sin(7.3 * la) * np.cos(5.1 * lo) +
                 150. * np.sin(300. * la + 170. * lo) * np.cos(90. * lo))
            z.round().astype(">i2").tofile(
                os.path.join(tiles, "N%02dE%03d.SRTMGL3.hgt" % (lat, lon)))
    geoid = os.path.join(tmp, "geoid.grd")
    with open(geoid, "w") as f:
        f.write("-90 90 0 360 10 10\n")
        for la in range(90, -91, -10):
            row = ["%.3f" % (20. * np.sin(np.radians(la) * 2) + 15. * np.cos(np.radians(lo)))
                   for lo in range(0, 361, 10)]
            for i in range(0, len(row), 8):
                f.write(" ".join(row[i:i + 8]) + "\n")
    with open(os.path.join(tmp, "fixed_time.c"), "w") as f:  # example-pthread: srand(time(NULL))
        f.write("#include <time.h>\ntime_t time(time_t * t) { if (t) *t = 42; return 42; }\n")
    subprocess.run(["gcc", "-shared", "-fPIC", "-o", os.path.join(tmp, "fixed_time.so"),
                    os.path.join(tmp, "fixed_time.c")], check=True)
    sides = {"reference": (os.path.join(H.REF_SOURCES, "include"), os.path.dirname(REF_LIB),
                           "turtle_ref"),
             "product": (os.path.join(ROOT, "include"), os.path.join(ROOT, "turtle_b200"),
                         "turtle_b200")}
    for side, (inc, libdir, lib) in sides.items():
        d = os.path.join(tmp, side)
        os.makedirs(os.path.join(d, "share", "data"))
        os.symlink(tiles, os.path.join(d, "share", "topography"))
        shutil.copy(geoid, os.path.join(d, "share", "data", "ww15mgh.grd"))
        for ex in ("projection", "demo", "stepper", "pthread"):
            subprocess.run(["gcc", "-O2", "-o", os.path.join(d, ex),
                            os.path.join(EXAMPLES, "example-%s.c" % ex), "-I" + inc, "-L" + libdir,
                            "-l" + lib, "-Wl,-rpath," + libdir, "-lm", "-lpthread"], check=True)
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = _shim(tmp) + ":" + env.get("LD_LIBRARY_PATH", "")

    def run(side, ex, *args, preload=None):
        e = dict(env, LD_PRELOAD=preload) if preload else env
        r = subprocess.run([os.path.join(tmp, side, ex)] + [str(a) for a in args],
                           cwd=os.path.join(tmp, side), env=e, stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True, timeout=120)
        assert r.returncode == 0, (side, ex, args, r.stderr)
        return r.stdout
    # example-projection writes the map the other examples load
    for side in sides:
        run(side, "projection")
    return tmp, run


def _nodes(path):
    m = tb.Map(path=path)
    info, tag = m.meta()
    z = np.array([[m.node(ix, iy)[2] for ix in range(info.nx)] for iy in range(info.ny)])
    return (info.nx, info.ny, tuple(info.x), tuple(info.y), tuple(info.z), tag), z


def test_example_projection_writes_the_same_map(world):
    tmp, run = world
    a = _nodes(os.path.join(tmp, "reference", "share", "data", "pdd-30m.png"))
    b = _nodes(os.path.join(tmp, "product", "share", "data", "pdd-30m.png"))
    assert a[0] == b[0] == (201, 201, (693530.7, 699530.7), (6515284.5, 6521284.5),
                            (500., 1500.), "Lambert 93")
    assert a[1].tobytes() == b[1].tobytes()
    assert a[1].max() - a[1].min() > 100.  # a real relief, not a clipped constant
    # ... and each library reads the other's file
    for side, other in (("reference", "product"), ("product", "reference")):
        shutil.copy(os.path.join(tmp, other, "share", "data", "pdd-30m.png"),
                    os.path.join(tmp, side, "share", "data", "pdd-30m.png"))
    assert run("reference", "demo") == run("product", "demo")
    run("reference", "projection")
    run("product", "projection")


def test_example_demo_prints_the_same(world):
    tmp, run = world
    text = run("product", "demo")
    assert text == run("reference", "demo")
    assert "Lambert 93" in text and "UTM 31N" in text and text.count("\n") >= 17


@pytest.mark.parametrize("args", [(), (120, 2, 1), (200, 10, 100, 1e-2, 0.4), (26, 5, 0),
                                  (310, 1, 10, 1e-3, 0.3), (75, 0.5), (0, 0), (180, -1, 1),
                                  (26, 5, 1, 1e-2, 0.4), (91, 3, 0, 1e-2, 0.4)])
def test_example_stepper_prints_the_same_rock_length(world, args):
    """azimuth, elevation, approximation range, resolution factor, slope factor
    (example-stepper.c:76-86): the rock length to six decimals."""
    tmp, run = world
    want, got = run("reference", "stepper", *args), run("product", "stepper", *args)
    assert got == want
    float(got)


def test_example_stepper_crosses_rock(world):
    tmp, run = world
    lengths = [float(run("product", "stepper", az, 1.)) for az in (0, 75, 200, 310)]
    assert max(lengths) > 1000. and min(lengths) >= 0.


def test_example_pthread_prints_the_same_tracks(world):
    """Four threads, one client each on a locked stack; tracks drawn from srand(time(NULL)),
    pinned for both runs by a preloaded time(). Lines come out in thread order of the run:
    compared as sets of `latitude longitude elevation`."""
    tmp, run = world
    preload = os.path.join(tmp, "fixed_time.so")

    def tracks(side):
        lines = run(side, "pthread", preload=preload).splitlines()
        assert len(lines) > 1000
        return sorted(l.split("] ")[1] for l in lines)
    assert tracks("product") == tracks("reference")
