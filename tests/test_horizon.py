"""The horizon of a station: turtle_stepper_horizon[_device], a K-ary search for the elevation
that separates the rays entering the ground from the rays reaching open sky, run on the device.

Without a GPU: the argument checks (before any device call, with a NULL plan), the loud failure
without a device, the layout of the record. On a B200: the bracket of an analytic horizon (steep
cones at known distances), bit-for-bit agreement of both ends with the tracer, a dense fan
around the bracket, the reference's own rays around it, determinism and the statuses."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.common import Scene, lambert_map, ulp_distance
from turtle_b200 import _lib
from turtle_b200.api import (HORIZON_ABOVE, HORIZON_BELOW, HORIZON_FOUND, HORIZON_INVALID,
                             HORIZON_RESULT)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RULE = dict(altitude_max=6000., max_steps=20000)


def raw_call(name, n=1, position=(0., 0., 0.), azimuth=True, window=(-90., 90.),
             tolerance=1e-6, rule=True, results=True):
    """The C entry point with a NULL plan; -> (code, message) or (0, '')."""
    az = np.zeros(n)
    out = np.zeros(n, dtype=HORIZON_RESULT)
    pos = (C.c_double * 3)(*position) if position is not None else None
    r = tb.trace_rule(6000.) if rule else None
    args = [None, 45., 2., pos, n, az.ctypes.data if azimuth else None, window[0], window[1],
            tolerance, C.byref(r) if r is not None else None,
            out.ctypes.data if results else None]
    if name.endswith("_device"):
        args.append(None)
    try:
        tb.api._check(getattr(_lib.lib, name)(*args))
    except tb.TurtleError as e:
        return e.code, str(e)
    return 0, ""


@pytest.mark.parametrize("name", ["turtle_stepper_horizon", "turtle_stepper_horizon_device"])
def test_arguments_are_checked_first(name):
    """Domain and address errors are raised before the plan or the device is touched."""
    domain = [dict(tolerance=0.), dict(tolerance=-1e-3), dict(tolerance=float("nan")),
              dict(window=(10., 5.)), dict(window=(5., 5.)), dict(window=(-90.5, 0.)),
              dict(window=(0., 91.)), dict(window=(float("nan"), 10.)), dict(rule=False)]
    for kw in domain:
        code, message = raw_call(name, **kw)
        assert code == 6, (kw, message)  # TURTLE_RETURN_DOMAIN_ERROR
        assert message.startswith("{ %s [#6], " % name), message
    for kw in (dict(position=None), dict(azimuth=False), dict(results=False)):
        code, message = raw_call(name, **kw)
        assert code == 1, (kw, message)  # TURTLE_RETURN_BAD_ADDRESS
        assert message.startswith("{ %s [#1], " % name), message
    # nothing to search: nothing is touched, not even the (NULL) plan
    assert raw_call(name, n=0) == (0, "")


@pytest.mark.parametrize("name", ["turtle_stepper_horizon", "turtle_stepper_horizon_device"])
def test_fails_loudly_without_gpu(name, has_gpu):
    if has_gpu:
        pytest.skip("a GPU is present")
    code, message = raw_call(name)
    assert code == 7 and "no CUDA device" in message and "no CPU fallback" in message


def test_header_declarations_compile(tmp_path):
    """A caller of the new declarations compiles as pedantic C99 and C++11; the record is the
    96 bytes the Python mirror reads."""
    src = ('#include <stddef.h>\n#include "turtle_b200.h"\n'
           'static enum turtle_return (*f)(struct turtle_plan *, double, double, const double *,'
           ' size_t, const double *, double, double, double, const struct turtle_trace_rule *,'
           ' struct turtle_horizon *) = turtle_stepper_horizon;\n'
           'static enum turtle_return (*g)(struct turtle_plan *, double, double, const double *,'
           ' size_t, const double *, double, double, double, const struct turtle_trace_rule *,'
           ' struct turtle_horizon *, void *) = turtle_stepper_horizon_device;\n'
           'int main(void) { return ((f != NULL) && (g != NULL) && '
           '(sizeof(struct turtle_horizon) == 96) && '
           '(offsetof(struct turtle_horizon, length) == 64) && '
           '(offsetof(struct turtle_horizon, medium) == 72) && '
           '(offsetof(struct turtle_horizon, n_iterations) == 92) && '
           '(TURTLE_HORIZON_FOUND == 0) && (TURTLE_HORIZON_INVALID == 3)) ? 0 : 1; }\n')
    for compiler, std, lang in (("gcc", "-std=c99", "c"), ("g++", "-std=c++11", "c++")):
        exe = str(tmp_path / ("horizon_" + lang.replace("+", "x")))
        subprocess.run([compiler, std, "-Wall", "-Wextra", "-pedantic", "-Werror",
                        "-I" + os.path.join(ROOT, "include"), "-x", lang, "-", "-x", "none",
                        _lib.LIB_PATH, "-o", exe], input=src, text=True, check=True)
        env = dict(os.environ, LD_LIBRARY_PATH=os.path.dirname(_lib.LIB_PATH))
        assert subprocess.run([exe], env=env).returncode == 0
    for k, offset in (("elevation", 0), ("direction", 16), ("length", 64), ("medium", 72),
                      ("status", 80), ("clear_status", 84), ("n_probes", 88),
                      ("n_iterations", 92)):
        assert HORIZON_RESULT.fields[k][1] == offset, k


# ---- scenes ---------------------------------------------------------------------------------

STATION = (45.45, 2.65)
AZIMUTHS = np.arange(48) * 7.5 + 0.3

# Steep cones on flat ground around (45.1, 2.1): (node offset east, node offset north, height,
# base radius in metres). The nodes are 5e-4 degrees apart (39 m east, 56 m north); the cones
# lie 3.3 - 5.2 km away, 57 degrees of azimuth or more apart, each narrower than its distance
# (so its apex is the highest point of its azimuth as seen from the station).
CONES_CENTRE = (45.1, 2.1)
CONES = [(100, 0, 600., 800.), (0, 80, 900., 800.), (-60, -60, 400., 800.),
         (50, -90, 1200., 800.), (-120, 40, 700., 800.)]


def cones_map():
    n = 401
    lon = np.linspace(2.0, 2.2, n)
    lat = np.linspace(45.0, 45.2, n)
    east = (lon - CONES_CENTRE[1]) * 111195. * np.cos(np.radians(CONES_CENTRE[0]))
    north = (lat - CONES_CENTRE[0]) * 111195.
    X, Y = np.meshgrid(east, north)
    z = np.zeros((n, n))
    for dx, dy, h, radius in CONES:
        x0, y0 = east[200 + dx], north[200 + dy]
        z = np.maximum(z, h * (1. - np.hypot(X - x0, Y - y0) / radius))
    return dict(nx=n, ny=n, x=(2.0, 2.2), y=(45.0, 45.2), z=(0., 3000.), projection=None,
                values=z)


class Case:
    def __init__(self, name, scene, station):
        self.name, self.scene, self.station = name, scene, station
        self.ora = scene.oracle()
        self.stepper, self.maps, self.stacks = scene.product()
        self.plan = self.stepper.freeze(0)
        self.origin, index = self.stepper.position(station[0], station[1], 1.0, 0)
        assert index >= 0
        self.rule = tb.trace_rule(**RULE)

    def horizon(self, azimuth=AZIMUTHS, **kw):
        return self.plan.horizon(self.station[0], self.station[1], self.origin, azimuth,
                                 self.rule, **kw)


def make_case(name, small_stack):
    A, F, S = H.ADD_MAP, H.ADD_FLAT, H.ADD_STACK
    if name == "stack":  # the single-stack kernel
        return Case(name, Scene(stacks=[small_stack], ops=[(S, 0, 0.)], range=0.), STATION)
    if name in ("generic_r0", "generic_r10"):  # projected map over stack over flat
        ora = H.Driver(H.best_oracle())
        maps = [lambert_map(ora, STATION[0], STATION[1], n=201, half=8000.)]
        ora.close()
        sc = Scene(maps=maps, stacks=[small_stack], ops=[(F, 0, 0.), (S, 0, 0.), (A, 0, 0.)],
                   range=0. if name == "generic_r0" else 10.)
        return Case(name, sc, STATION)
    if name == "cones":  # a geodetic test map
        sc = Scene(maps=[cones_map()], ops=[(A, 0, 0.)], range=0., resolution=1e-3)
        return Case(name, sc, CONES_CENTRE)
    raise KeyError(name)


_cases = {}


@pytest.fixture(scope="module", params=["stack", "generic_r0", "generic_r10", "cones"])
def case(request, small_stack):
    if request.param not in _cases:
        _cases[request.param] = make_case(request.param, small_stack)
    return _cases[request.param]


@pytest.fixture(scope="module")
def cones(small_stack):
    if "cones" not in _cases:
        _cases["cones"] = make_case("cones", small_stack)
    return _cases["cones"]


def obstructed(records):
    """The first medium change of the whole trace is into a medium >= 0 (a change into -1,
    leaving the data, ends the trace)."""
    return (records["n_changes"] >= 2) | ((records["n_changes"] == 1) & (records["index"][:, 0] >= 0))


def apex_angles(cones):
    ora = cones.ora
    ix = np.array([200 + c[0] for c in CONES])
    iy = np.array([200 + c[1] for c in CONES])
    lon, lat, z = ora.map_node(0, ix, iy)
    apex = ora.ecef_from_geodetic(lat, lon, z)
    n = len(CONES)
    la, lo = np.full(n, cones.station[0]), np.full(n, cones.station[1])
    return ora.ecef_to_horizontal(la, lo, apex - cones.origin[None])


# ---- on the GPU -----------------------------------------------------------------------------

@pytest.mark.gpu
def test_analytic_horizon(cones):
    """Toward the apex of each cone the horizon is the apex's elevation. elevation[0] is below
    it exactly (a ray above the apex node passes over every point of the bilinear surface).
    elevation[1] can only be below it by what the stepper fails to see: a ray that passes
    under the apex by d metres crosses a tip about 2 d / s wide (s: side slope, at most
    1.5 x sqrt(2) on a diagonal of the bilinear cells), and the steps shrink to the
    resolution r near the ground, so tips narrower than ~r can be stepped over. Hence
    eps = 4 r s / D (D: the distance of the apex), 0.9e-4 - 1.2e-4 degrees here; the
    misses measured on a B200 are 2e-6 - 5e-6 degrees."""
    az, el = apex_angles(cones)
    res = cones.horizon(az, tolerance=1e-6)
    assert (res["status"] == HORIZON_FOUND).all(), res["status"]
    slope = max(c[2] / c[3] for c in CONES) * np.sqrt(2.)
    distance = np.array([np.hypot(c[0] * 39.3, c[1] * 55.6) for c in CONES])
    eps = np.degrees(4. * 1e-3 * slope / distance)
    print("apex - elevation[1] (deg):", el - res["elevation"][:, 1], "eps:", eps)
    assert (res["elevation"][:, 0] <= el).all()
    assert (el <= res["elevation"][:, 1] + eps).all()
    assert (res["elevation"][:, 1] - res["elevation"][:, 0] <= 1e-6).all()


@pytest.mark.gpu
def test_ends_are_the_tracer_bit_for_bit(case):
    res = case.horizon(tolerance=1e-6)
    found = res["status"] == HORIZON_FOUND
    assert found.sum() >= len(res) // 2, res["status"]
    r = res[found]
    width = r["elevation"][:, 1] - r["elevation"][:, 0]
    assert ((width > 0) & (width <= 1e-6)).all()
    lat, lon = case.station
    n = len(r)
    for k in (0, 1):
        want = case.ora.ecef_from_horizontal(np.full(n, lat), np.full(n, lon),
                                             AZIMUTHS[found], r["elevation"][:, k])
        assert ulp_distance(r["direction"][:, k], want).max() <= 4
    origins = np.repeat(case.origin[None], n, 0)
    rec0, cross0 = case.plan.trace_crossings(origins, r["direction"][:, 0], case.rule, 1)
    assert (rec0["n_changes"] >= 1).all()
    assert cross0[:, 0]["length"].tobytes() == r["length"].tobytes()
    assert np.array_equal(cross0[:, 0]["to"], r["medium"][:, 1])
    assert (r["medium"][:, 1] >= 0).all() and (r["medium"][:, 1] != r["medium"][:, 0]).all()
    rec1, cross1 = case.plan.trace_crossings(origins, r["direction"][:, 1], case.rule, 1)
    assert not obstructed(rec1).any()
    assert np.array_equal(rec1["status"], r["clear_status"])
    assert (r["medium"][:, 0] == r["medium"][0, 0]).all()  # one station, one medium


@pytest.mark.gpu
def test_dense_fan_around_the_bracket(case):
    """0.01-degree steps of a fan: above elevation[1] clear, below elevation[0] obstructed."""
    res = case.horizon(tolerance=1e-6)
    lat, lon = case.station
    k = np.arange(1, 6) * 0.01
    checked = 0
    for i in np.flatnonzero(res["status"] == HORIZON_FOUND):
        lo, hi = res["elevation"][i]
        el = np.concatenate([lo - k[lo - k >= -90.], hi + k[hi + k <= 90.]])
        below = (el < lo)
        fan = tb.Plan.make_fan(lat, lon, case.origin, [AZIMUTHS[i]], el)
        rec = np.zeros(len(el), dtype=tb.TRACE_RESULT)
        case.plan.trace_fan(fan, case.rule, results=rec)
        assert np.array_equal(obstructed(rec), below), (i, lo, hi, obstructed(rec), below)
        checked += 1
    assert checked >= len(res) // 2


@pytest.mark.gpu
def test_against_the_reference(case):
    """With the reference's own directions, rays 1e-3 degrees below elevation[0] are obstructed
    and 1e-3 degrees above elevation[1] are clear, on every azimuth, for the C restatement and
    (its sources present) the compiled reference. At the bracket ends themselves -- grazing
    rays by construction -- agreement is reported, not asserted."""
    res = case.horizon(tolerance=1e-6)
    found = np.flatnonzero(res["status"] == HORIZON_FOUND)
    lat, lon = case.station
    n = len(found)
    origins = np.repeat(case.origin[None], n, 0)
    rule = H.rule(**RULE)
    libraries = [H.PORT] + ([H.REF] if os.path.exists(H.REF) else [])
    for library in libraries:
        ora = case.ora if library == H.best_oracle() else case.scene.oracle(library)
        for k, sign, want in ((0, -1., True), (1, 1., False)):
            el = res["elevation"][found, k]
            d = ora.ecef_from_horizontal(np.full(n, lat), np.full(n, lon), AZIMUTHS[found],
                                         el + sign * 1e-3)
            rec, _ = ora.trace_crossings(origins, d, rule, 1)
            assert (obstructed(rec) == want).all(), (library, k, np.flatnonzero(obstructed(rec) != want))
            rec, _ = ora.trace_crossings(origins, res["direction"][found, k], rule, 1)
            print("%s %s: %s end, the reference agrees on %d of %d rays" % (
                case.name, os.path.basename(library), "obstructed" if want else "clear",
                int((obstructed(rec) == want).sum()), n))


@pytest.mark.gpu
def test_deterministic(case):
    import torch
    want = case.horizon(tolerance=1e-5)
    for grid in ((1, 32), (2, 64), (3, 96), (0, 0)):
        case.plan.launch_set(*grid)
        assert case.horizon(tolerance=1e-5).tobytes() == want.tobytes(), grid
    case.plan.launch_set(0, 0)
    case.plan.specialise_set(0)
    try:
        assert case.horizon(tolerance=1e-5).tobytes() == want.tobytes()
    finally:
        case.plan.specialise_set(1)
    perm = np.random.default_rng(5).permutation(len(AZIMUTHS))
    got = case.horizon(AZIMUTHS[perm], tolerance=1e-5)
    # (n_iterations is the time of the warp that searched the azimuth: it depends on
    # nothing but the azimuth either)
    assert got.tobytes() == want[perm].tobytes()
    for i in range(0, len(AZIMUTHS), 5):
        assert case.horizon(AZIMUTHS[i:i + 1], tolerance=1e-5).tobytes() == want[i:i + 1].tobytes()
    out = torch.zeros(len(AZIMUTHS) * HORIZON_RESULT.itemsize, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        case.plan.horizon_device(case.station[0], case.station[1], case.origin, AZIMUTHS,
                                 case.rule, out, tolerance=1e-5, stream=stream.cuda_stream)
    stream.synchronize()
    assert out.cpu().numpy().tobytes() == want.tobytes()
    c = case.plan.counters(sync=True)
    assert c["rays"] == want["n_probes"].sum() and c["samples"] >= c["steps"] > 0


@pytest.mark.gpu
def test_statuses_and_counters(cones):
    lat, lon = cones.station
    rule = cones.rule
    # on the summit of the highest cone, nothing rises above the horizontal
    dx, dy = 50, -90
    top = (45.0 + (200 + dy) * 5e-4, 2.0 + (200 + dx) * 5e-4)
    summit, _ = cones.stepper.position(top[0], top[1], 1.0, 0)
    res = cones.plan.horizon(top[0], top[1], summit, AZIMUTHS, rule, elevation=(0., 90.))
    assert (res["status"] == HORIZON_BELOW).all()
    assert (res["elevation"][:, 1] == 0.).all() and np.isnan(res["elevation"][:, 0]).all()
    assert (res["clear_status"] >= 0).all() and (res["n_probes"] == 32).all()
    # a window entirely into the ground
    res = cones.horizon(elevation=(-90., -80.))
    assert (res["status"] == HORIZON_ABOVE).all()
    assert (res["elevation"][:, 0] == -80.).all() and np.isnan(res["elevation"][:, 1]).all()
    assert (res["medium"][:, 1] >= 0).all()
    # a station that is not finite, or off the data
    nan = float("nan")
    off_data = cones.ora.ecef_from_geodetic([45.5], [2.1], [10.])[0]  # north of the map
    for station, origin in (((lat, lon), (nan, 0., 0.)), ((nan, lon), cones.origin),
                            ((45.5, 2.1), off_data)):
        res = cones.plan.horizon(station[0], station[1], origin, AZIMUTHS[:4], rule)
        assert (res["status"] == HORIZON_INVALID).all(), station
    # the probes are the plan's rays
    res = cones.horizon(tolerance=1e-4)
    c = cones.plan.counters()
    assert c["rays"] == res["n_probes"].sum() > 0
    assert c["samples"] >= c["steps"] > 0
