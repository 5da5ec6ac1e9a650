"""Many stations in one call: turtle_stepper_trace_fans[_device] and
turtle_stepper_horizons[_device].

Each result is promised byte for byte equal to the one-station call (turtle_stepper_trace_fan,
turtle_stepper_horizon) on the same station, which the rest of the suite holds to the oracle.
So the one-station calls are the reference here.

Without a GPU: the argument checks (before any device call, with a NULL plan), the loud
failure without a device, and the declarations and struct layout from C99 and C++11.
On a B200: every scene of test_gpu_geometries.py with stations on its ground, far from every
map and stack, with a NaN position and twice the same; host slices that begin within a station;
thousands of small stations; many-station calls in flight with one-station calls.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import turtle_b200 as tb
from tests.test_fan import FIELDS
from tests.test_gpu_geometries import _draw, case, globe_stacks, tiles2  # noqa: F401
from tests.test_gpu_inflight import (Call, Hold, _bytes, _fields, assert_same, run_held, solo,
                                     warm, world)  # noqa: F401
from tests.test_scenes_extra import mixed_stack, sw_stack  # noqa: F401
from turtle_b200 import _lib
from turtle_b200.api import HORIZON_INVALID, HORIZON_RESULT, TRACE_INVALID

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FANS = ["turtle_stepper_trace_fans", "turtle_stepper_trace_fans_device"]
HORIZONS = ["turtle_stepper_horizons", "turtle_stepper_horizons_device"]
NAN = float("nan")


# ---- without a GPU --------------------------------------------------------------------------

def fans_call(name, struct=True, n_station=2, latitude=True, longitude=True, position=True,
              n_azimuth=3, azimuth=True, n_elevation=4, elevation=True, bundle=2, rule=True):
    """The C entry point with a NULL plan; -> (code, message) or (0, '')."""
    la, lo, pos = np.zeros(n_station), np.zeros(n_station), np.zeros((n_station, 3))
    az, el = np.zeros(n_azimuth), np.zeros(n_elevation)
    f = _lib.Fans(n_station, la.ctypes.data if latitude else None,
                  lo.ctypes.data if longitude else None, pos.ctypes.data if position else None,
                  n_azimuth, n_elevation, az.ctypes.data if azimuth else None,
                  el.ctypes.data if elevation else None, bundle)
    r = tb.trace_rule(6000.) if rule else None
    out = np.zeros(max(n_station * n_azimuth * n_elevation, 1), dtype=tb.TRACE_RESULT)
    args = [None, C.byref(f) if struct else None, C.byref(r) if r is not None else None,
            out.ctypes.data, None]
    if name.endswith("_device"):
        args.append(None)
    try:
        tb.api._check(getattr(_lib.lib, name)(*args))
    except tb.TurtleError as e:
        return e.code, str(e)
    return 0, ""


def horizons_call(name, n_station=2, latitude=True, longitude=True, position=True, n_azimuth=3,
                  azimuth=True, window=(-90., 90.), tolerance=1e-6, rule=True, results=True):
    la, lo, pos, az = np.zeros(n_station), np.zeros(n_station), np.zeros((n_station, 3)), \
        np.zeros(n_azimuth)
    out = np.zeros(max(n_station * n_azimuth, 1), dtype=HORIZON_RESULT)
    r = tb.trace_rule(6000.) if rule else None
    args = [None, n_station, la.ctypes.data if latitude else None,
            lo.ctypes.data if longitude else None, pos.ctypes.data if position else None,
            n_azimuth, az.ctypes.data if azimuth else None, window[0], window[1], tolerance,
            C.byref(r) if r is not None else None, out.ctypes.data if results else None]
    if name.endswith("_device"):
        args.append(None)
    try:
        tb.api._check(getattr(_lib.lib, name)(*args))
    except tb.TurtleError as e:
        return e.code, str(e)
    return 0, ""


def _expect(code, message, want, name, kw):
    assert code == want, (kw, message)
    assert message.startswith("{ %s [#%d], " % (name, want)), message


@pytest.mark.parametrize("name", FANS)
def test_fans_arguments_are_checked_first(name):
    """Address and domain errors are raised before the plan or the device is touched; an
    empty call touches nothing, not even the (NULL) plan."""
    for kw in (dict(struct=False), dict(latitude=False), dict(longitude=False),
               dict(position=False), dict(azimuth=False), dict(elevation=False)):
        _expect(*fans_call(name, **kw), 1, name, kw)  # TURTLE_RETURN_BAD_ADDRESS
    for kw in (dict(bundle=3), dict(n_elevation=5), dict(rule=False)):
        _expect(*fans_call(name, **kw), 6, name, kw)  # TURTLE_RETURN_DOMAIN_ERROR
    for kw in (dict(n_station=0), dict(n_station=0, latitude=False, longitude=False,
                                       position=False), dict(n_azimuth=0),
               dict(n_elevation=0), dict(n_azimuth=0, azimuth=False)):
        assert fans_call(name, **kw) == (0, ""), kw


@pytest.mark.parametrize("name", HORIZONS)
def test_horizons_arguments_are_checked_first(name):
    for kw in (dict(latitude=False), dict(longitude=False), dict(position=False),
               dict(azimuth=False), dict(results=False)):
        _expect(*horizons_call(name, **kw), 1, name, kw)
    for kw in (dict(tolerance=0.), dict(tolerance=NAN), dict(window=(10., 5.)),
               dict(window=(-90.5, 0.)), dict(window=(0., 91.)), dict(rule=False)):
        _expect(*horizons_call(name, **kw), 6, name, kw)
    for kw in (dict(n_station=0), dict(n_station=0, latitude=False, longitude=False,
                                       position=False, results=False),
               dict(n_azimuth=0), dict(n_azimuth=0, azimuth=False, results=False)):
        assert horizons_call(name, **kw) == (0, ""), kw


@pytest.mark.parametrize("name", FANS + HORIZONS)
def test_fails_loudly_without_gpu(name, has_gpu):
    if has_gpu:
        pytest.skip("a GPU is present")
    code, message = (fans_call if name in FANS else horizons_call)(name)
    assert code == 7 and "no CUDA device" in message and "no CPU fallback" in message


def test_header_declarations_compile(tmp_path):
    """Callers of the new declarations compile as pedantic C99 and C++11; struct turtle_fans
    has the size and offsets of its Python mirror."""
    offsets = {k: getattr(_lib.Fans, k).offset for k, _ in _lib.Fans._fields_}
    checks = " && ".join("(offsetof(struct turtle_fans, %s) == %d)" % kv for kv in offsets.items())
    src = ('#include <stddef.h>\n#include "turtle_b200.h"\n'
           'static enum turtle_return (*f)(struct turtle_plan *, const struct turtle_fans *,'
           ' const struct turtle_trace_rule *, struct turtle_trace_result *,'
           ' const struct turtle_trace_fields *) = turtle_stepper_trace_fans;\n'
           'static enum turtle_return (*g)(struct turtle_plan *, const struct turtle_fans *,'
           ' const struct turtle_trace_rule *, struct turtle_trace_result *,'
           ' const struct turtle_trace_fields *, void *) = turtle_stepper_trace_fans_device;\n'
           'static enum turtle_return (*h)(struct turtle_plan *, size_t, const double *,'
           ' const double *, const double *, size_t, const double *, double, double, double,'
           ' const struct turtle_trace_rule *, struct turtle_horizon *) = turtle_stepper_horizons;\n'
           'static enum turtle_return (*k)(struct turtle_plan *, size_t, const double *,'
           ' const double *, const double *, size_t, const double *, double, double, double,'
           ' const struct turtle_trace_rule *, struct turtle_horizon *, void *) ='
           ' turtle_stepper_horizons_device;\n'
           'int main(void) { return ((f != NULL) && (g != NULL) && (h != NULL) && (k != NULL) && '
           '(sizeof(struct turtle_fans) == %d) && %s) ? 0 : 1; }\n' % (C.sizeof(_lib.Fans), checks))
    for compiler, std, lang in (("gcc", "-std=c99", "c"), ("g++", "-std=c++11", "c++")):
        exe = str(tmp_path / ("stations_" + lang.replace("+", "x")))
        subprocess.run([compiler, std, "-Wall", "-Wextra", "-pedantic", "-Werror",
                        "-I" + os.path.join(ROOT, "include"), "-x", lang, "-", "-x", "none",
                        _lib.LIB_PATH, "-o", exe], input=src, text=True, check=True)
        env = dict(os.environ, LD_LIBRARY_PATH=os.path.dirname(_lib.LIB_PATH))
        assert subprocess.run([exe], env=env).returncode == 0
    assert C.sizeof(_lib.Fans) == 72


# ---- on a B200: the one-station calls are the reference ----------------------------------------

def one_by_one_fans(plan, stations, az, el, bundle, rule, names=FIELDS):
    """Records and fields of the per-station trace_fan calls, concatenated."""
    la, lo, pos = stations
    per = len(az) * len(el)
    rec = np.zeros(len(la) * per, dtype=tb.TRACE_RESULT)
    fields = tb.Plan.host_fields(len(rec), names)
    for s in range(len(la)):
        part = slice(s * per, (s + 1) * per)
        f = {k: v[part] for k, v in fields.items()}
        fan = tb.Plan.make_fan(la[s], lo[s], pos[s], az, el, bundle=bundle)
        plan.trace_fan(fan, rule, results=rec[part], fields=f)
    return rec, fields


def many_fans(plan, stations, az, el, bundle, rule, names=FIELDS):
    n = len(stations[0]) * len(az) * len(el)
    rec = np.zeros(n, dtype=tb.TRACE_RESULT)
    fields = tb.Plan.host_fields(n, names)
    plan.trace_fans(tb.Plan.make_fans(*stations, az, el, bundle=bundle), rule, results=rec,
                    fields=fields)
    return rec, fields


def many_fans_device(plan, stations, az, el, bundle, rule, names=FIELDS):
    import torch
    n = len(stations[0]) * len(az) * len(el)
    rec = torch.full((n * 96,), 0xa5, dtype=torch.uint8, device="cuda")
    fields = _fields(n, names)
    plan.trace_fans_device(tb.Plan.make_fans(*stations, az, el, bundle=bundle), rule,
                           results=rec, fields=fields)
    torch.cuda.synchronize()
    return _bytes(dict(fields, records=rec))


def same_fans(got, want):
    (g_rec, g_fields), (w_rec, w_fields) = got, want
    assert g_rec.tobytes() == w_rec.tobytes()
    for k in w_fields:
        assert g_fields[k].tobytes() == w_fields[k].tobytes(), k


def same_device(got_bytes, want):
    w_rec, w_fields = want
    assert got_bytes["records"] == w_rec.tobytes()
    for k in w_fields:
        assert got_bytes[k] == w_fields[k].tobytes(), k


def one_by_one_horizons(plan, stations, az, rule, **kw):
    la, lo, pos = stations
    return np.stack([plan.horizon(la[s], lo[s], pos[s], az, rule, **kw) for s in range(len(la))])


def scene_stations(c):
    """7 stations of a scene: four 1 m over the ground of layer 0 at points drawn over its
    boxes and ground bands, one far from every map and stack (only a flat layer can hold it),
    one with a NaN position and the first one again."""
    rng = np.random.default_rng(11)
    la, lo, pos = [], [], []
    regions = c.boxes + c.ground
    for attempt in range(60):  # (layer 0 need not have data over every region)
        if len(la) == 4:
            break
        a, b, _h = _draw([regions[attempt % len(regions)]], 8, rng)
        p, idx = c.plan.position(a, b, np.ones(len(a)), 0)
        ok = np.flatnonzero(idx >= 0)
        if len(ok):
            la.append(a[ok[0]])
            lo.append(b[ok[0]])
            pos.append(p[ok[0]])
    assert len(la) == 4, c.name
    far = (-60., -100.)  # the South Pacific: no scene has data there
    la += [far[0], la[1], la[0]]
    lo += [far[1], lo[1], lo[0]]
    pos += [c.ora.ecef_from_geodetic([far[0]], [far[1]], [1000.])[0], np.full(3, NAN), pos[0]]
    return np.array(la), np.array(lo), np.array(pos)


# (n_azimuth, n_elevation, bundle): 63 rays per station (warps hold rays of two stations),
# elevation-major, azimuth-major, and a band of 32 elevations
GRIDS = [(7, 9, 1), (7, 9, 9), (5, 32, 32)]


def _grid(n_az, n_el):
    az = 360. * (np.arange(n_az) + 0.37) / n_az
    el = -10. + 50. * (np.arange(n_el) + 0.5) / n_el
    return az, el


@pytest.mark.gpu
def test_scene_fans_and_horizons(case):  # noqa: F811
    """trace_fans / horizons and their _device variants equal the one-station calls byte for
    byte; permuting the stations permutes the blocks; host slices may begin within a
    station."""
    import torch
    st = scene_stations(case)
    n_st = len(st[0])
    plan, rule = case.plan, case.rule
    for n_az, n_el, bundle in GRIDS:
        az, el = _grid(n_az, n_el)
        want = one_by_one_fans(plan, st, az, el, bundle, rule)
        same_fans(many_fans(plan, st, az, el, bundle, rule), want)
        assert plan.counters()["rays"] == n_st * n_az * n_el
        same_device(many_fans_device(plan, st, az, el, bundle, rule), want)
        per = n_az * n_el
        blocks = want[0].reshape(n_st, per)
        assert (blocks[5]["status"] == TRACE_INVALID).all()  # the NaN position
        assert blocks[6].tobytes() == blocks[0].tobytes()    # the duplicate
        perm = np.random.default_rng(n_az + bundle).permutation(n_st)
        rec, _ = many_fans(plan, tuple(a[perm] for a in st), az, el, bundle, rule, ["status"])
        assert rec.tobytes() == blocks[perm].tobytes()
        # host slices of whole bands, beginning within a station
        os.environ["TURTLE_B200_FAN_SLICE_RAYS"] = str(max(per * n_st // 8, 1))
        try:
            same_fans(many_fans(plan, st, az, el, bundle, rule), want)
        finally:
            del os.environ["TURTLE_B200_FAN_SLICE_RAYS"]

    az = 360. * (np.arange(13) + 0.21) / 13
    kw = dict(elevation=(-30., 60.), tolerance=1e-4)
    want = one_by_one_horizons(plan, st, az, rule, **kw)
    got = plan.horizons(*st, az, rule, **kw)
    assert got.shape == (n_st, len(az)) and got.tobytes() == want.tobytes()
    assert plan.counters()["rays"] == want["n_probes"].sum()
    d_out = torch.full((got.size * 96,), 0xa5, dtype=torch.uint8, device="cuda")
    plan.horizons_device(*st, az, rule, d_out, **kw)
    torch.cuda.synchronize()
    assert d_out.cpu().numpy().tobytes() == want.tobytes()
    assert (want[5]["status"] == HORIZON_INVALID).all()
    assert want[6].tobytes() == want[0].tobytes()
    perm = np.random.default_rng(2).permutation(n_st)
    assert plan.horizons(*(a[perm] for a in st), az, rule, **kw).tobytes() == \
        want[perm].tobytes()


# ---- many small stations ----------------------------------------------------------------------

def _many(world, n, seed):
    rng = np.random.default_rng(seed)
    lat = rng.uniform(world.station[0] - 0.2, world.station[0] + 0.2, n)
    lon = rng.uniform(world.station[1] - 0.2, world.station[1] + 0.2, n)
    pos, idx = world.plan.position(lat, lon, np.ones(n), 0)
    assert (idx >= 0).all()
    return lat, lon, pos


@pytest.mark.gpu
def test_many_small_stations(world):  # noqa: F811
    """3000 stations x a 2 x 4 fan and x 8 azimuths, in one call each: a random 50 of them
    equal their one-station calls; the counters report every ray (probe) and, for the device
    call, one launch."""
    import torch
    plan, rule = world.plan, world.rule
    st = _many(world, 3000, 7)
    az, el = np.array([17., 203.]), np.array([-5., 3., 11., 25.])
    rec, fields = many_fans(plan, st, az, el, 2, rule)
    assert plan.counters()["rays"] == 3000 * 8
    got = many_fans_device(plan, st, az, el, 2, rule)
    c = plan.counters(sync=True)
    assert c["rays"] == 3000 * 8 and c["launches"] == 1
    same_device(got, (rec, fields))
    pick = np.sort(np.random.default_rng(8).choice(3000, 50, replace=False))
    sub = tuple(a[pick] for a in st)
    want = one_by_one_fans(plan, sub, az, el, 2, rule)
    rows = (pick[:, None] * 8 + np.arange(8)).reshape(-1)
    same_fans((rec[rows], {k: v[rows] for k, v in fields.items()}), want)

    az = np.arange(8) * 45. + 3.
    kw = dict(elevation=(-30., 60.), tolerance=1e-4)
    hz = plan.horizons(*st, az, rule, **kw)
    assert plan.counters()["rays"] == hz["n_probes"].sum()
    d_out = torch.empty(hz.size * 96, dtype=torch.uint8, device="cuda")
    plan.horizons_device(*st, az, rule, d_out, **kw)
    torch.cuda.synchronize()
    c = plan.counters(sync=True)
    assert c["launches"] == 1 and c["rays"] == hz["n_probes"].sum()
    assert d_out.cpu().numpy().tobytes() == hz.tobytes()
    assert one_by_one_horizons(plan, sub, az, rule, **kw).tobytes() == hz[pick].tobytes()


# ---- in flight --------------------------------------------------------------------------------

class Fans(Call):
    def __init__(self, plan, stations, az, el, rule, bundle=1, names=("length0", "status")):
        super().__init__(plan, "trace_fans_device %d x %dx%d" % (len(stations[0]), len(az), len(el)))
        self.fans = tb.Plan.make_fans(*stations, az, el, bundle=bundle)
        self.n, self.rule, self.names = len(stations[0]) * len(az) * len(el), rule, list(names)

    def prepare(self):
        import torch
        self.out = _fields(self.n, self.names)
        self.out["records"] = torch.full((self.n * 96,), 0xa5, dtype=torch.uint8, device="cuda")

    def issue(self, stream):
        fields = {k: v for k, v in self.out.items() if k != "records"}
        self.plan.trace_fans_device(self.fans, self.rule, results=self.out["records"],
                                    fields=fields, stream=stream.cuda_stream)

    def outputs(self):
        return _bytes(self.out)


class Horizons(Call):
    def __init__(self, plan, stations, az, rule):
        super().__init__(plan, "horizons_device %d x %d" % (len(stations[0]), len(az)))
        self.stations, self.az, self.rule = stations, np.asarray(az, dtype=float), rule

    def prepare(self):
        import torch
        self.out = dict(records=torch.full((len(self.stations[0]) * len(self.az) * 96,), 0xa5,
                                           dtype=torch.uint8, device="cuda"))

    def issue(self, stream):
        self.plan.horizons_device(*self.stations, self.az, self.rule, self.out["records"],
                                  elevation=(-30., 60.), tolerance=1e-4,
                                  stream=stream.cuda_stream)

    def outputs(self):
        return _bytes(self.out)


def _angles(seed, n_az, n_el=0):
    rng = np.random.default_rng(seed)
    return np.sort(rng.uniform(0., 360., n_az)), np.sort(rng.uniform(-10., 40., n_el))


@pytest.mark.gpu
def test_many_station_calls_in_flight(world):  # noqa: F811
    """Eight device calls, each on its own held stream: many-station fans and horizons mixed
    with one-station ones, each equal to its solo result."""
    p, rule = world.plan, world.rule
    calls = []
    for k in range(4):
        st = _many(world, 40 + 13 * k, 30 + k)
        az, el = _angles(40 + k, 9 + k, 7)
        calls.append(Fans(p, st, az, el, rule) if k % 2 == 0 else
                     Horizons(p, st, _angles(40 + k, 11 + k)[0], rule))
    calls += [world.fan(50), world.horizon(51), world.fan(52, n_az=23, n_el=11),
              world.horizon(53, n_az=29)]
    calls = [calls[i] for i in (0, 4, 1, 5, 2, 6, 3, 7)]
    warm(world, 500, 0)  # tables of 79 stations and 19 angles in every slot: none grows
    want = [solo(c) for c in calls]
    run_held(calls, 300)
    for c, w in zip(calls, want):
        assert_same(c, w)


@pytest.mark.gpu
def test_station_tables_grow_under_pending_calls(world):  # noqa: F811
    """A call with more stations than any before grows its slot's table while a smaller call
    holds another slot: neither is disturbed. The solo results come from a plan of its own."""
    import torch
    alone = world.stepper.freeze(0)
    az, el = _angles(60, 5, 3)

    def calls(plan):
        out = []
        for k, n in enumerate((30, 70, 150, 320)):
            small = Fans(plan, _many(world, 2, 61 + k), az, el, world.rule)
            st = _many(world, n, 70 + k)
            grow = Fans(plan, st, az, el, world.rule) if k % 2 == 0 else \
                Horizons(plan, st, az, world.rule)
            out.append((small, grow))
        return out

    want = [(solo(a), solo(b)) for a, b in calls(alone)]
    pairs = calls(world.plan)
    warm(world, 30, 0)
    for a, b in pairs:
        a.prepare()
        b.prepare()
    torch.cuda.synchronize()
    for a, b in pairs:
        hold = Hold(60)
        a.issue(hold.stream())
        assert hold.pending(), "the hold was over before %s was issued" % b.name
        b.issue(hold.stream())
    torch.cuda.synchronize()
    for (a, b), (wa, wb) in zip(pairs, want):
        assert_same(a, wa)
        assert_same(b, wb)
