"""The length of every ray in every cell of a voxel grid: turtle_stepper_trace_voxels[_device]
and turtle_stepper_trace_fans_voxels[_device], the matrix L of a density inversion.

The kernel walks each step's segment through the grid incrementally (a 3-D DDA). The reference
here is another algorithm: take the rock intervals of a ray from its medium crossings, compute
every cell-plane crossing inside each interval, sort them and take the differences. That
reference is first held to analytic cases, without a GPU.

Without a GPU: the reference clipping, the argument checks of the four calls (before any
device call, with a NULL plan), the loud failure without a device, and the declarations and
struct layouts from C99 and C++11.
On a B200, every scene of test_gpu_geometries.py: records byte for byte those of the plain
trace; entries against the GPU's own crossings (1 um) and against the reference's crossings
(1 mm, the test_crossings_vs_oracle rule); per-ray sums against length[m]; capacity, counting
only, media masks, fans against explicit rays, device forms against host forms; and device
calls in flight with trace_fans_device calls.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.test_fan import fan_rays
from tests.test_gpu_geometries import RULE, case, globe_stacks, tiles2  # noqa: F401
from tests.test_gpu_inflight import Call, _bytes, assert_same, run_held, solo, warm, world  # noqa: F401
from tests.test_scenes_extra import mixed_stack, sw_stack  # noqa: F401
from tests.test_stations import Fans, scene_stations
from turtle_b200 import _lib
from turtle_b200.api import (TRACE_ALTITUDE, TRACE_INVALID, TRACE_LENGTH, TRACE_STEPS,
                             VOXEL_ENTRY)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VOXELS = ["turtle_stepper_trace_voxels", "turtle_stepper_trace_voxels_device"]
FANS_VOXELS = ["turtle_stepper_trace_fans_voxels", "turtle_stepper_trace_fans_voxels_device"]
NAN, INF = float("nan"), float("inf")
ALL_MEDIA = 0xffffffff


# ---- the reference: all plane crossings, sorted, differences ---------------------------------

def frame(grid):
    """Origin and East / North / Up rows of the grid frame (turtle_ecef_from_geodetic and the
    vectors of turtle_ecef_from_horizontal)."""
    origin = tb.ecef_from_geodetic(grid.latitude, grid.longitude, grid.height)
    lam, phi = np.radians(grid.longitude), np.radians(grid.latitude)
    sl, cl, sp, cp = np.sin(lam), np.cos(lam), np.sin(phi), np.cos(phi)
    rows = np.array([[-sl, cl, 0.], [-cl * sp, -sl * sp, cp], [cl * cp, sl * cp, sp]])
    return origin, rows


def to_grid(fr, position, direction):
    """u0 = R (position - O) and v = R direction, in the kernel's order of operations."""
    origin, rows = fr
    d = np.asarray(position, dtype=float) - origin
    u0 = np.array([r[0] * d[0] + r[1] * d[1] + r[2] * d[2] for r in rows])
    v = np.array([r[0] * direction[0] + r[1] * direction[1] + r[2] * direction[2] for r in rows])
    return u0, v


def clip(u0, v, a, b, corner, size, n):
    """Pieces (cell, length) of the path lengths [a, b] of the line u0 + s v in the grid."""
    corner, size, n = (np.asarray(x, dtype=float) for x in (corner, size, n))
    ts = [np.array([a, b], dtype=float)]
    for k in range(3):
        if v[k] != 0.:
            t = (corner[k] + np.arange(int(n[k]) + 1) * size[k] - u0[k]) / v[k]
            ts.append(t[(t > a) & (t < b)])
    ts = np.unique(np.concatenate(ts))
    length = np.diff(ts)
    mid = 0.5 * (ts[:-1] + ts[1:])
    idx = np.floor((u0[None, :] + mid[:, None] * v[None, :] - corner) / size)
    keep = (idx >= 0).all(1) & (idx < n).all(1) & (length > 0.)
    cell = idx[:, 0] + n[0] * (idx[:, 1] + n[1] * idx[:, 2])
    return [(int(c), float(x)) for c, x in zip(cell[keep], length[keep])]


def grid_args(grid):
    return list(grid.corner), list(grid.size), list(grid.n)


def intervals(rec, cross):
    """(a, b, medium) of a ray from its record and its full crossings: the steps between two
    crossings started in the medium the first of them entered."""
    k = int(rec["n_changes"])
    if rec["status"] == TRACE_INVALID:
        return []
    c = cross[:k]
    bounds = [0.] + [float(x) for x in c["length"]] + [float(rec["total"])]
    media = [int(c["from"][0]) if k else int(rec["index"][0])] + [int(x) for x in c["to"]]
    return [(bounds[j], bounds[j + 1], media[j]) for j in range(k + 1)
            if bounds[j + 1] > bounds[j]]


def reference(fr, grid, position, direction, ivals):
    """(cell, medium) -> summed length of a ray."""
    u0, v = to_grid(fr, position, direction)
    out = {}
    for a, b, m in ivals:
        if 0 <= m < 32 and (grid.media >> m) & 1:
            for cell, x in clip(u0, v, a, b, *grid_args(grid)):
                out[(cell, m)] = out.get((cell, m), 0.) + x
    return out


def entry_map(entries, count):
    assert count <= len(entries)
    out = {}
    for e in entries[:count]:
        key = (int(e["voxel"]), int(e["medium"]))
        out[key] = out.get(key, 0.) + float(e["length"])
    return out


def same_map(got, want, tol, what=None):
    """Every key within tol (a function of the length); a key on one side only is <= tol."""
    for key in set(got) | set(want):
        g, w = got.get(key, 0.), want.get(key, 0.)
        assert abs(g - w) <= tol(max(abs(g), abs(w))), (key, g, w, what)


# ---- without a GPU: the reference against analytic cases --------------------------------------

def pieces(u0, v, a, b, n, corner=(0., 0., 0.), size=(1., 1., 1.)):
    return clip(np.asarray(u0, float), np.asarray(v, float), a, b, corner, size, n)


def cell(ix, iy, iz, n):
    return ix + n[0] * (iy + n[1] * iz)


def test_clip_axis_aligned():
    n = (4, 2, 2)
    got = pieces((0.5, 0.5, 0.5), (1., 0., 0.), 0., 3.2, n)
    assert [c for c, _ in got] == [cell(i, 0, 0, n) for i in range(4)]
    assert np.allclose([x for _, x in got], [0.5, 1., 1., 0.7], rtol=0, atol=1e-15)
    back = pieces((3.5, 1.5, 0.5), (-1., 0., 0.), 0., 2., n)
    assert back == [(cell(3, 1, 0, n), 0.5), (cell(2, 1, 0, n), 1.), (cell(1, 1, 0, n), 0.5)]
    up = pieces((0.25, 0.75, 0.), (0., 0., 1.), 0.5, 1.75, n)
    assert up == [(cell(0, 0, 0, n), 0.5), (cell(0, 0, 1, n), 0.75)]


def test_clip_diagonal_through_corners():
    n = (3, 3, 3)
    d = np.ones(3) / np.sqrt(3.)
    got = pieces((0., 0., 0.), d, 0., 3. * np.sqrt(3.), n)
    assert [c for c, _ in got] == [cell(i, i, i, n) for i in range(3)]
    assert np.allclose([x for _, x in got], np.sqrt(3.), rtol=1e-14)
    d2 = np.array([1., 1., 0.]) / np.sqrt(2.)  # through the vertical edges of the cells
    got = pieces((0., 0., 0.5), d2, 0., 2. * np.sqrt(2.), n)
    assert [c for c, _ in got] == [cell(0, 0, 0, n), cell(1, 1, 0, n)]


def test_clip_in_a_cell_plane():
    """A ray lying in a plane belongs to the cell above it (half-open cells); in the grid's
    last plane, to no cell."""
    n = (3, 3, 3)
    got = pieces((0.5, 1., 0.5), (1., 0., 0.), 0., 2., n)
    assert got == [(cell(0, 1, 0, n), 0.5), (cell(1, 1, 0, n), 1.), (cell(2, 1, 0, n), 0.5)]
    assert pieces((0.5, 3., 0.5), (1., 0., 0.), 0., 2., n) == []
    assert pieces((0.5, 0., 0.), (0., 0., 1.), 0., 0.5, n) == [(cell(0, 0, 0, n), 0.5)]


def test_clip_outside_ends():
    n = (4, 1, 1)
    got = pieces((-1.5, 0.5, 0.5), (1., 0., 0.), 0., 10., n)
    assert got == [(cell(i, 0, 0, n), 1.) for i in range(4)]
    assert pieces((-1.5, 0.5, 0.5), (1., 0., 0.), 0., 1., n) == []       # ends before
    assert pieces((5., 0.5, 0.5), (1., 0., 0.), 0., 3., n) == []         # starts after
    assert pieces((0.5, 1.5, 0.5), (1., 0., 0.), 0., 3., n) == []         # parallel, outside
    got = pieces((3.5, 0.5, 0.5), (1., 0., 0.), -2.25, 2., n)             # a < 0
    assert got == [(cell(1, 0, 0, n), 0.75), (cell(2, 0, 0, n), 1.), (cell(3, 0, 0, n), 1.)]


def slab(u0, v, a, b, corner, size, n):
    """Length of [a, b] inside the box of the grid (slab method)."""
    lo, hi = a, b
    for k in range(3):
        x0, x1 = corner[k], corner[k] + n[k] * size[k]
        if v[k] == 0.:
            if not (x0 <= u0[k] < x1):
                return 0.
            continue
        t0, t1 = sorted(((x0 - u0[k]) / v[k], (x1 - u0[k]) / v[k]))
        lo, hi = max(lo, t0), min(hi, t1)
    return max(hi - lo, 0.)


def test_clip_sums_to_the_clipped_interval():
    rng = np.random.default_rng(3)
    corner, size, n = (-3., -2., -1.), (0.7, 1.3, 0.4), (9, 5, 12)
    for k in range(300):
        u0 = rng.uniform(-6., 6., 3)
        v = rng.normal(size=3)
        v[rng.integers(3)] *= (k % 3 == 0)  # a zero component every third ray
        v /= np.linalg.norm(v)
        a, b = sorted(rng.uniform(-10., 10., 2))
        got = clip(u0, v, a, b, corner, size, n)
        assert abs(sum(x for _, x in got) - slab(u0, v, a, b, corner, size, n)) < 1e-12
        cells = [c for c, _ in got]
        assert all(0 <= c < 9 * 5 * 12 for c in cells)
        assert all(c0 != c1 for c0, c1 in zip(cells, cells[1:]))


def test_intervals_from_crossings():
    rec = np.zeros(1, dtype=tb.TRACE_RESULT)[0]
    cross = np.zeros(3, dtype=tb.api.TRACE_CROSSING)
    rec["total"], rec["n_changes"], rec["index"][0] = 10., 2, -1
    cross[0] = (4., 1, 0)
    cross[1] = (10., 0, -1)
    assert intervals(rec, cross) == [(0., 4., 1), (4., 10., 0)]
    rec["n_changes"], rec["index"][0] = 0, 2
    assert intervals(rec, cross) == [(0., 10., 2)]
    rec["status"] = TRACE_INVALID
    assert intervals(rec, cross) == []


# ---- without a GPU: argument checks -----------------------------------------------------------

def voxels_call(name, grid=True, position=True, direction=True, count=True, entries=True,
                capacity=4, n=3, cells=(2, 2, 2), size=(1., 1., 1.), origin=(45., 3., 0.),
                corner=(0., 0., 0.), media=1, rule=True, struct=True, n_station=2, n_azimuth=3):
    """The C entry point with a NULL plan; -> (code, message) or (0, '')."""
    fans = name in FANS_VOXELS
    if fans:
        la, lo, pos = np.zeros(n_station), np.zeros(n_station), np.zeros((n_station, 3))
        az, el = np.zeros(n_azimuth), np.zeros(4)
        f = _lib.Fans(n_station, la.ctypes.data, lo.ctypes.data, pos.ctypes.data, n_azimuth, 4,
                      az.ctypes.data, el.ctypes.data, 1)
        n = n_station * n_azimuth * 4
    p, d = np.zeros((max(n, 1), 3)), np.ones((max(n, 1), 3))
    ent = np.zeros((max(n, 1), max(capacity, 1)), dtype=VOXEL_ENTRY)
    cnt = np.zeros(max(n, 1), dtype=np.int32)
    g = tb.voxel_grid(*origin, corner, size, cells, media)
    r = tb.trace_rule(6000.) if rule else None
    args = [None]
    if fans:
        args.append(C.byref(f) if struct else None)
    else:
        args += [n, p.ctypes.data if position else None, d.ctypes.data if direction else None]
    args += [C.byref(r) if r is not None else None, C.byref(g) if grid else None, None,
             ent.ctypes.data if entries else None, capacity, cnt.ctypes.data if count else None]
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


@pytest.mark.parametrize("name", VOXELS + FANS_VOXELS)
def test_arguments_are_checked_first(name):
    """Address and domain errors are raised before the plan or the device is touched; an
    empty call touches nothing, not even the (NULL) plan."""
    fans = name in FANS_VOXELS
    bad = [dict(grid=False), dict(count=False), dict(entries=False)]
    bad += [dict(struct=False)] if fans else [dict(position=False), dict(direction=False)]
    for kw in bad:
        _expect(*voxels_call(name, **kw), 1, name, kw)  # TURTLE_RETURN_BAD_ADDRESS
    for kw in (dict(capacity=-1), dict(cells=(0, 2, 2)), dict(cells=(2, -1, 2)),
               dict(cells=(2, 2, 0)), dict(cells=(65536, 32768, 1)), dict(size=(0., 1., 1.)),
               dict(size=(1., -1., 1.)), dict(size=(1., 1., INF)), dict(size=(NAN, 1., 1.)),
               dict(origin=(NAN, 3., 0.)), dict(origin=(45., INF, 0.)),
               dict(origin=(45., 3., NAN)), dict(corner=(0., -INF, 0.)),
               dict(corner=(0., 0., NAN)), dict(media=0), dict(rule=False)):
        _expect(*voxels_call(name, **kw), 6, name, kw)  # TURTLE_RETURN_DOMAIN_ERROR
    assert "invalid voxel grid of 65536 x 32768 x 1 cells" in \
        voxels_call(name, cells=(65536, 32768, 1))[1]
    empty = [dict(n_station=0, count=False), dict(n_azimuth=0, count=False)] if fans else \
        [dict(n=0), dict(n=0, position=False, direction=False, count=False)]
    for kw in empty:
        assert voxels_call(name, **kw) == (0, ""), kw


@pytest.mark.parametrize("name", VOXELS + FANS_VOXELS)
def test_fails_loudly_without_gpu(name, has_gpu):
    if has_gpu:
        pytest.skip("a GPU is present")
    for kw in (dict(), dict(capacity=0, entries=False)):
        code, message = voxels_call(name, **kw)
        assert code == 7 and "no CUDA device" in message and "no CPU fallback" in message


def test_error_function_names():
    for name in VOXELS + FANS_VOXELS:
        fn = C.cast(getattr(_lib.lib, name), C.c_void_p)
        assert _lib.lib.turtle_error_function(fn) == name.encode()


def test_header_declarations_compile(tmp_path):
    """Callers of the new declarations compile as pedantic C99 and C++11; the two structs have
    the documented sizes and the offsets of their Python mirrors."""
    checks = []
    for struct, mirror in (("turtle_voxel_grid", _lib.VoxelGrid),
                           ("turtle_voxel_entry", _lib.VoxelEntry)):
        checks += ["(offsetof(struct %s, %s) == %d)" % (struct, k, getattr(mirror, k).offset)
                   for k, _ in mirror._fields_]
        checks.append("(sizeof(struct %s) == %d)" % (struct, C.sizeof(mirror)))
    common = ('struct turtle_plan *, const struct turtle_trace_rule *, '
              'const struct turtle_voxel_grid *, struct turtle_trace_result *, '
              'struct turtle_voxel_entry *, int, int32_t *')
    rays = common.replace("struct turtle_plan *,", "struct turtle_plan *, size_t, const double *, "
                          "const double *,")
    fans = common.replace("struct turtle_plan *,", "struct turtle_plan *, const struct turtle_fans *,")
    src = ('#include <stddef.h>\n#include "turtle_b200.h"\n'
           'static enum turtle_return (*f)(%s) = turtle_stepper_trace_voxels;\n'
           'static enum turtle_return (*g)(%s, void *) = turtle_stepper_trace_voxels_device;\n'
           'static enum turtle_return (*h)(%s) = turtle_stepper_trace_fans_voxels;\n'
           'static enum turtle_return (*k)(%s, void *) = turtle_stepper_trace_fans_voxels_device;\n'
           'int main(void) { return ((f != NULL) && (g != NULL) && (h != NULL) && (k != NULL) && '
           '%s) ? 0 : 1; }\n' % (rays, rays, fans, fans, " && ".join(checks)))
    for compiler, std, lang in (("gcc", "-std=c99", "c"), ("g++", "-std=c++11", "c++")):
        exe = str(tmp_path / ("voxels_" + lang.replace("+", "x")))
        subprocess.run([compiler, std, "-Wall", "-Wextra", "-pedantic", "-Werror",
                        "-I" + os.path.join(ROOT, "include"), "-x", lang, "-", "-x", "none",
                        _lib.LIB_PATH, "-o", exe], input=src, text=True, check=True)
        env = dict(os.environ, LD_LIBRARY_PATH=os.path.dirname(_lib.LIB_PATH))
        assert subprocess.run([exe], env=env).returncode == 0
    assert C.sizeof(_lib.VoxelGrid) == 88 and C.sizeof(_lib.VoxelEntry) == 16
    assert _lib.VoxelEntry.voxel.offset == 8 and _lib.VoxelEntry.medium.offset == 12


# ---- on a B200 --------------------------------------------------------------------------------

N_VOX = 1500   # rays of a scene compared with the reference clipping (Python: a few seconds)
CAP = 512      # entries per ray of the full-capacity calls


def check_entries(entries, count):
    """What holds whatever the geometry: positive lengths, consecutive entries that differ in
    cell or medium, untouched slots past the count."""
    for i in range(len(count)):
        e = entries[i, :min(count[i], entries.shape[1])]
        assert (e["length"] > 0.).all()
        same = (e["voxel"][1:] == e["voxel"][:-1]) & (e["medium"][1:] == e["medium"][:-1])
        assert not same.any()


def local_grid(c, media=ALL_MEDIA):
    """240 x 240 x 120 cells of 500 x 500 x 100 m around the scene's centre: rays start in and
    out of it, rays leave it."""
    lat, lon = c.center
    return tb.voxel_grid(lat, lon, 0., (-60e3, -60e3, -6e3), (500., 500., 100.), (240, 240, 120),
                         media)


def enclosing_grid(media):
    """Cells of 20 km around the whole Earth (origin at its centre)."""
    return tb.voxel_grid(0., 0., -6378137., (-7e6,) * 3, (2e4,) * 3, (700,) * 3, media)


@pytest.mark.gpu
def test_scene_voxels(case):  # noqa: F811
    plan, rule = case.plan, case.rule
    pos, dirs = case.pos[:N_VOX], case.dirs[:N_VOX]
    grid = local_grid(case)
    fr = frame(grid)
    rec, ent, cnt = plan.trace_voxels(pos, dirs, rule, grid, CAP)
    assert rec.tobytes() == case.got[:N_VOX].tobytes()
    assert (cnt <= CAP).all() and (cnt[rec["status"] == TRACE_INVALID] == 0).all()
    assert (cnt > 0).sum() > N_VOX // 20, case.name
    check_entries(ent, cnt)
    c = plan.counters()
    plan.trace(pos, dirs, rule)
    t = plan.counters()
    assert (c["rays"], c["steps"], c["samples"]) == (t["rays"], t["steps"], t["samples"])

    # against the GPU's own crossings: 1 um per key
    gres, gcross = plan.trace_crossings(pos, dirs, rule, 128)
    assert (gres["n_changes"] <= 128).all()
    for i in range(N_VOX):
        want = reference(fr, grid, pos[i], dirs[i], intervals(gres[i], gcross[i]))
        same_map(entry_map(ent[i], cnt[i]), want, lambda x: 1e-6,
                 (i, int(gres[i]["status"]), intervals(gres[i], gcross[i])[-3:]))

    # against the reference's crossings, on rays whose discrete outcome agrees
    m = N_VOX // 2
    wres, wcross = case.ora.trace_crossings(pos[:m], dirs[:m], H.rule(**RULE), 128,
                                            threads=case.threads)
    assert (wres["n_changes"] <= 128).all()
    same = (wres["n_steps"] == rec[:m]["n_steps"]) & \
        (wres["medium_hash"] == rec[:m]["medium_hash"]) & (wres["status"] == rec[:m]["status"])
    assert (~same).sum() <= max(3, m // 2000)
    compared = 0
    for i in np.flatnonzero(same):
        iv = intervals(wres[i], wcross[i])
        want = reference(fr, grid, pos[i], dirs[i], iv)
        got = entry_map(ent[i], cnt[i])
        if wres[i]["status"] in (TRACE_ALTITUDE, TRACE_LENGTH, TRACE_STEPS) and iv:
            # the end of the last stretch is placed by a threshold of the rule, not by a
            # located boundary (DESIGN.md section 5): its medium is not compared
            last = iv[-1][2]
            want = {k: x for k, x in want.items() if k[1] != last}
            got = {k: x for k, x in got.items() if k[1] != last}
        same_map(got, want, lambda x: 1e-3 + 1e-9 * x, (i, int(wres[i]["status"]), iv[-3:]))
        compared += len(want)
    assert compared > 0, case.name

    # per-ray sums equal length[m] of the unfolded media when the grid encloses the rays
    rec3, ent3, cnt3 = plan.trace_voxels(pos, dirs, rule, enclosing_grid(0b111), 64)
    assert rec3.tobytes() == rec.tobytes() and (cnt3 <= 64).all()
    valid = np.arange(64)[None, :] < cnt3[:, None]
    sums = np.where(valid, ent3["length"], 0.).sum(1)
    assert np.abs(sums - rec["length"][:, :3].sum(1)).max() < 1e-6


def station_fans(c):
    """A fan of 24 x 32 rays from a station 1 m over the ground of layer 0 (the first of
    test_stations.scene_stations)."""
    la, lo, pos = scene_stations(c)
    lat, lon, origin = la[0], lo[0], pos[:1]
    az = 360. * (np.arange(24) + 0.3) / 24
    el = -5. + 40. * (np.arange(32) + 0.5) / 32
    fans = tb.Plan.make_fans([lat], [lon], origin, az, el, bundle=32)
    dirs = fan_rays(c.ora, lat, lon, az, el, 32)
    return fans, np.repeat(origin, len(dirs), 0), dirs


def fan_grid(fans, media):
    """Cells of 50 x 50 x 25 m over the relief around the station, from 1.5 km below it to
    2.5 km above it."""
    lat, lon, height = tb.ecef_to_geodetic(list(fans[1][2][0]))
    return tb.voxel_grid(lat, lon, height, (-3000., -3000., -1500.), (50., 50., 25.),
                         (120, 120, 160), media)


def _host_call(plan, name, rays_or_fans, rule, grid, capacity, sentinel):
    """The host-memory C call on entries pre-filled with `sentinel` bytes."""
    fans = name == "turtle_stepper_trace_fans_voxels"
    n = len(rays_or_fans[0]) if not fans else \
        rays_or_fans[0].n_station * rays_or_fans[0].n_azimuth * rays_or_fans[0].n_elevation
    ent = np.frombuffer(bytes([sentinel]) * (n * capacity * 16), dtype=VOXEL_ENTRY).copy() \
        .reshape(n, capacity)
    cnt = np.full(n, -3, dtype=np.int32)
    rec = np.zeros(n, dtype=tb.TRACE_RESULT)
    head = [C.byref(rays_or_fans[0])] if fans else \
        [n, rays_or_fans[0].ctypes.data, rays_or_fans[1].ctypes.data]
    tb.api._check(getattr(_lib.lib, name)(plan.handle, *head, C.byref(rule), C.byref(grid),
                                          rec.ctypes.data, ent.ctypes.data if capacity else None,
                                          capacity, cnt.ctypes.data))
    return rec, ent, cnt


@pytest.mark.gpu
def test_scene_fans_capacity_and_media(case):  # noqa: F811
    import torch
    plan, rule = case.plan, case.rule
    fans, pos, dirs = station_fans(case)
    pos, dirs = np.ascontiguousarray(pos), np.ascontiguousarray(dirs)
    n = len(dirs)
    grid = fan_grid(fans, ALL_MEDIA)
    rec, ent, cnt = plan.trace_fans_voxels(fans, rule, grid, CAP)
    assert (cnt <= CAP).all()
    check_entries(ent, cnt)
    want_rec = np.zeros(n, dtype=tb.TRACE_RESULT)
    plan.trace_fans(fans, rule, results=want_rec)
    assert rec.tobytes() == want_rec.tobytes()
    # the fan is the rays of turtle_ecef_from_horizontal, byte for byte
    r2, e2, c2 = plan.trace_voxels(pos, dirs, rule, grid, CAP)
    assert (r2.tobytes(), e2.tobytes(), c2.tobytes()) == (rec.tobytes(), ent.tobytes(), cnt.tobytes())

    # the device forms are the host forms
    d_ent = torch.full((n * CAP * 16,), 0xa5, dtype=torch.uint8, device="cuda")
    d_cnt = torch.full((n,), -3, dtype=torch.int32, device="cuda")
    d_rec = torch.full((n * 96,), 0x5a, dtype=torch.uint8, device="cuda")
    plan.trace_fans_voxels_device(fans, rule, grid, CAP, d_ent, d_cnt, results=d_rec)
    torch.cuda.synchronize()
    assert plan.counters(sync=True)["launches"] == 1
    ents = d_ent.cpu().numpy().view(VOXEL_ENTRY).reshape(n, CAP)
    assert d_rec.cpu().numpy().tobytes() == rec.tobytes()
    assert d_cnt.cpu().numpy().tobytes() == cnt.tobytes()
    for i in range(n):
        k = cnt[i]
        assert ents[i, :k].tobytes() == ent[i, :k].tobytes()
        assert ents[i, k:].tobytes() == b"\xa5" * (16 * (CAP - k))
    d_ent.fill_(0xa5)
    d_cnt.fill_(-3)
    plan.trace_voxels_device(n, torch.from_numpy(pos).cuda(), torch.from_numpy(dirs).cuda(), rule,
                             grid, CAP, d_ent, d_cnt)
    torch.cuda.synchronize()
    assert d_cnt.cpu().numpy().tobytes() == cnt.tobytes()
    assert (d_ent.cpu().numpy().view(VOXEL_ENTRY).reshape(n, CAP) == ents).all()

    # capacity below the largest count: same counts, the first K entries, untouched slots
    top = int(cnt.max())
    assert top > 2, case.name
    k = top // 2
    for name, rays in (("turtle_stepper_trace_voxels", (pos, dirs)),
                       ("turtle_stepper_trace_fans_voxels", fans)):
        rk, ek, ck = _host_call(plan, name, rays, rule, grid, k, 0xee)
        assert rk.tobytes() == rec.tobytes() and ck.tobytes() == cnt.tobytes()
        for i in range(n):
            w = min(cnt[i], k)
            assert ek[i, :w].tobytes() == ent[i, :w].tobytes()
            assert ek[i, w:].tobytes() == b"\xee" * (16 * (k - w))
        r0, _, c0 = _host_call(plan, name, rays, rule, grid, 0, 0)
        assert r0.tobytes() == rec.tobytes() and c0.tobytes() == cnt.tobytes()

    # masks of the two media the fan crosses most (rock and air: 0b1, 0b10) partition the
    # entries of their union
    valid = np.arange(CAP)[None, :] < cnt[:, None]
    media, hits = np.unique(ent["medium"][valid], return_counts=True)
    ma, mb = (list(media[np.argsort(-hits)]) + [media[0] + 1])[:2]
    a, b = 1 << int(ma), 1 << int(mb)
    maps = {}
    for mask in (a, b, a | b):
        _, e, c = plan.trace_fans_voxels(fans, rule, fan_grid(fans, mask), CAP)
        assert (c <= CAP).all()
        maps[mask] = [entry_map(e[i], c[i]) for i in range(n)]
    for i in range(n):
        union = dict(maps[a][i])
        assert not set(union) & set(maps[b][i])
        union.update(maps[b][i])
        same_map(maps[a | b][i], union, lambda x: 1e-9 * x, i)
        assert all(m == ma for _, m in maps[a][i]) and all(m == mb for _, m in maps[b][i])
    assert sum(map(len, maps[a | b])) > 0, case.name


# ---- in flight ----------------------------------------------------------------------------------

class Voxels(Call):
    """turtle_stepper_trace_voxels_device or, with `fans`, turtle_stepper_trace_fans_voxels_device."""

    def __init__(self, plan, rule, grid, capacity, pos=None, dirs=None, fans=None):
        super().__init__(plan, "trace_%svoxels_device" % ("fans_" if fans else ""))
        self.rule, self.grid, self.capacity, self.fans = rule, grid, capacity, fans
        if fans is None:
            import torch
            self.n = len(pos)
            self.pos, self.dirs = (torch.from_numpy(np.ascontiguousarray(a)).cuda()
                                   for a in (pos, dirs))
        else:
            f = fans[0]
            self.n = f.n_station * f.n_azimuth * f.n_elevation

    def prepare(self):
        import torch
        self.out = dict(
            entries=torch.full((self.n * self.capacity * 16,), 0xa5, dtype=torch.uint8, device="cuda"),
            count=torch.full((self.n,), -3, dtype=torch.int32, device="cuda"),
            records=torch.full((self.n * 96,), 0x5a, dtype=torch.uint8, device="cuda"))

    def issue(self, stream):
        o = self.out
        if self.fans is None:
            self.plan.trace_voxels_device(self.n, self.pos, self.dirs, self.rule, self.grid,
                                          self.capacity, o["entries"], o["count"],
                                          results=o["records"], stream=stream.cuda_stream)
        else:
            self.plan.trace_fans_voxels_device(self.fans, self.rule, self.grid, self.capacity,
                                               o["entries"], o["count"], results=o["records"],
                                               stream=stream.cuda_stream)

    def outputs(self):
        return _bytes(self.out)


@pytest.mark.gpu
def test_voxel_calls_in_flight(world):  # noqa: F811
    """Eight device calls on their own held streams, voxel calls of both forms mixed with
    trace_fans_device calls: each gives its solo result."""
    p, rule = world.plan, world.rule
    lat, lon = world.station
    grid = tb.voxel_grid(lat, lon, 0., (-4000., -4000., -1000.), (40., 40., 20.), (200, 200, 150),
                         ALL_MEDIA)
    stations = (np.array([lat, lat]), np.array([lon, lon + 0.01]),
                np.stack([world.origin, world.plan.position([lat], [lon + 0.01], [1.], 0)[0][0]]))
    rng = np.random.default_rng(9)
    calls = []
    for k in range(4):
        az = np.sort(rng.uniform(0., 360., 9 + k))
        el = np.sort(rng.uniform(-10., 40., 7))
        fans = tb.Plan.make_fans(*stations, az, el)
        calls.append(Voxels(p, rule, grid, 24 + 8 * k, fans=fans) if k % 2 == 0 else
                     Voxels(p, rule, grid, 32, *world.rays(60 + k, 1500 + 7 * k)))
        calls.append(Fans(p, stations, az, el, rule))
    warm(world, 40, 0)
    want = [solo(c) for c in calls]
    run_held(calls, 300)
    for c, w in zip(calls, want):
        assert_same(c, w)
