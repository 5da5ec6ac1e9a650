"""Opacity and its gradient over a voxel grid without storing the matrix:
turtle_stepper_trace_opacity[_device] and turtle_stepper_trace_fans_opacity[_device].

These calls apply the L of turtle_stepper_trace_voxels (opacity = L @ density) and its
transpose (gradient += L.T @ weight) while they trace. The reference is L itself, read from the
entries of trace_voxels on the same rays and grid.

Without a GPU: the argument checks of the four calls (before any device call, with a NULL
plan), empty calls, the loud failure without a device, the error names, and the declarations
and the layout of struct turtle_voxel_opacity from C99 and C++11.
On a B200, every scene of test_gpu_geometries.py: records byte for byte those of trace_voxels;
the opacity bit for bit the host loop over its entries; the gradient within the bound of a
reordered sum of the same products, added to what the array held; the dot-product identity;
outside against the GPU's own crossings; forward, adjoint and both in one call; fans against
explicit rays, device forms against host forms; and device calls in flight adding into one
gradient, mixed with trace_fans_voxels_device calls.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import turtle_b200 as tb
from tests.test_gpu_geometries import case, globe_stacks, tiles2  # noqa: F401
from tests.test_gpu_inflight import Call, _bytes, assert_same, run_held, solo, warm, world  # noqa: F401
from tests.test_scenes_extra import mixed_stack, sw_stack  # noqa: F401
from tests.test_voxels import (ALL_MEDIA, FANS_VOXELS, VOXELS, Voxels, _expect, clip,
                               enclosing_grid, fan_grid, frame, grid_args, intervals,
                               local_grid, station_fans, to_grid)
from turtle_b200 import _lib
from turtle_b200.api import TRACE_INVALID

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPACITY = ["turtle_stepper_trace_opacity", "turtle_stepper_trace_opacity_device"]
FANS_OPACITY = ["turtle_stepper_trace_fans_opacity", "turtle_stepper_trace_fans_opacity_device"]
NAN, INF = float("nan"), float("inf")
EPS = np.finfo(float).eps


# ---- without a GPU: argument checks -----------------------------------------------------------

def opacity_call(name, grid=True, position=True, direction=True, struct=True, opacity=True,
                 density=True, outside=True, weight=True, gradient=True, n=3, cells=(2, 2, 2),
                 size=(1., 1., 1.), origin=(45., 3., 0.), corner=(0., 0., 0.), media=1, rule=True,
                 fans_struct=True, n_station=2, n_azimuth=3):
    """The C entry point with a NULL plan; -> (code, message) or (0, '')."""
    fans = name in FANS_OPACITY
    if fans:
        la, lo, pos = np.zeros(n_station), np.zeros(n_station), np.zeros((n_station, 3))
        az, el = np.zeros(n_azimuth), np.zeros(4)
        f = _lib.Fans(n_station, la.ctypes.data, lo.ctypes.data, pos.ctypes.data, n_azimuth, 4,
                      az.ctypes.data, el.ctypes.data, 1)
        n = n_station * n_azimuth * 4
    p, d = np.zeros((max(n, 1), 3)), np.ones((max(n, 1), 3))
    per_ray = [np.zeros(max(n, 1)) for _ in range(3)]
    per_cell = [np.zeros(max(int(np.prod(cells)), 1)) for _ in range(2)]
    arrays = dict(density=per_cell[0], opacity=per_ray[0], outside=per_ray[1],
                  weight=per_ray[2], gradient=per_cell[1])
    keep = dict(density=density, opacity=opacity, outside=outside, weight=weight,
                gradient=gradient)
    s = _lib.VoxelOpacity(*(arrays[k].ctypes.data if keep[k] else None
                            for k, _ in _lib.VoxelOpacity._fields_))
    g = tb.voxel_grid(*origin, corner, size, cells, media)
    r = tb.trace_rule(6000.) if rule else None
    args = [None]
    if fans:
        args.append(C.byref(f) if fans_struct else None)
    else:
        args += [n, p.ctypes.data if position else None, d.ctypes.data if direction else None]
    args += [C.byref(r) if r is not None else None, C.byref(g) if grid else None,
             C.byref(s) if struct else None, None]
    if name.endswith("_device"):
        args.append(None)
    try:
        tb.api._check(getattr(_lib.lib, name)(*args))
    except tb.TurtleError as e:
        return e.code, str(e)
    return 0, ""


@pytest.mark.parametrize("name", OPACITY + FANS_OPACITY)
def test_arguments_are_checked_first(name):
    """Address and domain errors are raised before the plan or the device is touched, the
    grid's with the messages of trace_voxels; an empty call touches nothing, not even the
    (NULL) plan."""
    fans = name in FANS_OPACITY
    bad = [dict(grid=False), dict(struct=False), dict(density=False),
           dict(weight=False), dict(density=False, weight=False, outside=False)]
    bad += [dict(fans_struct=False)] if fans else [dict(position=False), dict(direction=False)]
    for kw in bad:
        _expect(*opacity_call(name, **kw), 1, name, kw)  # TURTLE_RETURN_BAD_ADDRESS
    assert "missing voxel grid" in opacity_call(name, grid=False)[1]
    assert "missing voxel opacity arrays" in opacity_call(name, struct=False)[1]
    assert "missing voxel densities" in opacity_call(name, density=False)[1]
    assert "missing ray weights" in opacity_call(name, weight=False)[1]
    # each output needs only its own input
    for kw in (dict(opacity=False, density=False), dict(gradient=False, weight=False),
               dict(opacity=False, density=False, gradient=False, weight=False, outside=False)):
        code, message = opacity_call(name, **kw)
        assert ("missing plan" in message) or ("no CUDA device" in message), (kw, message)
    for kw in (dict(cells=(0, 2, 2)), dict(cells=(2, -1, 2)),
               dict(cells=(2, 2, 0)), dict(cells=(65536, 32768, 1)), dict(size=(0., 1., 1.)),
               dict(size=(1., -1., 1.)), dict(size=(1., 1., INF)), dict(size=(NAN, 1., 1.)),
               dict(origin=(NAN, 3., 0.)), dict(origin=(45., INF, 0.)),
               dict(origin=(45., 3., NAN)), dict(corner=(0., -INF, 0.)),
               dict(corner=(0., 0., NAN)), dict(media=0), dict(rule=False)):
        _expect(*opacity_call(name, **kw), 6, name, kw)  # TURTLE_RETURN_DOMAIN_ERROR
    # the grid's messages are those of trace_voxels
    from tests.test_voxels import voxels_call
    vname = name.replace("opacity", "voxels")
    for kw in (dict(cells=(65536, 32768, 1)), dict(size=(1., -1., 1.)), dict(corner=(0., 0., NAN)),
               dict(media=0), dict(grid=False)):
        got, want = opacity_call(name, **kw)[1], voxels_call(vname, **kw)[1]
        assert got.split("}", 1)[1] == want.split("}", 1)[1], (got, want)
    empty = [dict(n_station=0), dict(n_azimuth=0)] if fans else \
        [dict(n=0), dict(n=0, position=False, direction=False, opacity=False, outside=False,
                         weight=False, gradient=False)]
    for kw in empty:
        assert opacity_call(name, **kw) == (0, ""), kw


@pytest.mark.parametrize("name", OPACITY + FANS_OPACITY)
def test_fails_loudly_without_gpu(name, has_gpu):
    if has_gpu:
        pytest.skip("a GPU is present")
    for kw in (dict(), dict(opacity=False, density=False, outside=False),
               dict(gradient=False, weight=False)):
        code, message = opacity_call(name, **kw)
        assert code == 7 and "no CUDA device" in message and "no CPU fallback" in message


def test_error_function_names():
    for name in OPACITY + FANS_OPACITY:
        fn = C.cast(getattr(_lib.lib, name), C.c_void_p)
        assert _lib.lib.turtle_error_function(fn) == name.encode()
    for name in VOXELS + FANS_VOXELS:  # the names next to them are unchanged
        fn = C.cast(getattr(_lib.lib, name), C.c_void_p)
        assert _lib.lib.turtle_error_function(fn) == name.encode()


def test_header_declarations_compile(tmp_path):
    """Callers of the new declarations compile as pedantic C99 and C++11; the struct has the
    size and offsets of its Python mirror."""
    mirror = _lib.VoxelOpacity
    checks = ["(offsetof(struct turtle_voxel_opacity, %s) == %d)" % (k, getattr(mirror, k).offset)
              for k, _ in mirror._fields_]
    checks.append("(sizeof(struct turtle_voxel_opacity) == %d)" % C.sizeof(mirror))
    common = ('struct turtle_plan *, const struct turtle_trace_rule *, '
              'const struct turtle_voxel_grid *, const struct turtle_voxel_opacity *, '
              'struct turtle_trace_result *')
    rays = common.replace("struct turtle_plan *,", "struct turtle_plan *, size_t, const double *, "
                          "const double *,")
    fans = common.replace("struct turtle_plan *,", "struct turtle_plan *, const struct turtle_fans *,")
    src = ('#include <stddef.h>\n#include "turtle_b200.h"\n'
           'static enum turtle_return (*f)(%s) = turtle_stepper_trace_opacity;\n'
           'static enum turtle_return (*g)(%s, void *) = turtle_stepper_trace_opacity_device;\n'
           'static enum turtle_return (*h)(%s) = turtle_stepper_trace_fans_opacity;\n'
           'static enum turtle_return (*k)(%s, void *) = turtle_stepper_trace_fans_opacity_device;\n'
           'int main(void) {\n'
           '        double rho[1] = { 1. }, out[1];\n'
           '        struct turtle_voxel_opacity o = { rho, out, NULL, NULL, NULL };\n'
           '        return ((f != NULL) && (g != NULL) && (h != NULL) && (k != NULL) && '
           '(o.density == rho) && %s) ? 0 : 1;\n}\n' % (rays, rays, fans, fans, " && ".join(checks)))
    for compiler, std, lang in (("gcc", "-std=c99", "c"), ("g++", "-std=c++11", "c++")):
        exe = str(tmp_path / ("opacity_" + lang.replace("+", "x")))
        subprocess.run([compiler, std, "-Wall", "-Wextra", "-pedantic", "-Werror",
                        "-I" + os.path.join(ROOT, "include"), "-x", lang, "-", "-x", "none",
                        _lib.LIB_PATH, "-o", exe], input=src, text=True, check=True)
        env = dict(os.environ, LD_LIBRARY_PATH=os.path.dirname(_lib.LIB_PATH))
        assert subprocess.run([exe], env=env).returncode == 0
    assert C.sizeof(mirror) == 40
    assert [getattr(mirror, k).offset for k, _ in mirror._fields_] == [0, 8, 16, 24, 32]


# ---- the reference: L from the entries of trace_voxels ------------------------------------------

N_OP = 1500  # rays of a scene


def exact_entries(plan, rule, grid, pos=None, dirs=None, fans=None):
    """(records, entries, count) of trace_voxels (or trace_fans_voxels) with capacity = the
    counted maximum."""
    if fans is None:
        _, _, count = plan.trace_voxels(pos, dirs, rule, grid, 0)
        return plan.trace_voxels(pos, dirs, rule, grid, max(int(count.max()), 1))
    _, _, count = plan.trace_fans_voxels(fans, rule, grid, 0)
    return plan.trace_fans_voxels(fans, rule, grid, max(int(count.max()), 1))


def forward(entries, count, density):
    """acc = acc + density[voxel] * length over the entries of each ray, in order: one rounded
    product and one rounded sum per entry."""
    acc = np.zeros(len(count))
    for k in range(entries.shape[1]):
        live = k < count
        if not live.any():
            break
        e = entries[:, k]
        p = density[np.where(live, e["voxel"], 0)] * e["length"]
        acc = np.where(live, acc + p, acc)
    return acc


def products(entries, count, weight):
    """(cells, weight[i] * length) of every entry: the terms of L.T @ weight."""
    live = np.arange(entries.shape[1])[None, :] < count[:, None]
    rows = np.nonzero(live)[0]
    e = entries[live]
    return e["voxel"].astype(np.int64), weight[rows] * e["length"]


def check_gradient(got, start, terms):
    """got = start + the products of `terms` ([(cells, products)]), summed in any order: within
    (m_j - 1) eps sum |p| of the exact sum of the m_j terms of each cell (start included); the
    cells without a product hold `start` exactly."""
    cells = np.concatenate([t[0] for t in terms])
    p = np.concatenate([t[1] for t in terms])
    touched = np.zeros(len(got), dtype=bool)
    touched[cells] = True
    assert got[~touched].tobytes() == start[~touched].tobytes()
    order = np.argsort(cells, kind="stable")
    cells, p = cells[order], p[order]
    heads = np.flatnonzero(np.r_[True, cells[1:] != cells[:-1]])
    bad = 0
    for a, b in zip(heads, np.r_[heads[1:], len(cells)]):
        j = cells[a]
        exact = math.fsum([start[j]] + list(p[a:b]))
        bound = (b - a) * EPS * (abs(start[j]) + float(np.abs(p[a:b]).sum()))
        bad += abs(got[j] - exact) > bound
    assert bad == 0, "%d of %d cells off their bound" % (bad, len(heads))
    return len(heads)


def outside_reference(fr, grid, pos, dirs, gres, gcross):
    """Per ray: the selected stretches of the GPU's own crossings, less their pieces in cells."""
    out = np.zeros(len(pos))
    for i in range(len(pos)):
        u0, v = to_grid(fr, pos[i], dirs[i])
        for a, b, m in intervals(gres[i], gcross[i]):
            if 0 <= m < 32 and (grid.media >> m) & 1:
                out[i] += (b - a) - sum(x for _, x in clip(u0, v, a, b, *grid_args(grid)))
    return out


def scene_mask(case):
    """The medium that the scene's rays cross most in the local grid (of media 0, 1, 2: the
    folded length[m] of the records is then the selected length)."""
    _, ent, cnt = case.plan.trace_voxels(case.pos[:N_OP], case.dirs[:N_OP], case.rule,
                                         local_grid(case, 0b111), 64)
    live = np.arange(64)[None, :] < np.minimum(cnt, 64)[:, None]
    media, hits = np.unique(ent["medium"][live], return_counts=True)
    assert len(media) > 0, case.name
    return 1 << int(media[np.argmax(hits)])


# ---- on a B200 --------------------------------------------------------------------------------

@pytest.mark.gpu
def test_scene_opacity(case):  # noqa: F811
    plan, rule = case.plan, case.rule
    pos, dirs = case.pos[:N_OP], case.dirs[:N_OP]
    mask = scene_mask(case)
    grid = local_grid(case, mask)
    cells = 240 * 240 * 120
    rng = np.random.default_rng(len(case.name) * 1009 + mask)
    rho = rng.uniform(1.5, 3.0, cells)
    w = rng.normal(size=N_OP)
    start = rng.uniform(-1., 1., cells)

    rec_v, ent, cnt = exact_entries(plan, rule, grid, pos, dirs)
    assert (cnt > 0).sum() > N_OP // 50, case.name
    gradient = start.copy()
    rec, op, out, g = plan.trace_opacity(pos, dirs, rule, grid, density=rho, weight=w,
                                         gradient=gradient, outside=True)
    assert g is gradient
    assert rec.tobytes() == rec_v.tobytes() == case.got[:N_OP].tobytes()
    c = plan.counters()
    plan.trace(pos, dirs, rule)
    t = plan.counters()
    assert (c["rays"], c["steps"], c["samples"]) == (t["rays"], t["steps"], t["samples"])

    # forward: bit for bit the host loop over the entries; 0 without an entry
    want = forward(ent, cnt, rho)
    assert op.tobytes() == want.tobytes()
    assert (op[cnt == 0] == 0.).all() and (op[rec["status"] == TRACE_INVALID] == 0.).all()
    # adjoint: added to what the array held, within the bound of a reordered sum
    assert check_gradient(g, start, [products(ent, cnt, w)]) > 0

    # forward only, adjoint only, both: the same numbers
    r1, op1, out1, g1 = plan.trace_opacity(pos, dirs, rule, grid, density=rho)
    r2, op2, out2, g2 = plan.trace_opacity(pos, dirs, rule, grid, weight=w)
    r3, op3, out3, g3 = plan.trace_opacity(pos, dirs, rule, grid, density=rho, weight=w)
    assert r1.tobytes() == r2.tobytes() == r3.tobytes() == rec.tobytes()
    assert out1 is None and g1 is None and op2 is None and out2 is None and out3 is None
    assert op1.tobytes() == op3.tobytes() == op.tobytes()
    zero = np.zeros(cells)
    check_gradient(g2, zero, [products(ent, cnt, w)])
    check_gradient(g3, zero, [products(ent, cnt, w)])
    # <L rho, w> = <rho, L.T w>
    lhs, rhs = math.fsum(op3 * w), math.fsum(rho * g3)
    scale = max(math.fsum(np.abs(op3 * w)), math.fsum(np.abs(rho * g3)))
    assert abs(lhs - rhs) <= 1e-12 * scale, (lhs, rhs, scale)

    # outside: against the GPU's own crossings (1 um), and with the entries the selected length
    gres, gcross = plan.trace_crossings(pos, dirs, rule, 128)
    assert (gres["n_changes"] <= 128).all()
    fr = frame(grid)
    ref = outside_reference(fr, grid, pos, dirs, gres, gcross)
    assert np.abs(out - ref).max() <= 1e-6
    live = np.arange(ent.shape[1])[None, :] < cnt[:, None]
    inside = np.where(live, ent["length"], 0.).sum(1)
    m = int(mask).bit_length() - 1
    assert np.abs(out + inside - rec["length"][:, m]).max() <= 1e-6
    assert (out >= 0.).all()
    # a grid that encloses the rays leaves nothing outside
    _, _, out_e, _ = plan.trace_opacity(pos, dirs, rule, enclosing_grid(mask), outside=True)
    assert (out_e == 0.).all()


@pytest.mark.gpu
def test_scene_fans_and_device_forms(case):  # noqa: F811
    import torch
    plan, rule = case.plan, case.rule
    fans, pos, dirs = station_fans(case)
    pos, dirs = np.ascontiguousarray(pos), np.ascontiguousarray(dirs)
    n = len(dirs)
    grid = fan_grid(fans, ALL_MEDIA)
    cells = 120 * 120 * 160
    rng = np.random.default_rng(11)
    rho, w = rng.uniform(1.5, 3.0, cells), rng.normal(size=n)

    rec_v, ent, cnt = exact_entries(plan, rule, grid, fans=fans)
    assert (cnt > 0).sum() > 0, case.name
    rec, op, out, g = plan.trace_fans_opacity(fans, rule, grid, density=rho, weight=w,
                                              outside=True)
    assert rec.tobytes() == rec_v.tobytes()
    assert op.tobytes() == forward(ent, cnt, rho).tobytes()
    check_gradient(g, np.zeros(cells), [products(ent, cnt, w)])
    # the fan is the rays of turtle_ecef_from_horizontal
    r2, op2, out2, g2 = plan.trace_opacity(pos, dirs, rule, grid, density=rho, weight=w,
                                           outside=True)
    assert (r2.tobytes(), op2.tobytes(), out2.tobytes()) == (rec.tobytes(), op.tobytes(),
                                                             out.tobytes())
    check_gradient(g2, np.zeros(cells), [products(ent, cnt, w)])

    # the device forms are the host forms
    d_rho, d_w = torch.from_numpy(rho).cuda(), torch.from_numpy(w).cuda()
    for form in ("fans", "rays"):
        d_op = torch.full((n,), NAN, dtype=torch.float64, device="cuda")
        d_out = torch.full((n,), NAN, dtype=torch.float64, device="cuda")
        d_g = torch.zeros(cells, dtype=torch.float64, device="cuda")
        d_rec = torch.full((n * 96,), 0x5a, dtype=torch.uint8, device="cuda")
        kw = dict(density=d_rho, opacity=d_op, outside=d_out, weight=d_w, gradient=d_g,
                  results=d_rec)
        if form == "fans":
            plan.trace_fans_opacity_device(fans, rule, grid, **kw)
        else:
            plan.trace_opacity_device(n, torch.from_numpy(pos).cuda(),
                                      torch.from_numpy(dirs).cuda(), rule, grid, **kw)
        torch.cuda.synchronize()
        assert plan.counters(sync=True)["launches"] == 1
        assert d_rec.cpu().numpy().tobytes() == rec.tobytes()
        assert d_op.cpu().numpy().tobytes() == op.tobytes()
        assert d_out.cpu().numpy().tobytes() == out.tobytes()
        check_gradient(d_g.cpu().numpy(), np.zeros(cells), [products(ent, cnt, w)])


# ---- in flight ----------------------------------------------------------------------------------

class Opacity(Call):
    """turtle_stepper_trace_fans_opacity_device: opacity, outside and records of its own, the
    gradient added to `gradient` (a device tensor shared with other calls)."""

    def __init__(self, plan, rule, grid, fans, density, weight, gradient):
        super().__init__(plan, "trace_fans_opacity_device")
        self.rule, self.grid, self.fans = rule, grid, fans
        f = fans[0]
        self.n = f.n_station * f.n_azimuth * f.n_elevation
        self.density, self.weight, self.gradient = density, weight, gradient

    def prepare(self):
        import torch
        self.out = dict(
            opacity=torch.full((self.n,), NAN, dtype=torch.float64, device="cuda"),
            outside=torch.full((self.n,), NAN, dtype=torch.float64, device="cuda"),
            records=torch.full((self.n * 96,), 0x5a, dtype=torch.uint8, device="cuda"))

    def issue(self, stream):
        o = self.out
        self.plan.trace_fans_opacity_device(self.fans, self.rule, self.grid, density=self.density,
                                            opacity=o["opacity"], outside=o["outside"],
                                            weight=self.weight, gradient=self.gradient,
                                            results=o["records"], stream=stream.cuda_stream)

    def outputs(self):
        return _bytes(self.out)


@pytest.mark.gpu
def test_opacity_calls_in_flight(world):  # noqa: F811
    """Device calls on their own held streams add into ONE gradient: eight opacity calls, then
    opacity calls mixed with trace_fans_voxels_device calls. Each gives its solo opacity,
    outside and records, the voxel calls their solo results, and the shared gradient is the sum
    of the solo gradients within the bound of a reordered sum."""
    import torch
    p, rule = world.plan, world.rule
    lat, lon = world.station
    grid = tb.voxel_grid(lat, lon, 0., (-4000., -4000., -1000.), (40., 40., 20.), (200, 200, 150),
                         ALL_MEDIA)
    cells = 200 * 200 * 150
    stations = (np.array([lat, lat]), np.array([lon, lon + 0.01]),
                np.stack([world.origin, world.plan.position([lat], [lon + 0.01], [1.], 0)[0][0]]))
    rng = np.random.default_rng(19)
    rho = torch.from_numpy(rng.uniform(1.5, 3.0, cells)).cuda()
    shared = torch.zeros(cells, dtype=torch.float64, device="cuda")
    warm(world, 40, 0)

    def opacity_call(k):
        az = np.sort(rng.uniform(0., 360., 9 + k))
        el = np.sort(rng.uniform(-10., 40., 7))
        fans = tb.Plan.make_fans(*stations, az, el)
        w = rng.normal(size=2 * len(az) * len(el))
        return Opacity(p, rule, grid, fans, rho, torch.from_numpy(w).cuda(), shared), fans, w

    for mixed in (False, True):
        calls, terms = [], []
        for k in range(8):
            if mixed and k % 3 == 1:
                az = np.sort(rng.uniform(0., 360., 10 + k))
                el = np.sort(rng.uniform(-10., 40., 6))
                calls.append(Voxels(p, rule, grid, 32, fans=tb.Plan.make_fans(*stations, az, el)))
                continue
            call, fans, w = opacity_call(k)
            _, ent, cnt = exact_entries(p, rule, grid, fans=fans)
            terms.append(products(ent, cnt, w))
            calls.append(call)
        want = []
        for c in calls:
            want.append(solo(c))
        solo_sum = shared.cpu().numpy()  # the solo calls added into it one after the other
        check_gradient(solo_sum, np.zeros(cells), terms)
        shared.zero_()
        run_held(calls, 300)
        for c, w in zip(calls, want):
            assert_same(c, w)
        check_gradient(shared.cpu().numpy(), np.zeros(cells), terms)
        shared.zero_()
