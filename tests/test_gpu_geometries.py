"""GPU: the batched path on random and limit-sized geometries, against the oracle and
against itself.

The random-geometry suite on the host (test_random_geometries.py) runs the scalar
instantiation of tb_core.cuh: full-size local approximation blocks, eager Jacobians, no
footprint cull. What the kernels add on top of it depends on the geometry and only runs on
the device: the compact layout of the local approximation state (tb::lla_layout), the lazy
Jacobians and their rebuild over several stale transforms, the footprint cull of projected
transforms with its NaN x, y references, the one-entry x, y memo at range 0, the tile
tables of a second, third or fourth stack, and the choice of kernel. Every scene here goes
through all of them that it reaches:

  * against the oracle (the reference when it was built, else the C restatement): whole
    rays with the parity protocol of test_gpu_trace.check, medium crossings, one sample per
    particle, walks with and without device states, ray origins;
  * against the GPU itself, byte for byte: every entry point, schedule, launch shape and
    round structure of a batch, each ray on its own, a permutation, and a fan from a
    station on the ground (the COMPACT kernels, whose lanes take ray after ray from the
    same point: a state that survives from one ray to the next shows there);
  * the size of a particle's device state, from the layout rule of tb_core.cuh.
"""
import os
import zlib

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.common import Scene, geoid_map, lambert_map, random_scene, second_stack, \
    ulp_distance
from tests.test_crossings import _consistent
from tests.test_fan import FIELDS, columns, fan_rays
from tests.test_gpu_trace import check, noise_floor
from tests.test_scenes_extra import mixed_stack, sw_stack, utm_south_map  # noqa: F401
from turtle_b200 import synth

pytestmark = pytest.mark.gpu

N_RAYS = 4000 + 37        # ragged: not a multiple of the warp size
N_SAMPLES = 20000
N_WALKERS = 1000
K = 6                     # crossings kept per ray (test_crossings.K)
PS_FIELDS = 10            # per-particle fields ahead of the local approximation (tb_kernels.cu)
FRANCE = (44.9, 47.1, 1.9, 4.1)
CHILE = (-35.1, -32.9, -72.1, -69.9)
RANDOM_SEEDS = range(24)
NAMED = ["two_projections_r0", "three_projections_lla", "shared_projection_union",
         "map_first", "geodetic_map_first", "shared_map", "stacks_x4", "at_the_limits",
         "antimeridian_r0", "antimeridian_lla", "high_latitude", "polar_cap", "south_west_lla"]
RULE = dict(altitude_max=6000., length_max=3e4, max_steps=5000)


@pytest.fixture(scope="module")
def tiles2(tmp_path_factory):
    return second_stack(str(tmp_path_factory.mktemp("second_stack")))


@pytest.fixture(scope="module")
def globe_stacks(tmp_path_factory):
    """Stacks away from France: `seam` (write_seam_stack) and `arctic`, 2 x 2 tiles at
    N78 - N79, E015 - E016 (1/1200 deg cells of about 8 m in longitude)."""
    seam = write_seam_stack(str(tmp_path_factory.mktemp("seam_stack")))
    arctic = str(tmp_path_factory.mktemp("arctic_stack"))
    synth.write_hgt_stack(arctic, 78, 15, 2, 2, n=1201)
    return dict(seam=seam, arctic=arctic)


def write_seam_stack(directory):
    """2 x 2 tiles S01E179, S01W180, N00E179, N00W180 around the antimeridian on the equator:
    a tile table of 360 columns, 358 of them empty. The terrain is continuous across the
    seam, as in a real elevation model: the W180 tiles continue the node lattice of the E179
    ones. (With a step in the terrain exactly on the seam, a ray crossing it under the higher
    ground changes medium there, its bisection converges onto longitude 180, and which side a
    sample lands on hinges on the last ulp of its longitude, 3 nm: a grazing ray of the parity
    protocol in every such crossing.)"""
    os.makedirs(directory, exist_ok=True)
    for lat in (-1, 0):
        for lon, origin in ((179, 179), (-180, -181)):
            nodes = synth.tile_nodes(lat, lon, -1, origin, 1201)
            name = synth.hgt_name(lat, lon)[:-4] + ".SRTMGL3.hgt"
            nodes[::-1].astype(">i2").tofile(os.path.join(directory, name))
    return directory


def wrap(lon):
    """Longitudes in (-180, 180]."""
    lon = np.asarray(lon, dtype=np.float64)
    return np.where(lon > 180., lon - 360., np.where(lon <= -180., lon + 360., lon))


def dlon(a, b):
    """|a - b| modulo 360 (degrees): -180 and 180 are the same meridian."""
    return np.abs((np.asarray(a) - np.asarray(b) + 180.) % 360. - 180.)


class Case:
    """A scene, where its rays start (lat0, lat1, lon0, lon1 boxes, where lon0 > lon1 is a box
    across the antimeridian; `ground`: bands where a third of the rays and walkers start just
    over the ground of layer 0) and which of its stacks the oracle may share between threads
    (a lock makes the reference go through turtle_client, whose memo of a missing tile is
    history dependent for negative coordinates: see test_reference_client_memo_quirk)."""

    def __init__(self, scene, boxes=(FRANCE,), ground=(), locked=True, center=(45.6, 2.7)):
        self.scene, self.boxes, self.ground = scene, list(boxes), list(ground)
        self.locked, self.center = locked, center


def _map_at(ora, tag, lat, lon, half, n, seed):
    """A projected map of `n` x `n` nodes, 2 `half` metres wide, centred on (lat, lon)."""
    cx, cy = ora.project(tag, [lat], [lon])
    vals = synth.fbm_grid(np.arange(n) * 4., np.arange(n) * 4., seed=seed) * 2500.
    return dict(nx=n, ny=n, x=(cx[0] - half, cx[0] + half), y=(cy[0] - half, cy[0] + half),
                z=(0., 3000.), projection=tag, values=vals)


def seam_maps(ora):
    """The maps of the antimeridian scenes: a UTM 1N map wholly west of its zone (x 140 -
    166.02 km, y 40 - 70 km: 179.77 E to 8 - 25 m west of 180, whose unwrapped inverse
    projection lies at -180.23 - -180.0001), a UTM 60N map across 180 deg and a geodetic
    map whose east edge is the meridian 180 itself."""
    def fbm(n, seed):
        return synth.fbm_grid(np.arange(n) * 4., np.arange(n) * 4., seed=seed) * 2500.
    utm1 = dict(nx=131, ny=151, x=(140e3, 166020.), y=(40e3, 70e3), z=(0., 3000.),
                projection="UTM 1N", values=np.resize(fbm(151, 31), (151, 131)))
    cx, cy = ora.project("UTM 60N", [-0.3], [180.])
    utm60 = dict(nx=161, ny=161, x=(cx[0] - 16e3, cx[0] + 16e3), y=(cy[0] - 16e3, cy[0] + 16e3),
                 z=(0., 3000.), projection="UTM 60N", values=fbm(161, 32))
    geo = dict(nx=121, ny=61, x=(179.4, 180.), y=(-0.9, -0.6), z=(0., 3000.), projection=None,
               values=np.resize(fbm(121, 33), (61, 121)))
    return [utm1, utm60, geo]


def seam_ground(ora, utm1):
    """Ground bands within metres of the antimeridian (1.5E-04 deg = 17 m) and of the
    borders of the UTM 1N map."""
    bands = [(-0.9, 0.9, 180. - 1.5e-4, -180. + 1.5e-4)]
    (la0, la1), (lo0, lo1) = ora.project("UTM 1N", utm1["x"], utm1["y"], inverse=True)
    lo0, lo1 = wrap(lo0), wrap(lo1)
    bands += [(la0 - 2e-4, la0 + 2e-4, lo0, lo1), (la1 - 2e-4, la1 + 2e-4, lo0, lo1),
              (la0, la1, lo0 - 2e-4, lo0 + 2e-4), (la0, la1, lo1 - 2e-4, lo1 + 2e-4)]
    return bands


def named_case(name, ora, small, tiles2, mixed, sw, globe):
    A, F, S, L = H.ADD_MAP, H.ADD_FLAT, H.ADD_STACK, H.ADD_LAYER
    if name in ("antimeridian_r0", "antimeridian_lla"):
        # layer 0 evaluates the UTM 60N map (across 180: no box), the UTM 1N map, the
        # geodetic map, the stack (360 columns, over the equator) and the flat; layer 1 the
        # UTM 1N map again. At range 0 every sample over the UTM 1N map has a longitude near
        # +179.9 and must not be culled by a box taken at -180.1. At range 10 the references
        # of the UTM 60N transform, evaluated first, fall within 10 m of the seam, and the
        # longitude linearised from them is off by up to 360 deg for samples over the UTM 1N
        # map, whose union box comes within metres of 180: that box must not be used
        maps = seam_maps(ora)
        sc = Scene(maps=maps, stacks=[globe["seam"]],
                   ops=[(F, 0, -300.), (S, 0, 0.), (A, 2, 30.), (A, 0, 0.), (A, 1, 10.),
                        (L, 0, 0.), (A, 0, 700.)],
                   range=0. if name == "antimeridian_r0" else 10.)
        return Case(sc, boxes=[(-0.95, 0.95, 179.1, -179.1), (0.35, 0.65, 179.75, 179.95)],
                    ground=seam_ground(ora, maps[0]), locked=False, center=(0.5, 179.85))
    if name == "high_latitude":
        # UTM 33N far north: the grid is turned by up to 15 deg (convergence), the second map
        # reaches 84 N, the union box of the transform is widened by 1 / cos(lat)
        maps = [_map_at(ora, "UTM 33N", 78.9, 15.9, 15000., 151, 34),
                _map_at(ora, "UTM 33N", 83.78, 15.0, 25000., 151, 35), geoid_map()]
        sc = Scene(maps=maps, stacks=[globe["arctic"]],
                   ops=[(F, 0, -200.), (S, 0, 0.), (A, 0, 20.), (L, 0, 0.), (A, 1, 300.)],
                   geoid=2, range=1.)
        (la0, la1), (lo0, lo1) = ora.project("UTM 33N", maps[0]["x"], maps[0]["y"], inverse=True)
        ground = [(la0 - 2e-4, la0 + 2e-4, lo0, lo1), (la0, la1, lo1 - 5e-4, lo1 + 5e-4)]
        return Case(sc, boxes=[(77.9, 80.1, 14.9, 17.1), (83.5, 84.05, 14.0, 16.0)],
                    ground=ground, center=(78.9, 15.9))
    if name == "polar_cap":
        # a geodetic map over the whole cap: rays from within 55 m of the axis cross it, their
        # longitude flips by 180 deg, and the Jacobian of the longitude diverges there
        n = 361
        geo = dict(nx=n, ny=41, x=(-180., 180.), y=(89., 90.), z=(0., 3000.), projection=None,
                   values=np.resize(synth.fbm_grid(np.arange(n) * 3., np.arange(41) * 3.,
                                                   seed=36), (41, n)) * 1500.)
        sc = Scene(maps=[geo], ops=[(F, 0, -50.), (A, 0, 0.)], range=100.)
        return Case(sc, boxes=[(89.5, 90., -180., 180.)], ground=[(89.9995, 90., -180., 180.)],
                    center=(89.9999, 30.))
    if name == "south_west_lla":
        # the Chilean scene of test_scenes_extra (UTM 19S map over a stack in negative
        # coordinates) under the local approximation
        m = utm_south_map()
        sc = Scene(maps=[m], stacks=[sw], ops=[(S, 0, 0.), (A, 0, 0.), (L, 0, 0.), (S, 0, 800.)],
                   range=10.)
        (la0, la1), (lo0, lo1) = ora.project("UTM 19S", m["x"], m["y"], inverse=True)
        return Case(sc, boxes=[CHILE, (la0 - 0.01, la1 + 0.01, lo0 - 0.01, lo1 + 0.01)],
                    ground=[(la0 - 2e-4, la0 + 2e-4, lo0, lo1)], locked=False,
                    center=(0.5 * (la0 + la1), 0.5 * (lo0 + lo1)))
    if name == "two_projections_r0":
        # layer 0 evaluates the UTM 30N map first, then the Lambert map, then the stack. Far
        # from its central meridian the UTM grid is turned by ~4 degrees, so its geodetic
        # box holds slivers outside the map: a sample there evaluates UTM (not culled,
        # outside), then Lambert (which takes the one-entry memo), and when it is above
        # the ground of layer 0, UTM again for the second UTM map of layer 1
        maps = [_map_at(ora, "UTM 30N", 45.6, 2.7, 8000., 161, 11),
                lambert_map(ora, 45.6, 2.7, n=201, half=15000.),
                _map_at(ora, "UTM 30N", 45.6, 2.7, 25000., 201, 12)]
        sc = Scene(maps=maps, stacks=[small],
                   ops=[(S, 0, 0.), (A, 1, 0.), (A, 0, 20.), (L, 0, 0.), (A, 2, 400.)], range=0.)
        return Case(sc, boxes=[(45.4, 45.8, 2.45, 2.95)])
    if name == "three_projections_lla":
        maps = [lambert_map(ora, 46.3, 3.3, n=151, half=6000.),
                _map_at(ora, "UTM 31N", 45.6, 2.7, 15000., 151, 13),
                _map_at(ora, "Lambert II", 45.7, 2.8, 20000., 151, 14)]
        sc = Scene(maps=maps, stacks=[small],
                   ops=[(A, 0, 0.), (S, 0, 0.), (L, 0, 0.), (F, 0, 300.), (A, 1, 400.),
                        (L, 0, 0.), (A, 2, 800.)], range=10.)
        return Case(sc)
    if name == "shared_projection_union":
        # two disjoint Lambert 93 maps on its central meridian, the stack between and around
        # them: the footprint box of the transform is their union, rays cross the gap. The
        # north edge of the northern map and the upper part of its sides run within metres
        # of that box, so the rays that creep over the ground there take reference points
        # just outside the box -- which the cull widens by the range -- for samples inside
        maps = [lambert_map(ora, 45.45, 3.0, n=161, half=8000.),
                lambert_map(ora, 45.75, 3.0, n=161, half=8000.)]
        sc = Scene(maps=maps, stacks=[small],
                   ops=[(S, 0, 0.), (A, 0, 0.), (A, 1, 0.)], range=10.)
        (la0, la1), (lo0, lo1) = ora.project("Lambert 93", maps[1]["x"], [maps[1]["y"][1]] * 2,
                                             inverse=True)
        ground = [(la0 - 5e-4, la0 + 5e-4, lo0, lo1),
                  (la0 - 0.07, la0, lo0 - 7e-4, lo0 + 7e-4),
                  (la1 - 0.07, la1, lo1 - 7e-4, lo1 + 7e-4)]
        return Case(sc, boxes=[(45.3, 45.9, 2.7, 3.3)], ground=ground)
    if name == "map_first":
        maps = [_map_at(ora, "UTM 31N", 45.6, 2.7, 15000., 201, 15)]
        sc = Scene(maps=maps, stacks=[small],
                   ops=[(F, 0, -100.), (S, 0, 0.), (A, 0, 20.)], range=10.)
        return Case(sc, boxes=[(45.3, 45.9, 2.4, 3.0)])
    if name == "geodetic_map_first":
        geo = dict(nx=121, ny=91, x=(2.3, 3.1), y=(45.3, 45.9), z=(0., 3000.), projection=None,
                   values=synth.fbm_grid(np.arange(121) * 5., np.arange(91) * 5., seed=16) * 2500.)
        maps = [geo, lambert_map(ora, 45.6, 2.7, n=201, half=20000.), geoid_map()]
        sc = Scene(maps=maps, stacks=[small],
                   ops=[(S, 0, 0.), (A, 1, 0.), (A, 0, 30.)], geoid=2, range=10.)
        return Case(sc, boxes=[(45.2, 46.0, 2.2, 3.2)])
    if name == "shared_map":
        # ONE map: geoid, datum of layer 0 (under the stack, where a tile is missing) and
        # datum of layer 1
        sc = Scene(maps=[geoid_map()], stacks=[small],
                   ops=[(A, 0, -100.), (S, 0, 0.), (L, 0, 0.), (A, 0, 1500.)], geoid=0,
                   range=1.)
        return Case(sc)
    if name == "stacks_x4":
        # uniform (small), mixed 1201 / 3601 nodes, partial (tiles2) and the south-western
        # one, whose rays start over the southern hemisphere
        sc = Scene(stacks=[small, mixed, tiles2, sw],
                   ops=[(S, 0, 0.), (S, 1, 0.), (L, 0, 0.), (S, 2, 400.), (S, 3, 400.)],
                   range=0.)
        return Case(sc, boxes=[(44.9, 47.1, 0.9, 4.1), CHILE],
                    locked=[True, True, True, False])
    if name == "at_the_limits":
        # 8 layers, 24 metas, 12 data (4 stacks, the flat, 7 maps), 4 transforms
        maps = [lambert_map(ora, 45.5, 2.6, n=101, half=6000.),
                lambert_map(ora, 46.2, 3.2, n=101, half=6000.),
                _map_at(ora, "UTM 31N", 45.7, 2.9, 9000., 101, 17),
                _map_at(ora, "UTM 31N", 46.4, 2.5, 9000., 101, 18),
                _map_at(ora, "Lambert II", 45.4, 3.4, 9000., 101, 19),
                _map_at(ora, "Lambert II", 46.0, 2.4, 9000., 101, 20),
                dict(nx=81, ny=81, x=(2.8, 3.6), y=(45.2, 46.0), z=(0., 3000.), projection=None,
                     values=synth.fbm_grid(np.arange(81) * 6., np.arange(81) * 6., seed=21) * 2500.)]
        layers = [[(A, 0), (A, 2), (S, 0)], [(F, 0), (A, 4), (S, 1)], [(A, 6), (A, 1), (S, 2)],
                  [(A, 3), (A, 5), (S, 3)], [(S, 0), (A, 0), (A, 2)], [(S, 1), (A, 4), (A, 6)],
                  [(F, 0), (A, 1), (A, 3)], [(S, 2), (A, 5), (S, 3)]]
        ops = []
        for k, layer in enumerate(layers):
            if k:
                ops.append((L, 0, 0.))
            ops += [(kind, ref, 300. * k + 10. * j) for j, (kind, ref) in enumerate(layer)]
        sc = Scene(maps=maps, stacks=[small, tiles2, mixed, sw], ops=ops, range=1.)
        return Case(sc, locked=[True, True, True, False])
    raise KeyError(name)


def lla_rows(scene):
    """Rows of local approximation state per ray (tb::lla_layout): transforms are numbered
    in the order their first datum is added; the one of the first datum a sample evaluates
    (the last one added to layer 0) holds 3 + 4 ng rows, ng = 3 geodetic or 5 projected
    (+ 2 of x, y memo when projected); every other projected one 3 + 4 x 2 + 2 = 13 rows;
    other geodetic data need none."""
    names, seen, transform_of = [], set(), {}
    for kind, ref, _ in scene.ops:
        if kind == H.ADD_LAYER:
            continue
        key = (kind, 0 if kind == H.ADD_FLAT else ref)
        name = (scene.maps[ref]["projection"] if kind == H.ADD_MAP else None) or "geodetic"
        if key not in seen:
            seen.add(key)
            if name not in names:
                names.append(name)
        transform_of[key] = names.index(name)
    layer0 = []
    for kind, ref, _ in scene.ops:
        if kind == H.ADD_LAYER:
            break
        layer0.append((kind, 0 if kind == H.ADD_FLAT else ref))
    first = transform_of[layer0[-1]] if layer0 else 0
    rows = 0
    for t, name in enumerate(names):
        projected = name != "geodetic"
        if t == first:
            rows += 3 + 4 * (5 if projected else 3) + (2 if projected else 0)
        elif projected:
            rows += 13
    return rows


def _draw(boxes, n, rng, h=(-300., 4000.)):
    """Random points over the boxes, in equal shares: (lat, lon, height)."""
    parts = np.array_split(np.arange(n), len(boxes))
    la, lo = np.empty(n), np.empty(n)
    for b, idx in zip(boxes, parts):
        la[idx] = rng.uniform(b[0], b[1], len(idx))
        lo[idx] = wrap(rng.uniform(b[2], b[3] + (360. if b[3] < b[2] else 0.), len(idx)))
    return la, lo, rng.uniform(h[0], h[1], n)


def _origins(case, n, rng):
    """Ray origins over the boxes, and when the scene has ground bands, a third of them
    0.5 - 5 m over the ground of layer 0 there."""
    m = n // 3 if case.ground else 0
    la, lo, h = _draw(case.boxes, n - m, rng)
    pos = case.ora.ecef_from_geodetic(la, lo, h)
    if m:
        la, lo, h = _draw(case.ground, m, rng, h=(0.5, 5.))
        pos = np.concatenate([pos, case.ora.position(la, lo, h, 0)[0]])
    return pos


@pytest.fixture(scope="module", params=["random_%02d" % s for s in RANDOM_SEEDS] + NAMED)
def case(request, small_stack, tiles2, mixed_stack, sw_stack, globe_stacks):  # noqa: F811
    """One scene: its oracle, its plan, N_RAYS random rays and the oracle's records and
    crossings of them, shared by the tests of the scene."""
    ora0 = H.Driver(H.best_oracle())
    name = request.param
    if name.startswith("random_"):
        seed = int(name[-2:])
        c = Case(random_scene(np.random.default_rng(5000 + seed), ora0, small_stack, tiles2))
    else:
        c = named_case(name, ora0, small_stack, tiles2, mixed_stack, sw_stack, globe_stacks)
    c.name = name
    c.ora = c.scene.oracle(locked=c.locked)
    c.threads = os.cpu_count() if np.all(c.locked) else 1
    c.stepper, c.maps, c.stacks = c.scene.product()
    c.plan = c.stepper.freeze(0)
    c.n_layers = 1 + sum(op[0] == H.ADD_LAYER for op in c.scene.ops)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    c.pos = _origins(c, N_RAYS, rng)
    c.dirs = synth.random_unit(N_RAYS, 7)
    c.rule = tb.trace_rule(**RULE)
    c.want, c.wcross = c.ora.trace_crossings(c.pos, c.dirs, H.rule(**RULE), K,
                                             threads=c.threads)
    c.got = c.plan.trace(c.pos, c.dirs, c.rule)
    yield c
    del c.plan


# ---- against the oracle ---------------------------------------------------------------------

def test_rays_vs_oracle(case):
    floor = noise_floor(case.scene, case.want, case.pos, case.dirs, H.rule(**RULE),
                        locked=bool(np.all(case.locked)))
    check(case.want, case.got, max_grazing=max(3, N_RAYS // 2000), floor=floor)


def test_crossings_vs_oracle(case):
    got, gcross = case.plan.trace_crossings(case.pos, case.dirs, case.rule, K)
    _consistent(got, gcross)
    want, wcross = case.want, case.wcross
    same = (want["n_steps"] == got["n_steps"]) & (want["medium_hash"] == got["medium_hash"]) & \
        (want["status"] == got["status"])
    assert (~same).sum() <= max(3, N_RAYS // 2000)
    w, g = wcross[same], gcross[same]
    assert np.array_equal(w["from"], g["from"]) and np.array_equal(w["to"], g["to"])
    tol = np.maximum(1e-3, 1e-9 * np.abs(w["length"]))
    assert (np.abs(w["length"] - g["length"]) <= tol).all()


def test_samples_vs_oracle(case):
    """One sample per particle from a reset stepper (no direction): sample_geometry for
    every data kind of the scene, without the chaos of a whole trace."""
    rng = np.random.default_rng(17)
    la, lo, h = _draw(case.boxes, N_SAMPLES, rng)
    pos = case.ora.ecef_from_geodetic(la, lo, h)
    want = case.ora.step(pos, None)
    got = case.plan.step(pos.copy(), None)
    assert np.array_equal(got["position"], pos)

    def near_ground(o):
        e = o["elevation"]
        return (np.abs(o["altitude"][:, None] - e) < 1e-6).any(1)
    same = (want["index"] == got["index"]).all(1)
    assert (~same & ~near_ground(want) & ~near_ground(got)).sum() == 0
    assert np.abs(got["step"] - want["step"])[same].max() < 1e-6
    assert np.abs(got["altitude"] - want["altitude"])[same].max() < 1e-6
    assert ulp_distance(got["latitude"], want["latitude"])[same].max() <= 64
    # atan2 of a y of either sign of zero is +-180: the same meridian
    assert dlon(got["longitude"], want["longitude"])[same].max() <= 1e-11
    e_w, e_g = want["elevation"][same], got["elevation"][same]
    assert np.array_equal(np.abs(e_w) > 1e300, np.abs(e_g) > 1e300)  # +-DBL_MAX sentinels
    small = np.abs(e_w) < 1e300
    assert np.abs(e_w[small] - e_g[small]).max() < 1e-6


def _walkers(case, n, seed):
    rng = np.random.default_rng(seed)
    la, lo, h = _draw(case.boxes + case.ground, n, rng, h=(-50., 50.))
    ground, _ = case.ora.position(la, lo, h, 0)
    dirs = synth.random_unit(n * 12, seed).reshape(12, n, 3)
    dirs[3, ::97] = 0.   # standing still on a step: the cached sample
    return ground, dirs


def test_walks_vs_oracle(case):
    """Twelve steps with device states against the oracle's walk; the walk kernel over the
    same directions, 7 + 5, gives those twelve steps byte for byte."""
    n = N_WALKERS
    ground, dirs = _walkers(case, n, 41)
    want = case.ora.walk(ground, dirs, threads=case.threads)
    states = case.plan.states(n)
    pos = ground.copy()
    steps, bad = [], np.zeros(n, dtype=bool)
    for j in range(12):
        out = case.plan.step(pos, dirs[j], states=states)
        pos = out["position"]
        steps.append({k: v.copy() for k, v in out.items()})
        bad |= (out["index"] != want["index"][j]).any(1)
        ok = ~bad
        assert np.abs(out["step"] - want["step"][j])[ok].max(initial=0.) < 1e-5
        assert np.abs(out["altitude"] - want["altitude"][j])[ok].max(initial=0.) < 1e-5
    assert bad.sum() <= max(2, n // 500)
    assert np.abs(pos - want["position"])[~bad].max(initial=0.) < 1e-4
    s_b = case.plan.states(n)
    p_b = ground.copy()
    first = case.plan.walk(p_b, dirs[:7], states=s_b)
    second = case.plan.walk(p_b, dirs[7:], states=s_b)
    for j in range(12):
        got, jj = (first, j) if j < 7 else (second, j - 7)
        for f in ("altitude", "step", "index", "latitude", "longitude", "elevation"):
            assert np.array_equal(got[f][jj], steps[j][f]), (f, j)
    assert np.array_equal(p_b, pos)


def test_walks_without_states_vs_oracle(case):
    """No states: every call starts from a reset stepper, so the first step of a walk is a
    lone step_batch call, and the whole walk is the oracle's."""
    n = N_WALKERS
    ground, dirs = _walkers(case, n, 43)
    lone = case.plan.step(ground.copy(), dirs[0])
    walk = case.plan.walk(ground.copy(), dirs[:7])
    for f in ("altitude", "step", "index", "latitude", "longitude", "elevation"):
        assert np.array_equal(walk[f][0], lone[f]), f
    want = case.ora.walk(ground, dirs[:7], threads=case.threads)
    ok = np.logical_and.accumulate((walk["index"] == want["index"]).all(2), 0)
    assert (~ok[-1]).sum() <= max(2, n // 500)
    assert np.abs(walk["step"] - want["step"])[ok].max(initial=0.) < 1e-5
    assert np.abs(walk["altitude"] - want["altitude"])[ok].max(initial=0.) < 1e-5


def test_positions_vs_oracle(case):
    rng = np.random.default_rng(19)
    la, lo, h = _draw(case.boxes, 5000, rng, h=(-5., 50.))
    for layer in range(case.n_layers):
        wp, wi = case.ora.position(la, lo, h, layer)
        gp, gi = case.plan.position(la, lo, h, layer)
        assert np.array_equal(wi, gi), layer
        assert np.abs(wp - gp).max() < 1e-8, layer


# ---- against the GPU itself, byte for byte ---------------------------------------------------

def test_entry_points_and_schedules_agree(case):
    import torch
    plan, pos, dirs, rule, a = case.plan, case.pos, case.dirs, case.rule, case.got
    n = len(pos)
    d_res = torch.zeros((n, 96), dtype=torch.uint8, device="cuda:0")
    plan.trace_device(n, torch.from_numpy(pos).cuda(), torch.from_numpy(dirs).cuda(), rule, d_res)
    torch.cuda.synchronize()
    assert d_res.cpu().numpy().tobytes() == a.tobytes()
    fields = plan.trace_fields(pos, dirs, rule, tb.Plan.host_fields(n, FIELDS))
    for k, v in columns(a, FIELDS).items():
        assert np.array_equal(fields[k], v), k
    rec, _ = plan.trace_crossings(pos, dirs, rule, K)
    assert rec.tobytes() == a.tobytes()
    plan.schedule_set(1)    # longest-expected-first queue order
    assert plan.trace(pos, dirs, rule).tobytes() == a.tobytes()
    plan.schedule_set(0)
    plan.pipeline_set(1)    # one kernel per chunk
    assert plan.trace(pos, dirs, rule).tobytes() == a.tobytes()
    plan.pipeline_set(0)
    plan.launch_set(2, 64)  # another grid
    assert plan.trace(pos, dirs, rule).tobytes() == a.tobytes()
    plan.launch_set(0, 0)
    perm = np.random.default_rng(3).permutation(n)
    assert plan.trace(pos[perm], dirs[perm], rule).tobytes() == a[perm].tobytes()
    # above one streamed chunk (256 Ki rays) a batch goes through the streamed kernel, in
    # rounds of TURTLE_B200_STREAM_MAX_RAYS rays: three rounds here
    reps = (1 << 19) // n + 1
    big = plan.trace(np.tile(pos, (reps, 1)), np.tile(dirs, (reps, 1)), rule)
    assert big.tobytes() == np.tile(a, reps).tobytes()
    os.environ["TURTLE_B200_STREAM_MAX_RAYS"] = str(1 << 18)
    try:
        rounds = plan.trace(np.tile(pos, (reps, 1)), np.tile(dirs, (reps, 1)), rule)
    finally:
        del os.environ["TURTLE_B200_STREAM_MAX_RAYS"]
    assert rounds.tobytes() == big.tobytes() and plan.counters()["rays"] == reps * n


def test_each_ray_alone(case):
    """A ray in a batch of one gives the record it gets in the batch: no lane inherits
    anything from the ray it traced before."""
    for i in np.random.default_rng(5).choice(N_RAYS, 64, replace=False):
        one = case.plan.trace(case.pos[i:i + 1], case.dirs[i:i + 1], case.rule)
        assert one.tobytes() == case.got[i:i + 1].tobytes(), i


def test_fan_is_rays(case):
    """A fan from a station 1 m over the ground of layer 0, through the COMPACT kernels
    (fan in, records and all twelve fields out), equals the plain trace of the same rays
    with the reference's directions, in any order and one by one. Consecutive rays of a
    lane start from the same point, within range of the previous ray's reference points:
    a lane that kept them would take other steps, by far less than a millimetre, in each
    of these orders."""
    lat, lon = case.center
    origin, idx = case.plan.position([lat], [lon], [1.], 0)
    az = 360. * (np.arange(67) + 0.5) / 67
    el = 0.5 + 29.5 * (np.arange(64) + 0.5) / 64
    dirs = fan_rays(case.ora, lat, lon, az, el, 32)
    n = len(dirs)
    want = case.plan.trace(np.repeat(origin, n, 0), dirs, case.rule)
    fan = tb.Plan.make_fan(lat, lon, origin[0], az, el, bundle=32)
    rec = np.zeros(n, dtype=tb.TRACE_RESULT)
    fields = tb.Plan.host_fields(n, FIELDS)
    case.plan.trace_fan(fan, case.rule, results=rec, fields=fields)
    assert rec.tobytes() == want.tobytes()
    for k, v in columns(want, FIELDS).items():
        assert np.array_equal(fields[k], v), k
    perm = np.random.default_rng(6).permutation(n)
    p = case.plan.trace(np.repeat(origin, n, 0), dirs[perm], case.rule)
    assert p.tobytes() == want[perm].tobytes()
    for i in perm[:32]:
        one = case.plan.trace(origin, dirs[i:i + 1], case.rule)
        assert one.tobytes() == want[i:i + 1].tobytes(), i


def test_state_size(case):
    """Bytes of a particle's device state: PS_FIELDS, plus the compact local approximation
    rows at range > 0."""
    rows = lla_rows(case.scene) if case.scene.range > 0. else 0
    assert case.plan.states(8).bytes_per_particle == 8 * (PS_FIELDS + rows)
