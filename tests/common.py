"""Scenes shared by the tests: ONE description of maps / stacks / layers is turned
into (a) an oracle driver (reference .so or C restatement) and (b) the product's
objects, so both sides see the same bytes."""
import numpy as np

import turtle_b200 as tb
from oracle import harness as H
from turtle_b200 import synth


class Scene:
    def __init__(self, maps=(), stacks=(), ops=(), geoid=-1, range=1., slope=0.4,
                 resolution=1e-2):
        self.maps = list(maps)      # dict(nx, ny, x, y, z, projection, values[ny, nx])
        self.stacks = list(stacks)  # directories of .hgt tiles
        self.ops = list(ops)        # (kind, ref, offset) in add_* order
        self.geoid = geoid
        self.range, self.slope, self.resolution = range, slope, resolution

    def oracle(self, library=None, locked=False):
        """`locked`: one flag for all stacks, or one per stack."""
        d = H.Driver(library or H.best_oracle())
        for m in self.maps:
            d.map_create(m["nx"], m["ny"], m["x"], m["y"], m["z"], m["projection"], m["values"])
        for i, s in enumerate(self.stacks):
            d.stack_create(s, locked=locked[i] if isinstance(locked, (list, tuple)) else locked)
        d.geometry(self.ops, geoid=self.geoid, range=self.range, slope=self.slope,
                   resolution=self.resolution)
        return d

    def product(self):
        """-> (Stepper, maps, stacks) built through the product's C ABI."""
        maps = [tb.Map(m["nx"], m["ny"], m["x"], m["y"], m["z"], m["projection"],
                       np.asarray(m["values"]).reshape(m["ny"], m["nx"])) for m in self.maps]
        stacks = [tb.Stack(s) for s in self.stacks]
        s = tb.Stepper(range=self.range, slope=self.slope, resolution=self.resolution,
                       geoid=maps[self.geoid] if self.geoid >= 0 else None)
        for kind, ref, offset in self.ops:
            if kind == H.ADD_LAYER:
                s.add_layer()
            elif kind == H.ADD_FLAT:
                s.add_flat(offset)
            elif kind == H.ADD_MAP:
                s.add_map(maps[ref], offset)
            else:
                s.add_stack(stacks[ref], offset)
        return s, maps, stacks


def utm_map(n=301, pitch=10., x0=486000., y0=5057000., zscale=3000., seed=synth.SEED):
    """Config-1 style map: n x n nodes, `pitch` metres, UTM 31N, synthetic terrain."""
    vals = synth.fbm_grid(np.arange(n) * 3., np.arange(n) * 3., seed) * zscale
    return dict(nx=n, ny=n, x=(x0, x0 + pitch * (n - 1)), y=(y0, y0 + pitch * (n - 1)),
                z=(0., 3000.), projection="UTM 31N", values=vals)


def lambert_map(oracle, lat_c=45.6, lon_c=2.7, n=301, half=4000., nodes_per_degree=1200,
                lat0=45, lon0=2, tag="Lambert 93"):
    """Config-3 style local map: projected grid resampled from the SAME synthetic terrain
    as the tile stack (global lattice origin at (lat0, lon0))."""
    cx, cy = oracle.project(tag, [lat_c], [lon_c])
    x = (cx[0] - half, cx[0] + half)
    y = (cy[0] - half, cy[0] + half)
    X, Y = np.meshgrid(np.linspace(x[0], x[1], n), np.linspace(y[0], y[1], n))
    la, lo = oracle.project(tag, X.ravel(), Y.ravel(), inverse=True)
    vals = np.rint(synth.fbm_points((lo - lon0) * nodes_per_degree,
                                    (la - lat0) * nodes_per_degree) * 3000.) + 0.0
    return dict(nx=n, ny=n, x=x, y=y, z=(0., 6553.5), projection=tag, values=vals)


def geoid_map():
    lon = np.linspace(0, 360, 361)
    lat = np.linspace(-90, 90, 181)
    vals = 30. + 10. * np.sin(np.radians(lon))[None, :] * np.cos(np.radians(lat))[:, None]
    return dict(nx=361, ny=181, x=(0., 360.), y=(-90., 90.), z=(-100., 100.), projection=None,
                values=vals)


TAGS = ["Lambert 93", "Lambert I", "Lambert II", "Lambert IIe", "Lambert III", "Lambert IV",
        "UTM 31N", "UTM 3.0N", None]


def second_stack(directory):
    """A tile stack that differs from conftest's `small_stack` in extent (1 x 3 tiles from
    N45 E001), tile resolution (3601 nodes) and the missing tile (45, 1), so that a wrong
    tile table offset or a wrong per-stack tile shape changes the answer. Its terrain has
    another seed."""
    synth.write_hgt_stack(directory, 45, 1, 1, 3, n=3601, seed=synth.SEED + 1, skip=((45, 1),))
    return directory


def random_map(rng, ref):
    tag = TAGS[rng.integers(len(TAGS))]
    nx, ny = int(rng.integers(20, 120)), int(rng.integers(20, 120))
    lat_c, lon_c = rng.uniform(45.3, 46.7), rng.uniform(2.3, 3.7)
    if tag is None:
        half = rng.uniform(0.02, 0.3)
        x, y = (lon_c - half, lon_c + half), (lat_c - half, lat_c + half)
    else:
        cx, cy = ref.project(tag, [lat_c], [lon_c])
        half = rng.uniform(1000., 20000.)
        x, y = (cx[0] - half, cx[0] + half), (cy[0] - half, cy[0] + half)
    values = np.resize(synth.fbm_grid(np.arange(nx) * rng.uniform(1, 8),
                                      np.arange(ny) * rng.uniform(1, 8),
                                      seed=int(rng.integers(1 << 30))), (ny, nx))
    return dict(nx=nx, ny=ny, x=x, y=y, z=(0., 3000.), projection=tag,
                values=values * rng.uniform(500, 3000))


def random_scene(rng, ref, tiles, tiles2=None):
    """1 - 3 layers of 1 - 3 data each: flat, tile stacks and maps in nine projections
    (geodetic maps included), offsets, geoid on or off, local approximation range 0 / 1 /
    10 / 100, random slope and resolution factors. With `tiles2` every stack datum is one
    of the two stacks at random. Rays over lat 44.9 - 47.1, lon 1.9 - 4.1 see all of it."""
    n_maps = int(rng.integers(0, 4))
    maps = [random_map(rng, ref) for _ in range(n_maps)]
    geoid = -1
    if rng.random() < 0.4:
        maps.append(geoid_map())
        geoid = len(maps) - 1
    stacks = [tiles] if tiles2 is None else [tiles, tiles2]
    ops = []
    for layer in range(int(rng.integers(1, 4))):
        if layer > 0:
            ops.append((H.ADD_LAYER, 0, 0.))
        for _ in range(int(rng.integers(1, 4))):
            kind = rng.integers(3)
            offset = float(rng.uniform(-50, 50) + 400. * layer)
            if (kind == 1) and (n_maps > 0):
                ops.append((H.ADD_MAP, int(rng.integers(n_maps)), offset))
            elif (kind == 0) and (rng.random() < 0.5):
                ops.append((H.ADD_FLAT, 0, float(rng.uniform(-100, 500) + 400 * layer)))
            else:
                ops.append((H.ADD_STACK, int(rng.integers(len(stacks))) if tiles2 else 0,
                            offset))
    return Scene(maps=maps, stacks=stacks, ops=ops, geoid=geoid,
                 range=[0., 1., 10., 100.][rng.integers(4)], slope=float(rng.uniform(0.1, 1.)),
                 resolution=float(10 ** rng.uniform(-3, 0)))


def ulp_distance(a, b):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    ia, ib = a.view(np.int64), b.view(np.int64)
    # map the sign-magnitude order of IEEE doubles onto a monotonic integer line
    ia = np.where(ia < 0, np.int64(-2 ** 63) - ia, ia)
    ib = np.where(ib < 0, np.int64(-2 ** 63) - ib, ib)
    return np.abs(ia - ib)


def compare_traces(ref, got, rel=1e-9, absolute=1e-3):
    """Parity report of two result arrays. `exact` = rays whose discrete outcome
    (steps, status, index, media sequence) is identical; among those, lengths are
    compared with the north-star tolerance (1e-9 relative / 1 mm)."""
    n = len(ref)
    discrete = np.ones(n, dtype=bool)
    for f in ("n_steps", "status", "medium_hash", "n_changes"):
        discrete &= (ref[f] == got[f])
    discrete &= (ref["index"] == got["index"]).all(1)
    tol = np.maximum(absolute, rel * np.abs(ref["length"]))
    len_ok = (np.abs(ref["length"] - got["length"]) <= tol).all(1)
    tot_ok = np.abs(ref["total"] - got["total"]) <= np.maximum(absolute, rel * np.abs(ref["total"]))
    dpos = np.abs(ref["position"] - got["position"]).max(1)
    bit = np.array([ref[i].tobytes() == got[i].tobytes() for i in range(n)]) if n else np.zeros(0, bool)
    return dict(n=n, discrete_mismatch=int((~discrete).sum()),
                length_mismatch=int((discrete & ~(len_ok & tot_ok)).sum()),
                bit_identical=int(bit.sum()),
                max_dpos=float(dpos[discrete].max()) if discrete.any() else 0.,
                max_dlen=float(np.abs(ref["length"] - got["length"])[discrete].max()) if discrete.any() else 0.)
