"""The DEM node path of the device, format by format: tiles ingested on the device from
`.hgt`, `.png`, `.tif`, `.grd` and `.asc` files (ingest_kernel), decoded by tb::node_decode
(NODE_DIRECT_I16 for `.hgt` / `.tif`, NODE_AFFINE_U16 for the others), gathered globally,
from the cell-packed copy (pack_cells_kernel) or from the shared-memory window
(NodesWindow), and the same files loaded as maps.

The reference is ONE integer terrain over a 2 x 2 stack of 1 degree tiles (tile (46, 3)
missing) that every format stores without loss: int16 nodes spanning the whole range
[-32768, 32767] in every tile, so that the scaled formats get z0 = -32768 and dz = 1
exactly and every node decodes to the same double as the `.hgt` node. Every header gives
the `.hgt` tile's x0, y0, dx, dy doubles (checked on the host below), so every result on
the device must be BYTE-IDENTICAL to the `.hgt` stack's, which the oracle holds. Node
values are checked against the int16 grid the test wrote, bilinear values against numpy
evaluated in the order of map.c:272-273 (+ - * / only: bit-exact), and everything against
the product's host scalar calls.
"""
import ctypes as C
import os

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from oracle import parity as P
from tests.common import Scene, geoid_map
from turtle_b200 import synth

FORMATS = ["png", "tif", "grd", "asc"]       # each held to the `.hgt` stack of the same size
MISSING = (46, 3)
TILES = [(45, 2), (45, 3), (46, 2)]
MIXED = {(45, 2): "grd", (45, 3): "png", (46, 2): "hgt"}  # one format per tile: not uniform
LAT0, LON0 = 45, 2


# ---- the terrain and its writers ------------------------------------------------------

def terrain(n):
    """int16 nodes [2n-1, 2n-1] (rows SOUTH first) of the 2 x 2 degree area from (45, 2):
    tile (la, lo) is the [n, n] block at ((la - 45)(n - 1), (lo - 2)(n - 1)), so that shared
    edges are identical. Relief shifted down by 400 m, two basins below sea level, a
    4 km cliff between neighbouring nodes, and one -32768 and one 32767 node per tile."""
    m, k = 2 * n - 1, n - 1
    g = np.arange(m) * (3600 // k)  # one relief at any tile size
    z = np.empty((m, m), dtype=np.int32)
    for r in range(0, m, 512):      # row blocks: bounded memory at 3601 nodes
        z[r:r + 512] = synth.elevation_grid(g, g[r:r + 512]).astype(np.int32) - 400
    t = np.arange(m) / k            # degrees from the corner
    ty, tx = t[:, None], t[None, :]
    for cy, cx, radius, depth in ((0.35, 0.7, 0.12, 3000.), (1.3, 0.4, 0.2, 1500.)):
        r2 = ((tx - cx) ** 2 + (ty - cy) ** 2) / radius ** 2
        z -= np.rint(depth * np.maximum(0., 1. - r2)).astype(np.int32)
    z += np.where((tx > 1.2) & (tx < 1.5) & (ty > 0.2) & (ty < 0.8), 4000, 0).astype(np.int32)
    for la, lo in TILES + [MISSING]:
        oy, ox = (la - LAT0) * k, (lo - LON0) * k
        z[oy + round(0.85 * k), ox + round(0.1 * k)] = -32768
        z[oy + round(0.1 * k), ox + round(0.85 * k)] = 32767
    assert -32768 <= z.min() and z.max() <= 32767
    return z.astype(np.int16)


def tile_of(z, la, lo):
    n = (len(z) + 1) // 2
    oy, ox = (la - LAT0) * (n - 1), (lo - LON0) * (n - 1)
    return z[oy:oy + n, ox:ox + n]


def _text(values, per_line):
    """Whitespace separated integers, `per_line` to a line (the `.grd` reader tokenises
    127-character chunks: lines stay well below)."""
    v = values.ravel()
    lines = [" ".join(map(str, v[i:i + per_line].tolist())) for i in range(0, len(v), per_line)]
    return "\n".join(lines) + "\n"


def write_tile(directory, fmt, la, lo, t):
    """Tile (la, lo) with nodes t [n, n] (int16, rows SOUTH first) in format `fmt`."""
    n = len(t)
    dx = 1. / (n - 1)
    base = "n%02de%03d" % (la, lo)
    if fmt == "hgt":  # big-endian, north first; 1201 nodes need the SRTMGL3 name
        name = synth.hgt_name(la, lo)
        if n != 3601:
            name = name[:-4] + ".SRTMGL3.hgt"
        t[::-1].astype(">i2").tofile(os.path.join(directory, name))
    elif fmt == "png":
        tb.Map(n, n, (float(lo), lo + 1.), (float(la), la + 1.), (-32768., 32767.), None,
               t.astype(np.float64)).dump(os.path.join(directory, base + ".png"))
    elif fmt == "tif":  # the product's writer only stores z0 = -32767: Pillow writes it
        from PIL import Image, TiffImagePlugin
        ifd = TiffImagePlugin.ImageFileDirectory_v2()
        ifd[33550] = (dx, dx, 0.)                            # ModelPixelScale
        ifd.tagtype[33550] = 12
        ifd[33922] = (0., 0., 0., float(lo), la + 1., 0.)    # ModelTiepoint: north-west corner
        ifd.tagtype[33922] = 12
        Image.fromarray(np.ascontiguousarray(t[::-1]).view(np.uint16)).save(
            os.path.join(directory, base + ".tif"), tiffinfo=ifd)
    elif fmt == "grd":  # header y0 y1 x0 x1 dy dx, rows SOUTH first
        head = " ".join(repr(float(v)) for v in (la, la + 1, lo, lo + 1, dx, dx))
        with open(os.path.join(directory, base + ".grd"), "w") as f:
            f.write(head + "\n" + _text(t, 16))
    elif fmt == "asc":  # cell-corner header (the reader adds half a cell), rows NORTH first
        with open(os.path.join(directory, base + ".asc"), "w") as f:
            f.write("ncols %d\nnrows %d\nxllcorner %r\nyllcorner %r\ncellsize %r\n"
                    "NODATA_value -99999\n" % (n, n, lo - 0.5 * dx, la - 0.5 * dx, dx))
            f.write(_text(t[::-1], n))
    else:
        raise ValueError(fmt)


class Files:
    """Stacks written once per module: fmt in FORMATS + ["hgt", "mixed"]."""

    def __init__(self, root):
        self.root, self._z, self._dirs = root, {}, {}

    def z(self, n):
        if n not in self._z:
            self._z[n] = terrain(n)
        return self._z[n]

    def stack(self, fmt, n=1201):
        key = (fmt, n)
        if key not in self._dirs:
            if fmt == "tif":
                pytest.importorskip("PIL")
            d = os.path.join(self.root, "%s%d" % (fmt, n))
            os.makedirs(d)
            for la, lo in TILES:
                write_tile(d, MIXED[(la, lo)] if fmt == "mixed" else fmt, la, lo,
                           tile_of(self.z(n), la, lo))
            self._dirs[key] = d
        return self._dirs[key]

    def tile_path(self, fmt, la, lo, n=1201):
        d = self.stack(fmt, n)
        return os.path.join(d, sorted(f for f in os.listdir(d)
                                      if f.lower().startswith(("n%02de%03d" % (la, lo)).lower()))[0])


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    return Files(str(tmp_path_factory.mktemp("dem_formats")))


# ---- query points and the numpy reference -----------------------------------------------

def node_points(n):
    """Every node of every tile: (latitude, longitude) = (y0 + iy dy, x0 + ix dx)."""
    d = 1. / (n - 1)
    i = np.arange(n)
    la, lo = [], []
    for y0, x0 in TILES:
        la.append(np.repeat(y0 + i * d, n))
        lo.append(np.tile(x0 + i * d, n))
    return np.concatenate(la), np.concatenate(lo)


def edge_points(rng, k=20000):
    """On and next to the tile edges and corners (integer degrees), +-1e-13 off them, a
    fraction of a cell off them, and outside of the stack."""
    off = np.array([0., 1e-13, -1e-13, 0.3 / 1200, -0.3 / 1200])
    la = rng.uniform(44.95, 47.05, k)
    lo = rng.uniform(1.95, 4.05, k)
    a, b = k // 3, 2 * k // 3
    la[:a] = rng.integers(45, 48, a) + rng.choice(off, a)
    lo[a:b] = rng.integers(2, 5, b - a) + rng.choice(off, b - a)
    la[b:] = rng.integers(45, 48, k - b) + rng.choice(off, k - b)   # corners
    lo[b:] = rng.integers(2, 5, k - b) + rng.choice(off, k - b)
    return la, lo


def random_points(rng, k=200000):
    return rng.uniform(44.9, 47.1, k), rng.uniform(1.9, 4.1, k)


def bilinear(z, n, la, lo):
    """numpy reference of a stack query strictly inside a tile (no edge handling), in the
    order of map.c:272-273. -> (values, mask of the points it applies to)."""
    gy, gx = la - LAT0, lo - LON0
    ty, tx = np.floor(gy), np.floor(gx)
    ok = (np.abs(gy - np.rint(gy)) > 1e-9) & (np.abs(gx - np.rint(gx)) > 1e-9) & \
        (ty >= 0) & (ty <= 1) & (tx >= 0) & (tx <= 1) & ~((ty == 1) & (tx == 1))
    ty, tx = np.where(ok, ty, 0).astype(int), np.where(ok, tx, 0).astype(int)
    d = 1. / (n - 1)
    hx = (lo - (LON0 + tx)) / d
    hy = (la - (LAT0 + ty)) / d
    ix = np.where(ok, hx, 0).astype(int)
    iy = np.where(ok, hy, 0).astype(int)
    fx, fy = hx - ix, hy - iy
    gx_, gy_ = tx * (n - 1) + ix, ty * (n - 1) + iy
    zf = z.astype(np.float64)
    z00, z10 = zf[gy_, gx_], zf[gy_, gx_ + 1]
    z01, z11 = zf[gy_ + 1, gx_], zf[gy_ + 1, gx_ + 1]
    v = z00 * (1. - fx) * (1. - fy) + z01 * (1. - fx) * fy + z10 * fx * (1. - fy) + z11 * fx * fy
    return v, ok


def host_stack(directory):
    """The product's host scalar calls on a stack of `directory` (a C loop over
    turtle_stack_elevation / turtle_stack_gradient)."""
    d = H.Driver(H.PRODUCT)
    return d, d.stack_create(directory)


# ---- host: the fixtures themselves ------------------------------------------------------

@pytest.mark.parametrize("fmt", ["hgt"] + FORMATS)
def test_written_tiles_load_as_written(files, fmt):
    """Each written tile, loaded as a map: the expected shape, extents and z span, and at a
    dense sample of nodes (edge rows and columns, the extremes, 20 000 random nodes) the
    int16 node the test wrote."""
    n = 1201
    z = files.z(n)
    rng = np.random.default_rng(1)
    for la, lo in TILES:
        m = tb.Map(path=files.tile_path(fmt, la, lo))
        info, tag = m.meta()
        assert (info.nx, info.ny, tag) == (n, n, None)
        assert (info.x[0], info.x[1], info.y[0], info.y[1]) == (lo, lo + 1., la, la + 1.)
        zspan = (-32767., 32768.) if fmt in ("hgt", "tif") else (-32768., 32767.)
        assert (info.z[0], info.z[1]) == zspan
        t = tile_of(z, la, lo)
        ix = np.concatenate([np.arange(n)] * 4 + [[0, 1, n - 2, n - 1] * n,
                                                   rng.integers(0, n, 20000)])
        iy = np.concatenate([np.full(n, v) for v in (0, 1, n - 2, n - 1)] +
                            [np.repeat(np.arange(n), 4), rng.integers(0, n, 20000)])
        ex = np.argwhere((t == -32768) | (t == 32767))
        assert len(ex) == 2
        ix, iy = np.concatenate([ix, ex[:, 1]]), np.concatenate([iy, ex[:, 0]])
        got = np.array([m.node(int(i), int(j)) for i, j in zip(ix, iy)])
        assert (got[:, 2] == t[iy, ix]).all()
        d = 1. / (n - 1)
        assert (got[:, 0] == lo + ix * d).all() and (got[:, 1] == la + iy * d).all()


@pytest.mark.parametrize("fmt", FORMATS + ["mixed"])
def test_host_stacks_answer_like_hgt(files, fmt):
    """The host scalar path of every format's stack gives the `.hgt` stack's answer bit for
    bit: at every node of every tile, at random points, on and next to tile edges and
    corners and outside; and the numpy reference in cell interiors."""
    n = 1201
    rng = np.random.default_rng(2)
    la, lo = [np.concatenate(v) for v in zip(node_points(n), random_points(rng, 50000),
                                             edge_points(rng))]
    d, s = host_stack(files.stack(fmt))
    dh, sh = host_stack(files.stack("hgt"))
    z, inside = d.stack_elevation(s, la, lo)
    zh, inside_h = dh.stack_elevation(sh, la, lo)
    assert np.array_equal(inside, inside_h) and z.tobytes() == zh.tobytes()
    want, ok = bilinear(files.z(n), n, la, lo)
    assert ok.sum() > len(la) // 2 and (inside[ok] == 1).all()
    assert z[ok].tobytes() == want[ok].tobytes()
    g = d.stack_gradient(s, la[::7], lo[::7])
    gh = dh.stack_gradient(sh, la[::7], lo[::7])
    for a, b in zip(g, gh):
        assert a.tobytes() == b.tobytes()
    # the Python binding's scalar call is the same host path
    st = tb.Stack(files.stack(fmt))
    for i in range(0, len(la), len(la) // 500):
        assert st.elevation(la[i], lo[i]) == (zh[i] if inside_h[i] else 0., inside_h[i])


# ---- GPU: ingestion and decoding, node by node ------------------------------------------

def stack_plan(directory, load=False, region=None):
    st = tb.Stack(directory)
    if load:
        st.load()  # host-resident tiles: uploaded as they are
    s = tb.Stepper(range=0.)
    s.add_stack(st, 0.)
    return s, s.freeze(0, region=region)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS)
def test_ingestion_and_decoding_node_by_node(files, fmt):
    """Tiles ingested on the device from the files and tiles uploaded from the host answer
    turtle_stack_elevation_batch / _gradient_batch like the numpy reference in cell
    interiors, like the host scalar path everywhere and like the `.hgt` plan, bit for bit;
    a plan of two tiles answers the same inside its box."""
    n = 1201
    rng = np.random.default_rng(3)
    sets = [node_points(n), random_points(rng), edge_points(rng)]
    _, ingested = stack_plan(files.stack(fmt))
    r = ingested.residency()
    assert r["tiles_resident"] == 3 and r["tiles_ingested"] == 3
    _, uploaded = stack_plan(files.stack(fmt), load=True)
    assert uploaded.residency()["tiles_ingested"] == 0
    _, hgt = stack_plan(files.stack("hgt"))
    d, s = host_stack(files.stack(fmt))
    box = (44.9, 47.1, 1.9, 2.98)
    _, part = stack_plan(files.stack(fmt), region=box)
    assert part.residency()["tiles_resident"] == 2
    for la, lo in sets:
        want, ok = bilinear(files.z(n), n, la, lo)
        hz, hin = d.stack_elevation(s, la, lo)
        hg = d.stack_gradient(s, la, lo)
        ref_z = hgt.stack_elevation(0, la, lo)
        ref_g = hgt.stack_gradient(0, la, lo)
        assert np.array_equal(ref_z[1], hin) and ref_z[0].tobytes() == hz.tobytes()
        for plan in (ingested, uploaded):
            z, inside = plan.stack_elevation(0, la, lo)
            assert np.array_equal(inside, hin) and z.tobytes() == hz.tobytes()
            assert z[ok].tobytes() == want[ok].tobytes()
            g = plan.stack_gradient(0, la, lo)
            for a, b, c in zip(g, hg, ref_g):
                assert a.tobytes() == b.tobytes() == c.tobytes()
        keep = (lo < box[3] - 1e-3)
        z, inside = part.stack_elevation(0, la[keep], lo[keep])
        assert np.array_equal(inside, hin[keep]) and z.tobytes() == hz[keep].tobytes()
    assert (hin == 0).any() and ok.any()


# ---- GPU: whole rays through every format -------------------------------------------------

RULE = dict(altitude_max=9000., length_max=5e4, max_steps=20000)
STATION = (45.4, 2.6)


def flagship(directory):
    """One uniform stack, range 0, no geoid: SHAPE_STACK (the single-stack kernel)."""
    return Scene(stacks=[directory], ops=[(H.ADD_STACK, 0, 0.)], range=0.)


def layered(directory):
    """A flat layer below the stack, a geoid, the local approximation (range 10)."""
    return Scene(maps=[geoid_map()], stacks=[directory],
                 ops=[(H.ADD_FLAT, 0, -1000.), (H.ADD_LAYER, 0, 0.), (H.ADD_STACK, 0, 0.)],
                 geoid=0, range=10.)


def rays(stepper, n=30000):
    """A fan from the station and n random rays over the whole stack."""
    origin, _ = stepper.position(STATION[0], STATION[1], 1., 0)
    fan = synth.fan_directions(STATION[0], STATION[1], 128, 64)
    rng = np.random.default_rng(4)
    pos = tb.ecef_from_geodetic_batch(rng.uniform(44.9, 47.1, n), rng.uniform(1.9, 4.1, n),
                                      rng.uniform(-500., 5000., n))
    return (np.concatenate([np.repeat(origin[None], len(fan), 0), pos]),
            np.concatenate([fan, synth.random_unit(n, 6)]), origin)


def every_entry_point(stepper, plan, pos, dirs, origin):
    """The records of every batched entry point on these rays -> dict name -> bytes."""
    rule = tb.trace_rule(**RULE)
    out = {}
    for spec in (1, 0):
        for pipe in (0, 1):
            plan.specialise_set(spec)
            plan.pipeline_set(pipe)
            out["trace_%d%d" % (spec, pipe)] = plan.trace(pos, dirs, rule).tobytes()
    plan.specialise_set(1)
    plan.pipeline_set(0)
    az = np.arange(96) * 3.75 + 0.1
    el = np.linspace(-5., 30., 48)
    rec = np.zeros(len(az) * len(el), dtype=tb.api.TRACE_RESULT)
    fields = tb.Plan.host_fields(len(rec), ["length0", "total", "position", "status", "index"])
    plan.trace_fan(tb.Plan.make_fan(STATION[0], STATION[1], origin, az, el, bundle=8), rule,
                   results=rec, fields=fields)
    out["fan"] = rec.tobytes() + b"".join(v.tobytes() for v in fields.values())
    f2 = plan.trace_fields(pos, dirs, rule, tb.Plan.host_fields(len(pos), ["total", "n_steps",
                                                                           "medium_hash"]))
    out["fields"] = b"".join(v.tobytes() for v in f2.values())
    res, cross = plan.trace_crossings(pos, dirs, rule, 6)
    out["crossings"] = res.tobytes() + cross.tobytes()
    k = 4096
    states = plan.states(k)
    p = pos[-k:].copy()
    for j in range(3):
        step = plan.step(p, dirs[j:j + k], states=states)
        out["step%d" % j] = b"".join(v.tobytes() for v in step.values())
    walk = plan.walk(p, np.stack([np.roll(dirs[-k:], j, 0) for j in range(5)]), states=states)
    out["walk"] = b"".join(v.tobytes() for v in walk.values())
    out["horizon"] = plan.horizon(STATION[0], STATION[1], origin, az[::4],
                                  tb.trace_rule(6000., length_max=3e4, max_steps=5000)).tobytes()
    return out


@pytest.fixture(scope="module")
def hgt_runs(files):
    """The `.hgt` stack through every entry point, once per geometry; the random rays held
    to the oracle."""
    runs = {}
    for name, make in (("flagship", flagship), ("layered", layered)):
        sc = make(files.stack("hgt"))
        stepper, _, _ = sc.product()
        plan = stepper.freeze(0)
        pos, dirs, origin = rays(stepper)
        runs[name] = every_entry_point(stepper, plan, pos, dirs, origin)
        want, _, _ = sc.oracle(locked=True).trace(pos, dirs, H.rule(**RULE),
                                                  threads=os.cpu_count())
        got = np.frombuffer(runs[name]["trace_10"], dtype=tb.api.TRACE_RESULT)
        rep = P.report(want, got)
        grazing = max(3, len(pos) // 2000)
        assert rep["discrete_mismatch"] <= grazing, P.table(rep)
        assert rep["located_rays_over"] <= grazing, P.table(rep)
    return runs


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS + ["mixed"])
@pytest.mark.parametrize("geometry", ["flagship", "layered"])
def test_whole_rays_like_hgt(files, hgt_runs, fmt, geometry):
    """Every batched entry point through every format's stack (tiles ingested on the
    device) gives the `.hgt` stack's records byte for byte. In the flagship geometry the
    packed gather is accepted on the uniform stacks (so the single-stack kernel is the one
    that ran and decoded scaled nodes) and refused on the mixed stack."""
    sc = (flagship if geometry == "flagship" else layered)(files.stack(fmt))
    stepper, _, _ = sc.product()
    plan = stepper.freeze(0)
    assert plan.residency()["tiles_ingested"] == 3
    pos, dirs, origin = rays(stepper)
    got = every_entry_point(stepper, plan, pos, dirs, origin)
    want = hgt_runs[geometry]
    for k in want:
        assert got[k] == want[k], k
    for k in ("trace_00", "trace_01", "trace_11"):
        assert got[k] == got["trace_10"], k
    if geometry == "layered" or fmt == "mixed":
        with pytest.raises(tb.TurtleError):
            plan.gather_set(1)
    else:
        plan.gather_set(1)
        rule = tb.trace_rule(**RULE)
        assert plan.trace(pos, dirs, rule).tobytes() == want["trace_10"]
        plan.gather_set(0)


# ---- GPU: the packed and windowed gathers at tile borders -----------------------------------

K = 3600  # cells per tile side of the 3601-node stacks
WINDOW_STATIONS = {
    "interior": (45.4, 2.6),
    "south": (45. + 10. / K, 2.5),
    "north": (46. - 10. / K, 2.5),
    "west": (45.5, 2. + 10. / K),
    "east": (45.5, 3. - 10. / K),
    "last_cell": (46. - 0.5 / K, 3. - 0.5 / K),
    "corner_45_3": (45., 3.),  # corners on the rim of the stack: the rays start 2e-6
    "corner_46_2": (46., 2.),  # degrees inside (the corner itself may round outside)
    "x0_not_multiple_of_8": (45.5, 2. + 1803. / K),
}


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["hgt", "png"])
def test_gathers_at_tile_borders(files, fmt):
    """The single-stack kernel with its nodes from the cell-packed copy (mode 1) and from
    a window clamped to the tile (mode 2) gives the records of the global gather (mode 0)
    byte for byte, for windows in the tile interior, at each edge, in the last cell, at
    tile corners and at a node index that is not a multiple of 8; fans cross into the
    neighbouring tiles, the missing tile and out of the stack, and the same fans start from
    the same place in the other tiles."""
    import torch
    stepper, plan = stack_plan(files.stack(fmt, 3601))
    rule = tb.trace_rule(6000., length_max=3e4, max_steps=20000)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    for name, (lat, lon) in WINDOW_STATIONS.items():
        at = (lat + 2e-6, lon + 2e-6) if name.startswith("corner") else (lat, lon)
        # the same fan from the same place in every other tile: its cells have the node
        # indices of the window's cells but not its nodes (NodesWindow's tile test)
        pos, dirs = [], []
        for dla, dlo in ((0, 0), (0, 1), (0, -1), (1, 0), (-1, 0)):
            la, lo = at[0] + dla, at[1] + dlo
            if (int(np.floor(la)), int(np.floor(lo))) not in TILES:
                continue
            origin, idx = stepper.position(la, lo, 1., 0)
            assert idx >= 0, name
            dirs.append(synth.fan_directions(la, lo, 128, 32))
            pos.append(np.repeat(origin[None], len(dirs[-1]), 0))
        assert len(pos) >= 2, name
        pos, dirs = np.concatenate(pos), np.concatenate(dirs)
        n = len(dirs)
        d_pos, d_dir = dev(pos), dev(dirs)
        records = {}
        for mode in (0, 1, 2):
            plan.gather_set(mode, lat, lon)
            d_res = torch.zeros((n, 96), dtype=torch.uint8, device="cuda")
            before = plan.counters(sync=True)["window_hits"]
            plan.trace_device(n, d_pos, d_dir, rule, d_res)
            torch.cuda.synchronize()
            records[mode] = d_res.cpu().numpy().tobytes()
            if mode == 2:
                assert plan.counters(sync=True)["window_hits"] > before, name
        plan.gather_set(0)
        assert records[1] == records[0], name
        assert records[2] == records[0], name
        res = np.frombuffer(records[0], dtype=tb.api.TRACE_RESULT)
        assert (res["n_changes"] > 0).sum() > n // 20, name  # the fan meets the ground
    # refusals: no such mode, no tile under the window, a geometry that is not one stack
    with pytest.raises(tb.TurtleError):
        plan.gather_set(3, 45.4, 2.6)
    for lat, lon in ((46.5, 3.5), (46., 3.), (44.5, 2.5), (45.5, 4.5), (47.5, 2.5), (45.5, 1.5)):
        with pytest.raises(tb.TurtleError):
            plan.gather_set(2, lat, lon)
    flat = tb.Stepper(range=0.)
    flat.add_flat(-1000.)
    flat.add_layer()
    flat.add_stack(tb.Stack(files.stack(fmt, 3601)), 0.)
    fplan = flat.freeze(0)
    for mode in (1, 2):
        with pytest.raises(tb.TurtleError):
            fplan.gather_set(mode, 45.4, 2.6)
    fplan.gather_set(0)


# ---- GPU: maps loaded from files ------------------------------------------------------------

def map_points(rng, n):
    """Every node of tile (45, 2), its closed upper edges and corners, just outside, NaN,
    the first row of cells (the gradient quirk of map.c:353) and random points."""
    d = 1. / (n - 1)
    i = np.arange(n)
    x = [np.tile(2. + i * d, n), rng.uniform(1.999, 3.001, 100000),
         np.full(n, 3.), rng.uniform(2., 3., n), np.array([2., 3., 3., 2., 3. + 1e-12, 2. - 1e-12,
                                                           np.nan, 2.5])]
    y = [np.repeat(45. + i * d, n), rng.uniform(44.999, 46.001, 100000),
         rng.uniform(45., 46., n), np.full(n, 46.), np.array([45., 46., 45., 46., 45.5, 45.5,
                                                              45.5, np.nan])]
    x.append(rng.uniform(2., 3., 20000))
    y.append(45. + rng.uniform(0., 0.6 * d, 20000))
    return np.concatenate(x), np.concatenate(y)


def map_reference(t, x, y):
    """numpy: map.c:229-277 on the closed domain of one tile at (45, 2)."""
    n = len(t)
    d = 1. / (n - 1)
    hx, hy = (x - 2.) / d, (y - 45.) / d
    inside = (hx <= n - 1) & (hx >= 0) & (hy <= n - 1) & (hy >= 0)
    hx, hy = np.where(inside, hx, 0.), np.where(inside, hy, 0.)
    ix, iy = hx.astype(int), hy.astype(int)
    fx = np.where(ix == n - 1, 1., hx - ix)
    fy = np.where(iy == n - 1, 1., hy - iy)
    ix, iy = np.minimum(ix, n - 2), np.minimum(iy, n - 2)
    zf = t.astype(np.float64)
    z00, z10, z01, z11 = zf[iy, ix], zf[iy, ix + 1], zf[iy + 1, ix], zf[iy + 1, ix + 1]
    z = z00 * (1. - fx) * (1. - fy) + z01 * (1. - fx) * fy + z10 * fx * (1. - fy) + z11 * fx * fy
    return np.where(inside, z, 0.), inside.astype(np.int32)


def host_map(m, x, y):
    """The host scalar turtle_map_elevation / turtle_map_gradient of the same map."""
    lib = tb.api.lib
    z, gx, gy = np.zeros(len(x)), np.zeros(len(x)), np.zeros(len(x))
    inside = np.zeros(len(x), dtype=np.int32)
    a, b, c = C.c_double(), C.c_double(), C.c_int()
    for i in range(len(x)):
        z[i], inside[i] = m.elevation(x[i], y[i])
        a.value, b.value = 0., 0.
        tb.api._check(lib.turtle_map_gradient(m.handle, x[i], y[i], C.byref(a), C.byref(b),
                                              C.byref(c)))
        gx[i], gy[i] = a.value, b.value
    return z, inside, gx, gy


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["hgt"] + FORMATS)
def test_maps_loaded_from_files(files, fmt):
    """A tile loaded as a map: turtle_map_elevation_batch from the row-major and from the
    cell-packed mirror, turtle_map_gradient_batch and the fused ECEF kernel in both modes
    against the numpy reference, the host scalar calls and the `.hgt` map, bit for bit
    (the fused kernel: within the tolerance of its transcendental functions). A re-fill
    reaches both mirrors."""
    from turtle_b200._lib import lib
    n = 1201
    t = tile_of(files.z(n), 45, 2)
    m = tb.Map(path=files.tile_path(fmt, 45, 2))
    ref = tb.Map(path=files.tile_path("hgt", 45, 2))
    rng = np.random.default_rng(7)
    x, y = map_points(rng, n)
    want, win = map_reference(t, x, y)
    sample = np.concatenate([np.arange(len(x) - 20008, len(x)),
                             rng.integers(0, len(x) - 20008, 20000)])
    hz, hin, hgx, hgy = host_map(m, x[sample], y[sample])
    assert np.array_equal(hin, win[sample]) and hz.tobytes() == want[sample].tobytes()
    for mode in (0, 1):
        lib.turtle_map_gather_set(m.handle, mode)
        z, inside = m.elevation_batch(x, y)
        assert np.array_equal(inside, win) and z.tobytes() == want.tobytes(), mode
    gx, gy, gin = m.gradient_batch(x, y)
    assert np.array_equal(gin, win)
    assert gx[sample].tobytes() == hgx.tobytes() and gy[sample].tobytes() == hgy.tobytes()
    rgx, rgy, _ = ref.gradient_batch(x, y)
    assert gx.tobytes() == rgx.tobytes() and gy.tobytes() == rgy.tobytes()
    first_row = (win == 1) & ((y - 45.) * (n - 1) <= 0.5)
    assert first_row.sum() > 10000 and (gy[first_row] == 0.).all()  # map.c:353: gy untouched
    # the fused kernel, at the map's own coordinates (longitude, latitude)
    keep = ~(np.isnan(x) | np.isnan(y))
    ecef = tb.ecef_from_geodetic_batch(y[keep], x[keep], rng.uniform(0., 5000., keep.sum()))
    fused = []
    for mode in (0, 1):
        lib.turtle_map_gather_set(m.handle, mode)
        fused.append(m.elevation_ecef_batch(ecef))
    lib.turtle_map_gather_set(ref.handle, 0)
    assert all(a.tobytes() == b.tobytes() for a, b in zip(fused[0], fused[1]))
    assert all(a.tobytes() == b.tobytes() for a, b in zip(fused[0], ref.elevation_ecef_batch(ecef)))
    la, lo, _, fz, fin = fused[0]
    sub = rng.integers(0, len(ecef), 5000)
    geo = np.array([tb.ecef_to_geodetic(e) for e in ecef[sub]])
    hz2 = np.array([m.elevation(b, a) for a, b in geo[:, :2]])
    assert np.abs(geo[:, 0] - la[sub]).max() < 1e-12 and np.abs(geo[:, 1] - lo[sub]).max() < 1e-12
    both = (fin[sub] == 1) & (hz2[:, 1] == 1)
    assert (fin[sub] != hz2[:, 1]).sum() <= 2
    assert np.abs(fz[sub][both] - hz2[both, 0]).max() < 1e-5  # 4 ulp of a degree, 65 km steps
    # a re-fill reaches both mirrors (the packed one exists from the calls above)
    t2 = np.clip(t[::-1, ::-1].astype(np.int32), -32767, 32767).astype(np.int16)
    m.fill(t2.astype(np.float64))
    want2, _ = map_reference(t2, x, y)
    for mode in (1, 0):
        lib.turtle_map_gather_set(m.handle, mode)
        z, inside = m.elevation_batch(x, y)
        assert np.array_equal(inside, win) and z.tobytes() == want2.tobytes(), mode


@pytest.mark.gpu
def test_asc_nodata_node(files, tmp_path):
    """An `.asc` NODATA node is left out of the z range and quantised like any value
    (asc.c:84-145): the device answers like the host scalar path around it."""
    n = 1201
    t = tile_of(files.z(n), 45, 2).copy()
    write_tile(str(tmp_path), "asc", 45, 2, t)
    path = str(tmp_path / "n45e002.asc")
    text = open(path).read().split("\n")
    row = text[6 + (n - 1 - 600)].split(" ")  # rows north first after the 6 header lines
    row[600] = "-99999"
    text[6 + (n - 1 - 600)] = " ".join(row)
    open(path, "w").write("\n".join(text))
    m = tb.Map(path=path)
    info, _ = m.meta()
    assert (info.z[0], info.z[1]) == (-32768., 32767.)  # the NODATA value is not in the span
    d = 1. / (n - 1)
    rng = np.random.default_rng(8)
    x = 2. + (600 + rng.uniform(-2., 2., 2000)) * d
    y = 45. + (600 + rng.uniform(-2., 2., 2000)) * d
    hz, hin, hgx, hgy = host_map(m, x, y)
    z, inside = m.elevation_batch(x, y)
    gx, gy, _ = m.gradient_batch(x, y)
    assert np.array_equal(inside, hin) and z.tobytes() == hz.tobytes()
    assert gx.tobytes() == hgx.tobytes() and gy.tobytes() == hgy.tobytes()
    st = tb.Stepper(range=0.)
    st.add_stack(tb.Stack(str(tmp_path)), 0.)
    sz, sin = st.freeze(0).stack_elevation(0, y, x)
    dh, sh = host_stack(str(tmp_path))
    wz, wsin = dh.stack_elevation(sh, y, x)
    assert np.array_equal(sin, wsin) and sz.tobytes() == wz.tobytes()
    assert m.node(600, 600)[2] != t[600, 600]
