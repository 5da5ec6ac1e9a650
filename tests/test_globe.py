"""The frame, projection and query kernels and the stepper away from France: at the
antimeridian, on the equator, at the poles and over the whole domain of each transform,
against the oracle (the reference when it was built, else the C restatement).

Longitudes are compared modulo 360 where the sign of a zero y decides between -180 and
+180 (atan2(+-0, x < 0)): that is the same meridian, not a defect."""
import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.common import Scene, compare_traces, ulp_distance
from tests.test_gpu_geometries import dlon, named_case, write_seam_stack
from tests.test_horizon import HORIZON_FOUND, obstructed
from turtle_b200 import synth

B = 6356752.3142


@pytest.fixture(scope="module")
def ora():
    return H.Driver(H.best_oracle())


@pytest.fixture(scope="module")
def seam_stack(tmp_path_factory):
    return write_seam_stack(str(tmp_path_factory.mktemp("seam")))


def seam_case(name, seam_stack):
    c = named_case(name, H.Driver(H.best_oracle()), None, None, None, None,
                   dict(seam=seam_stack, arctic=None))
    c.ora = c.scene.oracle(locked=False)
    c.stepper, c.maps, c.stacks = c.scene.product()
    return c


def _rays(c, n, seed):
    rng = np.random.default_rng(seed)
    la = rng.uniform(-0.9, 0.9, n)
    lo = rng.uniform(179.1, 180.9, n)
    lo = np.where(lo > 180., lo - 360., lo)
    return c.ora.ecef_from_geodetic(la, lo, rng.uniform(-200., 4000., n)), synth.random_unit(n, seed)


# ---- on the host: the footprint cull is the same code ----------------------------------------

def test_host_antimeridian_map_is_seen(seam_stack):
    """The product's scalar calls flatten the geometry with the same footprint boxes as the
    device plan and cull at range 0 with the same test: a UTM 1N map west of its zone, whose
    unwrapped inverse projection lies at -180.23 .. -180.0001 deg while its samples have
    longitudes of 179.77 .. 179.9999, must be seen as the oracle sees it."""
    c = seam_case("antimeridian_r0", seam_stack)
    prod = c.scene.oracle(H.PRODUCT)
    pos, dirs = _rays(c, 1000, 3)
    rule = H.rule(6000., length_max=3e4, max_steps=5000)
    want, s0, _ = c.ora.trace(pos, dirs, rule)
    got, s1, _ = prod.trace(pos, dirs, rule)
    rep = compare_traces(want, got)
    assert rep["discrete_mismatch"] == 0 and rep["length_mismatch"] == 0, rep
    # samples over the UTM 1N map answer with it (layer 0: meta 1, the map)
    ml = c.scene.maps[0]
    x = np.random.default_rng(4).uniform(ml["x"][0], ml["x"][1], 2000)
    y = np.random.default_rng(5).uniform(ml["y"][0], ml["y"][1], 2000)
    la, lo = c.ora.project("UTM 1N", x, y, inverse=True)
    assert (lo < -180.).all()  # not wrapped by the inverse projection
    p = c.ora.ecef_from_geodetic(la, lo, np.full(2000, -100.))
    w, g = c.ora.step(p, None), prod.step(p, None)
    assert np.array_equal(w["index"], g["index"]) and (w["index"][:, 1] == 1).all()
    assert np.array_equal(w["elevation"], g["elevation"])
    assert (g["longitude"] > 179.).all()


# ---- ECEF -> geodetic over its whole domain --------------------------------------------------

def _geodetic_edges(ora):
    """Points on and around every branch switch of ecef_to_geodetic at 50 km and more from
    the centre of the Earth, plus the general cases (axis, denormal, huge, NaN, Inf)."""
    rng = np.random.default_rng(31)
    pts = []
    # the polar axis, and just off it: w^2 on both sides of 1E-200
    for z in (B + 25., -(B + 25.), 0., -0., 1e5, -1e5, 1e8):
        pts.append((0., 0., z))
        for w in (1e-100 * (1. - 4e-16), 1e-100, 1e-100 * (1. + 4e-16), 1e-99, 1e-101, 1e-3):
            pts += [(w, 0., z), (0., w, z), (-w, 0., z), (w / np.sqrt(2.), -w / np.sqrt(2.), z)]
    # z = +-0, |x| = |y| and the quadrant boundaries, y = +-0 with x < 0
    for r in (6378137., 6378137. + 5000., 1e5, 1e7):
        for z in (0., -0., 1e3, -1e3):
            for x, y in ((r, 0.), (-r, 0.), (-r, -0.), (0., r), (0., -r), (r, r), (-r, r),
                         (r, -r), (-r, -r), (-r, 1e-300), (-r, -1e-300), (-r, 5e-324)):
                pts.append((x, y, z))
    pts = [np.array(pts)]
    # the c2 = 0.3 switch (geocentric cos^2 = 0.3) and s = 0.55 in asin_latitude (about
    # 33.37 deg of geodetic latitude at the surface), densely, at several heights
    n = 40000
    az = rng.uniform(-np.pi, np.pi, n)
    r = np.where(rng.random(n) < 0.5, rng.uniform(6.35e6, 6.4e6, n), 10 ** rng.uniform(4.7, 8, n))
    gc = np.arccos(np.sqrt(0.3)) + rng.uniform(-1e-9, 1e-9, n) * np.where(rng.random(n) < 0.5, 1., 1e6)
    gc *= np.where(rng.random(n) < 0.5, 1., -1.)
    pts.append(np.stack([r * np.cos(gc) * np.cos(az), r * np.cos(gc) * np.sin(az), r * np.sin(gc)], 1))
    la = rng.uniform(33.2, 33.6, n) * np.where(rng.random(n) < 0.5, 1., -1.)
    pts.append(ora.ecef_from_geodetic(la, rng.uniform(-180., 180., n), rng.uniform(-1e4, 1e5, n)))
    # radii from 50 km to 1e8 m in every direction
    d = synth.random_unit(n, 32)
    pts.append(d * 10 ** rng.uniform(np.log10(5e4), 8, n)[:, None])
    # the general branch: huge, denormal coordinates, NaN, Inf
    pts.append(np.array([(1e101, 2e101, 3e101), (-1e150, 1e149, -1e150), (3e200, 0., 1e200),
                         (1e-160, -1e-160, 1e-160), (1e-300, 0., B), (np.nan, 0., B),
                         (0., np.nan, B), (1e6, 1e6, np.nan), (0., 0., np.inf),
                         (0., 0., -np.inf)]))
    return np.concatenate(pts)


# The device arctangent divides through a reciprocal: with a denormal or infinite x or y
# it makes 0 x inf, and the longitude is NaN where the reference's is finite
# (turtle_b200.h). Latitude and altitude are the reference's there.
ATAN2_NAN = np.array([(5e-324, 0., B), (5e-324, 5e-324, 0.), (np.inf, 0., 0.)])


def _same(a, b):
    return (a == b) | (np.isnan(a) & np.isnan(b))


@pytest.mark.gpu
def test_to_geodetic_whole_domain(ora):
    """Altitude bit-exact, latitude and longitude within 4 ulp (turtle_b200.h states the
    domain: at least 50 km from the centre of the Earth), NaN where the oracle gives NaN."""
    ecef = _geodetic_edges(ora)
    want = ora.ecef_to_geodetic(ecef)
    got = tb.ecef_to_geodetic_batch(ecef)
    assert _same(want[2], got[2]).all(), ecef[~_same(want[2], got[2])][:8]
    for k in (0, 1):
        nan = np.isnan(want[k])
        assert np.array_equal(nan, np.isnan(got[k])), (k, ecef[nan != np.isnan(got[k])][:8])
        u = ulp_distance(want[k][~nan], got[k][~nan])
        if k == 1:  # +-180: the same meridian
            u = np.where(dlon(want[k][~nan], got[k][~nan]) == 0., 0, u)
        assert u.max() <= 4, (k, u.max(), ecef[~nan][u > 4][:8])
    want = ora.ecef_to_geodetic(ATAN2_NAN)
    got = tb.ecef_to_geodetic_batch(ATAN2_NAN)
    assert np.isfinite(want[1]).all() and np.isnan(got[1]).all()
    assert _same(want[0], got[0]).all() and _same(want[2], got[2]).all()


@pytest.mark.gpu
def test_to_geodetic_near_the_centre(ora):
    """Closer than 50 km to the centre of the Earth Olson's method leaves the range its
    device arcsine polynomial was fitted for (and the reference's own acos / asin take
    arguments beyond 1 below about 40 km). Outside the stated domain the latitude is not
    bounded, only reported; the longitude, which does not go through Olson's method, stays
    within 4 ulp."""
    d = synth.random_unit(200000, 33)
    ecef = d * 10 ** np.random.default_rng(34).uniform(3, np.log10(5e4), len(d))[:, None]
    want = ora.ecef_to_geodetic(ecef)
    got = tb.ecef_to_geodetic_batch(ecef)
    ok = np.isfinite(want[0]) & np.isfinite(want[2])
    print("near the centre: %d of %d finite in the oracle, max |dlat| %.3g deg" % (
        ok.sum(), len(ok), np.abs(want[0] - got[0])[ok].max()))
    assert ulp_distance(want[1], got[1]).max() <= 4


@pytest.mark.gpu
def test_from_geodetic_and_horizontal_edges(ora):
    """Poles, the antimeridian and the equator, exactly and within 1e-13 deg."""
    la = np.array([-90., 90., 0., -0., 1e-13, -1e-13, 90. - 1e-13, -90. + 1e-13, 45., 84.])
    lo = np.array([-180., 180., 0., -0., 180. - 1e-13, -180. + 1e-13, 1e-13, 179.9999, -179.9999,
                   90.])
    L, O = np.meshgrid(la, lo)
    L, O = L.ravel(), O.ravel()
    rng = np.random.default_rng(35)
    n = len(L)
    for h in (0., -1e3, 1e5):
        want = ora.ecef_from_geodetic(L, O, np.full(n, h))
        got = tb.ecef_from_geodetic_batch(L, O, np.full(n, h))
        assert np.abs(want - got).max() <= 1e-15 * 6.4e6 * 4
    for az, el in ((0., 0.), (90., 30.), (180., -90.), (270., 90.), (359.9999, 1e-13)):
        want = ora.ecef_from_horizontal(L, O, np.full(n, az), np.full(n, el))
        got = tb.ecef_from_horizontal_batch(L, O, np.full(n, az), np.full(n, el))
        assert np.abs(want - got).max() <= 4e-16 * 4
    az, el = rng.uniform(0, 360, n), rng.uniform(-90, 90, n)
    want = ora.ecef_from_horizontal(L, O, az, el)
    assert np.abs(want - tb.ecef_from_horizontal_batch(L, O, az, el)).max() <= 4e-16 * 4


# ---- projections over their whole domain -----------------------------------------------------

def _projection_errors(ora, tag, la, lo):
    p = tb.Projection(tag)
    wx, wy = ora.project(tag, la, lo)
    gx, gy = p.project_batch(la, lo)
    wla, wlo = ora.project(tag, wx, wy, inverse=True)
    gla, glo = p.unproject_batch(wx, wy)
    return (max(np.abs(wx - gx).max(), np.abs(wy - gy).max()), np.abs(wla - gla).max(),
            dlon(wlo, glo).max())


@pytest.mark.gpu
def test_utm_every_zone(ora):
    """Every UTM zone, north and south, at latitudes -80 .. 84 and out to 10 deg beyond the
    edges of the zone (where the eta of the Krueger series, and the error of the device's
    recurrences with it, grow), and a free central meridian on the antimeridian. Tolerances
    of test_gpu_frames.test_projection_batches: x, y within 2e-8 m, latitude and longitude
    within 1e-12 deg."""
    rng = np.random.default_rng(36)
    n = 4096
    worst = np.zeros(3)
    tags = ["UTM %d%s" % (z, h) for z in range(1, 61) for h in "NS"] + ["UTM 180.0N", "UTM 180.0S"]
    for tag in tags:
        lon0 = 180. if "." in tag else -183. + 6. * int(tag.split()[1][:-1])
        la = rng.uniform(-80., 84., n)
        lo = lon0 + rng.uniform(-13., 13., n)
        lo = np.where(lo > 180., lo - 360., np.where(lo <= -180., lo + 360., lo))
        err = _projection_errors(ora, tag, la, lo)
        worst = np.maximum(worst, err)
        assert err[0] < 2e-8 and err[1] < 1e-12 and err[2] < 1e-12, (tag, err)
    print("UTM, largest error: x, y %.3g m, latitude %.3g deg, longitude %.3g deg" % tuple(worst))


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["Lambert 93", "Lambert I", "Lambert II", "Lambert IIe",
                                 "Lambert III", "Lambert IV"])
def test_lambert_domain(ora, tag):
    """The six Lambert tags over France and its margins (test_projection_batches bounds)."""
    rng = np.random.default_rng(37)
    n = 1 << 16
    err = _projection_errors(ora, tag, rng.uniform(40., 53., n), rng.uniform(-7., 11., n))
    print(tag, "largest error: x, y %.3g m, latitude %.3g deg, longitude %.3g deg" % err)
    assert err[0] < 2e-8 and err[1] < 2e-8 and err[2] < 1e-12


# ---- stack queries and positions on the seam -------------------------------------------------

@pytest.mark.gpu
def test_stack_on_the_seam(seam_stack):
    """Elevation and gradient of a stack whose tile table spans 360 columns, bit-exact at
    longitude +-180 exactly, on the equator and within 1e-13 deg of both."""
    ref = H.Driver(H.best_oracle())
    st = ref.stack_create(seam_stack)
    stepper = tb.Stepper(range=0.)
    stepper.add_stack(tb.Stack(seam_stack), 0.)
    plan = stepper.freeze(0)
    rng = np.random.default_rng(38)
    n = 1 << 16
    la = rng.uniform(-1.1, 1.1, n)
    lo = rng.uniform(178.9, 181.1, n)
    lo = np.where(lo > 180., lo - 360., lo)
    k = n // 4
    eps = rng.choice([0., 1e-13, -1e-13, 2e-14], k)
    lo[:k] = rng.choice([-180., 180., 179., -179.], k) + eps
    la[k:2 * k] = rng.choice([0., -1., 1.], k) + rng.choice([0., 1e-13, -1e-13], k)
    lo[2 * k:2 * k + 64] = 180.
    la[2 * k:2 * k + 64] = 0.
    lo[2 * k + 64:2 * k + 128] = -180.
    wz, win = ref.stack_elevation(st, la, lo)
    gz, gin = plan.stack_elevation(0, la, lo)
    assert np.array_equal(win, gin) and np.array_equal(wz, gz)
    wla, wlo, win = ref.stack_gradient(st, la, lo)
    gla, glo, gin = plan.stack_gradient(0, la, lo)
    assert np.array_equal(win, gin)
    assert np.array_equal(wla, gla) and np.array_equal(wlo, glo)
    assert 0.3 < gin.mean() < 1.


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["antimeridian_r0", "high_latitude"])
def test_positions_at_the_seam_and_far_north(name, seam_stack, tmp_path):
    rng = np.random.default_rng(39)
    if name == "antimeridian_r0":
        c = seam_case(name, seam_stack)
        la = rng.uniform(-1., 1., 4000)
        lo = np.concatenate([np.full(1000, 180.), np.full(1000, -180.),
                             180. - rng.uniform(0., 1e-4, 1000), -180. + rng.uniform(0., 1e-4, 1000)])
        la[:200] = 0.
    else:
        arctic = str(tmp_path / "arctic")
        synth.write_hgt_stack(arctic, 78, 15, 2, 2, n=1201)
        c = named_case(name, H.Driver(H.best_oracle()), None, None, None, None,
                       dict(seam=None, arctic=arctic))
        c.ora = c.scene.oracle()
        c.stepper, c.maps, c.stacks = c.scene.product()
        la = np.concatenate([np.full(2000, 84.), rng.uniform(83.5, 84.05, 1000),
                             rng.uniform(78., 80., 1000)])
        lo = rng.uniform(14., 17., 4000)
    plan = c.stepper.freeze(0)
    h = rng.uniform(-5., 50., len(la))
    for layer in range(2):
        wp, wi = c.ora.position(la, lo, h, layer)
        gp, gi = plan.position(la, lo, h, layer)
        assert np.array_equal(wi, gi), layer
        assert np.abs(wp - gp).max() < 1e-8, layer


# ---- residency and the horizon on the seam ---------------------------------------------------

@pytest.mark.gpu
def test_residency_across_the_seam(seam_stack):
    """A plan made for the box of a set of rays answers like the plan of the whole stack:
    rays that stay east of the seam (a box of one side), and rays across it (whose box has
    no longitude bounds)."""
    c = seam_case("antimeridian_r0", seam_stack)
    full = c.stepper.freeze(0)
    rule = tb.trace_rule(6000., length_max=1.5e4, max_steps=5000)
    for lon, cross in ((179.5, False), (179.9995, True)):
        origin, idx = c.stepper.position(0.5, lon, 1., 0)
        assert idx >= 0
        dirs = synth.fan_directions(0.5, lon, 128, 32)
        pos = np.repeat(origin[None], len(dirs), 0)
        box = tb.residency_from_rays(pos, dirs, rule, margin=0.001)
        assert np.isnan(box.longitude_min) == cross
        part = c.stepper.freeze(0, region=box)
        if not cross:
            assert part.residency()["tiles_skipped"] > 0
        assert part.trace(pos, dirs, rule).tobytes() == full.trace(pos, dirs, rule).tobytes()


@pytest.mark.gpu
def test_horizon_at_the_seam(seam_stack):
    """One horizon search from a station 20 m west of the antimeridian: both bracket ends are
    the rays trace_batch traces, bit for bit."""
    c = seam_case("antimeridian_lla", seam_stack)
    plan = c.stepper.freeze(0)
    lat, lon = 0.2, 180. - 1.8e-4
    origin, idx = c.stepper.position(lat, lon, 1., 0)
    assert idx >= 0
    rule = tb.trace_rule(6000., length_max=3e4, max_steps=5000)
    az = np.arange(48) * 7.5 + 0.3
    res = plan.horizon(lat, lon, origin, az, rule, tolerance=1e-6)
    found = res["status"] == HORIZON_FOUND
    assert found.sum() >= len(res) // 2, res["status"]
    r = res[found]
    assert ((r["elevation"][:, 1] - r["elevation"][:, 0] > 0) &
            (r["elevation"][:, 1] - r["elevation"][:, 0] <= 1e-6)).all()
    n = len(r)
    origins = np.repeat(origin[None], n, 0)
    rec0, cross0 = plan.trace_crossings(origins, r["direction"][:, 0], rule, 1)
    assert (rec0["n_changes"] >= 1).all()
    assert cross0[:, 0]["length"].tobytes() == r["length"].tobytes()
    assert np.array_equal(cross0[:, 0]["to"], r["medium"][:, 1])
    rec1, _ = plan.trace_crossings(origins, r["direction"][:, 1], rule, 1)
    assert not obstructed(rec1).any()
    assert np.array_equal(rec1["status"], r["clear_status"])
    for k in (0, 1):
        want = c.ora.ecef_from_horizontal(np.full(n, lat), np.full(n, lon), az[found],
                                          r["elevation"][:, k])
        assert ulp_distance(r["direction"][:, k], want).max() <= 4
