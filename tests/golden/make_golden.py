"""Generate the golden vectors of tests/golden/ from the UNMODIFIED reference.

Run where oracle/Makefile has built oracle/_ref/libturtle_ref.so from the reference's
sources (TURTLE_REF):

    python tests/golden/make_golden.py

The reference's own test-suite holds no absolute vectors (SURVEY.md section 8c), so
these fixtures are what pins the C restatement (oracle/turtle_oracle.c) and the
product on machines where the reference is absent. Inputs are stored with the
outputs; everything is float64 / int32, bit-exact (npz keeps the raw bytes).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import harness as H  # noqa: E402
from tests.common import Scene, geoid_map, lambert_map, utm_map  # noqa: E402
from turtle_b200 import synth  # noqa: E402

TAGS = ["Lambert I", "Lambert II", "Lambert IIe", "Lambert III", "Lambert IV",
        "Lambert 93", "UTM 31N", "UTM 31S", "UTM 3.0N", "UTM 3.0S"]


def geodesy(ref, out):
    rng = np.random.default_rng(20261018)
    n = 4096
    lat = np.concatenate([rng.uniform(-90, 90, n - 6), [90., -90., 0., 0., 45.5, -33.25]])
    lon = np.concatenate([rng.uniform(-180, 180, n - 6), [0., 0., 0., 180., 3.5, 151.2]])
    alt = np.concatenate([rng.uniform(-1000, 9000, n - 6), [0., 0., 0., 100., 1000., -50.]])
    ecef = ref.ecef_from_geodetic(lat, lon, alt)
    # exact pole / axis inputs of the special case, ecef.c:77-84
    ecef_special = np.array([[0., 0., 6356752.3142], [0., 0., -6356752.3142],
                             [0., 0., 7e6], [6378137., 0., 0.], [0., 6378137., 0.]])
    ecef_all = np.concatenate([ecef, ecef_special])
    la, lo, al = ref.ecef_to_geodetic(ecef_all)
    az = rng.uniform(0, 360, n)
    el = rng.uniform(-90, 90, n)
    d = ref.ecef_from_horizontal(lat, lon, az, el)
    az2, el2 = ref.ecef_to_horizontal(lat, lon, d)
    out.update(geo_lat=lat, geo_lon=lon, geo_alt=alt, geo_ecef=ecef, geo_ecef_all=ecef_all,
               geo_back_lat=la, geo_back_lon=lo, geo_back_alt=al, hor_az=az, hor_el=el,
               hor_dir=d, hor_back_az=az2, hor_back_el=el2)
    shrink_geodesy(out, n)
    pla = rng.uniform(41., 51., 1024)
    plo = rng.uniform(-5., 9., 1024)
    out.update(proj_lat=pla, proj_lon=plo)
    for t in TAGS:
        x, y = ref.project(t, pla, plo)
        bla, blo = ref.project(t, x, y, inverse=True)
        key = t.replace(" ", "_").replace(".", "p")
        out["proj_%s_x" % key], out["proj_%s_y" % key] = x, y
        out["proj_%s_lat" % key], out["proj_%s_lon" % key] = bla, blo


def shrink_geodesy(out, n):
    """Keep every other random row (and all the special ones) of the n-row geodesy
    vectors, so that the stored file stays under 1 MB."""
    keep = np.r_[0:n - 6:2, n - 6:n]
    keep_all = np.r_[keep, n:n + 5]  # + the pole / axis inputs of ecef_all
    for k in ("geo_lat", "geo_lon", "geo_alt", "geo_ecef", "hor_az", "hor_el", "hor_dir",
              "hor_back_az", "hor_back_el"):
        out[k] = out[k][keep]
    for k in ("geo_ecef_all", "geo_back_lat", "geo_back_lon", "geo_back_alt"):
        out[k] = out[k][keep_all]


def maps(ref, out):
    # Appendix D vector M: 5 x 4 map with an analytic fill
    ix, iy = np.meshgrid(np.arange(5), np.arange(4))
    vals = 37. * ix + 101. * iy + 13. * ix * iy
    m = ref.map_create(5, 4, (10., 14.), (20., 23.), (0., 1000.), None, vals)
    qx = np.array([11.3, 14., 13.999, 14.0000001, 10., 9.9999, 12.5, np.nan])
    qy = np.array([21.7, 23., 22.5, 21., 20., 20., 23.0000001, 21.])
    z, inside = ref.map_elevation(m, qx, qy)
    nx_, ny_, nz_ = ref.map_node(m, ix.ravel(), iy.ravel())
    out.update(map_vals=vals, map_qx=qx, map_qy=qy, map_z=z, map_inside=inside, map_node_x=nx_,
               map_node_y=ny_, map_node_z=nz_)


def traces(ref_lib, out, stack_dir):
    rng = np.random.default_rng(7)
    # (a) config-1 style: UTM map over a flat bottom, fan from the map centre
    mp = utm_map(n=201)
    for rg in (0., 10.):
        sc = Scene(maps=[mp], ops=[(H.ADD_FLAT, 0, -100.), (H.ADD_LAYER, 0, 0.),
                                   (H.ADD_MAP, 0, 0.)], range=rg)
        d = sc.oracle(ref_lib)
        cx, cy = 0.5 * (mp["x"][0] + mp["x"][1]), 0.5 * (mp["y"][0] + mp["y"][1])
        lat, lon = d.project("UTM 31N", [cx], [cy], inverse=True)
        pos, idx = d.position(lat, lon, [1.0], 1)
        n = 256
        az, el = synth.golden_fan(n)
        dirs = d.ecef_from_horizontal(np.full(n, lat[0]), np.full(n, lon[0]), az, el)
        res, steps, _ = d.trace(np.repeat(pos, n, 0), dirs, H.rule(3100.))
        key = "c1_r%d" % int(rg)
        out[key + "_pos"], out[key + "_dir"], out[key + "_res"] = np.repeat(pos, n, 0), dirs, res
    # (b) config-3 style: flat / stack / Lambert map, two layers, geoid, LLA
    d0 = H.Driver(ref_lib)
    lm = lambert_map(d0, n=201)
    for rg, geoid in ((0., -1), (10., 1)):
        sc = Scene(maps=[lm, geoid_map()], stacks=[stack_dir],
                   ops=[(H.ADD_FLAT, 0, 0.), (H.ADD_STACK, 0, 0.), (H.ADD_MAP, 0, 0.),
                        (H.ADD_LAYER, 0, 0.), (H.ADD_STACK, 0, 500.), (H.ADD_MAP, 0, 600.)],
                   geoid=geoid, range=rg)
        d = sc.oracle(ref_lib)
        n = 512
        olat = rng.uniform(44.9, 47.1, n)
        olon = rng.uniform(1.9, 4.1, n)
        oalt = rng.uniform(-500, 5000, n)
        pos = d.ecef_from_geodetic(olat, olon, oalt)
        dirs = synth.random_unit(n, 11)
        res, steps, _ = d.trace(pos, dirs, H.rule(9000., length_max=5e4))
        key = "c3_r%d" % int(rg)
        out[key + "_pos"], out[key + "_dir"], out[key + "_res"] = pos, dirs, res
        one = d.step(pos, dirs)
        for f in ("position", "latitude", "longitude", "altitude", "elevation", "step", "index"):
            out[key + "_step_" + f] = one[f]
    # Appendix D vector S: flat only, three consecutive steps
    sc = Scene(ops=[(H.ADD_FLAT, 0, 0.)], range=0.)
    d = sc.oracle(ref_lib)
    pos, _ = d.position([45.], [3.], [100.], 0)
    dirs = d.ecef_from_horizontal([45.], [3.], [90.], [-2.])
    w = d.walk(pos, np.repeat(dirs[None], 3, 0))
    out.update(flat_pos=pos, flat_dir=dirs, flat_step=w["step"], flat_alt=w["altitude"],
               flat_index=w["index"], flat_final=w["position"])


def main():
    if not os.path.exists(H.REF):
        raise SystemExit("build oracle/_ref first: make -C oracle ref")
    ref = H.Driver(H.REF)
    out = {}
    geodesy(ref, out)
    maps(ref, out)
    stack_dir = "/tmp/turtle_golden_stack1201"
    synth.write_hgt_stack(stack_dir, 45, 2, 2, 2, n=1201, skip=((46, 3),))
    traces(H.REF, out, stack_dir)
    path = os.path.join(HERE, "reference_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "%.1f kB" % (os.path.getsize(path) / 1e3), len(out), "arrays")


if __name__ == "__main__":
    main()
