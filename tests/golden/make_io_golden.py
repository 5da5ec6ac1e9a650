"""Generate the file-format fixtures of tests/golden/io/ with the UNMODIFIED reference.

Run where oracle/_ref/libturtle_ref.so is built and the reference's sources are present:

    python tests/golden/make_io_golden.py

The reference reaches PNG and GeoTIFF through libpng / libtiff, which it dlopen()s by
their bare names; this container only has the copies bundled with Pillow, so the script
re-executes itself with a shim directory of symlinks on LD_LIBRARY_PATH. What it writes:

  tests/golden/io/*.png *.tif     written by the reference's turtle_map_dump
  tests/golden/io/*.grd *.asc     written here (text), read back by the reference
  tests/golden/io_vectors.npz     for every file: the meta data and ALL node values as the
                                  reference's turtle_map_load + turtle_map_node report them

tests/test_io_formats.py holds the product's readers to these, bit for bit.
"""
import ctypes as C
import glob
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "io")
SHIM = "/tmp/turtle_io_shim"


def _reexec_with_shim():
    if os.environ.get("TURTLE_IO_SHIM") == "1":
        return
    os.makedirs(SHIM, exist_ok=True)
    site = [p for p in sys.path if p.endswith("site-packages")][0]
    for name, pattern in (("libpng.so", "pillow.libs/libpng16-*.so*"),
                          ("libtiff.so", "pillow.libs/libtiff-*.so*")):
        found = glob.glob(os.path.join(site, pattern))
        link = os.path.join(SHIM, name)
        if found and not os.path.exists(link):
            os.symlink(found[0], link)
    env = dict(os.environ, TURTLE_IO_SHIM="1")
    env["LD_LIBRARY_PATH"] = SHIM + ":" + os.path.dirname(glob.glob(
        os.path.join(site, "pillow.libs"))[0] + "/x") + ":" + env.get("LD_LIBRARY_PATH", "")
    os.execve(sys.executable, [sys.executable] + sys.argv, env)


class MapInfo(C.Structure):
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("x", C.c_double * 2), ("y", C.c_double * 2),
                ("z", C.c_double * 2), ("encoding", C.c_char_p)]


def reference():
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libturtle_ref.so"))
    lib.turtle_error_handler_set(None)
    lib.turtle_map_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(MapInfo), C.c_char_p]
    lib.turtle_map_fill.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double]
    lib.turtle_map_dump.argtypes = [C.c_void_p, C.c_char_p]
    lib.turtle_map_load.argtypes = [C.POINTER(C.c_void_p), C.c_char_p]
    lib.turtle_map_node.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double),
                                    C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.turtle_map_meta.argtypes = [C.c_void_p, C.POINTER(MapInfo), C.POINTER(C.c_char_p)]
    lib.turtle_map_meta.restype = None
    lib.turtle_map_destroy.argtypes = [C.POINTER(C.c_void_p)]
    lib.turtle_map_destroy.restype = None
    return lib


def make_map(lib, nx, ny, x, y, z, projection, values):
    info = MapInfo(nx, ny, (C.c_double * 2)(*x), (C.c_double * 2)(*y), (C.c_double * 2)(*z), None)
    m = C.c_void_p()
    assert lib.turtle_map_create(C.byref(m), C.byref(info), projection) == 0
    for iy in range(ny):
        for ix in range(nx):
            assert lib.turtle_map_fill(m, ix, iy, float(values[iy, ix])) == 0
    return m


def describe(lib, path):
    """What the reference makes of a file: (meta vector, projection, node values)."""
    m = C.c_void_p()
    rc = lib.turtle_map_load(C.byref(m), path.encode())
    assert rc == 0, (path, rc)
    info, proj = MapInfo(), C.c_char_p()
    lib.turtle_map_meta(m, C.byref(info), C.byref(proj))
    z = np.empty((info.ny, info.nx))
    x0, y0, x1, y1, zz = (C.c_double() for _ in range(5))
    lib.turtle_map_node(m, 0, 0, C.byref(x0), C.byref(y0), C.byref(zz))
    lib.turtle_map_node(m, info.nx - 1, info.ny - 1, C.byref(x1), C.byref(y1), C.byref(zz))
    for iy in range(info.ny):
        for ix in range(info.nx):
            lib.turtle_map_node(m, ix, iy, None, None, C.byref(zz))
            z[iy, ix] = zz.value
    meta = np.array([info.nx, info.ny, info.x[0], info.x[1], info.y[0], info.y[1], info.z[0],
                     info.z[1], x0.value, y0.value, x1.value, y1.value])
    tag = proj.value.decode() if proj.value else ""
    enc = info.encoding.decode() if info.encoding else ""
    lib.turtle_map_destroy(C.byref(m))
    return meta, tag, enc, z


def terrain(nx, ny, lo, hi, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:ny, 0:nx]
    v = np.sin(xx * 0.31) * np.cos(yy * 0.17) + 0.3 * rng.standard_normal((ny, nx))
    v = (v - v.min()) / (v.max() - v.min())
    return lo + v * (hi - lo)


def main():
    _reexec_with_shim()
    os.makedirs(OUT, exist_ok=True)
    lib = reference()
    files = []

    # 1. projected map, affine 16-bit scale, PNG with the JSON header
    m = make_map(lib, 37, 23, (486000., 486360.), (5057000., 5057220.), (-50., 3200.),
                 b"UTM 31N", terrain(37, 23, -50., 3200., 1))
    assert lib.turtle_map_dump(m, os.path.join(OUT, "utm31n.png").encode()) == 0
    lib.turtle_map_destroy(C.byref(m))
    files.append("utm31n.png")
    # 2. Lambert map with non-dyadic bounds (hex-float header must round trip)
    m = make_map(lib, 11, 29, (650000.1, 651000.7), (6860000.3, 6862800.9), (0.1, 4810.45),
                 b"Lambert 93", terrain(11, 29, 0.1, 4810.45, 2))
    assert lib.turtle_map_dump(m, os.path.join(OUT, "lambert93.png").encode()) == 0
    lib.turtle_map_destroy(C.byref(m))
    files.append("lambert93.png")
    # 3. geodetic tile on the GeoTIFF integer scale (z0 = -32767, dz = 1), as PNG and TIFF
    vals = np.rint(terrain(41, 31, -420., 8848., 3))
    m = make_map(lib, 41, 31, (3., 4.), (44., 45.), (-32767., 32768.), None, vals)
    assert lib.turtle_map_dump(m, os.path.join(OUT, "n44e003.tif").encode()) == 0
    assert lib.turtle_map_dump(m, os.path.join(OUT, "n44e003.png").encode()) == 0
    lib.turtle_map_destroy(C.byref(m))
    files += ["n44e003.tif", "n44e003.png"]
    # 4. GRD text grid: "y0 y1 x0 x1 dy dx" then the values, 8 per line. (Lines must stay
    # below the 127 characters the reference reads at a time, grd.c:134: a longer line is
    # cut inside a number, yields extra tokens and overruns the reference's map.)
    g = terrain(19, 9, -107., 85.4, 4)
    with open(os.path.join(OUT, "geoid.grd"), "w") as f:
        f.write("  -10.000000   10.000000   20.000000   65.000000    2.500000    2.500000\n")
        for row in g:
            for k in range(0, len(row), 8):
                f.write(" ".join("%9.3f" % v for v in row[k:k + 8]) + "\n")
    files.append("geoid.grd")
    # 5. ESRI ASCII grid with NODATA cells
    a = np.round(terrain(13, 7, 120., 1893., 5), 2)
    a[2, 3] = a[5, 11] = -9999.
    with open(os.path.join(OUT, "esri.asc"), "w") as f:
        f.write("ncols 13\nnrows 7\nxllcorner 700000.0\nyllcorner 4300000.0\ncellsize 25.0\n"
                "NODATA_value -9999\n")
        for row in a:
            f.write(" ".join("%.2f" % v for v in row) + "\n")
    files.append("esri.asc")

    out = {"files": np.array(files)}
    for name in files:
        meta, tag, enc, z = describe(lib, os.path.join(OUT, name))
        key = name.replace(".", "_")
        out[key + "_meta"], out[key + "_z"] = meta, z
        out[key + "_projection"], out[key + "_encoding"] = np.array(tag), np.array(enc)
        print("%-18s %3d x %3d  projection=%-10r encoding=%r z in [%g, %g]" % (
            name, int(meta[0]), int(meta[1]), tag, enc, z.min(), z.max()))
    np.savez_compressed(os.path.join(HERE, "io_vectors.npz"), **out)


if __name__ == "__main__":
    main()
