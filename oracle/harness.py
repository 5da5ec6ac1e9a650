"""ctypes wrapper of oracle/libtrace_driver.so -- TEST INFRASTRUCTURE.

``Driver(lib)`` drives any library exporting the turtle.h interface through the
pthread ray loop of trace_driver.c. Three libraries are of interest:

  REF     oracle/_ref/libturtle_ref.so  the unmodified reference (built by
          oracle/Makefile from REF_SOURCES below)
  REF_FMA oracle/_ref/libturtle_ref_fma.so  the same sources built with FMA contraction:
          the rounding-noise floor of the path (oracle/parity.py), never the checker
  PORT    oracle/liboracle.so           the plain-C restatement (turtle_oracle.c)
  PRODUCT turtle_b200/libturtle_b200.so the product's own scalar (host) calls

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs import this module.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# the unmodified reference's sources, which oracle/Makefile builds _ref/ from (same default)
REF_SOURCES = os.environ.get("TURTLE_REF") or os.path.join(os.path.dirname(os.path.dirname(HERE)),
                                                           "reference")
REF = os.path.join(HERE, "_ref", "libturtle_ref.so")
# the same sources with FMA contraction: the rounding-noise floor, not an oracle
REF_FMA = os.path.join(HERE, "_ref", "libturtle_ref_fma.so")
PORT = os.path.join(HERE, "liboracle.so")
PRODUCT = os.path.join(os.path.dirname(HERE), "turtle_b200", "libturtle_b200.so")
DRIVER = os.path.join(HERE, "libtrace_driver.so")

ADD_LAYER, ADD_FLAT, ADD_MAP, ADD_STACK = range(4)

RESULT = np.dtype([
    ("position", "<f8", (3,)), ("altitude", "<f8"), ("length", "<f8", (4,)),
    ("total", "<f8"), ("n_steps", "<i4"), ("status", "<i4"), ("index", "<i4", (2,)),
    ("medium_hash", "<u4"), ("n_changes", "<i4")])
CROSSING = np.dtype([("length", "<f8"), ("from", "<i4"), ("to", "<i4")])


class Op(C.Structure):
    _fields_ = [("kind", C.c_int), ("ref", C.c_int), ("offset", C.c_double)]


class Rule(C.Structure):
    _fields_ = [("altitude_min", C.c_double), ("altitude_max", C.c_double),
                ("length_max", C.c_double), ("max_steps", C.c_int32),
                ("reserved", C.c_int32)]


def rule(altitude_max, altitude_min=-1.7976931348623157e308,
         length_max=1.7976931348623157e308, max_steps=100000):
    return Rule(altitude_min, altitude_max, length_max, max_steps, 0)


def available(which):
    return os.path.exists(which) and os.path.exists(DRIVER)


def best_oracle():
    """The reference itself when it was compiled, else the restatement."""
    return REF if os.path.exists(REF) else PORT


_P = C.c_void_p


def _load_driver():
    d = C.CDLL(DRIVER)
    d.td_open.restype = _P
    d.td_open.argtypes = [C.c_char_p]
    d.td_close.argtypes = [_P]
    d.td_last_error.restype = C.c_char_p
    d.td_last_error.argtypes = [_P]
    d.td_map_create.argtypes = [_P, C.c_int, C.c_int] + [C.c_double] * 6 + [C.c_char_p, _P]
    d.td_stack_create.argtypes = [_P, C.c_char_p, C.c_int]
    d.td_geometry.argtypes = [_P, C.POINTER(Op), C.c_int, C.c_int] + [C.c_double] * 3
    d.td_trace.restype = C.c_longlong
    d.td_trace.argtypes = [_P, C.c_size_t, _P, _P, C.POINTER(Rule), _P, C.c_int,
                           C.POINTER(C.c_double)]
    d.td_trace_crossings.restype = C.c_longlong
    d.td_trace_crossings.argtypes = [_P, C.c_size_t, _P, _P, C.POINTER(Rule), _P, _P, C.c_int,
                                     C.c_int, C.POINTER(C.c_double)]
    d.td_walk.argtypes = [_P, C.c_size_t, C.c_int, _P, _P, _P, _P, _P, C.c_int,
                          C.POINTER(C.c_double)]
    d.td_step.argtypes = [_P, C.c_size_t] + [_P] * 8
    d.td_position.argtypes = [_P, C.c_size_t, _P, _P, _P, C.c_int, _P, _P]
    d.td_ecef_to_geodetic.argtypes = [_P, C.c_size_t] + [_P] * 4
    d.td_ecef_from_geodetic.argtypes = [_P, C.c_size_t] + [_P] * 4
    d.td_ecef_from_horizontal.argtypes = [_P, C.c_size_t] + [_P] * 5
    d.td_ecef_to_horizontal.argtypes = [_P, C.c_size_t] + [_P] * 5
    d.td_project.argtypes = [_P, C.c_char_p, C.c_int, C.c_size_t] + [_P] * 4
    d.td_map_elevation.argtypes = [_P, C.c_int, C.c_size_t] + [_P] * 4
    d.td_map_node.argtypes = [_P, C.c_int, C.c_size_t] + [_P] * 5
    d.td_stack_elevation.argtypes = [_P, C.c_int, C.c_size_t] + [_P] * 4
    d.td_map_gradient.argtypes = [_P, C.c_int, C.c_size_t] + [_P] * 5
    d.td_stack_gradient.argtypes = [_P, C.c_int, C.c_size_t] + [_P] * 5
    d.td_map_pointer.restype = _P
    d.td_map_pointer.argtypes = [_P, C.c_int]
    d.td_stack_pointer.restype = _P
    d.td_stack_pointer.argtypes = [_P, C.c_int]
    return d


def _f8(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a.reshape(shape) if shape is not None else a


def _p(a):
    return a.ctypes.data_as(_P) if a is not None else None


class Driver:
    def __init__(self, library):
        self.d = _load_driver()
        self.library = library
        self.h = self.d.td_open(library.encode())
        self._unlocked_stacks = 0
        if not self.h:
            raise OSError("could not open %s" % library)
        if os.path.realpath(library) == os.path.realpath(PRODUCT):
            # the driver installs its own error handler; the product library keeps ONE
            # handler per process, so hand it back to the Python binding
            try:
                from turtle_b200 import api
                api.install_handler()
            except ImportError:
                pass

    def close(self):
        if self.h:
            self.d.td_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- objects -----------------------------------------------------------------
    def map_create(self, nx, ny, x, y, z, projection, values):
        v = _f8(values)
        assert v.size == nx * ny
        i = self.d.td_map_create(self.h, nx, ny, x[0], x[1], y[0], y[1], z[0], z[1],
                                 projection.encode() if projection else None, _p(v))
        if i < 0:
            raise RuntimeError("map_create failed: %s" % self.d.td_last_error(self.h).decode())
        return i

    def stack_create(self, path, locked=False):
        i = self.d.td_stack_create(self.h, path.encode(), int(locked))
        self._unlocked_stacks += 0 if locked else 1
        if i < 0:
            raise RuntimeError("stack_create failed: %s" % self.d.td_last_error(self.h).decode())
        return i

    def geometry(self, ops, geoid=-1, range=1., slope=0.4, resolution=1e-2):
        """ops: list of (kind, ref, offset) in turtle_stepper_add_* order."""
        arr = (Op * len(ops))(*[Op(k, r, o) for (k, r, o) in ops])
        if self.d.td_geometry(self.h, arr, len(ops), geoid, range, slope, resolution) != 0:
            raise RuntimeError("geometry failed")

    # ---- stepping ----------------------------------------------------------------
    def trace(self, position, direction, rule_, threads=1):
        position, direction = _f8(position, (-1, 3)), _f8(direction, (-1, 3))
        n = len(position)
        if threads > 1 and self._unlocked_stacks:
            # the reference's stack mutates its MRU list on every lookup (stack.c:325):
            # threads need a locked stack (=> one client per stepper)
            raise ValueError("multi-threaded tracing needs stack_create(..., locked=True)")
        out = np.zeros(n, dtype=RESULT)
        seconds = C.c_double()
        steps = self.d.td_trace(self.h, n, _p(position), _p(direction), C.byref(rule_), _p(out),
                                threads, C.byref(seconds))
        if steps < 0:
            raise RuntimeError("trace failed: %s" % self.d.td_last_error(self.h).decode())
        return out, steps, seconds.value

    def trace_crossings(self, position, direction, rule_, max_crossings, threads=1):
        """trace() + the first `max_crossings` medium changes of every ray."""
        position, direction = _f8(position, (-1, 3)), _f8(direction, (-1, 3))
        n = len(position)
        out = np.zeros(n, dtype=RESULT)
        cross = np.zeros((n, max_crossings), dtype=CROSSING)
        seconds = C.c_double()
        steps = self.d.td_trace_crossings(self.h, n, _p(position), _p(direction), C.byref(rule_),
                                          _p(out), _p(cross), max_crossings, threads,
                                          C.byref(seconds))
        if steps < 0:
            raise RuntimeError("trace failed: %s" % self.d.td_last_error(self.h).decode())
        return out, cross

    def walk(self, position, direction, threads=1):
        """direction[k, i, :]: n_steps x n particles. Returns per (k, i) step, altitude, index
        and the final positions."""
        position = _f8(position, (-1, 3)).copy()
        direction = _f8(direction)
        n_steps, n = direction.shape[0], direction.shape[1]
        if threads > 1 and self._unlocked_stacks:
            raise ValueError("multi-threaded walks need stack_create(..., locked=True)")
        step = np.empty((n_steps, n))
        altitude = np.empty((n_steps, n))
        index = np.empty((n_steps, n, 2), dtype=np.int32)
        seconds = C.c_double()
        if self.d.td_walk(self.h, n, n_steps, _p(position), _p(direction), _p(step),
                          _p(altitude), _p(index), threads, C.byref(seconds)) != 0:
            raise RuntimeError("walk failed")
        return dict(position=position, step=step, altitude=altitude, index=index,
                    seconds=seconds.value)

    def step(self, position, direction=None):
        position = _f8(position, (-1, 3)).copy()
        n = len(position)
        d = _f8(direction, (-1, 3)) if direction is not None else None
        out = dict(position=position, latitude=np.empty(n), longitude=np.empty(n),
                   altitude=np.empty(n), elevation=np.empty((n, 2)), step=np.empty(n),
                   index=np.empty((n, 2), dtype=np.int32))
        if self.d.td_step(self.h, n, _p(position), _p(d), _p(out["latitude"]),
                          _p(out["longitude"]), _p(out["altitude"]), _p(out["elevation"]),
                          _p(out["step"]), _p(out["index"])) != 0:
            raise RuntimeError("step failed")
        return out

    def position(self, latitude, longitude, height, layer):
        la, lo, h = _f8(latitude), _f8(longitude), _f8(height)
        pos = np.zeros((len(la), 3))
        idx = np.empty(len(la), dtype=np.int32)
        if self.d.td_position(self.h, len(la), _p(la), _p(lo), _p(h), layer, _p(pos), _p(idx)) != 0:
            raise RuntimeError("position failed")
        return pos, idx

    # ---- frames / projections / elevation -------------------------------------------
    def ecef_to_geodetic(self, ecef):
        ecef = _f8(ecef, (-1, 3))
        n = len(ecef)
        la, lo, al = np.empty(n), np.empty(n), np.empty(n)
        self.d.td_ecef_to_geodetic(self.h, n, _p(ecef), _p(la), _p(lo), _p(al))
        return la, lo, al

    def ecef_from_geodetic(self, latitude, longitude, elevation):
        la, lo, el = _f8(latitude), _f8(longitude), _f8(elevation)
        out = np.empty((len(la), 3))
        self.d.td_ecef_from_geodetic(self.h, len(la), _p(la), _p(lo), _p(el), _p(out))
        return out

    def ecef_from_horizontal(self, latitude, longitude, azimuth, elevation):
        la, lo, az, el = _f8(latitude), _f8(longitude), _f8(azimuth), _f8(elevation)
        out = np.empty((len(la), 3))
        self.d.td_ecef_from_horizontal(self.h, len(la), _p(la), _p(lo), _p(az), _p(el), _p(out))
        return out

    def ecef_to_horizontal(self, latitude, longitude, direction):
        la, lo, d = _f8(latitude), _f8(longitude), _f8(direction, (-1, 3))
        az, el = np.zeros(len(la)), np.zeros(len(la))
        self.d.td_ecef_to_horizontal(self.h, len(la), _p(la), _p(lo), _p(d), _p(az), _p(el))
        return az, el

    def project(self, name, latitude, longitude, inverse=False):
        a, b = _f8(latitude), _f8(longitude)
        c, d = np.empty(len(a)), np.empty(len(a))
        if self.d.td_project(self.h, name.encode(), int(inverse), len(a), _p(a), _p(b), _p(c),
                             _p(d)) != 0:
            raise RuntimeError("bad projection %s" % name)
        return c, d

    def map_elevation(self, map_, x, y):
        x, y = _f8(x), _f8(y)
        z = np.zeros(len(x))
        inside = np.zeros(len(x), dtype=np.int32)
        self.d.td_map_elevation(self.h, map_, len(x), _p(x), _p(y), _p(z), _p(inside))
        return z, inside

    def map_node(self, map_, ix, iy):
        ix = np.ascontiguousarray(ix, dtype=np.int32)
        iy = np.ascontiguousarray(iy, dtype=np.int32)
        x, y, z = np.empty(len(ix)), np.empty(len(ix)), np.empty(len(ix))
        self.d.td_map_node(self.h, map_, len(ix), _p(ix), _p(iy), _p(x), _p(y), _p(z))
        return x, y, z

    def stack_elevation(self, stack, latitude, longitude):
        la, lo = _f8(latitude), _f8(longitude)
        z = np.zeros(len(la))
        inside = np.zeros(len(la), dtype=np.int32)
        self.d.td_stack_elevation(self.h, stack, len(la), _p(la), _p(lo), _p(z), _p(inside))
        return z, inside

    def map_gradient(self, map_, x, y, fill=0.):
        x, y = _f8(x), _f8(y)
        gx, gy = np.full(len(x), fill), np.full(len(x), fill)
        inside = np.zeros(len(x), dtype=np.int32)
        self.d.td_map_gradient(self.h, map_, len(x), _p(x), _p(y), _p(gx), _p(gy), _p(inside))
        return gx, gy, inside

    def stack_gradient(self, stack, latitude, longitude, fill=0.):
        la, lo = _f8(latitude), _f8(longitude)
        glat, glon = np.full(len(la), fill), np.full(len(la), fill)
        inside = np.zeros(len(la), dtype=np.int32)
        self.d.td_stack_gradient(self.h, stack, len(la), _p(la), _p(lo), _p(glat), _p(glon),
                                 _p(inside))
        return glat, glon, inside

    def map_pointer(self, map_):
        return C.c_void_p(self.d.td_map_pointer(self.h, map_))

    def stack_pointer(self, stack):
        return C.c_void_p(self.d.td_stack_pointer(self.h, stack))
