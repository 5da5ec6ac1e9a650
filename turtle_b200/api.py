"""Thin Python mirror of the C interface (turtle.h + turtle_b200.h), for tests and
bench.py. Names follow the C objects: Map, Stack, Stepper, Plan, States.

numpy arrays are passed as HOST pointers (the ``*_batch`` calls), torch CUDA
tensors as DEVICE pointers (the ``*_batch_device`` calls). Nothing is computed in
Python.
"""
import ctypes as C

import numpy as np

from ._lib import (ERROR_HANDLER, Fan, Fans, MapInfo, PlanCounters, TraceFields, Residency, ResidencyReport, TraceRule,
                   lib)

TRACE_RESULT = np.dtype([
    ("position", "<f8", (3,)), ("altitude", "<f8"), ("length", "<f8", (4,)),
    ("total", "<f8"), ("n_steps", "<i4"), ("status", "<i4"), ("index", "<i4", (2,)),
    ("medium_hash", "<u4"), ("n_changes", "<i4")])
assert TRACE_RESULT.itemsize == 96

TRACE_CROSSING = np.dtype([("length", "<f8"), ("from", "<i4"), ("to", "<i4")])
assert TRACE_CROSSING.itemsize == 16

TRACE_ALTITUDE, TRACE_DOMAIN, TRACE_LENGTH, TRACE_STEPS, TRACE_INVALID = range(5)

HORIZON_RESULT = np.dtype([
    ("elevation", "<f8", (2,)), ("direction", "<f8", (2, 3)), ("length", "<f8"),
    ("medium", "<i4", (2,)), ("status", "<i4"), ("clear_status", "<i4"), ("n_probes", "<i4"),
    ("n_iterations", "<i4")])
assert HORIZON_RESULT.itemsize == 96

HORIZON_FOUND, HORIZON_BELOW, HORIZON_ABOVE, HORIZON_INVALID = range(4)


class TurtleError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(message)
        self.code = code


_last_error = []


@ERROR_HANDLER
def _on_error(code, function, message):
    _last_error.append((code, message.decode(errors="replace") if message else ""))


def install_handler():
    """(Re)install the Python error handler: it is a process-wide setting of the library
    (turtle_error_handler_set) that other users of the same .so may have replaced."""
    lib.turtle_error_handler_set(C.cast(_on_error, C.c_void_p))


install_handler()


def _check(rc):
    if rc != 0:
        if not _last_error:
            install_handler()  # someone replaced the handler: be loud next time at least
        code, message = _last_error.pop() if _last_error else (rc, "turtle error %d" % rc)
        del _last_error[:]
        raise TurtleError(code, message)
    del _last_error[:]


def _f8(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a):
    """Host pointer of a numpy array, device pointer of a torch tensor, or NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if isinstance(a, int):  # a raw device pointer (e.g. a peer mapping, dist.PeerRecords)
        return C.c_void_p(a)
    return C.c_void_p(a.data_ptr())


def device_count():
    return lib.turtle_b200_device_count()


def kernel_info(role):
    """(registers per thread, static shared bytes) of a built kernel, or None."""
    r, sh = C.c_int(), C.c_int()
    if lib.turtle_b200_kernel_info(role.encode(), C.byref(r), C.byref(sh)) != 0:
        return None
    return r.value, sh.value


def dfma_peak(repeats=3):
    return lib.turtle_b200_dfma_peak(repeats)


# ---- frames -------------------------------------------------------------------

def ecef_from_geodetic(latitude, longitude, elevation):
    out = (C.c_double * 3)()
    lib.turtle_ecef_from_geodetic(latitude, longitude, elevation, out)
    return np.array(out)


def ecef_to_geodetic(ecef):
    e = (C.c_double * 3)(*ecef)
    la, lo, al = C.c_double(), C.c_double(), C.c_double()
    lib.turtle_ecef_to_geodetic(e, C.byref(la), C.byref(lo), C.byref(al))
    return la.value, lo.value, al.value


def ecef_from_horizontal(latitude, longitude, azimuth, elevation):
    out = (C.c_double * 3)()
    lib.turtle_ecef_from_horizontal(latitude, longitude, azimuth, elevation, out)
    return np.array(out)


def ecef_to_geodetic_batch(ecef):
    ecef = _f8(ecef, (-1, 3))
    n = len(ecef)
    la, lo, al = np.empty(n), np.empty(n), np.empty(n)
    _check(lib.turtle_ecef_to_geodetic_batch(n, _ptr(ecef), _ptr(la), _ptr(lo), _ptr(al)))
    return la, lo, al


def ecef_from_geodetic_batch(latitude, longitude, elevation):
    la, lo, el = _f8(latitude), _f8(longitude), _f8(elevation)
    out = np.empty((len(la), 3))
    _check(lib.turtle_ecef_from_geodetic_batch(len(la), _ptr(la), _ptr(lo), _ptr(el), _ptr(out)))
    return out


def ecef_from_horizontal_batch(latitude, longitude, azimuth, elevation):
    la, lo, az, el = _f8(latitude), _f8(longitude), _f8(azimuth), _f8(elevation)
    out = np.empty((len(la), 3))
    _check(lib.turtle_ecef_from_horizontal_batch(
        len(la), _ptr(la), _ptr(lo), _ptr(az), _ptr(el), _ptr(out)))
    return out


# ---- objects --------------------------------------------------------------------

class Projection:
    def __init__(self, name):
        self._p = C.c_void_p()
        _check(lib.turtle_projection_create(C.byref(self._p), name.encode()))

    def project(self, latitude, longitude):
        x, y = C.c_double(), C.c_double()
        _check(lib.turtle_projection_project(self._p, latitude, longitude, C.byref(x), C.byref(y)))
        return x.value, y.value

    def unproject(self, x, y):
        la, lo = C.c_double(), C.c_double()
        _check(lib.turtle_projection_unproject(self._p, x, y, C.byref(la), C.byref(lo)))
        return la.value, lo.value

    def project_batch(self, latitude, longitude):
        la, lo = _f8(latitude), _f8(longitude)
        x, y = np.empty(len(la)), np.empty(len(la))
        _check(lib.turtle_projection_project_batch(self._p, len(la), _ptr(la), _ptr(lo),
                                                   _ptr(x), _ptr(y)))
        return x, y

    def unproject_batch(self, x, y):
        x, y = _f8(x), _f8(y)
        la, lo = np.empty(len(x)), np.empty(len(x))
        _check(lib.turtle_projection_unproject_batch(self._p, len(x), _ptr(x), _ptr(y),
                                                     _ptr(la), _ptr(lo)))
        return la, lo

    def __del__(self):
        if getattr(self, "_p", None):
            lib.turtle_projection_destroy(C.byref(self._p))


class Map:
    """turtle_map: 16-bit node grid. ``values[iy, ix]`` fills every node."""

    def __init__(self, nx=None, ny=None, x=None, y=None, z=None, projection=None,
                 values=None, path=None):
        self._p = C.c_void_p()
        if path is not None:
            _check(lib.turtle_map_load(C.byref(self._p), path.encode()))
            return
        info = MapInfo(nx, ny, (C.c_double * 2)(*x), (C.c_double * 2)(*y),
                       (C.c_double * 2)(*z), None)
        _check(lib.turtle_map_create(C.byref(self._p), C.byref(info),
                                     projection.encode() if projection else None))
        if values is not None:
            self.fill(values)

    @property
    def handle(self):
        return self._p

    def fill(self, values):
        v = _f8(values)
        _check(lib.turtle_map_fill_batch(self._p, _ptr(v)))

    def meta(self):
        info = MapInfo()
        name = C.c_char_p()
        lib.turtle_map_meta(self._p, C.byref(info), C.byref(name))
        return info, (name.value.decode() if name.value else None)

    def resample(self, plan, layer=0):
        """turtle_map_resample: fill every node from layer `layer` of the plan's geometry
        (example-projection.c:88-104 as one kernel). Returns the number of nodes the
        geometry has no data for (left untouched)."""
        outside = C.c_size_t()
        _check(lib.turtle_map_resample(self._p, plan.handle, layer, C.byref(outside)))
        return outside.value

    def dump(self, path):
        """turtle_map_dump: `.png` (any map) or `.tif` (integer metre scale, geodetic)."""
        _check(lib.turtle_map_dump(self._p, path.encode()))

    def node(self, ix, iy):
        x, y, z = C.c_double(), C.c_double(), C.c_double()
        _check(lib.turtle_map_node(self._p, ix, iy, C.byref(x), C.byref(y), C.byref(z)))
        return x.value, y.value, z.value

    def elevation(self, x, y):
        z, inside = C.c_double(), C.c_int()
        _check(lib.turtle_map_elevation(self._p, x, y, C.byref(z), C.byref(inside)))
        return z.value, inside.value

    def elevation_batch(self, x, y):
        x, y = _f8(x), _f8(y)
        z = np.zeros(len(x))
        inside = np.zeros(len(x), dtype=np.int32)
        _check(lib.turtle_map_elevation_batch(self._p, len(x), _ptr(x), _ptr(y), _ptr(z),
                                              _ptr(inside)))
        return z, inside

    def gradient_batch(self, x, y):
        x, y = _f8(x), _f8(y)
        gx, gy = np.zeros(len(x)), np.zeros(len(x))
        inside = np.zeros(len(x), dtype=np.int32)
        _check(lib.turtle_map_gradient_batch(self._p, len(x), _ptr(x), _ptr(y), _ptr(gx),
                                             _ptr(gy), _ptr(inside)))
        return gx, gy, inside

    def elevation_ecef_batch(self, ecef):
        ecef = _f8(ecef, (-1, 3))
        n = len(ecef)
        la, lo, al, z = np.empty(n), np.empty(n), np.empty(n), np.zeros(n)
        inside = np.zeros(n, dtype=np.int32)
        _check(lib.turtle_map_elevation_ecef_batch(
            self._p, n, _ptr(ecef), _ptr(la), _ptr(lo), _ptr(al), _ptr(z), _ptr(inside)))
        return la, lo, al, z, inside

    def __del__(self):
        if getattr(self, "_p", None):
            lib.turtle_map_destroy(C.byref(self._p))


class Stack:
    """turtle_stack over a directory of tiles (.hgt .png .tif .grd .asc)."""

    def __init__(self, path, size=0):
        self._p = C.c_void_p()
        _check(lib.turtle_stack_create(C.byref(self._p), path.encode(), size, None, None))

    @property
    def handle(self):
        return self._p

    def load(self):
        _check(lib.turtle_stack_load(self._p))

    def elevation(self, latitude, longitude):
        z, inside = C.c_double(), C.c_int()
        _check(lib.turtle_stack_elevation(self._p, latitude, longitude, C.byref(z),
                                          C.byref(inside)))
        return z.value, inside.value

    def __del__(self):
        if getattr(self, "_p", None):
            lib.turtle_stack_destroy(C.byref(self._p))


class Stepper:
    """turtle_stepper: geometry description + tunables (+ scalar set-up calls)."""

    def __init__(self, range=None, slope=None, resolution=None, geoid=None):
        self._p = C.c_void_p()
        self._keep = []
        _check(lib.turtle_stepper_create(C.byref(self._p)))
        if geoid is not None:
            self._keep.append(geoid)
            lib.turtle_stepper_geoid_set(self._p, geoid.handle)
        if slope is not None:
            lib.turtle_stepper_slope_set(self._p, slope)
        if resolution is not None:
            lib.turtle_stepper_resolution_set(self._p, resolution)
        if range is not None:
            lib.turtle_stepper_range_set(self._p, range)

    @property
    def handle(self):
        return self._p

    def add_layer(self):
        _check(lib.turtle_stepper_add_layer(self._p))

    def add_flat(self, offset=0.):
        _check(lib.turtle_stepper_add_flat(self._p, offset))

    def add_map(self, map_, offset=0.):
        self._keep.append(map_)
        _check(lib.turtle_stepper_add_map(self._p, map_.handle, offset))

    def add_stack(self, stack, offset=0.):
        self._keep.append(stack)
        _check(lib.turtle_stepper_add_stack(self._p, stack.handle, offset))

    def reset(self):
        lib.turtle_stepper_reset(self._p)

    def position(self, latitude, longitude, height, layer):
        pos = (C.c_double * 3)()
        index = C.c_int()
        _check(lib.turtle_stepper_position(self._p, latitude, longitude, height, layer, pos,
                                           C.byref(index)))
        return np.array(pos), index.value

    def step(self, position, direction=None):
        """Scalar turtle_stepper_step (host, set-up path). Returns a dict."""
        pos = (C.c_double * 3)(*position)
        d = (C.c_double * 3)(*direction) if direction is not None else None
        la, lo, al, st = C.c_double(), C.c_double(), C.c_double(), C.c_double()
        el = (C.c_double * 2)()
        idx = (C.c_int * 2)()
        _check(lib.turtle_stepper_step(self._p, pos, d, C.byref(la), C.byref(lo), C.byref(al),
                                       el, C.byref(st), idx))
        return dict(position=np.array(pos), latitude=la.value, longitude=lo.value,
                    altitude=al.value, elevation=(el[0], el[1]), step=st.value,
                    index=(idx[0], idx[1]))

    def freeze(self, device=0, region=None, memory_limit=0):
        """Residency plan on `device`. ``region`` = (lat_min, lat_max, lon_min, lon_max)
        (None / NaN = open) or a Residency from ``residency_from_rays``: only the stack
        tiles that meet it are uploaded (turtle_stepper_freeze_region)."""
        return Plan(self, device, region, memory_limit)

    def __del__(self):
        if getattr(self, "_p", None):
            lib.turtle_stepper_destroy(C.byref(self._p))


def residency_from_rays(position, direction, rule, step=1000., margin=0.):
    """Bounding box (a Residency) of the ground tracks of the rays under `rule`."""
    position, direction = _f8(position, (-1, 3)), _f8(direction, (-1, 3))
    r = Residency()
    _check(lib.turtle_residency_from_rays(len(position), _ptr(position), _ptr(direction),
                                          C.byref(rule), step, margin, C.byref(r)))
    return r


def trace_rule(altitude_max, altitude_min=-1.7976931348623157e308,
               length_max=1.7976931348623157e308, max_steps=100000):
    return TraceRule(altitude_min, altitude_max, length_max, max_steps, 0)


class Plan:
    """turtle_plan: a stepper geometry resident on one GPU."""

    def __init__(self, stepper, device=0, region=None, memory_limit=0):
        self._p = C.c_void_p()
        self.stepper = stepper
        if region is None and not memory_limit:
            _check(lib.turtle_stepper_freeze(stepper.handle, device, C.byref(self._p)))
            return
        if not isinstance(region, Residency):
            nan = float("nan")
            box = [nan if v is None else float(v) for v in (region or (None,) * 4)]
            region = Residency(box[0], box[1], box[2], box[3], 0)
        region.memory_limit = int(memory_limit)
        _check(lib.turtle_stepper_freeze_region(stepper.handle, device, C.byref(region),
                                                C.byref(self._p)))

    def residency(self):
        r = ResidencyReport()
        lib.turtle_plan_residency_get(self._p, C.byref(r))
        return dict(tiles_resident=r.tiles_resident, tiles_skipped=r.tiles_skipped,
                    tiles_ingested=r.tiles_ingested, bytes=r.bytes, read_ms=r.read_ms,
                    upload_ms=r.upload_ms)

    @property
    def handle(self):
        return self._p

    @property
    def device(self):
        return lib.turtle_plan_device(self._p)

    @property
    def bytes(self):
        return lib.turtle_plan_bytes(self._p)

    def launch_set(self, ctas_per_sm=0, threads=0):
        lib.turtle_plan_launch_set(self._p, ctas_per_sm, threads)

    def schedule_set(self, mode):
        lib.turtle_plan_schedule_set(self._p, mode)

    def pipeline_set(self, mode):
        lib.turtle_plan_pipeline_set(self._p, int(mode))

    def specialise_set(self, enable):
        lib.turtle_plan_specialise_set(self._p, int(enable))

    def counters(self, sync=False):
        if sync:
            lib.turtle_plan_counters_sync(self._p)
        c = PlanCounters()
        lib.turtle_plan_counters_get(self._p, C.byref(c))
        return dict(rays=c.rays, steps=c.steps, samples=c.samples, launches=c.launches,
                    kernel_ms=c.kernel_ms, rebuilds=c.rebuilds, window_hits=c.window_hits)

    def gather_set(self, mode, latitude=0., longitude=0.):
        """turtle_plan_gather_set: 0 global 16-bit loads, 1 cell-packed copy, 2 window."""
        _check(lib.turtle_plan_gather_set(self._p, mode, latitude, longitude))

    def trace(self, position, direction, rule, results=None):
        """Host arrays in, host records out (turtle_stepper_trace_batch)."""
        position, direction = _f8(position, (-1, 3)), _f8(direction, (-1, 3))
        n = len(position)
        if results is None:
            results = np.zeros(n, dtype=TRACE_RESULT)
        _check(lib.turtle_stepper_trace_batch(self._p, n, _ptr(position), _ptr(direction),
                                              C.byref(rule), _ptr(results)))
        return results

    def trace_crossings(self, position, direction, rule, max_crossings):
        """turtle_stepper_trace_crossings: the trace records and, per ray, its first
        `max_crossings` medium changes (structured array [n, max_crossings])."""
        position, direction = _f8(position, (-1, 3)), _f8(direction, (-1, 3))
        n = len(position)
        results = np.zeros(n, dtype=TRACE_RESULT)
        crossings = np.zeros((n, max_crossings), dtype=TRACE_CROSSING)
        _check(lib.turtle_stepper_trace_crossings(
            self._p, n, _ptr(position), _ptr(direction), C.byref(rule), _ptr(results),
            _ptr(crossings), max_crossings))
        return results, crossings

    # ---- compact input / output (turtle_stepper_trace_fan / _fields) ---------------------
    FIELD_DTYPES = dict(length0="<f8", length1="<f8", length2="<f8", length3="<f8", total="<f8",
                        altitude="<f8", position="<f8", n_steps="<i4", status="<i4",
                        index="<i4", medium_hash="<u4", n_changes="<i4")

    @classmethod
    def host_fields(cls, n, names):
        """Host arrays for the named columns of a trace result -> dict name -> array."""
        shape = dict(position=(n, 3), index=(n, 2))
        return {k: np.zeros(shape.get(k, (n,)), dtype=cls.FIELD_DTYPES[k]) for k in names}

    @staticmethod
    def _fields_struct(arrays):
        """dict name -> array (numpy) or tensor (torch, device) -> struct turtle_trace_fields"""
        f = TraceFields()
        for k, a in arrays.items():
            p = _ptr(a).value
            if k.startswith("length"):
                f.length[int(k[-1])] = p
            else:
                setattr(f, k, p)
        return f

    @staticmethod
    def make_fan(latitude, longitude, position, azimuth, elevation, bundle=1):
        """struct turtle_fan over host arrays of angles (kept alive by the returned pair)."""
        az, el = _f8(azimuth), _f8(elevation)
        fan = Fan(latitude, longitude, (C.c_double * 3)(*[float(x) for x in position]),
                  len(az), len(el), _ptr(az), _ptr(el), bundle)
        return fan, (az, el)

    def trace_fan(self, fan, rule, results=None, fields=None):
        """turtle_stepper_trace_fan: host records and / or host field arrays out."""
        f = self._fields_struct(fields) if fields else None
        _check(lib.turtle_stepper_trace_fan(
            self._p, C.byref(fan[0]), C.byref(rule), _ptr(results) if results is not None else None,
            C.byref(f) if f is not None else None))
        return results, fields

    def trace_fan_device(self, fan, rule, results=None, fields=None, stream=None):
        f = self._fields_struct(fields) if fields else None
        _check(lib.turtle_stepper_trace_fan_device(
            self._p, C.byref(fan[0]), C.byref(rule), _ptr(results) if results is not None else None,
            C.byref(f) if f is not None else None, C.c_void_p(stream) if stream else None))

    @staticmethod
    def make_fans(latitude, longitude, position, azimuth, elevation, bundle=1):
        """struct turtle_fans: one angle grid from every station (latitude[s], longitude[s],
        position[s]), over host arrays (kept alive by the returned pair). Ray
        s * len(azimuth) * len(elevation) + q is ray q of station s's make_fan."""
        la, lo = _f8(latitude).reshape(-1), _f8(longitude).reshape(-1)
        pos = _f8(position, (-1, 3))
        az, el = _f8(azimuth).reshape(-1), _f8(elevation).reshape(-1)
        if not len(la) == len(lo) == len(pos):
            raise ValueError("one latitude, longitude and position per station")
        fans = Fans(len(la), _ptr(la), _ptr(lo), _ptr(pos), len(az), len(el), _ptr(az), _ptr(el),
                    bundle)
        return fans, (la, lo, pos, az, el)

    def trace_fans(self, fans, rule, results=None, fields=None):
        """turtle_stepper_trace_fans: host records and / or host field arrays out."""
        f = self._fields_struct(fields) if fields else None
        _check(lib.turtle_stepper_trace_fans(
            self._p, C.byref(fans[0]), C.byref(rule), _ptr(results) if results is not None else None,
            C.byref(f) if f is not None else None))
        return results, fields

    def trace_fans_device(self, fans, rule, results=None, fields=None, stream=None):
        """turtle_stepper_trace_fans_device: device records / fields, one launch, asynchronous."""
        f = self._fields_struct(fields) if fields else None
        _check(lib.turtle_stepper_trace_fans_device(
            self._p, C.byref(fans[0]), C.byref(rule), _ptr(results) if results is not None else None,
            C.byref(f) if f is not None else None, C.c_void_p(stream) if stream else None))

    def trace_fields(self, position, direction, rule, fields):
        """turtle_stepper_trace_fields: host rays in, host field arrays out."""
        position, direction = _f8(position, (-1, 3)), _f8(direction, (-1, 3))
        f = self._fields_struct(fields)
        _check(lib.turtle_stepper_trace_fields(self._p, len(position), _ptr(position),
                                               _ptr(direction), C.byref(rule), C.byref(f)))
        return fields

    def trace_fields_device(self, n, position, direction, rule, fields, stream=None):
        f = self._fields_struct(fields)
        _check(lib.turtle_stepper_trace_fields_device(
            self._p, n, _ptr(position), _ptr(direction), C.byref(rule), C.byref(f),
            C.c_void_p(stream) if stream else None))

    def trace_device(self, n, position, direction, rule, results, stream=None):
        """Device tensors in / out (turtle_stepper_trace_batch_device), asynchronous."""
        _check(lib.turtle_stepper_trace_batch_device(
            self._p, n, _ptr(position), _ptr(direction), C.byref(rule), _ptr(results),
            C.c_void_p(stream) if stream else None))

    # ---- the horizon of a station (turtle_stepper_horizon) -------------------------------
    def horizon(self, latitude, longitude, position, azimuth, rule, elevation=(-90., 90.),
                tolerance=1e-6):
        """Horizon bracket of the station for each azimuth (degrees): a HORIZON_RESULT array."""
        az = _f8(azimuth).reshape(-1)
        pos = (C.c_double * 3)(*[float(x) for x in position])
        results = np.zeros(len(az), dtype=HORIZON_RESULT)
        _check(lib.turtle_stepper_horizon(self._p, latitude, longitude, pos, len(az), _ptr(az),
                                          elevation[0], elevation[1], tolerance, C.byref(rule),
                                          _ptr(results)))
        return results

    def horizon_device(self, latitude, longitude, position, azimuth, rule, results,
                       elevation=(-90., 90.), tolerance=1e-6, stream=None):
        """turtle_stepper_horizon_device: `azimuth` on the host, `results` a device tensor of
        len(azimuth) * 96 bytes; asynchronous on `stream`."""
        az = _f8(azimuth).reshape(-1)
        pos = (C.c_double * 3)(*[float(x) for x in position])
        _check(lib.turtle_stepper_horizon_device(
            self._p, latitude, longitude, pos, len(az), _ptr(az), elevation[0], elevation[1],
            tolerance, C.byref(rule), _ptr(results), C.c_void_p(stream) if stream else None))

    @staticmethod
    def _stations(latitude, longitude, position):
        la, lo = _f8(latitude).reshape(-1), _f8(longitude).reshape(-1)
        pos = _f8(position, (-1, 3))
        if not len(la) == len(lo) == len(pos):
            raise ValueError("one latitude, longitude and position per station")
        return la, lo, pos

    def horizons(self, latitude, longitude, position, azimuth, rule, elevation=(-90., 90.),
                 tolerance=1e-6):
        """turtle_stepper_horizons: the horizon of every station (latitude[s], longitude[s],
        position[s]) for each azimuth -> HORIZON_RESULT array [n_station, n_azimuth]."""
        la, lo, pos = self._stations(latitude, longitude, position)
        az = _f8(azimuth).reshape(-1)
        results = np.zeros((len(la), len(az)), dtype=HORIZON_RESULT)
        _check(lib.turtle_stepper_horizons(self._p, len(la), _ptr(la), _ptr(lo), _ptr(pos),
                                           len(az), _ptr(az), elevation[0], elevation[1],
                                           tolerance, C.byref(rule), _ptr(results)))
        return results

    def horizons_device(self, latitude, longitude, position, azimuth, rule, results,
                        elevation=(-90., 90.), tolerance=1e-6, stream=None):
        """turtle_stepper_horizons_device: stations and azimuths on the host, `results` a
        device tensor of n_station * len(azimuth) * 96 bytes; asynchronous on `stream`."""
        la, lo, pos = self._stations(latitude, longitude, position)
        az = _f8(azimuth).reshape(-1)
        _check(lib.turtle_stepper_horizons_device(
            self._p, len(la), _ptr(la), _ptr(lo), _ptr(pos), len(az), _ptr(az), elevation[0],
            elevation[1], tolerance, C.byref(rule), _ptr(results),
            C.c_void_p(stream) if stream else None))

    def step(self, position, direction=None, states=None):
        """One turtle_stepper_step per particle, host arrays. Returns a dict of arrays;
        ``position`` is advanced in place when a direction is given."""
        position = _f8(position, (-1, 3))
        n = len(position)
        d = _f8(direction, (-1, 3)) if direction is not None else None
        out = dict(position=position, latitude=np.empty(n), longitude=np.empty(n),
                   altitude=np.empty(n), elevation=np.empty((n, 2)), step=np.empty(n),
                   index=np.empty((n, 2), dtype=np.int32))
        _check(lib.turtle_stepper_step_batch(
            self._p, states.handle if states else None, n, _ptr(position), _ptr(d),
            _ptr(out["latitude"]), _ptr(out["longitude"]), _ptr(out["altitude"]),
            _ptr(out["elevation"]), _ptr(out["step"]), _ptr(out["index"])))
        return out

    def step_device(self, n, position, direction, states=None, latitude=None,
                    longitude=None, altitude=None, elevation=None, step=None, index=None,
                    stream=None):
        _check(lib.turtle_stepper_step_batch_device(
            self._p, states.handle if states else None, n, _ptr(position), _ptr(direction),
            _ptr(latitude), _ptr(longitude), _ptr(altitude), _ptr(elevation), _ptr(step),
            _ptr(index), C.c_void_p(stream) if stream else None))

    def walk_device(self, n, n_steps, position, direction, states=None, latitude=None,
                    longitude=None, altitude=None, elevation=None, step=None, index=None,
                    stream=None):
        """turtle_stepper_walk_batch_device: n_steps steps per particle in one launch;
        direction is [n_steps, n, 3], the per-step outputs [n_steps, n(, 2)]."""
        _check(lib.turtle_stepper_walk_batch_device(
            self._p, states.handle if states else None, n, n_steps, _ptr(position),
            _ptr(direction), _ptr(latitude), _ptr(longitude), _ptr(altitude), _ptr(elevation),
            _ptr(step), _ptr(index), C.c_void_p(stream) if stream else None))

    def walk(self, position, direction, states=None):
        """turtle_stepper_walk_batch on host arrays: direction [n_steps, n, 3]. Returns a
        dict of per-step arrays; ``position`` is advanced in place."""
        position = _f8(position, (-1, 3))
        d = _f8(direction)
        k, n = d.shape[0], d.shape[1]
        out = dict(position=position, altitude=np.empty((k, n)), step=np.empty((k, n)),
                   index=np.empty((k, n, 2), dtype=np.int32), latitude=np.empty((k, n)),
                   longitude=np.empty((k, n)), elevation=np.empty((k, n, 2)))
        _check(lib.turtle_stepper_walk_batch(
            self._p, states.handle if states else None, n, k, _ptr(position), _ptr(d),
            _ptr(out["latitude"]), _ptr(out["longitude"]), _ptr(out["altitude"]),
            _ptr(out["elevation"]), _ptr(out["step"]), _ptr(out["index"])))
        return out

    def position(self, latitude, longitude, height, layer):
        la, lo, h = _f8(latitude), _f8(longitude), _f8(height)
        pos = np.zeros((len(la), 3))
        idx = np.empty(len(la), dtype=np.int32)
        _check(lib.turtle_stepper_position_batch(self._p, len(la), _ptr(la), _ptr(lo), _ptr(h),
                                                 layer, _ptr(pos), _ptr(idx)))
        return pos, idx

    def stack_elevation(self, stack, latitude, longitude):
        """turtle_stack_elevation_batch on stack `stack` of the plan -> (z, inside)."""
        la, lo = _f8(latitude), _f8(longitude)
        z, inside = np.zeros(len(la)), np.zeros(len(la), dtype=np.int32)
        _check(lib.turtle_stack_elevation_batch(self._p, stack, len(la), _ptr(la), _ptr(lo),
                                                _ptr(z), _ptr(inside)))
        return z, inside

    def stack_gradient(self, stack, latitude, longitude):
        """turtle_stack_gradient_batch -> (glat, glon, inside)."""
        la, lo = _f8(latitude), _f8(longitude)
        glat, glon = np.zeros(len(la)), np.zeros(len(la))
        inside = np.zeros(len(la), dtype=np.int32)
        _check(lib.turtle_stack_gradient_batch(self._p, stack, len(la), _ptr(la), _ptr(lo),
                                               _ptr(glat), _ptr(glon), _ptr(inside)))
        return glat, glon, inside

    def states(self, n):
        return States(self, n)

    def __del__(self):
        if getattr(self, "_p", None):
            lib.turtle_plan_destroy(C.byref(self._p))


class States:
    """turtle_states: per-particle stepper memory on the device."""

    def __init__(self, plan, n):
        self._p = C.c_void_p()
        self.plan = plan
        _check(lib.turtle_states_create(plan.handle, n, C.byref(self._p)))

    @property
    def handle(self):
        return self._p

    def reset(self):
        _check(lib.turtle_states_reset(self._p))

    @property
    def bytes_per_particle(self):
        return lib.turtle_states_bytes_per_particle(self._p)

    def __del__(self):
        if getattr(self, "_p", None):
            lib.turtle_states_destroy(C.byref(self._p))
