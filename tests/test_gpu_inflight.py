"""GPU: asynchronous entry points with several calls in flight on one plan.

Device-pointer calls (`*_device`) are asynchronous and up to 8 of them may be in flight on
one plan, each on its own stream (include/turtle_b200.h). Each call holds a slot of the
plan's ring of device resources (the queue cursor of its kernel, its schedule buffers, its
fan / azimuth tables) until it completes. Every call here is first made alone and
synchronously: that path is held to the oracle by test_gpu_trace.py, test_gpu_geometries.py,
test_fan.py and test_horizon.py. The same call made while others are in flight must give
the same bytes: records, field arrays, crossings, horizon records, walk outputs, final
positions, and the particle states left behind (one more step from them).

The overlap does not depend on timing. A stream is held back by an event that a side stream
records after `torch.cuda._sleep`: what is queued behind it is still pending while the later
calls are issued. Each test asserts that the hold was still pending after those calls; a test
that could pass without an overlap would show nothing. Holds last a few hundred ms at most.
Only non-blocking streams are held, so calls on the legacy default stream (the host horizon
and the host crossings) are not serialised behind them.
"""
import ctypes
import os

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.common import Scene
from tests.test_gpu_trace import c3
from turtle_b200 import synth

pytestmark = pytest.mark.gpu

FIELDS = ["length0", "length1", "length2", "length3", "total", "altitude", "position",
          "n_steps", "status", "index", "medium_hash", "n_changes"]
FIELD_WIDTH = dict(position=3, index=2)
SLOTS = 8  # device-pointer calls that may be in flight on a plan


# ---- holding streams back ------------------------------------------------------------------

_CYCLES_PER_MS = []


def cycles_per_ms():
    """Clock cycles of torch.cuda._sleep per millisecond on this device (measured once)."""
    import torch
    if not _CYCLES_PER_MS:
        side = torch.cuda.Stream()
        rate = 0.
        for _ in range(2):  # the first one loads the kernel
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(side):
                e0.record()
                torch.cuda._sleep(20_000_000)
                e1.record()
            side.synchronize()
            rate = 20_000_000 / e0.elapsed_time(e1)
        _CYCLES_PER_MS.append(rate)
    return _CYCLES_PER_MS[0]


def non_blocking(stream):
    """The stream does not synchronise with the legacy default stream (CU_STREAM_NON_BLOCKING)."""
    cuda = ctypes.CDLL("libcuda.so.1")
    flags = ctypes.c_uint()
    assert cuda.cuStreamGetFlags(ctypes.c_void_p(stream.cuda_stream), ctypes.byref(flags)) == 0
    return bool(flags.value & 1)


class Hold:
    """An event recorded on a side stream after a sleep of `ms` milliseconds: the streams
    made to wait on it run nothing queued after that wait before the sleep is over."""

    def __init__(self, ms):
        import torch
        self.side = torch.cuda.Stream()
        self.event = torch.cuda.Event()
        with torch.cuda.stream(self.side):
            torch.cuda._sleep(int(ms * cycles_per_ms()))
        self.event.record(self.side)

    def stream(self):
        import torch
        s = torch.cuda.Stream()
        assert non_blocking(s)
        s.wait_event(self.event)
        return s

    def pending(self):
        return not self.event.query()


def streams(n):
    import torch
    out = [torch.cuda.Stream() for _ in range(n)]
    assert all(non_blocking(s) for s in out)
    return out


# ---- the calls -----------------------------------------------------------------------------

def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bytes(outputs):
    """dict name -> torch tensor (device) or numpy array -> dict name -> bytes"""
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v).tobytes() for k, v in outputs.items()}


class Call:
    """One entry point and its inputs. prepare() allocates fresh outputs (and particle
    states), issue() queues the call on a stream (a host-pointer call runs to its end),
    outputs() reads what it wrote, after() does what is checked once it is over."""
    host = False

    def __init__(self, plan, name):
        self.plan, self.name = plan, name

    def after(self):
        return {}


class Trace(Call):
    def __init__(self, plan, pos, dirs, rule, schedule=0, gather=(0,)):
        super().__init__(plan, "trace_device" + (" schedule %d" % schedule if schedule else "") +
                         (" gather %d" % gather[0] if gather[0] else ""))
        self.n, self.pos, self.dirs, self.rule = len(pos), _dev(pos), _dev(dirs), rule
        self.schedule, self.gather = schedule, gather

    def prepare(self):
        import torch
        self.out = dict(records=torch.full((self.n * 96,), 0xa5, dtype=torch.uint8, device="cuda"))

    def issue(self, stream):
        self.plan.schedule_set(self.schedule)
        self.plan.gather_set(*self.gather)
        try:
            self.plan.trace_device(self.n, self.pos, self.dirs, self.rule, self.out["records"],
                                   stream=stream.cuda_stream)
        finally:
            self.plan.schedule_set(0)
            self.plan.gather_set(0)

    def outputs(self):
        return _bytes(self.out)


class Crossings(Trace):
    """turtle_stepper_trace_crossings_device (no wrapper of its own: through the C ABI)."""

    def __init__(self, plan, pos, dirs, rule, max_crossings=3):
        super().__init__(plan, pos, dirs, rule)
        self.name, self.max_crossings = "trace_crossings_device", max_crossings

    def prepare(self):
        import torch
        super().prepare()
        self.out["crossings"] = torch.full((self.n * self.max_crossings * 16,), 0x5a,
                                           dtype=torch.uint8, device="cuda")

    def issue(self, stream):
        p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
        tb.api._check(tb._lib.lib.turtle_stepper_trace_crossings_device(
            self.plan.handle, self.n, p(self.pos), p(self.dirs), ctypes.byref(self.rule),
            p(self.out["records"]), p(self.out["crossings"]), self.max_crossings,
            ctypes.c_void_p(stream.cuda_stream)))


def _fields(n, names):
    import torch
    out = {}
    for k in names:
        dtype = torch.float64 if tb.Plan.FIELD_DTYPES[k] == "<f8" else torch.int32
        out[k] = torch.full((n * FIELD_WIDTH.get(k, 1),), -7, dtype=dtype, device="cuda")
    return out


class Fields(Trace):
    def __init__(self, plan, pos, dirs, rule, names):
        super().__init__(plan, pos, dirs, rule)
        self.name, self.names = "trace_fields_device", names

    def prepare(self):
        self.out = _fields(self.n, self.names)

    def issue(self, stream):
        self.plan.trace_fields_device(self.n, self.pos, self.dirs, self.rule, self.out,
                                      stream=stream.cuda_stream)


class Fan(Call):
    def __init__(self, plan, station, origin, az, el, rule, bundle=1, records=True,
                 names=FIELDS):
        super().__init__(plan, "trace_fan_device %dx%d" % (len(az), len(el)))
        self.fan = tb.Plan.make_fan(station[0], station[1], origin, az, el, bundle=bundle)
        self.n, self.rule, self.records, self.names = len(az) * len(el), rule, records, names

    def prepare(self):
        import torch
        self.out = _fields(self.n, self.names)
        if self.records:
            self.out["records"] = torch.full((self.n * 96,), 0xa5, dtype=torch.uint8,
                                             device="cuda")

    def issue(self, stream):
        fields = {k: v for k, v in self.out.items() if k != "records"}
        self.plan.trace_fan_device(self.fan, self.rule, results=self.out.get("records"),
                                   fields=fields or None, stream=stream.cuda_stream)

    def outputs(self):
        return _bytes(self.out)


class Horizon(Call):
    def __init__(self, plan, station, origin, az, rule, tolerance=1e-4):
        super().__init__(plan, "horizon_device %d" % len(az))
        self.station, self.origin, self.az = station, origin, np.asarray(az, dtype=float)
        self.rule, self.tolerance = rule, tolerance

    def prepare(self):
        import torch
        self.out = dict(records=torch.full((len(self.az) * 96,), 0xa5, dtype=torch.uint8,
                                           device="cuda"))

    def issue(self, stream):
        self.plan.horizon_device(self.station[0], self.station[1], self.origin, self.az,
                                 self.rule, self.out["records"], elevation=(-30., 60.),
                                 tolerance=self.tolerance, stream=stream.cuda_stream)

    def outputs(self):
        return _bytes(self.out)


class Walk(Call):
    """k steps per particle with device states: turtle_stepper_step_batch_device (k = 1) or
    turtle_stepper_walk_batch_device. after(): one more step from the states left behind."""

    def __init__(self, plan, ground, dirs, more):
        k = len(dirs)
        super().__init__(plan, "step_batch_device" if k == 1 else "walk_batch_device %d" % k)
        self.ground, self.dirs, self.more = ground, _dev(dirs), _dev(more)
        self.n, self.k = ground.shape[0], k

    def _outs(self, k):
        import torch
        f8 = lambda *s: torch.full(s, -7., dtype=torch.float64, device="cuda")  # noqa: E731
        return dict(latitude=f8(k, self.n), longitude=f8(k, self.n), altitude=f8(k, self.n),
                    elevation=f8(k, self.n, 2), step=f8(k, self.n),
                    index=torch.full((k, self.n, 2), -7, dtype=torch.int32, device="cuda"))

    def prepare(self):
        self.states = self.plan.states(self.n)
        self.position = _dev(self.ground)
        self.out = self._outs(self.k)

    def _run(self, dirs, out, stream):
        if self.k == 1:
            self.plan.step_device(self.n, self.position, dirs[0], self.states, stream=stream,
                                  **out)
        else:
            self.plan.walk_device(self.n, self.k, self.position, dirs, self.states,
                                  stream=stream, **out)

    def issue(self, stream):
        self._run(self.dirs, self.out, stream.cuda_stream)

    def outputs(self):
        return _bytes(dict(self.out, position=self.position))

    def after(self):
        import torch
        position = self.position.clone()
        out = self._outs(1)
        self.plan.step_device(self.n, self.position, self.more[0], self.states, **out)
        torch.cuda.synchronize()
        got = _bytes(dict(out, position=self.position))
        self.position = position
        return {"next step " + k: v for k, v in got.items()}


# host-pointer calls: they return when their results are in place

class HostFan(Fan):
    """turtle_stepper_trace_fan cut in 8 slices on two streams, on a grid of one 32-lane CTA
    per SM: the slices of both streams run side by side, each with rays left in its queue."""
    host = True

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.name = "trace_fan %dx%d (8 slices)" % (self.fan[0].n_azimuth, self.fan[0].n_elevation)
        band = self.fan[0].n_azimuth * self.fan[0].bundle
        assert self.fan[0].n_elevation % (8 * self.fan[0].bundle) == 0
        self.slice_rays = self.n // 8
        assert self.slice_rays % band == 0

    def prepare(self):
        self.out = {k: v.reshape(-1) for k, v in tb.Plan.host_fields(self.n, self.names).items()}
        for v in self.out.values():
            v.view(np.uint8)[:] = 0xa5
        if self.records:
            self.out["records"] = np.full(self.n * 96, 0xa5, dtype=np.uint8)

    def issue(self, stream):
        fields = {k: v for k, v in self.out.items() if k != "records"}
        records = self.out["records"].view(tb.TRACE_RESULT) if self.records else None
        os.environ["TURTLE_B200_FAN_SLICE_RAYS"] = str(self.slice_rays)
        self.plan.launch_set(1, 32)
        try:
            self.plan.trace_fan(self.fan, self.rule, results=records, fields=fields or None)
        finally:
            del os.environ["TURTLE_B200_FAN_SLICE_RAYS"]
            self.plan.launch_set(0, 0)


class HostTrace(Call):
    host = True

    def __init__(self, plan, pos, dirs, rule, pipeline):
        super().__init__(plan, "trace (%s)" % ("streamed", "chunked")[pipeline])
        self.pos, self.dirs, self.rule, self.pipeline = pos, dirs, rule, pipeline

    def prepare(self):
        self.out = dict(records=np.zeros(len(self.pos), dtype=tb.TRACE_RESULT))

    def issue(self, stream):
        self.plan.pipeline_set(self.pipeline)
        try:
            self.plan.trace(self.pos, self.dirs, self.rule, results=self.out["records"])
        finally:
            self.plan.pipeline_set(0)

    def outputs(self):
        return _bytes(self.out)


class HostCrossings(HostTrace):
    def __init__(self, plan, pos, dirs, rule, max_crossings=3):
        super().__init__(plan, pos, dirs, rule, 0)
        self.name, self.max_crossings = "trace_crossings", max_crossings

    def issue(self, stream):
        self.out = dict(zip(("records", "crossings"), self.plan.trace_crossings(
            self.pos, self.dirs, self.rule, self.max_crossings)))


class HostHorizon(Horizon):
    host = True

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.name = "horizon %d" % len(self.az)

    def prepare(self):
        self.out = {}

    def issue(self, stream):
        self.out = dict(records=self.plan.horizon(self.station[0], self.station[1], self.origin,
                                                  self.az, self.rule, elevation=(-30., 60.),
                                                  tolerance=self.tolerance))


class HostWalk(Walk):
    host = True

    def __init__(self, *args):
        super().__init__(*args)
        self.name = "step" if self.k == 1 else "walk %d" % self.k
        self.dirs_host = self.dirs.cpu().numpy()

    def issue(self, stream):
        pos = self.ground.copy()
        out = (self.plan.step(pos, self.dirs_host[0], states=self.states) if self.k == 1 else
               self.plan.walk(pos, self.dirs_host, states=self.states))
        self.position = _dev(pos)
        self.out = {k: v for k, v in out.items() if k != "position"}

    def outputs(self):
        return _bytes(dict(self.out, position=self.position.cpu().numpy()))


# ---- running them --------------------------------------------------------------------------

def solo(call):
    """The call alone, synchronously: the reference of every other run of it."""
    import torch
    call.prepare()
    torch.cuda.synchronize()
    call.issue(torch.cuda.Stream())
    torch.cuda.synchronize()
    got = call.outputs()
    call.counters = call.plan.counters(sync=not call.host)
    got.update(call.after())
    return got


def assert_same(call, want):
    got = call.outputs()
    got.update(call.after())
    assert sorted(got) == sorted(want), call.name
    for k in want:
        if got[k] != want[k]:
            a = np.frombuffer(got[k], np.uint8)
            b = np.frombuffer(want[k], np.uint8)
            width = 96 if k == "records" else 1
            bad = np.flatnonzero((a != b).reshape(-1, width).any(1)) if len(a) == len(b) else []
            raise AssertionError("%s: %s differs from the call made alone (%d of %d %s, first %s)" % (
                call.name, k, len(bad), len(b) // width, "records" if width > 1 else "bytes",
                [int(i) for i in bad[:5]]))


def warm(world, angles, rays):
    """Go round the ring of device slots with the largest fan tables and schedule buffers the
    test uses: later calls neither allocate nor free, which would wait for the device."""
    import torch
    az = np.linspace(0., 359., angles - 8)
    for _ in range(SLOTS):
        world.plan.trace_fan_device(tb.Plan.make_fan(world.station[0], world.station[1],
                                                     world.origin, az, np.arange(8.)),
                                    world.rule, fields=_fields(8 * len(az), ["status"]))
        torch.cuda.synchronize()
    t = Trace(world.plan, world.pos[:rays], world.dirs[:rays], world.rule, schedule=1)
    for _ in range(SLOTS if rays else 0):
        t.prepare()
        t.issue(torch.cuda.current_stream())
        torch.cuda.synchronize()


class World:
    """A plan, a station on its ground, ragged batches of rays and particles."""

    def __init__(self, name, stepper, station, box):
        self.name, self.stepper, self.station = name, stepper, station
        self.plan = stepper.freeze(0)
        self.origin = stepper.position(station[0], station[1], 1.0, 0)[0]
        rng = np.random.default_rng(41)
        n = 6000 + 17
        la, lo = rng.uniform(box[0], box[1], n), rng.uniform(box[2], box[3], n)
        self.pos, _ = self.plan.position(la, lo, rng.uniform(-50., 2000., n), 0)
        self.dirs = synth.random_unit(n, 42)
        self.ground, _ = self.plan.position(la[:3001], lo[:3001], rng.uniform(-20, 20, 3001), 0)
        self.steps = synth.random_unit(3001 * 8, 43).reshape(8, 3001, 3)
        self.rule = tb.trace_rule(6000., length_max=2e4, max_steps=5000)

    def rays(self, seed, n):
        rng = np.random.default_rng(seed)
        i = rng.choice(len(self.pos), n, replace=False)
        return self.pos[i], self.dirs[i]

    def fan(self, seed, n_az=67, n_el=33, host=False, plan=None, **kwargs):
        rng = np.random.default_rng(seed)
        az = np.sort(rng.uniform(0., 360., n_az))
        el = np.sort(rng.uniform(-10., 40., n_el))
        return (HostFan if host else Fan)(plan or self.plan, self.station, self.origin, az, el,
                                          self.rule, **kwargs)

    def horizon(self, seed, n_az=67, host=False, plan=None):
        az = np.sort(np.random.default_rng(seed).uniform(0., 360., n_az))
        return (HostHorizon if host else Horizon)(plan or self.plan, self.station, self.origin,
                                                  az, self.rule)

    def walk(self, k, offset=0, host=False, n=3001):
        return (HostWalk if host else Walk)(self.plan, self.ground[:n], self.steps[offset:offset + k, :n],
                                            self.steps[7:8, :n])


@pytest.fixture(scope="module", params=["small_stack", "c3_r10"])
def world(request, small_stack):
    if request.param == "small_stack":  # the specialised single-stack kernels
        sc = Scene(stacks=[small_stack], ops=[(H.ADD_STACK, 0, 0.)], range=0.)
        return World("small_stack", sc.product()[0], (45.4, 2.6), (45.1, 45.9, 2.1, 2.9))
    # layered, Lambert map, geoid, local approximation: the LLA + projected kernels with
    # dynamic shared memory and device states
    return World("c3_r10", c3(small_stack, 10., 1).product()[0], (45.6, 2.7),
                 (45.5, 45.7, 2.6, 2.8))


def run_held(calls, hold_ms, same_stream=False):
    """Issue `calls` on held streams (one each, or all on one), check that the hold outlived
    the issuing, then synchronise."""
    import torch
    for c in calls:
        c.prepare()
    torch.cuda.synchronize()
    hold = Hold(hold_ms)
    held = [hold.stream()] * len(calls) if same_stream else [hold.stream() for _ in calls]
    for c, s in zip(calls, held):
        c.issue(s)
    assert hold.pending(), "the hold was over before the last call was issued: no overlap shown"
    torch.cuda.synchronize()


# ---- 1. eight in flight, all kinds ---------------------------------------------------------

def eight_calls(world):
    p = world.plan
    return [
        Trace(p, *world.rays(1, 4000 + 3), world.rule),
        Crossings(p, *world.rays(2, 3000 + 5), world.rule),
        world.fan(3),
        Fields(p, *world.rays(4, 2000 + 11), world.rule, FIELDS),
        world.horizon(5),
        world.walk(1),
        world.walk(5, offset=1),
        Trace(p, *world.rays(6, 5000 + 1), world.rule, schedule=1),
    ]


def test_eight_in_flight_all_kinds(world):
    calls = eight_calls(world)
    warm(world, 100, 5001)
    want = [solo(c) for c in calls]
    run_held(calls, 300)
    got = world.plan.counters(sync=True)  # before after() makes one more step
    for c, w in zip(calls, want):
        assert_same(c, w)
    # the counters are those of the call issued last
    last = calls[-1].counters
    assert got["rays"] == last["rays"] == 5001
    assert (got["steps"], got["samples"]) == (last["steps"], last["samples"])


def test_a_ninth_call_waits_for_the_oldest(world):
    """Nine device calls with eight slots: the ninth takes the slot of the call issued first
    once that call is over -- the longest of the eight here."""
    import torch
    calls = eight_calls(world)
    calls[0] = world.fan(11, n_az=199, n_el=99)  # 19701 rays
    ninth = world.fan(12, n_az=199, n_el=99)     # same tables, other angles
    warm(world, 298, 5001)
    want = [solo(c) for c in calls + [ninth]]
    for c in calls + [ninth]:
        c.prepare()
    torch.cuda.synchronize()
    hold = Hold(300)
    for c in calls:
        c.issue(hold.stream())
    assert hold.pending(), "the hold was over before the eighth call was issued"
    ninth.issue(streams(1)[0])
    torch.cuda.synchronize()
    got = world.plan.counters(sync=True)
    for c, w in zip(calls + [ninth], want):
        assert_same(c, w)
    assert (got["steps"], got["samples"]) == (ninth.counters["steps"], ninth.counters["samples"])


# ---- 2. uneven lifetimes -------------------------------------------------------------------

def test_uneven_lifetimes(world):
    """One call held on stream A while stream B makes twelve short calls one after the other
    (synchronising B after each): at most two in flight, but B goes round the ring while A's
    fan tables are still to be uploaded. B's fans and horizons have A's numbers of angles,
    so no table is reallocated."""
    import torch
    p = world.plan
    a = world.fan(20)
    b = [world.fan(21), Trace(p, *world.rays(22, 1000 + 1), world.rule), world.horizon(23),
         Fields(p, *world.rays(24, 777), world.rule, ["length0", "n_steps"]), world.fan(25),
         world.walk(1, n=999), Crossings(p, *world.rays(26, 1500 + 9), world.rule),
         world.fan(27),  # the eighth: round-robin would give it A's slot
         world.horizon(28), world.fan(29), Trace(p, *world.rays(30, 2001), world.rule),
         world.walk(3, offset=2, n=999)]
    warm(world, 100, 0)
    want_a, want_b = solo(a), [solo(c) for c in b]
    for c in [a] + b:
        c.prepare()
    torch.cuda.synchronize()
    hold = Hold(500)
    s_a = hold.stream()
    a.issue(s_a)
    a_done = torch.cuda.Event()
    a_done.record(s_a)
    s_b = streams(1)[0]
    for c in b:
        c.issue(s_b)
        s_b.synchronize()
    assert hold.pending() and not a_done.query(), "A was over before B's last call"
    torch.cuda.synchronize()
    assert_same(a, want_a)
    for c, w in zip(b, want_b):
        assert_same(c, w)


# ---- 3. host-pointer calls while device calls are pending ----------------------------------

def test_host_calls_while_device_calls_pend(world):
    """The host-pointer calls have resources of their own: made while device calls are held
    on the caller's stream, both sides give their solo results."""
    import torch
    p = world.plan
    held = [Trace(p, *world.rays(40, 3000 + 7), world.rule), world.fan(41)]
    # short rules keep the host calls well within the hold
    short = tb.trace_rule(6000., length_max=2e3, max_steps=64)
    # slices of 20 000 rays, four per lane of their launch: each kernel pulls rays from its
    # queue cursor for as long as it runs, so slices that ran on one cursor would lose rays
    fan_dev = world.fan(42, n_az=400, n_el=400)
    host_fan = world.fan(42, n_az=400, n_el=400, host=True)
    fan_dev.rule = host_fan.rule = short
    # > 256 Ki rays: the streamed pipeline (mode 0)
    rng = np.random.default_rng(43)
    i = rng.integers(0, len(world.pos), (1 << 18) + 1001)
    quick = [host_fan, HostTrace(p, world.pos[i], world.dirs[i], short, 0),
             HostTrace(p, world.pos[i[:50001]], world.dirs[i[:50001]], short, 1)]
    waiting = [world.horizon(44, host=True), world.walk(1, host=True),
               world.walk(4, offset=3, host=True),
               HostCrossings(p, *world.rays(45, 2500 + 3), world.rule)]
    warm(world, 160, 0)
    want = [solo(c) for c in held + quick + waiting]
    # the fan cut in slices is the device fan
    assert want[2] == solo(fan_dev)
    for c in held + quick + waiting:
        c.prepare()
    torch.cuda.synchronize()
    hold = Hold(600)
    caller = hold.stream()
    for c in held:
        c.issue(caller)
    for c in quick:
        c.issue(None)
    assert hold.pending(), "the device calls were over before the host calls were made"
    # (these free device buffers of their own before they return, which waits for the device)
    for c in waiting:
        c.issue(None)
    torch.cuda.synchronize()
    for c, w in zip(held + quick + waiting, want):
        assert_same(c, w)


# ---- 4. tables that grow while earlier calls are pending -----------------------------------

def test_tables_grow_under_pending_calls(world):
    """Fans and horizons with more angles than any before, each issued while a smaller call
    is held: a slot's tables are reallocated, never under a call that is still in flight.
    (Freeing the smaller tables waits for the device: one growth per hold.) The calls made
    alone run on a plan of their own, whose tables grow apart."""
    import torch
    alone = world.stepper.freeze(0)

    def calls(plan):
        out = []
        for k, n_az in enumerate((40, 90, 150, 260, 420)):
            small = world.fan(50 + k, n_az=7, n_el=k + 3, plan=plan)
            grow = (world.fan(60 + k, n_az=n_az, n_el=k + 5, plan=plan) if k % 2 == 0 else
                    world.horizon(70 + k, n_az=n_az + 7, plan=plan))
            out.append((small, grow))
        return out

    want = [(solo(a), solo(b)) for a, b in calls(alone)]
    pairs = calls(world.plan)
    warm(world, 30, 0)
    for a, b in pairs:
        a.prepare()
        b.prepare()
    torch.cuda.synchronize()
    for a, b in pairs:
        hold = Hold(60)
        a.issue(hold.stream())
        assert hold.pending(), "the hold was over before %s was issued" % b.name
        b.issue(hold.stream())
    torch.cuda.synchronize()
    for (a, b), (wa, wb) in zip(pairs, want):
        assert_same(a, wa)
        assert_same(b, wb)


# ---- 5. gather modes -----------------------------------------------------------------------

def test_gather_modes_in_flight(small_stack):
    """Shared-memory window gathers (mode 2) in flight with global gathers (mode 0) on the
    same plan and on another one: same records, and each call's window hits are its own."""
    sc = Scene(stacks=[small_stack], ops=[(H.ADD_STACK, 0, 0.)], range=0.)
    w = World("small_stack", sc.product()[0], (45.4, 2.6), (45.1, 45.9, 2.1, 2.9))
    other = w.stepper.freeze(0)
    n = 20000 + 13
    pos = np.repeat(w.origin[None], n, 0)
    dirs_a, dirs_b = synth.random_unit(n, 51), synth.random_unit(n, 52)
    window = (2, w.station[0], w.station[1])
    for order in ((2, 0), (0, 2)):
        calls = [Trace(w.plan, pos, dirs_a, w.rule, gather=window if order[0] else (0,)),
                 Trace(other, pos, dirs_a, w.rule, gather=window if order[1] else (0,)),
                 Trace(w.plan, pos, dirs_b, w.rule, gather=window if order[1] else (0,)),
                 Trace(other, pos, dirs_b, w.rule, gather=window if order[0] else (0,))]
        want = [solo(c) for c in calls]
        for c in calls:
            assert (c.counters["window_hits"] > 0) == (c.gather[0] == 2), c.name
        assert want[0] == want[1] and want[2] == want[3]
        run_held(calls, 300)
        for c, x in zip(calls, want):
            assert_same(c, x)
        for plan, last in ((w.plan, calls[2]), (other, calls[3])):
            got = plan.counters(sync=True)
            assert (got["window_hits"], got["samples"]) == \
                (last.counters["window_hits"], last.counters["samples"]), last.name
