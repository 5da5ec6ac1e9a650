"""Compact input / output of whole rays: turtle_stepper_trace_fan (one station + two tables
of angles instead of 48 bytes per ray) and field arrays (the columns a caller wants instead
of 96-byte records). ref: the caller being batched is examples/example-stepper.c:102-140 --
one origin, turtle_ecef_from_horizontal per ray, one number kept per ray.

The fan's directions must be those of the reference's turtle_ecef_from_horizontal TO THE
BIT: the records of a fan are compared byte for byte with the records of the same rays
handed in as arrays whose directions the REFERENCE computed."""
import os

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.common import Scene

FIELDS = ["length0", "length1", "length2", "length3", "total", "altitude", "position",
          "n_steps", "status", "index", "medium_hash", "n_changes"]


def columns(records, names):
    out = {}
    for k in names:
        out[k] = records["length"][:, int(k[-1])] if k.startswith("length") else records[k]
    return out


def fan_rays(ora, lat, lon, az, el, bundle):
    """(i, j) of every ray in the order of struct turtle_fan, and the reference's directions."""
    n_az, n_el = len(az), len(el)
    r = np.arange(n_az * n_el)
    band, rem = r // (n_az * bundle), r % (n_az * bundle)
    i, k = rem // bundle, rem % bundle
    j = band * bundle + k
    return ora.ecef_from_horizontal(np.full(len(r), lat), np.full(len(r), lon), az[i], el[j])


def test_fan_arguments_are_checked_without_a_gpu(small_stack):
    """(runs everywhere: the argument checks come before any CUDA call)"""
    sc = Scene(stacks=[small_stack], ops=[(H.ADD_STACK, 0, 0.)], range=0.)
    stepper, _, _ = sc.product()
    if tb.device_count() == 0:
        pytest.skip("needs a plan, i.e. a device; see test_abi for the no-device behaviour")
    plan = stepper.freeze(0)
    fan = tb.Plan.make_fan(45.4, 2.6, [0., 0., 0.], np.arange(4.), np.arange(6.), bundle=4)
    with pytest.raises(tb.TurtleError, match="multiple of its bundle"):
        plan.trace_fan(fan, tb.trace_rule(6000.), fields=tb.Plan.host_fields(24, ["status"]))


@pytest.mark.gpu
@pytest.mark.parametrize("bundle", [1, 32, 96])
def test_fan_equals_rays_with_reference_directions(small_stack, bundle):
    sc = Scene(stacks=[small_stack], ops=[(H.ADD_STACK, 0, 0.)], range=0.)
    ora = sc.oracle()
    stepper, _, _ = sc.product()
    plan = stepper.freeze(0)
    lat, lon = 45.4, 2.6
    origin, _ = stepper.position(lat, lon, 1.0, 0)
    az = 360. * (np.arange(331) + 0.5) / 331
    el = 0.5 + 29.5 * (np.arange(96) + 0.5) / 96
    dirs = fan_rays(ora, lat, lon, az, el, bundle)
    n = len(dirs)
    rule = tb.trace_rule(6000., max_steps=20000)
    want = plan.trace(np.repeat(origin[None], n, 0), dirs, rule)
    fan = tb.Plan.make_fan(lat, lon, origin, az, el, bundle=bundle)
    rec = np.zeros(n, dtype=tb.TRACE_RESULT)
    fields = tb.Plan.host_fields(n, FIELDS)
    plan.trace_fan(fan, rule, results=rec, fields=fields)
    assert rec.tobytes() == want.tobytes()
    for k, v in columns(want, FIELDS).items():
        assert np.array_equal(fields[k], v), k
    # ... and against the reference stepper itself, discrete outcome
    ref, _, _ = ora.trace(np.repeat(origin[None], n, 0), dirs, H.rule(6000., max_steps=20000))
    assert (ref["n_steps"] != rec["n_steps"]).sum() <= 2


@pytest.mark.gpu
def test_fields_only_and_rounds(small_stack):
    """Only what is asked for is written; host fans go in slices and calls above the staging
    bound in rounds (the field arrays of each begin at its first ray); device-pointer variants
    agree."""
    import torch
    sc = Scene(stacks=[small_stack], ops=[(H.ADD_STACK, 0, 0.)], range=0.)
    stepper, _, _ = sc.product()
    plan = stepper.freeze(0)
    lat, lon = 45.4, 2.6
    origin, _ = stepper.position(lat, lon, 1.0, 0)
    az = 360. * (np.arange(2048) + 0.5) / 2048
    el = 0.5 + 29.5 * (np.arange(320) + 0.5) / 320
    n = len(az) * len(el)
    rule = tb.trace_rule(6000., max_steps=20000)
    fan = tb.Plan.make_fan(lat, lon, origin, az, el, bundle=32)
    rec = np.zeros(n, dtype=tb.TRACE_RESULT)
    plan.trace_fan(fan, rule, results=rec)
    two = tb.Plan.host_fields(n, ["length0", "status"])
    two["length0"][:] = -7.
    os.environ["TURTLE_B200_FAN_SLICE_RAYS"] = str(1 << 17)  # five slices on two streams
    plan.trace_fan(fan, rule, fields=two)
    del os.environ["TURTLE_B200_FAN_SLICE_RAYS"]
    assert np.array_equal(two["length0"], rec["length"][:, 0])
    c = plan.counters()
    assert c["rays"] == n and c["steps"] == int(rec["n_steps"].sum())
    # arrays of rays in, fields out
    ora = sc.oracle()
    dirs = fan_rays(ora, lat, lon, az, el, 32)
    pos = np.repeat(origin[None], n, 0)
    # (the streamed kernel, in rounds: the field arrays of each round begin at its first ray)
    os.environ["TURTLE_B200_STREAM_MAX_RAYS"] = str(1 << 18)  # three rounds
    rounds = tb.Plan.host_fields(n, ["length0", "status"])
    rounds["length0"][:] = -7.
    plan.trace_fields(pos, dirs, rule, rounds)
    del os.environ["TURTLE_B200_STREAM_MAX_RAYS"]
    assert np.array_equal(rounds["length0"], rec["length"][:, 0])
    assert np.array_equal(rounds["status"], rec["status"])
    assert plan.counters()["rays"] == n
    three = plan.trace_fields(pos, dirs, rule, tb.Plan.host_fields(n, ["total", "n_steps", "index"]))
    assert np.array_equal(three["total"], rec["total"])
    assert np.array_equal(three["n_steps"], rec["n_steps"])
    assert np.array_equal(three["index"], rec["index"])
    # device variants
    d_len = torch.full((n,), -1., dtype=torch.float64, device="cuda:0")
    d_hash = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    plan.trace_fan_device(fan, rule, fields=dict(length0=d_len, medium_hash=d_hash))
    torch.cuda.synchronize()
    assert np.array_equal(d_len.cpu().numpy(), rec["length"][:, 0])
    assert np.array_equal(d_hash.cpu().numpy().view(np.uint32), rec["medium_hash"])
    d_alt = torch.zeros(n, dtype=torch.float64, device="cuda:0")
    plan.trace_fields_device(n, torch.from_numpy(pos).cuda(), torch.from_numpy(dirs).cuda(), rule,
                             dict(altitude=d_alt))
    torch.cuda.synchronize()
    assert np.array_equal(d_alt.cpu().numpy(), rec["altitude"])
