"""GPU: one turtle_stepper_step for n independent particles (turtle_stepper_step_batch)
and ray origins (turtle_stepper_position_batch) against the oracle."""
import os

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.common import ulp_distance
from tests.test_gpu_trace import c3
from turtle_b200 import synth

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.npz"))


@pytest.mark.parametrize("rg,geoid", [(0., -1), (10., 1)])
def test_single_steps_golden(small_stack, rg, geoid):
    """Fresh stepper per particle (states = NULL): the committed reference outputs."""
    stepper, maps, stacks = c3(small_stack, rg, geoid).product()
    plan = stepper.freeze(0)
    key = "c3_r%d" % int(rg)
    got = plan.step(GOLD[key + "_pos"].copy(), GOLD[key + "_dir"])
    want = {f: GOLD[key + "_step_" + f] for f in got}
    same_medium = (got["index"] == want["index"]).all(1)
    assert (~same_medium).sum() <= 1
    assert np.array_equal(got["altitude"][same_medium], want["altitude"][same_medium]) or \
        np.abs(got["altitude"] - want["altitude"])[same_medium].max() < 1e-6
    assert np.abs(got["step"] - want["step"])[same_medium].max() < 1e-6
    assert np.abs(got["position"] - want["position"])[same_medium].max() < 1e-6
    assert ulp_distance(got["latitude"], want["latitude"])[same_medium].max() <= 64
    fin = same_medium & (want["index"][:, 0] >= 0)
    e_w, e_g = want["elevation"][fin], got["elevation"][fin]
    assert np.array_equal(np.abs(e_w) > 1e300, np.abs(e_g) > 1e300)  # +-DBL_MAX sentinels
    small = np.abs(e_w) < 1e300
    assert np.abs(e_w[small] - e_g[small]).max() < 1e-6
    # query mode: no direction, position untouched, step = slope * distance
    q = plan.step(GOLD[key + "_pos"].copy(), None)
    assert np.array_equal(q["position"], GOLD[key + "_pos"])
    out = q["index"][:, 0] < 0
    assert (q["step"][out] == 0.).all() and (q["elevation"][out] == 0.).all()


def test_particle_walk_with_states(small_stack):
    """Config-4 shape: many consecutive steps with a fresh direction each, stepper state
    (last sample + local approximation) kept per particle on the device."""
    sc = c3(small_stack, 1., -1)
    ora = sc.oracle(locked=True)
    stepper, maps, stacks = sc.product()
    plan = stepper.freeze(0)
    rng = np.random.default_rng(31)
    n, k = 4000, 12
    la, lo = rng.uniform(45.2, 45.9, n), rng.uniform(2.2, 2.9, n)
    ground, idx = ora.position(la, lo, rng.uniform(-50, 50, n), 0)
    dirs = synth.random_unit(n * k, 4).reshape(k, n, 3)
    want = ora.walk(ground, dirs, threads=os.cpu_count())
    states = plan.states(n)
    pos = ground.copy()
    bad = np.zeros(n, dtype=bool)
    for j in range(k):
        out = plan.step(pos, dirs[j], states=states)
        pos = out["position"]
        bad |= (out["index"] != want["index"][j]).any(1)
        ok = ~bad
        assert np.abs(out["step"] - want["step"][j])[ok].max() < 1e-5
        assert np.abs(out["altitude"] - want["altitude"][j])[ok].max() < 1e-5
    assert bad.sum() <= max(2, n // 500)
    assert np.abs(pos - want["position"])[~bad].max() < 1e-4


@pytest.mark.parametrize("rg", [0., 1.])
@pytest.mark.parametrize("with_states", [True, False])
def test_walk_batch_is_k_steps(small_stack, rg, with_states):
    """turtle_stepper_walk_batch: k steps per particle in one launch, the stepper state on chip
    in between. Every output of every step, the final position and the state left behind
    are those of k turtle_stepper_step_batch calls, byte for byte (and thereby the oracle's
    walk, see test_particle_walk_with_states)."""
    sc = c3(small_stack, rg, -1)
    stepper, maps, stacks = sc.product()
    plan = stepper.freeze(0)
    rng = np.random.default_rng(33)
    n, k1, k2 = 3001, 7, 5
    la, lo = rng.uniform(45.2, 45.9, n), rng.uniform(2.2, 2.9, n)
    ground, idx = plan.position(la, lo, rng.uniform(-50, 50, n), 0)
    dirs = synth.random_unit(n * (k1 + k2), 5).reshape(k1 + k2, n, 3)
    # a few particles stand still on a step (direction 0 0 0 is legal: the cached sample)
    dirs[3, ::97] = 0.
    s_a = plan.states(n) if with_states else None
    pos = ground.copy()
    steps = []
    for j in range(k1 + k2):
        out = plan.step(pos, dirs[j], states=s_a)
        pos = out["position"]
        steps.append(out)
    s_b = plan.states(n) if with_states else None
    p_b = ground.copy()
    first = plan.walk(p_b, dirs[:k1], states=s_b)
    if not with_states:
        # no states: every WALK starts from a reset stepper, every step_batch call as well;
        # compare the first step only, then the walk against the oracle
        for f in ("altitude", "step", "index", "latitude", "longitude", "elevation"):
            assert np.array_equal(first[f][0], steps[0][f]), f
        ora = sc.oracle(locked=True)
        want = ora.walk(ground, dirs[:k1], threads=os.cpu_count())
        ok = np.logical_and.accumulate((first["index"] == want["index"]).all(2), 0)
        assert (~ok[-1]).sum() <= max(2, n // 500)
        assert np.abs(first["step"] - want["step"])[ok].max() < 1e-5
        assert np.abs(first["altitude"] - want["altitude"])[ok].max() < 1e-5
        return
    second = plan.walk(p_b, dirs[k1:], states=s_b)
    for j in range(k1 + k2):
        got = first if j < k1 else second
        jj = j if j < k1 else j - k1
        for f in ("altitude", "step", "index", "latitude", "longitude", "elevation"):
            assert np.array_equal(got[f][jj], steps[j][f]), (f, j)
    assert np.array_equal(p_b, pos)


def test_position_batch(small_stack):
    sc = c3(small_stack, 0., 1)
    ora = sc.oracle()
    stepper, maps, stacks = sc.product()
    plan = stepper.freeze(0)
    rng = np.random.default_rng(32)
    n = 20000
    la, lo, h = rng.uniform(44.9, 47.1, n), rng.uniform(1.9, 4.1, n), rng.uniform(-5, 50, n)
    for layer in (0, 1):
        wp, wi = ora.position(la, lo, h, layer)
        gp, gi = plan.position(la, lo, h, layer)
        assert np.array_equal(wi, gi)
        assert np.abs(wp - gp).max() < 1e-8  # sin / cos of from_geodetic: a few ulp of 6.4e6 m
    assert (wi == -1).any()
    with pytest.raises(tb.TurtleError):
        plan.position(la, lo, h, 5)


def test_states_outlive_their_plan(small_stack):
    """Particle states may be destroyed after their plan (a garbage collector finalises
    the two in any order): that leaves no CUDA error behind for the next call to report."""
    import ctypes
    sc = c3(small_stack, 1., -1)
    stepper, maps, stacks = sc.product()
    plan = stepper.freeze(0)
    states = plan.states(100)
    tb.api.lib.turtle_plan_destroy(ctypes.byref(plan.handle))
    assert not plan.handle
    del states
    other = stepper.freeze(0)
    pos, idx = other.position([45.5], [2.5], [1.], 0)
    assert idx[0] >= 0
