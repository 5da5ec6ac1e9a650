"""More geometries, on the CPU (host scalar calls + C restatement vs the compiled
reference) and on the GPU (batched path vs the oracle): southern / western hemisphere
tiles, a stack mixing 1201- and 3601-node tiles of the same span (non uniform tile
shape), a southern-hemisphere UTM map, limits of the flattened geometry."""
import os

import numpy as np
import pytest

import turtle_b200 as tb
from oracle import harness as H
from tests.common import Scene, compare_traces
from turtle_b200 import synth

needs_ref = pytest.mark.skipif(not os.path.exists(H.REF), reason="oracle/_ref not built")


@pytest.fixture(scope="module")
def sw_stack(tmp_path_factory):
    """2 x 2 tiles around (-34, -71): names S34W071 ... (negative coordinates)."""
    d = str(tmp_path_factory.mktemp("sw"))
    synth.write_hgt_stack(d, -35, -72, 2, 2, n=1201)
    return d


@pytest.fixture(scope="module")
def mixed_stack(tmp_path_factory):
    """1 x 2 tiles with the same 1 degree span but 1201 and 3601 nodes."""
    d = str(tmp_path_factory.mktemp("mixed"))
    synth.write_hgt_stack(d, 45, 2, 1, 1, n=1201)
    nodes = synth.tile_nodes(45, 3, 45, 2, 3601)
    nodes[::-1].astype(">i2").tofile(os.path.join(d, synth.hgt_name(45, 3)))
    return d


def utm_south_map():
    n = 151
    vals = 500. + synth.fbm_grid(np.arange(n) * 2., np.arange(n) * 2., seed=5) * 2000.
    return dict(nx=n, ny=n, x=(340000., 343000.), y=(6230000., 6233000.), z=(0., 3000.),
                projection="UTM 19S", values=vals)


def rays(ora, lat0, lat1, lon0, lon1, n, seed):
    rng = np.random.default_rng(seed)
    pos = ora.ecef_from_geodetic(rng.uniform(lat0, lat1, n), rng.uniform(lon0, lon1, n),
                                 rng.uniform(-200, 4000, n))
    return pos, synth.random_unit(n, seed)


def scenes(sw_stack, mixed_stack):
    return {
        "south_west": (Scene(maps=[utm_south_map()], stacks=[sw_stack],
                             ops=[(H.ADD_STACK, 0, 0.), (H.ADD_MAP, 0, 0.), (H.ADD_LAYER, 0, 0.),
                                  (H.ADD_STACK, 0, 800.)], range=0.),
                       (-35.1, -32.9, -72.1, -69.9)),
        "mixed_tiles": (Scene(stacks=[mixed_stack], ops=[(H.ADD_FLAT, 0, -50.),
                                                         (H.ADD_STACK, 0, 0.)], range=5.),
                        (44.95, 46.05, 1.95, 4.05)),
    }


@needs_ref
@pytest.mark.parametrize("name", ["south_west", "mixed_tiles"])
@pytest.mark.parametrize("lib", [H.PORT, H.PRODUCT], ids=["port", "product"])
def test_host_matches_reference(sw_stack, mixed_stack, name, lib):
    scene, box = scenes(sw_stack, mixed_stack)[name]
    ref, d = scene.oracle(H.REF), scene.oracle(lib)
    pos, dirs = rays(ref, *box, 1500, 3)
    want, s0, _ = ref.trace(pos, dirs, H.rule(6000., length_max=5e4, max_steps=20000))
    got, s1, _ = d.trace(pos, dirs, H.rule(6000., length_max=5e4, max_steps=20000))
    assert s0 == s1 and want.tobytes() == got.tobytes()
    assert (want["n_changes"] > 0).sum() > 100
    if name == "south_west":  # no flat layer there: rays do leave the data
        assert (want["status"] == 1).any()
    rng = np.random.default_rng(4)
    la, lo = rng.uniform(box[0], box[1], 20000), rng.uniform(box[2], box[3], 20000)
    z0, i0 = ref.stack_elevation(0, la, lo)
    z1, i1 = d.stack_elevation(0, la, lo)
    assert np.array_equal(i0, i1) and np.array_equal(z0, z1) and 0.2 < i0.mean() < 1.


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["south_west", "mixed_tiles"])
def test_gpu_matches_oracle(sw_stack, mixed_stack, name):
    scene, box = scenes(sw_stack, mixed_stack)[name]
    # single thread, no lock: with a lock the reference goes through turtle_client, whose
    # "known missing tile" memo is history dependent for negative coordinates (see
    # test_reference_client_memo_quirk)
    ora = scene.oracle(locked=False)
    pos, dirs = rays(ora, *box, 20000, 5)
    want, steps, _ = ora.trace(pos, dirs, H.rule(6000., length_max=5e4, max_steps=20000))
    stepper, maps, stacks = scene.product()
    got = stepper.freeze(0).trace(pos, dirs, tb.trace_rule(6000., length_max=5e4, max_steps=20000))
    rep = compare_traces(want, got)
    assert rep["discrete_mismatch"] <= 10, rep
    la = np.random.default_rng(6).uniform(box[0], box[1], 5000)
    lo = np.random.default_rng(7).uniform(box[2], box[3], 5000)
    wp, wi = ora.position(la, lo, np.full(5000, 2.), 0)
    gp, gi = stepper.freeze(0).position(la, lo, np.full(5000, 2.), 0)
    assert np.array_equal(wi, gi) and np.abs(wp - gp).max() < 1e-8


@needs_ref
def test_reference_client_memo_quirk(sw_stack, mixed_stack):
    """DESIGN.md section 4: the reference's turtle_client remembers the (int)-truncated
    coordinates of its last miss (client.c:117-124, 163-165). C truncation is toward
    zero, so for NEGATIVE coordinates a ray that left the stack at longitude -70.0 makes
    the next ray starting at -70.1 look outside. The stack itself (no lock) has no such
    memory, and neither has the batched path, which follows the stack."""
    scene, box = scenes(sw_stack, mixed_stack)["south_west"]
    with_client, plain = scene.oracle(H.REF, locked=True), scene.oracle(H.REF, locked=False)
    pos, dirs = rays(plain, *box, 4000, 5)
    rule = H.rule(6000., length_max=5e4, max_steps=20000)
    a, _, _ = with_client.trace(pos, dirs, rule)
    b, _, _ = plain.trace(pos, dirs, rule)
    differ = a["n_steps"] != b["n_steps"]
    assert 0 < differ.sum() < 100
    assert (a["status"][differ] == 1).all() and (a["n_steps"][differ] == 0).all()
    ours, _, _ = scene.oracle(H.PRODUCT, locked=True).trace(pos, dirs, rule)
    assert ours.tobytes() == b.tobytes()  # the product follows the memoryless stack


def _small_map(projection, x=(0., 1.), y=(0., 1.)):
    return tb.Map(2, 2, x, y, (0., 10.), projection, np.zeros((2, 2)))


def _over_the_limit(tmp_path, over, excess):
    """A stepper holding the limit of `over` + `excess`."""
    s = tb.Stepper(range=0.)
    if over == "layers":
        for k in range(8 + excess):
            s.add_layer()
            s.add_flat(float(k))
    elif over == "metas":  # data in the layers, one flat datum
        for k in range(24 + excess):
            s.add_flat(float(k))
    elif over == "data":
        for k in range(12 + excess):
            s.add_map(_small_map(None, (2. + 0.01 * k, 2.5), (45., 45.5)))
    elif over == "transforms":  # distinct projections
        for p in ("Lambert 93", "Lambert II", "UTM 31N", "UTM 32N", "Lambert IV")[:4 + excess]:
            s.add_map(_small_map(p, (5e5, 5.1e5), (5e6, 5.1e6)))
    else:
        for k in range(4 + excess):
            d = str(tmp_path / ("stack%d" % k))
            synth.write_hgt_stack(d, 45, 2 + k, 1, 1, n=11)
            s.add_stack(tb.Stack(d))
    return s


def test_geometry_limits_are_reported(tmp_path):
    """One more layer, meta, datum, transform or stack than the flattened geometry holds
    (8, 24, 12, 4, 4): an error, not a truncation. At the limit it is accepted."""
    for over in ("layers", "metas", "data", "transforms", "stacks"):
        with pytest.raises(tb.TurtleError) as e:
            _over_the_limit(tmp_path, over, 1).step(tb.ecef_from_geodetic(45., 3., 100.))
        assert "geometry too large" in str(e.value), over
        _over_the_limit(tmp_path, over, 0).step(tb.ecef_from_geodetic(45., 3., 100.))


def test_pole_and_axis_positions():
    """ecef.c:77-84: exact special case on the polar axis; a flat-only stepper there."""
    s = tb.Stepper(range=0.)
    s.add_flat(0.)
    out = s.step(np.array([0., 0., 6356752.3142 + 25.]))
    assert out["latitude"] == 90. and out["longitude"] == 0.
    assert abs(out["altitude"] - 25.) < 1e-9 and out["index"] == (1, 0)
    assert abs(out["step"] - 0.4 * 25.) < 1e-9
