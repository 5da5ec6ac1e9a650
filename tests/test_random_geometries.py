"""Random geometries, host side: 1 - 3 layers of 1 - 3 data each (flat / two distinct tile
stacks / maps in nine projections, geodetic maps included), offsets, geoid on or off, local
approximation range 0 / 1 / 10 / 100, random slope and resolution factors, stacks with and without a lock
(= through turtle_client). Whole rays and short random walks through the product's scalar
path (the tb_core.cuh the kernels are built from, instantiated for the host) and through the
oracle's C restatement give the reference's records byte for byte.

ref: src/turtle/stepper.c:85-197 (transforms and their memo), :617-775 (sampling the layers),
:780-875 (the step); the reference's own geometry tests are tests/test-turtle.c:255-410."""
import os

import numpy as np
import pytest

from oracle import harness as H
from tests.common import random_scene, second_stack
from turtle_b200 import synth

pytestmark = pytest.mark.skipif(not os.path.exists(H.REF), reason="oracle/_ref not built")


@pytest.fixture(scope="module")
def tiles(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("random_geometries"))
    synth.write_hgt_stack(d, 45, 2, 2, 2, n=1201)
    return d


@pytest.fixture(scope="module")
def tiles2(tmp_path_factory):
    return second_stack(str(tmp_path_factory.mktemp("random_geometries_2")))


@pytest.mark.parametrize("lib", [H.PRODUCT, H.PORT], ids=["product", "restatement"])
@pytest.mark.parametrize("seed", range(24))
def test_host_paths_are_the_reference(tiles, tiles2, seed, lib):
    rng = np.random.default_rng(1000 + seed)
    scene = random_scene(rng, H.Driver(H.REF), tiles, tiles2)
    locked = bool(rng.random() < 0.3)
    ref, ours = scene.oracle(H.REF, locked=locked), scene.oracle(lib, locked=locked)
    n = 300
    pos = ref.ecef_from_geodetic(rng.uniform(44.9, 47.1, n), rng.uniform(1.9, 4.1, n),
                                 rng.uniform(-300, 4000, n))
    rule = H.rule(6000., length_max=3e4, max_steps=5000)
    want, steps, _ = ref.trace(pos, synth.random_unit(n, seed), rule)
    got, steps_ours, _ = ours.trace(pos, synth.random_unit(n, seed), rule)
    assert steps == steps_ours  # (a lone small map: every ray starts outside, 0 steps)
    assert want.tobytes() == got.tobytes(), (scene.ops, scene.range,
                                             [m["projection"] for m in scene.maps])
    turns = synth.random_unit(100 * 6, seed + 1).reshape(6, 100, 3)
    a, b = ref.walk(pos[:100], turns), ours.walk(pos[:100], turns)
    for field in ("step", "altitude", "index", "position"):
        assert np.array_equal(a[field], b[field], equal_nan=True), field
