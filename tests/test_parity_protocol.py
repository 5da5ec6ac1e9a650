"""The parity protocol itself (oracle/parity.py) and the rounding-noise floor it rests on,
on the CPU: the reference against ITSELF built with FMA contraction
(oracle/_ref/libturtle_ref_fma.so, SURVEY.md 8c).

What the GPU tests assume is pinned here without a GPU: between two builds of the reference
that differ only in the rounding of a*b + c, (1) the discrete outcome of a ray and every
boundary-LOCATED quantity agree to 1 mm / 1e-9, (2) quantities of rays stopped by an altitude /
length THRESHOLD do not -- by metres on long rays --, which is why those are held to a multiple
of this floor instead of 1 mm, and (3) the report sorts the fields of a ray accordingly."""
import os

import numpy as np
import pytest

from oracle import harness as H
from oracle import parity as P
from turtle_b200 import synth

needs_floor = pytest.mark.skipif(
    not (H.available(H.REF) and H.available(H.REF_FMA)),
    reason="needs oracle/_ref (built where the reference's sources are found)")


def records(n):
    r = np.zeros(n, dtype=H.RESULT)
    r["index"] = [[1, 0]] * n
    r["status"] = 0
    r["n_steps"] = 10
    r["length"][:, 0] = 100.
    r["length"][:, 1] = 5000.
    r["total"] = 5100.
    r["position"] = [[4e6, 1e5, 4.5e6]] * n
    r["altitude"] = 9000.
    return r


def test_report_classes_and_tolerances():
    ref = records(8)
    got = ref.copy()
    got["length"][[1, 6, 7], 0] += 5e-2  # rock length, a medium the ray has left: located
    got["length"][2, 1] += 0.5       # final medium of a threshold exit
    got["total"][2] += 0.5
    got["position"][3, 0] += 4e6 * 0.5e-9  # within 1e-9 relative of 4e6 m
    got["n_steps"][4] += 1           # discrete mismatch: not compared any further
    got["length"][4, 0] += 7.
    ref["status"][5] = got["status"][5] = P.STATUS_DOMAIN  # left the data: everything located
    got["total"][5] += 2e-3
    rep = P.report(ref, got)
    assert rep["discrete_mismatch"] == 1 and rep["rays"] == 8
    assert rep["located"]["length0"]["over"] == 3 and rep["located_rays_over"] == 4
    assert rep["located"]["total"]["n"] == 1 and rep["located"]["total"]["over"] == 1
    assert rep["threshold"]["length1"]["over"] == 1 and rep["threshold"]["total"]["over"] == 1
    assert rep["threshold"]["position"]["over"] == 0
    assert abs(rep["threshold"]["total"]["max"] - 0.5) < 1e-9
    # against a floor: the same report is its own floor; a quiet floor flags it
    assert P.against_floor(rep, rep) == []
    quiet = P.report(ref, ref)
    assert any("located.length0" in b for b in P.against_floor(rep, quiet))
    assert any("threshold.total" in b for b in P.against_floor(rep, quiet))
    assert "located" in P.table(rep, quiet)


@needs_floor
def test_the_reference_against_its_fma_build(small_stack):
    """40 000 random rays through flat / stack, range 0 and the reference's default range."""
    rng = np.random.default_rng(11)
    n = 40000
    dirs = synth.random_unit(n, 17)
    for rg in (0., 1.):
        drv = []
        for lib in (H.REF, H.REF_FMA):
            d = H.Driver(lib)
            st = d.stack_create(small_stack, locked=True)
            d.geometry([(H.ADD_FLAT, 0, 0.), (H.ADD_STACK, st, 0.)], range=rg)
            drv.append(d)
        pos = drv[0].ecef_from_geodetic(rng.uniform(45.0, 47.0, n), rng.uniform(2.0, 4.0, n),
                                        rng.uniform(-500., 5000., n))
        rule = H.rule(9000., length_max=1e5)
        a, _, _ = drv[0].trace(pos, dirs, rule, threads=os.cpu_count())
        b, _, _ = drv[1].trace(pos, dirs, rule, threads=os.cpu_count())
        rep = P.report(a, b)
        assert rep["discrete_mismatch"] <= 2
        assert rep["located_rays_over"] == 0                # boundaries: 1 mm / 1e-9 holds
        assert rep["located"]["length0"]["max"] < 1e-3
        assert rep["threshold"]["total"]["over"] > n // 100  # threshold exits: it cannot
        assert rep["threshold"]["total"]["max"] > 0.05       # ... by far
        assert rep["bit_identical"] < n // 2
