"""Horizon search (turtle_stepper_horizon) on the C2 geometry and station of bench.py: the
3 x 3 stack of 3601-node tiles seen from (DET_LAT, DET_LON, DET_HEIGHT).

For 3600 azimuths over the whole window [-90, 90] at tolerances of 1e-3 and 1e-6 degrees it
prints, one JSON line each:
  - the device time of the search (CUDA events, after a warm-up), probes per azimuth, steps,
    samples, samples/s and the active lanes per loop iteration (samples / warp iterations);
  - samples/s of the whole-ray trace kernel of a single stack (trace_stack) on a sample of
    the bench fan, for comparison;
  - the device time of the dense fan (turtle_stepper_trace_fan, 0.01 degree) that brute force
    needs over the band of elevations where the horizons fall;
  - the reference on the host cores running the same K-ary search for a fixed sample of
    azimuths (its probes are whole rays: the reference has no first-change stop).
Every line carries the card's name and power limit.

    python tools/bench_horizon.py [--azimuths 3600] [--repeats 5] [--ref-azimuths 8]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (geometry and station of the C2 configuration, unchanged)


def card():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out) if out else None
    except (OSError, ValueError, subprocess.SubprocessError):
        info["power_limit_w"] = None
    return info


def timed(fn, repeats):
    """Mean device time (ms) of `fn` on the current stream, after one warm-up call."""
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(repeats):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / repeats


def reference_search(d, H, origin, azimuth, window, tolerance, rule, cores):
    """The device's K-ary search with the reference's rays: 32 probes per round, the bracket
    narrowed to [highest obstructed probe, next probe above it]. -> (elevations, probes)."""
    lo, hi = window
    probes = 0
    for rnd in range(64):
        if rnd == 0:
            el = lo + (hi - lo) * (np.arange(32) / 31.)
            el[31] = hi
        else:
            el = lo + (hi - lo) * ((np.arange(32) + 1.) / 33.)
        dirs = d.ecef_from_horizontal(np.full(32, bench.DET_LAT), np.full(32, bench.DET_LON),
                                      np.full(32, azimuth), el)
        rec, cross = d.trace_crossings(np.repeat(origin, 32, 0), dirs, rule, 1, threads=cores)
        probes += 32
        hit = (rec["n_changes"] >= 1) & (cross[:, 0]["to"] >= 0)
        if rnd == 0 and (not hit[0] or hit[31]):
            return (np.nan, np.nan), probes
        k = np.flatnonzero(hit)
        old = (lo, hi)
        if len(k) == 0:
            hi = el[0]
        else:
            lo = el[k[-1]]
            if k[-1] < 31:
                hi = el[k[-1] + 1]
        if not (hi - lo > tolerance) or (lo, hi) == old:
            break
    return (lo, hi), probes


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--azimuths", type=int, default=3600)
    p.add_argument("--repeats", type=int, default=5)
    p.add_argument("--ref-azimuths", type=int, default=8)
    args = p.parse_args()

    import torch
    import turtle_b200 as tb
    from turtle_b200.api import HORIZON_FOUND

    who = card()
    bench.make_stack()
    stack = tb.Stack(bench.stack_dir())
    stepper = tb.Stepper(range=0., slope=0.4, resolution=1e-2)
    stepper.add_stack(stack, 0.)
    plan = stepper.freeze(0)
    rule = tb.trace_rule(bench.ALTITUDE_MAX, max_steps=bench.MAX_STEPS)
    lat, lon = bench.DET_LAT, bench.DET_LON
    origin, index = stepper.position(lat, lon, bench.DET_HEIGHT, 0)
    assert index == 0
    stream = torch.cuda.current_stream()
    n = args.azimuths
    azimuth = (np.arange(n) + 0.5) * (360. / n)
    d_out = torch.empty(n * 96, dtype=torch.uint8, device="cuda")

    def emit(line):
        line.update(who)
        print(json.dumps(line), flush=True)

    found = None
    for tolerance in (1e-3, 1e-6):
        res = plan.horizon(lat, lon, origin, azimuth, rule, tolerance=tolerance)
        c = plan.counters()

        def search():
            plan.horizon_device(lat, lon, origin, azimuth, rule, d_out, tolerance=tolerance,
                                stream=stream.cuda_stream)
        ms = timed(search, args.repeats)
        assert d_out.cpu().numpy().tobytes() == res.tobytes()
        iterations = int(res["n_iterations"].sum())
        emit({"what": "horizon", "azimuths": n, "window": [-90., 90.], "tolerance_deg": tolerance,
              "ms": ms, "probes_per_azimuth": float(res["n_probes"].mean()),
              "probes_max": int(res["n_probes"].max()), "rays": c["rays"], "steps": c["steps"],
              "samples": c["samples"], "samples_per_s": c["samples"] / (ms * 1e-3),
              "active_lanes_per_iteration": c["samples"] / max(iterations, 1),
              "status_counts": np.bincount(res["status"], minlength=4).tolist()})
        if tolerance == 1e-6:
            found = res

    # the whole-ray kernel of the same geometry, on a 4 Mi-ray sample of the bench fan
    m = 1 << 22
    dirs = bench.fan_subsample(0, 1, (bench.N_AZ * bench.N_EL) // m, bench.N_AZ * bench.N_EL)[:m]
    d_pos = torch.tensor(np.repeat(origin[None], m, 0), device="cuda")
    d_dir = torch.tensor(dirs, device="cuda")
    d_res = torch.empty((m, 96), dtype=torch.uint8, device="cuda")
    ms = timed(lambda: plan.trace_device(m, d_pos, d_dir, rule, d_res,
                                         stream=stream.cuda_stream), args.repeats)
    c = plan.counters(sync=True)
    emit({"what": "trace_stack", "rays": m, "ms": ms, "samples": c["samples"],
          "samples_per_s": c["samples"] / (ms * 1e-3)})
    del d_pos, d_dir, d_res

    # brute force: a 0.01-degree fan over the band where the horizons fall
    ok = found["status"] == HORIZON_FOUND
    band = (np.floor(found["elevation"][ok, 0].min() * 100.) / 100.,
            np.ceil(found["elevation"][ok, 1].max() * 100.) / 100.)
    el = np.arange(int(round((band[1] - band[0]) * 100.)) + 1) * 0.01 + band[0]
    fan = tb.Plan.make_fan(lat, lon, origin, azimuth, el, bundle=1)
    rays = n * len(el)
    d_changes = torch.empty(rays, dtype=torch.int32, device="cuda")
    ms = timed(lambda: plan.trace_fan_device(fan, rule, fields=dict(n_changes=d_changes),
                                             stream=stream.cuda_stream), args.repeats)
    c = plan.counters(sync=True)
    emit({"what": "dense_fan", "band_deg": list(band), "step_deg": 0.01,
          "elevations": len(el), "rays": rays, "ms": ms, "steps": c["steps"],
          "samples": c["samples"]})
    del d_changes

    # the reference on the host cores, same search, a fixed sample of azimuths
    d, H, kind = bench.reference_driver()
    cores = os.cpu_count() or 1
    ref_pos, _ = d.position([lat], [lon], [bench.DET_HEIGHT], 0)
    sample = np.arange(args.ref_azimuths) * (n // args.ref_azimuths)
    t0 = time.perf_counter()
    brackets, probes = [], 0
    for i in sample:
        b, k = reference_search(d, H, ref_pos, azimuth[i], (-90., 90.), 1e-6,
                                H.rule(bench.ALTITUDE_MAX, max_steps=bench.MAX_STEPS), cores)
        brackets.append(b)
        probes += k
    seconds = time.perf_counter() - t0
    brackets = np.array(brackets)
    emit({"what": "reference_search", "kind": kind, "cores": cores, "azimuths": len(sample),
          "tolerance_deg": 1e-6, "seconds": seconds, "ms_per_azimuth": 1e3 * seconds / len(sample),
          "probes": probes, "note": "probes traced to the rule's end (no first-change stop)",
          "max_abs_diff_vs_gpu_deg": float(np.nanmax(np.abs(brackets - found["elevation"][sample])))})
    return 0


if __name__ == "__main__":
    sys.exit(main())
