"""Many stations, three ways, on the C2 geometry of bench.py (3 x 3 stack of 3601-node tiles):

  loop      one host-pointer call per station (turtle_stepper_trace_fan / _horizon), one after
            the other: what a caller without the station dimension writes first;
  inflight  one device-pointer call per station, 8 in flight on 8 streams (the most a plan
            takes), results in device memory;
  stations  ONE call for all the stations (turtle_stepper_trace_fans / _horizons), host- and
            device-pointer variants.

Workloads: stations 1 m over the ground at seeded random points of the stack,
  fans      --stations x (64 azimuths x 16 elevations), field length[0] only;
  horizons  --stations x 360 azimuths over [-90, 90], tolerance 1e-4 degrees.
Each way is timed on the host clock around work that ends in a device synchronise, after a
warm-up, as the mean of --repeats runs; every way must give the bytes of the loop. One JSON
line per (workload, way), with rays (probes) per second and the card's name and power limit.

    python tools/bench_stations.py [--stations 2000] [--repeats 3]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (geometry of the C2 configuration, unchanged)
from bench_horizon import card  # noqa: E402

N_AZ_FAN, N_EL_FAN = 64, 16
N_AZ_HORIZON, TOLERANCE = 360, 1e-4
SLOTS = 8  # device-pointer calls in flight on one plan


def timed(fn, repeats):
    """Mean wall time (s) of fn() followed by a device synchronise, after one warm-up."""
    import torch
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(repeats):
        fn()
        torch.cuda.synchronize()
    return (time.perf_counter() - t0) / repeats


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--stations", type=int, default=2000)
    p.add_argument("--repeats", type=int, default=3)
    args = p.parse_args()

    import torch
    import turtle_b200 as tb

    who = card()
    bench.make_stack()
    stack = tb.Stack(bench.stack_dir())
    stepper = tb.Stepper(range=0., slope=0.4, resolution=1e-2)
    stepper.add_stack(stack, 0.)
    plan = stepper.freeze(0)
    rule = tb.trace_rule(bench.ALTITUDE_MAX, max_steps=bench.MAX_STEPS)
    rng = np.random.default_rng(2024)
    n = args.stations
    la = rng.uniform(bench.STACK_LAT0 + 0.5, bench.STACK_LAT0 + bench.STACK_N - 0.5, n)
    lo = rng.uniform(bench.STACK_LON0 + 0.5, bench.STACK_LON0 + bench.STACK_N - 0.5, n)
    pos, index = plan.position(la, lo, np.full(n, bench.DET_HEIGHT), 0)
    assert (index >= 0).all()
    streams = [torch.cuda.Stream() for _ in range(SLOTS)]

    def emit(line):
        line.update(who)
        print(json.dumps(line), flush=True)

    # ---- fans: length[0] of every ray --------------------------------------------------------
    az = (np.arange(N_AZ_FAN) + 0.5) * (360. / N_AZ_FAN)
    el = -10. + 50. * (np.arange(N_EL_FAN) + 0.5) / N_EL_FAN
    per = N_AZ_FAN * N_EL_FAN
    rays = n * per
    fans = [tb.Plan.make_fan(la[s], lo[s], pos[s], az, el) for s in range(n)]
    many = tb.Plan.make_fans(la, lo, pos, az, el)
    h_len = np.zeros(rays)
    d_len = torch.zeros(rays, dtype=torch.float64, device="cuda")

    def fan_loop():
        for s in range(n):
            plan.trace_fan(fans[s], rule, fields=dict(length0=h_len[s * per:(s + 1) * per]))

    def fan_inflight():
        for s in range(n):
            plan.trace_fan_device(fans[s], rule, fields=dict(length0=d_len[s * per:(s + 1) * per]),
                                  stream=streams[s % SLOTS].cuda_stream)

    def fan_stations_host():
        plan.trace_fans(many, rule, fields=dict(length0=h_len))

    def fan_stations_device():
        plan.trace_fans_device(many, rule, fields=dict(length0=d_len))

    want = None
    for way, fn, out in (("loop", fan_loop, h_len), ("inflight", fan_inflight, d_len),
                         ("stations_host", fan_stations_host, h_len),
                         ("stations_device", fan_stations_device, d_len)):
        h_len[:] = np.nan
        d_len.fill_(float("nan"))
        seconds = timed(fn, args.repeats)
        got = (out.cpu().numpy() if hasattr(out, "cpu") else out).tobytes()
        if want is None:
            want = got
        emit({"workload": "fans", "way": way, "stations": n, "grid": [N_AZ_FAN, N_EL_FAN],
              "rays": rays, "s": seconds, "rays_per_s": rays / seconds,
              "same_as_loop": got == want})

    # ---- horizons ----------------------------------------------------------------------------
    az = (np.arange(N_AZ_HORIZON) + 0.5) * (360. / N_AZ_HORIZON)
    kw = dict(elevation=(-90., 90.), tolerance=TOLERANCE)
    h_res = np.zeros((n, N_AZ_HORIZON), dtype=tb.HORIZON_RESULT)
    d_res = torch.zeros(n * N_AZ_HORIZON * 96, dtype=torch.uint8, device="cuda")
    row = N_AZ_HORIZON * 96

    def horizon_loop():
        for s in range(n):
            h_res[s] = plan.horizon(la[s], lo[s], pos[s], az, rule, **kw)

    def horizon_inflight():
        for s in range(n):
            plan.horizon_device(la[s], lo[s], pos[s], az, rule, d_res[s * row:(s + 1) * row],
                                stream=streams[s % SLOTS].cuda_stream, **kw)

    def horizon_stations_host():
        h_res[:] = plan.horizons(la, lo, pos, az, rule, **kw)

    def horizon_stations_device():
        plan.horizons_device(la, lo, pos, az, rule, d_res, **kw)

    want, probes = None, 0
    for way, fn, out in (("loop", horizon_loop, h_res), ("inflight", horizon_inflight, d_res),
                         ("stations_host", horizon_stations_host, h_res),
                         ("stations_device", horizon_stations_device, d_res)):
        h_res[:] = np.zeros(1, dtype=tb.HORIZON_RESULT)
        d_res.zero_()
        seconds = timed(fn, args.repeats)
        got = (out.cpu().numpy() if hasattr(out, "cpu") else out).tobytes()
        if want is None:
            want = got
            probes = int(h_res["n_probes"].sum())
        emit({"workload": "horizons", "way": way, "stations": n, "azimuths": N_AZ_HORIZON,
              "tolerance_deg": TOLERANCE, "probes": probes, "s": seconds,
              "probes_per_s": probes / seconds, "same_as_loop": got == want})
    return 0


if __name__ == "__main__":
    sys.exit(main())
