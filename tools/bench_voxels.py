"""Rock length per voxel against the plain fan trace, on the same rays of a muography survey.

Scene (C3-like): the 3 x 3 stack of 3601-node tiles of bench.py with a Lambert 93 map of the
same terrain over it, both in layer 0: rays 1 m over the ground start in medium 1 (air) and
cross medium 0 (rock). Workload: --stations stations (default 8) 1 m over the ground around
(46.5 N, 3.5 E), one --n x --n fan each (azimuth 0-360 deg, elevation -5-45 deg) as ONE
struct turtle_fans. Grid: cells of --cell metres (default 50) over 20 x 20 km and from 1000 m
below to 4000 m above the frame's origin, which covers the relief under the stations.

Timed, alternately, with CUDA events after one warm-up of each:
  fans    turtle_stepper_trace_fans_device, field length[0] (the rock length of every ray);
  voxels  turtle_stepper_trace_fans_voxels_device, media = rock, entries and counts, with the
          exact capacity found by a counting pass (capacity 0).
One JSON line: Mrays/s of each and their ratio, entries per ray (mean, p99, max), bytes of
entries and counts written per second, and the card's name and power limit.

    python tools/bench_voxels.py [--stations 8] [--n 256] [--repeats 5]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (the stack of the C2 / C3 configurations, unchanged)
from bench_horizon import card  # noqa: E402


class Survey:
    """The scene, stations, fans and grid of the module docstring: plan, rule, fans, grid, n
    (rays) and cells (along E, N, U)."""

    def __init__(self, stations=8, n=256, cell=50.):
        import turtle_b200 as tb
        from oracle import harness as H
        from tests.common import lambert_map

        bench.make_stack()
        lat0, lon0 = bench.DET_LAT, bench.DET_LON
        lm = lambert_map(H.Driver(H.best_oracle()), lat_c=lat0, lon_c=lon0, n=401, half=12000.,
                         nodes_per_degree=3600, lat0=bench.STACK_LAT0, lon0=bench.STACK_LON0)
        stack = tb.Stack(bench.stack_dir())
        lmap = tb.Map(lm["nx"], lm["ny"], lm["x"], lm["y"], lm["z"], lm["projection"], lm["values"])
        stepper = tb.Stepper(range=0.)
        stepper.add_stack(stack, 0.)
        stepper.add_map(lmap, 0.)
        self.plan = plan = stepper.freeze(0)
        self.rule = tb.trace_rule(bench.ALTITUDE_MAX, max_steps=bench.MAX_STEPS)

        rng = np.random.default_rng(2025)
        la = lat0 + rng.uniform(-0.04, 0.04, stations)
        lo = lon0 + rng.uniform(-0.05, 0.05, stations)
        pos, index = plan.position(la, lo, np.ones(stations), 0)
        assert (index >= 0).all()
        az = (np.arange(n) + 0.5) * (360. / n)
        el = -5. + 50. * (np.arange(n) + 0.5) / n
        self.fans = tb.Plan.make_fans(la, lo, pos, az, el, bundle=32 if n % 32 == 0 else 1)
        self.n = stations * n * n
        half = 10000.
        c = int(round(2 * half / cell))
        self.cells = [c, c, int(round(5000. / cell))]
        self.grid = tb.voxel_grid(lat0, lon0, 0., (-half, -half, -1000.), (cell,) * 3,
                                  self.cells, 0b1)


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--stations", type=int, default=8)
    p.add_argument("--n", type=int, default=256)
    p.add_argument("--cell", type=float, default=50.)
    p.add_argument("--repeats", type=int, default=5)
    args = p.parse_args()

    import torch

    who = card()
    sv = Survey(args.stations, args.n, args.cell)
    plan, rule, fans, grid, n = sv.plan, sv.rule, sv.fans, sv.grid, sv.n
    cells = sv.cells[0]

    count = torch.empty(n, dtype=torch.int32, device="cuda")
    plan.trace_fans_voxels_device(fans, rule, grid, 0, None, count)  # counting pass
    torch.cuda.synchronize()
    c = count.cpu().numpy()
    capacity = max(int(c.max()), 1)
    entries = torch.empty(n * capacity * 16, dtype=torch.uint8, device="cuda")
    length = torch.empty(n, dtype=torch.float64, device="cuda")

    def fans_call():
        plan.trace_fans_device(fans, rule, fields={"length0": length})

    def voxels_call():
        plan.trace_fans_voxels_device(fans, rule, grid, capacity, entries, count)

    times = {"fans": [], "voxels": []}
    calls = {"fans": fans_call, "voxels": voxels_call}
    for name in calls:  # warm-up
        calls[name]()
    torch.cuda.synchronize()
    for _ in range(args.repeats):
        for name, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e-3)
    # the counts of the timed calls are those of the counting pass
    assert np.array_equal(count.cpu().numpy(), c)
    t_f, t_v = float(np.median(times["fans"])), float(np.median(times["voxels"]))
    written = int(c.sum()) * 16 + 4 * n
    line = dict(bench="voxels", scene="C3-like: 3x3 stack of 3601-node tiles + Lambert 93 map",
                stations=args.stations, fan="%d x %d" % (args.n, args.n), rays=n,
                cell_m=args.cell, grid_cells=[cells, cells, int(round(5000. / args.cell))],
                capacity=capacity, repeats=args.repeats,
                fans_s=t_f, voxels_s=t_v, fans_mrays_s=n / t_f * 1e-6,
                voxels_mrays_s=n / t_v * 1e-6, voxels_over_fans_time=t_v / t_f,
                entries_per_ray_mean=float(c.mean()),
                entries_per_ray_p99=float(np.percentile(c, 99)), entries_per_ray_max=int(c.max()),
                rays_with_entries=int((c > 0).sum()), entry_bytes_written=written,
                entry_gb_s=written / t_v * 1e-9, fans_times_s=times["fans"],
                voxels_times_s=times["voxels"])
    line.update(who)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
