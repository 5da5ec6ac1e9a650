"""L @ rho and L.T @ w applied while tracing, against building L and multiplying by it.

Scene, stations, fans and grid of tools/bench_voxels.py (its Survey): the C3-like stack with a
Lambert 93 map, --stations stations (default 8) with one --n x --n fan each, cells of --cell
metres (default 50), media = rock. Densities uniform in [2, 3], weights normal, seeded.

Timed, alternately, with CUDA events after one warm-up of each:
  count     the counting pass alone (capacity 0 of turtle_stepper_trace_fans_voxels_device);
  matrix    the recipe of INTEGRATION.md section 12 on the device: the counting pass
            (capacity 0) of turtle_stepper_trace_fans_voxels_device, the largest count read
            back, the fill pass into an [n, max count] buffer, the torch.sparse CSR matrix built
            from it, L @ rho, L.T converted to CSR and L.T @ w;
  forward   turtle_stepper_trace_fans_opacity_device, opacity only;
  adjoint   the same, gradient only;
  both      the same, opacity and gradient in one call.
One JSON line: the median times, the bytes L takes (exact: 16 per entry; padded: the
[n, max count] buffer of the recipe), gradient atomics (entries) per second, the largest
relative difference of the opacity and gradient from the CSR products, and the card's name and
power limit.

    python tools/bench_opacity.py [--stations 8] [--n 256] [--repeats 5]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_horizon import card  # noqa: E402
from bench_voxels import Survey  # noqa: E402


def csr(count, entries, capacity, cells):
    """The torch.sparse CSR matrix of the entries of a [n, capacity] buffer."""
    import torch
    n = len(count)
    length = entries.view(torch.float64).view(n, 2 * capacity)[:, 0::2]
    voxel = entries.view(torch.int32).view(n, 4 * capacity)[:, 2::4]
    live = torch.arange(capacity, device=count.device)[None, :] < count[:, None]
    crow = torch.zeros(n + 1, dtype=torch.int64, device=count.device)
    crow[1:] = torch.cumsum(count, 0)
    return torch.sparse_csr_tensor(crow, voxel[live].to(torch.int64), length[live],
                                   size=(n, cells))


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
    cells = int(np.prod(sv.cells))
    rng = np.random.default_rng(7)
    rho = torch.from_numpy(rng.uniform(2., 3., cells)).cuda()
    w = torch.from_numpy(rng.normal(size=n)).cuda()

    count = torch.empty(n, dtype=torch.int32, device="cuda")
    plan.trace_fans_voxels_device(fans, rule, grid, 0, None, count)
    torch.cuda.synchronize()
    c = count.cpu().numpy()
    capacity = max(int(c.max()), 1)
    entries = torch.empty(n * capacity * 16, dtype=torch.uint8, device="cuda")
    out = {}

    def matrix():
        plan.trace_fans_voxels_device(fans, rule, grid, 0, None, count)  # counting pass
        cap = max(int(count.max().item()), 1)
        assert cap == capacity
        plan.trace_fans_voxels_device(fans, rule, grid, cap, entries, count)
        L = csr(count, entries, cap, cells)
        out["L_rho"] = torch.mv(L, rho)
        out["Lt_w"] = torch.mv(L.t().to_sparse_csr(), w)

    opacity = torch.empty(n, dtype=torch.float64, device="cuda")
    gradient = torch.zeros(cells, dtype=torch.float64, device="cuda")

    def forward():
        plan.trace_fans_opacity_device(fans, rule, grid, density=rho, opacity=opacity)

    def adjoint():
        plan.trace_fans_opacity_device(fans, rule, grid, weight=w, gradient=gradient)

    def both():
        plan.trace_fans_opacity_device(fans, rule, grid, density=rho, opacity=opacity, weight=w,
                                       gradient=gradient)

    def counting():
        plan.trace_fans_voxels_device(fans, rule, grid, 0, None, count)

    calls = dict(count=counting, matrix=matrix, forward=forward, adjoint=adjoint, both=both)
    times = {k: [] for k in calls}
    for fn in calls.values():  # warm-up
        fn()
    torch.cuda.synchronize()
    for _ in range(args.repeats):
        for name, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e-3)

    # the numbers: one forward and one adjoint from zero against the CSR products
    gradient.zero_()
    both()
    torch.cuda.synchronize()
    L_rho, Lt_w = out["L_rho"], out["Lt_w"]
    op_diff = float(((opacity - L_rho).abs() / L_rho.abs().clamp_min(1e-300)).max())
    g_scale = float(Lt_w.abs().max())
    g_diff = float((gradient - Lt_w).abs().max()) / g_scale
    t = {k: float(np.median(v)) for k, v in times.items()}
    n_entries = int(c.sum())
    line = dict(bench="opacity", scene="C3-like: 3x3 stack of 3601-node tiles + Lambert 93 map",
                stations=args.stations, fan="%d x %d" % (args.n, args.n), rays=n,
                cell_m=args.cell, grid_cells=sv.cells, repeats=args.repeats,
                count_s=t["count"], matrix_s=t["matrix"], forward_s=t["forward"], adjoint_s=t["adjoint"],
                both_s=t["both"], forward_mrays_s=n / t["forward"] * 1e-6,
                matrix_over_both_time=t["matrix"] / t["both"],
                adjoint_over_forward_time=t["adjoint"] / t["forward"],
                forward_over_count_time=t["forward"] / t["count"],
                entries=n_entries, entries_per_ray_max=int(c.max()),
                L_bytes_exact=n_entries * 16, L_bytes_padded=n * capacity * 16,
                gradient_atomics_per_s=n_entries / t["adjoint"],
                opacity_max_rel_diff_vs_csr=op_diff, gradient_max_diff_vs_csr_over_max=g_diff,
                times_s=times)
    line.update(who)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
