#!/usr/bin/env python
"""bench.py -- Mrays/s of the batched DEM ray stepper on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[1], SURVEY.md section 8d "C2"): a muography fan of
4096 x 4096 = 16 Mi rays (lowest elevations first, in azimuth-coherent bundles of 32:
turtle_b200.synth.fan_angles) from a detector at (46.5 N, 3.5 E) + 1 m through a synthetic
SRTMGL1-shaped 3 x 3 stack of 3601 x 3601 one-arc-second tiles, geodetic coordinates,
range 0 (no local approximation), slope 0.4, resolution 1e-2. A ray stops when it
leaves the stack (index[0] < 0), rises above 9000 m or after 1e5 steps.

One "step" of this bench = one pass of the hot path over the whole batch of rays of
every rank. Scaling is weak: each rank (one per GPU, DEM replicated) traces its own
16 Mi rays -- with N ranks the fan has N x 4096 azimuths and rank r takes azimuths
r, r + N, ... --; the 96-byte result records of all ranks land in rank 0's memory inside the
timed region: each rank's trace kernel stores them there itself over NVLink (CUDA IPC peer
mapping, turtle_b200.dist.PeerRecords), with an NCCL gather as the fall-back.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--rays R] [--impl reference]
                    [--dump-outputs DIR]

prints ONE JSON line (see the keys at the bottom of main()).
  value      whole-job Mrays/s with rays resident in HBM (device-pointer C ABI call,
             96-byte records delivered to rank 0)
  e2e        end to end through turtle_stepper_trace_fan, the batched form of the caller
             of examples/example-stepper.c: the station and two tables of angles go in
             from pinned HOST memory, rock length + status + step count per ray come back
             to pinned HOST memory, all inside the timed region, every step
  e2e_full_records  the same through turtle_stepper_trace_batch: 48 B per ray in, the
             96-byte record per ray out, pinned host buffers
  strong_scaling    ONE 16 Mi-ray fan split over the ranks (the headline numbers are weak)
  roofline   the trace kernel against the measured FP64 FMA peak of this GPU (the
             path is FP64-pipe / issue bound, not HBM bound: DESIGN.md) -- plus the
             HBM side for reference. Operation counts and DRAM traffic come from the
             committed ncu capture (profiles/r02_kernels.json), refused when stale
  cpu_baseline  the reference's own CPU stepper (oracle/_ref, else the C port) on all
             host cores, on a strided sample of the same rays, with the parity of those
             rays (every field) next to the reference-vs-FMA-reference noise floor
`--impl reference` times that CPU path alone, same metric / unit / config.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DET_LAT, DET_LON, DET_HEIGHT = 46.5, 3.5, 1.0
STACK_LAT0, STACK_LON0, STACK_N = 45, 2, 3
ALTITUDE_MAX, MAX_STEPS = 9000.0, 100000
N_AZ = N_EL = 4096
BYTES_PER_RAY = 48 + 96  # position + direction in, result record out
BYTES_PER_SAMPLE = 8     # four 16-bit nodes
# --dump-outputs: a fixed, seeded sample of the records (120 B per ray as float64: 32 MB)
DUMP_RAYS, DUMP_SEED = 1 << 18, 0x7075727474


def _synth():
    """turtle_b200/synth.py (numpy input generators) loaded as a plain module: importing
    the PACKAGE would load libturtle_b200.so, which the reference arm must not touch."""
    import importlib.util
    if "turtle_b200_synth" not in sys.modules:
        spec = importlib.util.spec_from_file_location(
            "turtle_b200_synth", os.path.join(ROOT, "turtle_b200", "synth.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        sys.modules["turtle_b200_synth"] = mod
    return sys.modules["turtle_b200_synth"]


def stack_dir():
    return os.environ.get("TURTLE_BENCH_STACK", "/tmp/turtle_b200_stack3601")


def make_stack():
    synth = _synth()
    return synth.write_hgt_stack(stack_dir(), STACK_LAT0, STACK_LON0, STACK_N, STACK_N, n=3601)


def fan(rank, world, first, count, n_az=N_AZ, n_el=N_EL):
    """Directions of rays [first, first + count) of the part of the fan traced by `rank`:
    the azimuths of the `world` ranks interleave into one fan of world * n_az azimuths."""
    synth = _synth()
    return DET_LAT, DET_LON, synth.fan_directions(
        DET_LAT, DET_LON, n_az, n_el, first=first, count=count, part=rank, parts=world)


def fan_tables(synth, rank, world):
    """The azimuths and elevations (degrees) of the rank's part of the fan: what
    turtle_stepper_trace_fan takes instead of one direction per ray (bundle = 32)."""
    i = np.arange(N_AZ, dtype=np.int64) * 32   # first ray of every azimuth of band 0
    az, _ = synth.fan_angles(i, N_AZ, N_EL, part=rank, parts=world)
    j = np.arange(N_EL, dtype=np.int64)
    r = (j // 32) * (N_AZ * 32) + j % 32       # azimuth 0, elevation j
    _, el = synth.fan_angles(r, N_AZ, N_EL, part=rank, parts=world)
    return np.ascontiguousarray(az), np.ascontiguousarray(el)


def fan_subsample(rank, world, stride, n_total):
    """Every `stride`-th ray of the rank's part of the fan (ray index order preserved)."""
    synth = _synth()
    r = np.arange(0, n_total, stride, dtype=np.int64)
    az, el = synth.fan_angles(r, N_AZ, N_EL, part=rank, parts=world)
    return synth.np_from_horizontal(np.full(len(r), DET_LAT), np.full(len(r), DET_LON), az, el)


def dump_sample(n):
    """Rows of a batch of n rays that --dump-outputs writes: all of them up to DUMP_RAYS,
    else the same seeded sample of DUMP_RAYS rows on every run (ascending)."""
    if n <= DUMP_RAYS:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_RAYS, replace=False))


def dump_outputs(directory, rays, records):
    """DIR/<field>.npy for every field of the result records (float64; the integer fields
    are exact in it) and DIR/ray.npy, the index of each record's ray in the rank's fan of
    N_AZ x N_EL rays: the same numbering in both arms, whatever part of the fan they trace."""
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "ray.npy"), rays.astype(np.float64))
    for name in records.dtype.names:
        np.save(os.path.join(directory, name + ".npy"),
                np.ascontiguousarray(records[name], dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.2 and len(r) >= 7] or \
               [r for (_, r) in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower() == "active" for r in rows)]
        power = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]),
                "power_w_max": max(power) if power else None, "samples": len(rows),
                "reasons": reasons}


def reference_driver():
    """The reference CPU stepper (oracle/_ref when it was compiled, else the C port)
    behind the pthread ray loop of oracle/trace_driver.c, on the bench geometry."""
    from oracle import harness as H
    lib = H.best_oracle()
    d = H.Driver(lib)
    st = d.stack_create(stack_dir(), locked=True)  # mutex lock => one client per thread
    d.geometry([(H.ADD_STACK, st, 0.)], range=0., slope=0.4, resolution=1e-2)
    kind = "reference" if lib == H.REF else "port"
    return d, H, kind


def cpu_trace(d, H, rank, world, stride, n_total, cores):
    pos, _ = d.position([DET_LAT], [DET_LON], [DET_HEIGHT], 0)
    dirs = fan_subsample(rank, world, stride, n_total)
    res, steps, seconds = d.trace(np.repeat(pos, len(dirs), 0), dirs,
                                  H.rule(ALTITUDE_MAX, max_steps=MAX_STEPS), threads=cores)
    return res, steps, seconds, len(dirs)


def run_reference(args):
    """--impl reference: the reference's CPU path, all host cores, bounded sample/step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    make_stack()
    d, H, kind = reference_driver()
    cores = os.cpu_count() or 1
    n_total = args.rays
    stride = max(1, n_total // args.ref_rays)
    for _ in range(max(args.warmup, 0)):
        cpu_trace(d, H, 0, args.gpus, stride * 8, n_total, cores)
    t_all, rays_all, steps_all = 0., 0, 0
    for _ in range(args.steps):
        res, steps, seconds, n = cpu_trace(d, H, 0, args.gpus, stride, n_total, cores)
        t_all += seconds
        rays_all += n
        steps_all += steps
    if args.dump_outputs:
        rows = dump_sample(len(res))
        dump_outputs(args.dump_outputs, rows * stride, res[rows])
    value = rays_all / t_all / 1e6
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "ns_per_step": 1e9 * t_all / max(steps_all, 1),
        "config": workload_config(n_total, args.gpus),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": kind,
                         "sample": "every %d-th ray of the fan (%d rays per step), "
                                   "one stepper + client per pthread" % (stride, rays_all // args.steps)},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def workload_config(n_rays, gpus):
    return {"workload": "C2: %d-ray muography fan per GPU (4096 az x 4096 el, el 0.5-30 deg, "
                        "lowest elevations first in 32-ray azimuth bundles) from "
                        "(46.5N, 3.5E)+1 m through a synthetic SRTMGL1-shaped 3x3 stack of "
                        "3601x3601 int16 tiles (233 MB), geodetic, range 0, slope 0.4, "
                        "resolution 1e-2; stop: leaves stack | alt > 9000 m | 1e5 steps" % n_rays,
            "rays_per_gpu": n_rays, "parallelism": "rays sharded x%d, DEM replicated" % gpus,
            "l2": "inputs + outputs per step (%.0f MB per GPU) exceed the 126 MB L2; "
                  "no explicit flush" % (n_rays * BYTES_PER_RAY / 1e6)}


def kernel_profile(name):
    """The committed ncu measurement of a kernel (profiles/r02_kernels.json, written by
    tools/kernel_profiles.py from the .ncu-rep captures): executed FP64-pipe lane slots
    per sample and DRAM bytes of the captured launch. Refused -- so that a stale number
    cannot be reported silently -- when the registers per thread of the built kernel are
    not the ones of the capture."""
    path = os.path.join(ROOT, "profiles", "r02_kernels.json")
    if not os.path.exists(path):
        return None, "profiles/r02_kernels.json is missing"
    entry = json.load(open(path)).get(name)
    if entry is None:
        return None, "no entry `%s' in profiles/r02_kernels.json" % name
    import turtle_b200 as tb
    info = tb.kernel_info(entry["role"])
    if info is None or info[0] != entry["registers"]:
        return None, "profile `%s' is stale: captured at %s registers, the built %s has %s" % (
            name, entry["registers"], entry["role"], info[0] if info else None)
    return entry, "profiles/%s" % entry.get("source", "r02_kernels.json")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rays", type=int, default=N_AZ * N_EL, help="rays per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-rays", type=int, default=1 << 20,
                    help="rays per step of the --impl reference arm")
    ap.add_argument("--cpu-rays", type=int, default=1 << 22,
                    help="rays of the cpu_baseline sample (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result records of the last one "
                         "(rank 0's rays, at most %d of them: a fixed seeded sample) as "
                         "DIR/<field>.npy in float64, and DIR/ray.npy: the index of each "
                         "ray in the fan" % DUMP_RAYS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps

    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import turtle_b200 as tb
    synth = _synth()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if tb.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: turtle_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout: keep stdout to the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/turtle_b200_nccl.%h.%p.log")
        dist.init_process_group("nccl", device_id=dev)

    # ---- geometry: rank 0 writes the tiles once, every rank freezes its own copy ------
    if rank == 0:
        make_stack()
    if world > 1:
        dist.barrier()
    stack = tb.Stack(stack_dir())
    stepper = tb.Stepper(range=0., slope=0.4, resolution=1e-2)
    stepper.add_stack(stack, 0.)
    plan = stepper.freeze(local)
    plan.launch_set(args.ctas_per_sm, args.threads)
    rule = tb.trace_rule(ALTITUDE_MAX, max_steps=MAX_STEPS)

    # ---- rays of this rank (pinned host copies for the full-record e2e leg) --------------
    n = args.rays
    full = n == N_AZ * N_EL
    lat, lon, dirs = fan(rank, world, 0, n) if full else (
        DET_LAT, DET_LON, fan_subsample(rank, world, (N_AZ * N_EL) // n, N_AZ * N_EL)[:n])
    origin, data_index = stepper.position(lat, lon, DET_HEIGHT, 0)
    assert data_index == 0
    h_pos = torch.empty((n, 3), dtype=torch.float64, pin_memory=True)
    h_dir = torch.empty((n, 3), dtype=torch.float64, pin_memory=True)
    h_pos.numpy()[:] = origin[None, :]
    h_dir.numpy()[:] = dirs
    del dirs
    h_res = torch.empty((n, 96), dtype=torch.uint8, pin_memory=True)
    d_pos = h_pos.to(dev)
    d_dir = h_dir.to(dev)
    d_res = torch.empty((n, 96), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    # N > 1: the records of every rank land in rank 0's memory. The trace kernel of rank r
    # stores them there itself, over NVLink, as its rays end (turtle_b200.dist.PeerRecords:
    # rank 0's array mapped into every process by CUDA IPC): no gather after the kernel.
    # Should the GPUs not reach each other, fall back to an NCCL gather of the records.
    peer, gathered, exchange = None, None, "none (1 GPU)"
    if world > 1:
        from turtle_b200.dist import PeerRecords
        ok = torch.ones(1, device=dev)
        try:
            peer = PeerRecords([n] * world, dst=0)
        except Exception as err:  # noqa: BLE001 -- reported, then the gather path is used
            sys.stderr.write("rank %d: peer mapping failed (%s)\n" % (rank, err))
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() > 0:
            exchange = "peer stores from the trace kernel into rank 0's HBM (CUDA IPC over NVLink)"
        else:
            peer = None
            exchange = "NCCL gather of the records on rank 0 after the kernel"
            gathered = [torch.empty((n, 96), dtype=torch.uint8, device=dev)
                        for _ in range(world)] if rank == 0 else None
    out_ptr = peer.view if peer is not None else d_res

    def step_device():
        plan.trace_device(n, d_pos, d_dir, rule, out_ptr, stream=stream.cuda_stream)
        if world > 1 and peer is None:
            dist.gather(d_res, gathered, dst=0)

    def timed(fn, steps):
        """EXACTLY `steps` calls bracketed by barrier + synchronize, max over ranks."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t1 = time.time()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), t0, t1

    def timed_host(fn, steps):
        """Host-pointer calls return when their results are in place: wall clock around
        EXACTLY `steps` calls, barrier + synchronize on both sides, max over ranks."""
        fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        w = torch.tensor([time.perf_counter() - w0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(w, op=dist.ReduceOp.MAX)
        return float(w.item())

    # ---- device-resident throughput ------------------------------------------------------
    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    if peer is not None:  # mark every slot unwritten (status -1) before the timed steps
        peer.ready()
        if rank == 0:
            peer.tensor.fill_(0xff)
            torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    ms_total, t0, t1 = timed(step_device, args.steps)
    clocks = sampler.stop(t0, t1) if sampler else None
    counters = plan.counters(sync=True)  # of the last launch
    launches = args.steps
    ms_step = ms_total / args.steps
    value = world * n / (ms_step * 1e-3) / 1e6
    if peer is not None and rank == 0:
        # every rank's records are in rank 0's array: none of the slots is left unwritten
        status = peer.tensor.view(world, n, 96)[:, :, 76:80].contiguous().view(torch.int32)
        assert int((status < 0).sum().item()) == 0 and int((status > 4).sum().item()) == 0
        d_res.copy_(peer.tensor[:n])
    if args.dump_outputs and rank == 0:
        rows = dump_sample(n)
        picked = d_res.index_select(0, torch.from_numpy(rows).to(dev)).cpu().numpy()
        rays = rows if full else rows * ((N_AZ * N_EL) // n)
        dump_outputs(args.dump_outputs, rays, picked.view(tb.TRACE_RESULT).reshape(len(rows)))

    # kernel alone (no gather), CUDA events on the launching stream: the roofline input
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    k0.record(stream)
    for _ in range(args.steps):
        plan.trace_device(n, d_pos, d_dir, rule, d_res, stream=stream.cuda_stream)
    k1.record(stream)
    torch.cuda.synchronize()
    kernel_ms = k0.elapsed_time(k1) / args.steps
    launches += args.steps
    rank_ms = torch.tensor([kernel_ms], device=dev, dtype=torch.float64)
    all_ms = [torch.zeros_like(rank_ms) for _ in range(world)]
    if world > 1:
        dist.all_gather(all_ms, rank_ms)
    else:
        all_ms = [rank_ms]
    per_rank_kernel_ms = [round(float(t.item()), 3) for t in all_ms]

    # ---- strong scaling: the SAME 16 Mi-ray fan split over the ranks ---------------------
    # (rank r takes azimuths r, r + N, ... of the 4096: 1 / N of the rays each; what limits
    # it is the lone-lane tail of a launch, which does not shrink with the ray count)
    strong = None
    if full:
        az_all, el_all = fan_tables(synth, 0, 1)
        az_mine = np.ascontiguousarray(az_all[rank::world])
        m = len(az_mine) * len(el_all)
        fan_s = tb.Plan.make_fan(DET_LAT, DET_LON, origin, az_mine, el_all, bundle=32)
        d_len = torch.empty(m, dtype=torch.float64, device=dev)

        def step_strong():
            plan.trace_fan_device(fan_s, rule, fields=dict(length0=d_len),
                                  stream=stream.cuda_stream)
        for _ in range(2):
            step_strong()
        ms_s, _, _ = timed(step_strong, args.steps)
        launches += 2 + args.steps
        strong = {"rays_total": world * m, "rays_per_gpu": m, "ms_per_step": ms_s / args.steps,
                  "Mrays_per_s": world * m / (ms_s / args.steps) / 1e3,
                  "note": "one 4096 x 4096 fan over all ranks, device-resident, rock length "
                          "per ray kept on each rank"}

    # ---- end to end, the caller of examples/example-stepper.c batched ----------------------
    # turtle_stepper_trace_fan: the station and the two tables of angles go in (pinned host
    # memory), rock length + stop status + step count come back (pinned host memory), every
    # step. No per-ray input exists for this caller: the directions ARE the two tables.
    e2e, e2e_full = None, None
    if not args.no_e2e:
        az_t, el_t = fan_tables(synth, rank, world)
        if not full:  # reduced runs: the lowest elevation bands of the same fan
            el_t = np.ascontiguousarray(el_t[:max(32, (n // len(az_t)) // 32 * 32)])
        h_az = torch.from_numpy(az_t).pin_memory()
        h_el = torch.from_numpy(el_t).pin_memory()
        n_fan = len(az_t) * len(el_t)
        fan_h = tb.Plan.make_fan(DET_LAT, DET_LON, origin, h_az.numpy(), h_el.numpy(), bundle=32)
        h_len = torch.empty(n_fan, dtype=torch.float64, pin_memory=True)
        h_status = torch.empty(n_fan, dtype=torch.int32, pin_memory=True)
        h_steps = torch.empty(n_fan, dtype=torch.int32, pin_memory=True)
        out = dict(length0=h_len.numpy(), status=h_status.numpy(), n_steps=h_steps.numpy())

        def step_fan():
            plan.trace_fan(fan_h, rule, fields=out)
        w = timed_host(step_fan, args.steps)
        hc = plan.counters()
        launches += hc["launches"] * (args.steps + 1)
        e2e = {"value": world * n_fan * args.steps / w / 1e6, "unit": "Mrays/s",
               "h2d_bytes_per_step": int(16 * (len(az_t) + len(el_t)) + 8),
               "d2h_bytes_per_step": int(n_fan * 16), "ms_per_step": 1e3 * w / args.steps,
               "rays_per_gpu": n_fan, "kernel_ms_per_step": hc["kernel_ms"],
               "launches_per_step": hc["launches"],
               "api": "turtle_stepper_trace_fan: pinned host tables of %d azimuths + %d "
                      "elevations in, rock length (8 B) + status (4 B) + step count (4 B) per "
                      "ray out to pinned host memory; up to 8 resident slices on two streams, the "
                      "copy of a slice under the kernel of the next" % (len(az_t), len(el_t))}
        # the compact path against the full records of the same fan traced on the device
        d_chk = torch.empty((n_fan, 96), dtype=torch.uint8, device=dev)
        plan.trace_fan_device(fan_h, rule, results=d_chk, stream=stream.cuda_stream)
        torch.cuda.synchronize()
        chk = d_chk.cpu().numpy().view(tb.TRACE_RESULT).reshape(n_fan)
        e2e["matches_device_records"] = bool(
            np.array_equal(chk["length"][:, 0], out["length0"]) and
            np.array_equal(chk["status"], out["status"]) and
            np.array_equal(chk["n_steps"], out["n_steps"]))
        del d_chk, chk

        # ---- ... and with arbitrary rays in, full records out (48 B + 96 B per ray) --------
        res_np = h_res.numpy().view(tb.TRACE_RESULT).reshape(n)

        def step_host():
            plan.trace(h_pos.numpy(), h_dir.numpy(), rule, results=res_np)
        w = timed_host(step_host, args.steps)
        hc = plan.counters()
        launches += hc["launches"] * (args.steps + 1)
        e2e_full = {"value": world * n * args.steps / w / 1e6, "unit": "Mrays/s",
                    "h2d_bytes_per_step": int(n * 48), "d2h_bytes_per_step": int(n * 96),
                    "ms_per_step": 1e3 * w / args.steps, "kernel_ms_per_step": hc["kernel_ms"],
                    "launches_per_step": hc["launches"],
                    "api": "turtle_stepper_trace_batch (pinned host buffers; one persistent "
                           "kernel streamed by the copy engines in 256 Ki-ray pieces)"}
        # the two paths must agree bit for bit
        e2e_full["matches_device_path"] = bool(
            (torch.from_numpy(h_res.numpy()) == d_res.cpu()).all())

    if peer is not None:  # collective: the peers unmap before rank 0 frees
        peer.close()
        peer = None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel ------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak, hbm_src = 6650.0, "fallback"
    if os.path.exists(peaks_path):
        hbm_peak, hbm_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured"
    dfma = tb.dfma_peak(3)  # G FP64-pipe instructions / s, measured now on this GPU
    samples, steps = counters["samples"], counters["steps"]
    prof, prof_src = kernel_profile("c2_trace_stack")
    ops = prof["fp64_lane_slots_per_sample"] if prof else None
    achieved_ops = ops * samples / (kernel_ms * 1e-3) / 1e12 if prof else None
    alg_bytes = n * BYTES_PER_RAY + samples * BYTES_PER_SAMPLE
    regs = tb.kernel_info("trace_stack")
    roofline = {
        "kernel": "trace_kernel<LLA=0, PROJ=0, MINB=6, SHAPE_STACK>", "bound": "fp64",
        "achieved": achieved_ops, "peak": dfma / 1e3, "unit": "Tinst/s (FP64 pipe; FMA = 1)",
        "frac": achieved_ops / (dfma / 1e3) if (prof and dfma > 0) else None,
        "peak_source": "turtle_b200_dfma_peak() measured in this run (MEASURED_PEAKS.json has "
                       "no FP64 entry; nominal 148 SM x 64 / clk x 1.965 GHz = 18.6)",
        "ops_per_sample": ops, "samples_per_launch": samples,
        "ops_source": "executed FP64-pipe warp instructions x 32 / samples of the captured "
                      "launch (ncu --set full): " + prof_src,
        "issue_ceiling": prof.get("issue_ceiling") if prof else None,
        "kernel_registers": regs[0] if regs else None,
        "kernel_ms": kernel_ms,
        "traffic": prof["dram_bytes"] * (n / prof["rays"]) if prof and prof.get("rays") else None,
        "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of the captured launch "
                          "(scaled by rays when the capture was smaller): " + prof_src,
        "hbm": {"achieved": alg_bytes / (kernel_ms * 1e-3) / 1e9, "peak": hbm_peak,
                "unit": "GB/s", "frac": alg_bytes / (kernel_ms * 1e-3) / 1e9 / hbm_peak,
                "algorithmic_bytes": alg_bytes, "peak_source": hbm_src},
    }

    # ---- the reference's CPU path on this box, bounded sample; parity of the same rays -------
    cpu = None
    if args.cpu_rays > 0:
        from oracle import parity as P
        d, H, kind = reference_driver()
        cores = os.cpu_count() or 1
        stride = max(1, (N_AZ * N_EL) // args.cpu_rays)
        ref, ref_steps, seconds, m = cpu_trace(d, H, 0, world, stride, N_AZ * N_EL, cores)
        cpu = {"value": m / seconds / 1e6, "unit": "Mrays/s", "cores": cores, "kind": kind,
               "ns_per_step": 1e9 * seconds / max(ref_steps, 1), "seconds": seconds,
               "sample": "every %d-th ray of the rank-0 fan (%d rays)" % (stride, m)}
        if full:  # parity of the same rays: every field, next to the rounding-noise floor
            got = d_res.cpu().numpy().view(tb.TRACE_RESULT).reshape(n)[::stride]
            rep = P.report(ref, got)
            floor = None
            if H.available(H.REF_FMA) and kind == "reference":
                f = H.Driver(H.REF_FMA)
                st = f.stack_create(stack_dir(), locked=True)
                f.geometry([(H.ADD_STACK, st, 0.)], range=0., slope=0.4, resolution=1e-2)
                fma, _, _, _ = cpu_trace(f, H, 0, world, stride, N_AZ * N_EL, cores)
                floor = P.report(ref, fma)
            cpu["parity"] = {"gpu_vs_reference": rep, "reference_vs_reference_fma": floor,
                             "violations": P.against_floor(rep, floor) if floor else None,
                             "protocol": "oracle/parity.py: located = ends on a bisected "
                                         "boundary, held to 1 mm / 1e-9; threshold = stopped "
                                         "by the altitude rule, held to the FMA noise floor"}
            sys.stderr.write(P.table(rep, floor) + "\n")

    line = {
        "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(n, world), "exchange": exchange,
        "ns_per_step": kernel_ms * 1e6 / max(steps, 1),
        "steps_per_ray": steps / n, "samples_per_step": samples / max(steps, 1),
        "per_rank_kernel_ms": per_rank_kernel_ms,
        "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e,
        "e2e_full_records": e2e_full, "strong_scaling": strong, "roofline": roofline,
        "cpu_baseline": cpu, "plan_bytes": plan.bytes,
    }
    sys.stdout.flush()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
