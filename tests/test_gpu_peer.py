"""GPU: delivery of the result records into ONE rank's memory by the trace kernels of all
ranks (turtle_b200.dist.PeerRecords, turtle_b200_peer_* in the C ABI).

World size 1 exercises the allocation / raw-pointer path on any GPU box; world size 2
(skipped with fewer than 2 GPUs) runs one process per GPU over NCCL: each rank traces
its shard straight into rank 0's array over NVLink and rank 0 compares the whole array,
byte for byte, with a single-GPU trace of all the rays."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import turtle_b200 as tb
from oracle import harness as H
from tests.common import Scene
from turtle_b200 import synth
from turtle_b200.dist import PeerRecords, shard_bounds

pytestmark = pytest.mark.gpu


def _plan_and_rays(stack_dir, n, device):
    sc = Scene(stacks=[stack_dir], ops=[(H.ADD_STACK, 0, 0.)], range=0.)
    stepper, maps, stacks = sc.product()
    plan = stepper.freeze(device)
    origin, _ = stepper.position(45.4, 2.6, 1.0, 0)
    dirs = synth.fan_directions(45.4, 2.6, 512, 512)[:n]
    pos = np.repeat(origin[None], n, 0)
    return (stepper, maps, stacks), plan, pos, dirs


def test_peer_records_world1(small_stack):
    n = 20000 + 5
    keep, plan, pos, dirs = _plan_and_rays(small_stack, n, 0)
    rule = tb.trace_rule(6000., max_steps=20000)
    want = plan.trace(pos, dirs, rule)
    torch.cuda.set_device(0)
    peer = PeerRecords([n])
    assert peer.first == 0 and peer.tensor.shape == (n, 96)
    peer.tensor.fill_(0xff)
    plan.trace_device(n, torch.from_numpy(pos).cuda(), torch.from_numpy(dirs).cuda(), rule,
                      peer.view)
    peer.ready()
    assert peer.tensor.cpu().numpy().tobytes() == want.tobytes()
    peer.close()


def _worker(rank, size, port, stack_dir, n, out_path):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=size,
                            device_id=torch.device("cuda", rank))
    keep, plan, pos, dirs = _plan_and_rays(stack_dir, n, rank)
    bounds = [shard_bounds(n, r, size) for r in range(size)]
    first, last = bounds[rank]
    peer = PeerRecords([b - a for a, b in bounds], dst=0)
    assert peer.first == first
    if rank == 0:
        peer.tensor.fill_(0xff)
    peer.ready()
    rule = tb.trace_rule(6000., max_steps=20000)
    d_pos = torch.from_numpy(pos[first:last]).cuda()
    d_dir = torch.from_numpy(dirs[first:last]).cuda()
    plan.trace_device(last - first, d_pos, d_dir, rule, peer.view)
    peer.ready()
    if rank == 0:
        np.save(out_path, peer.tensor.cpu().numpy())
    peer.close()
    dist.destroy_process_group()


def test_peer_records_world2(small_stack, tmp_path):
    if tb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    n = 60000 + 3
    out = str(tmp_path / "peer.npy")
    mp.spawn(_worker, args=(2, 29731 + os.getpid() % 1000, small_stack, n, out), nprocs=2,
             join=True)
    keep, plan, pos, dirs = _plan_and_rays(small_stack, n, 0)
    want = plan.trace(pos, dirs, tb.trace_rule(6000., max_steps=20000))
    got = np.load(out)
    assert got.shape == (n, 96)
    assert got.tobytes() == want.tobytes()
