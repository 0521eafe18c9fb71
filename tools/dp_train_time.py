#!/usr/bin/env python3
"""The data-parallel learner, timed (DESIGN §5f).  Run under torchrun with one process per GPU of the box:

    python -m torch.distributed.run --nproc-per-node <GPUs> tools/dp_train_time.py [out.json]

For every R in 1, 2, 4, 8 that fits the box, the first R ranks form a LearnerGroup and time its update at a global minibatch
of B = 64, 1,024 and 6,250 transitions split evenly over the R ranks (CUDA events on each rank's stream around `reps`
updates; the slowest rank is reported).  Rank 0 times the plain QNet.train_step at the same B in the same run.  Then every
rank runs a Trainer(world = all ranks) at 65,536 envs per GPU and the iteration time is taken on the host around a device
synchronise.  Rank 0 prints one JSON object with the card's name and power limit; an R larger than the box is reported as
not measured.
"""
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as graft  # noqa: E402

S = graft.load_package()
BATCHES = (64, 1024, 6250)
REPS = {64: 100, 1024: 20, 6250: 10}


def card(dev):
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        line = subprocess.check_output(["nvidia-smi", "-i", str(dev.index), "--query-gpu=" + q, "--format=csv,noheader"],
                                       text=True).strip()
        return dict(zip(q.split(","), [v.strip() for v in line.split(",")]))
    except (OSError, subprocess.CalledProcessError):
        return {"name": torch.cuda.get_device_name(dev), "power.limit": "unknown"}


def minibatch(ring, net, B):
    b = ring.stack_exp(ring.sample_indices(B))
    b["targets"] = S.masked_target(net(b["next_states"]), b["mask"], b["rewards"], b["dones"])
    return b


def events_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    env = S.SnakeGame(16384, device=dev.index, auto_reset=True, seed=42 + rank)
    ring = S.ReplayBuffer(capacity=50000, device=dev.index, seed=rank)
    net0 = S.qnet.QNet(S.qnet.glorot_layers(0), dev)
    ro = S.rollout.Rollout(env, net0, net0, ring, epsilon=0.3)
    for _ in range(4):
        ro.step()
    res = {"world": world, "card": card(dev), "group_update_ms": {}, "train_step_ms": {}}
    for R in (1, 2, 4, 8):
        sub = dist.new_group(list(range(R))) if R <= world else None
        if R > world:
            res["group_update_ms"][str(R)] = "not measured: the box has %d GPUs" % world
            continue
        if rank >= R:
            continue
        row = {}
        for B in BATCHES:
            Br = B // R + (1 if rank < B % R else 0)
            net = S.qnet.QNet(S.qnet.glorot_layers(0), dev)
            group = S.qnet.DistributedLearnerGroup(net, group=sub)
            opt = S.qnet.RMSProp()
            b = minibatch(ring, net, Br)
            dist.barrier(group=sub)
            ms = events_ms(lambda: group.train_step(b["states"], b["actions"], b["targets"], opt), REPS[B])
            group.check()
            every = [None] * R
            dist.all_gather_object(every, ms, group=sub)
            row[str(B)] = round(max(every), 4)
            dist.barrier(group=sub)
            group.close()
        res["group_update_ms"][str(R)] = row
    if rank == 0:
        for B in BATCHES:
            net = S.qnet.QNet(S.qnet.glorot_layers(0), dev)
            opt = S.qnet.RMSProp()
            b = minibatch(ring, net, B)
            res["train_step_ms"][str(B)] = round(events_ms(lambda: net.train_step(b["states"], b["actions"], b["targets"], opt),
                                                           REPS[B]), 4)
    dist.barrier()
    # the Trainer iteration at 65,536 envs per GPU, all ranks in one group
    tr = S.train.Trainer(n_envs=65536, device=dev.index, fill=65536, world=world, rank=rank)
    if world > 1:
        handles = [None] * world
        dist.all_gather_object(handles, tr.handle())
        tr.connect(handles)
    tr.fill_buffer()
    for _ in range(3):
        tr.iteration()
    torch.cuda.synchronize(dev)
    dist.barrier()
    iters = 50
    t0 = time.perf_counter()
    for _ in range(iters):
        tr.iteration()
    torch.cuda.synchronize(dev)
    ms = 1e3 * (time.perf_counter() - t0) / iters
    every = [None] * world
    dist.all_gather_object(every, ms)
    res["trainer_iteration_ms"] = {"n_envs_per_gpu": 65536, "batch_size_per_gpu": tr.replay.batch_size, "world": world,
                                   "per_rank": [round(v, 4) for v in every]}
    res["card_after"] = card(dev)
    if rank == 0:
        print(json.dumps(res))
        if len(sys.argv) > 1:
            with open(sys.argv[1], "w") as f:
                f.write(json.dumps(res, indent=1) + "\n")
    dist.barrier()
    if tr.learner is not None:
        tr.learner.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
