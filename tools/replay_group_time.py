#!/usr/bin/env python3
"""The replay group, timed (DESIGN §5g).

    python tools/replay_group_time.py [out.json]                                       one GPU: 1, 2 and 4 virtual ranks
    python -m torch.distributed.run --nproc-per-node <GPUs> tools/replay_group_time.py [out.json]   one rank per GPU

Every rank holds a full 50,000-record ring (a seeded rollout of 16,384 games, four steps, so the ring has wrapped).  At a share
of B_r = 64, 1,024 and 6,250 transitions per rank, CUDA events time `reps` calls of ReplayGroup.sample() against
ReplayBuffer.sample() of B_r transitions on one ring in the same run.  With virtual ranks every rank is driven from its own
stream of ONE GPU: those figures time the flag hand-overs between streams of one device and R gathers on one device, not
NVLink.  Under torchrun each rank times its own stream and the slowest rank is reported; run as one process, the multi-GPU
figures are reported as not measured.  Run as one process, the Trainer iteration at 65,536 envs (world 1) is also timed with and
without shared_replay, alternating, on the host around a device synchronise.  The card's name and power limit are read in the
same run.
"""
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as graft  # noqa: E402

S = graft.load_package()
SHARES = (64, 1024, 6250)
REPS = {64: 200, 1024: 100, 6250: 40}


def card(dev):
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        line = subprocess.check_output(["nvidia-smi", "-i", str(dev.index), "--query-gpu=" + q, "--format=csv,noheader"],
                                       text=True).strip()
        return dict(zip(q.split(","), [v.strip() for v in line.split(",")]))
    except (OSError, subprocess.CalledProcessError):
        return {"name": torch.cuda.get_device_name(dev), "power.limit": "unknown"}


def full_ring(dev, seed, batch_size=64):
    env = S.SnakeGame(16384, device=dev.index, auto_reset=True, seed=42 + seed)
    ring = S.ReplayBuffer(capacity=50000, device=dev.index, batch_size=batch_size, seed=seed)
    net = S.qnet.QNet(S.qnet.glorot_layers(0), dev)
    ro = S.rollout.Rollout(env, net, net, ring, epsilon=0.3)
    for _ in range(4):
        ro.step()
    torch.cuda.synchronize(dev)
    return ring


def events_ms(fn, reps, warm=5):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def trainer_iteration_ms(shared, iters=50):
    tr = S.train.Trainer(n_envs=65536, device=0, fill=65536, shared_replay=shared)
    tr.fill_buffer()
    for _ in range(3):
        tr.iteration()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        tr.iteration()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0) / iters


def single_process():
    dev = torch.device("cuda", 0)
    res = {"card": card(dev), "ring_capacity": 50000, "replay_buffer_sample_ms": {}, "virtual_ranks_sample_ms": {},
           "note": "virtual ranks: R groups on ONE GPU, each on its own stream; the time of one call of every rank, enqueued "
                   "together. This times flag hand-overs between streams of one device, not NVLink.",
           "real_gpus_sample_ms": "not measured: run as one process on a box with %d GPU(s)" % torch.cuda.device_count()}
    rings = [full_ring(dev, r) for r in range(4)]
    for B in SHARES:
        rb = rings[0]
        rb.batch_size = B
        res["replay_buffer_sample_ms"][str(B)] = round(events_ms(rb.sample, REPS[B]), 4)
    for R in (1, 2, 4):
        row = {}
        for B in SHARES:
            g = S.LocalReplayGroup(rings[:R], [B] * R, 5)
            row[str(B)] = round(events_ms(g.sample, REPS[B]), 4)
            g.check()
            g.close()
        res["virtual_ranks_sample_ms"][str(R)] = row
    del rings
    it = {"n_envs": 65536, "batch_size": 64, "world": 1, "plain": [], "shared_replay": []}
    for _ in range(2):
        it["plain"].append(round(trainer_iteration_ms(False), 4))
        it["shared_replay"].append(round(trainer_iteration_ms(True), 4))
    res["trainer_iteration_ms"] = it
    res["card_after"] = card(dev)
    return res


def distributed():
    import torch.distributed as dist
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    ring = full_ring(dev, rank)
    res = {"world": world, "card": card(dev), "ring_capacity": 50000, "real_gpus_sample_ms": {}}
    for B in SHARES:
        g = S.DistributedReplayGroup(ring, [B] * world, 5)
        dist.barrier()
        ms = events_ms(g.sample, REPS[B])
        g.check()
        every = [None] * world
        dist.all_gather_object(every, ms)
        res["real_gpus_sample_ms"][str(B)] = round(max(every), 4)
        dist.barrier()
        g.close()
    dist.destroy_process_group()
    return res if rank == 0 else None


def main():
    res = distributed() if "WORLD_SIZE" in os.environ else single_process()
    if res is not None:
        print(json.dumps(res))
        if len(sys.argv) > 1:
            with open(sys.argv[1], "w") as f:
                f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
