#!/usr/bin/env python3
"""The replay group across real GPUs (one process per GPU, under torchrun): every rank fills its own ring from a seeded rollout
(rank r: capacity 3,000 + 500 r, 512 + 256 r games, so the rings differ in size and fill), connects a DistributedReplayGroup
through connect_host and draws 5 union minibatches with uneven shares (rank r: 40 + 23 r transitions).  Rank 0 gathers every
ring's checkpoint blob and every rank's outputs, builds ONE full ring of the concatenated records with the group's seed and draw
counter, and compares the bits of its sample_indices + stack_exp with the ranks' outputs concatenated in rank order.  Prints
one JSON line.

    python -m torch.distributed.run --nproc-per-node 2 tools/replay_group_check.py
"""
import json
import os
import struct
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as graft  # noqa: E402

CALLS = 5
SEED = 11
KEYS = ("idx", "states", "next_states", "actions", "rewards", "dones", "mask", "ep_return", "score")


def same(x, y):
    return x.shape == y.shape and torch.equal(x.reshape(-1).view(torch.uint8), y.reshape(-1).view(torch.uint8))


def main():
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    S = graft.load_package()
    n_envs = 512 + 256 * rank
    env = S.SnakeGame(n_envs, device=dev.index, auto_reset=True, seed=200 + rank)
    ring = S.ReplayBuffer(capacity=3000 + 500 * rank, device=dev.index, seed=rank)
    net = S.qnet.QNet(S.qnet.glorot_layers(rank), dev)
    ro = S.rollout.Rollout(env, net, net, ring, epsilon=0.5)
    for _ in range(5):
        ro.step()
    batch_all = [40 + 23 * q for q in range(world)]
    group = S.DistributedReplayGroup(ring, batch_all, SEED)
    outs = []
    for _ in range(CALLS):
        o = group.sample(want_idx=True, ep_stats=True)
        outs.append({k: o[k].cpu() for k in KEYS})
    torch.cuda.synchronize(dev)
    group.check()
    every = [None] * world
    dist.all_gather_object(every, {"blob": ring.state_dict()["blob"], "outs": outs})
    if rank == 0:
        recs = b"".join(e["blob"].numpy().tobytes()[40:] for e in every)
        n = len(recs) // 128
        ok = True
        for c in range(CALLS):
            blob = torch.frombuffer(bytearray(b"snk-rpl\0" + struct.pack("<IIqqQ", 1, 128, n, n, c) + recs), dtype=torch.uint8)
            ref = S.ReplayBuffer(n, dev.index, sum(batch_all), SEED)
            ref.load_state_dict({"blob": blob, "seed": SEED, "batch_size": sum(batch_all)})
            idx = ref.sample_indices()
            want = ref.stack_exp(idx, ep_stats=True)
            want["idx"] = idx
            for k in KEYS:
                ok &= same(torch.cat([e["outs"][c][k] for e in every]), want[k].cpu())
        print(json.dumps({"world": world, "calls": CALLS, "batch_all": batch_all, "union": n, "same_bits_as_one_ring": bool(ok)}))
    dist.barrier()                       # nobody still reads a peer's ring
    group.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
