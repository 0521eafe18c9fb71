#!/usr/bin/env python3
"""The data-parallel learner across real GPUs (one process per GPU, under torchrun): every rank brings its own seeded
minibatch (rank r: 40 + 23 r transitions of its own rollout) and runs 5 updates through a DistributedLearnerGroup.  Rank 0
gathers the minibatches, re-runs them concatenated in rank order with QNet.train_step on its GPU, and compares the bits of
every update's loss and g and of the final θ and RMSProp state; θ must also be equal on every rank.  Prints one JSON line.

    python -m torch.distributed.run --nproc-per-node 2 tools/dp_learner_check.py
"""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as graft  # noqa: E402

UPDATES = 5


def transitions(S, dev, B, seed):
    """B transitions out of a replay ring filled by a seeded rollout, with their masked targets"""
    env = S.SnakeGame(512, device=dev.index, auto_reset=True, seed=seed)
    ring = S.ReplayBuffer(capacity=512 * 8, device=dev.index, batch_size=B, seed=seed)
    net = S.qnet.QNet(S.qnet.glorot_layers(seed), dev)
    ro = S.rollout.Rollout(env, net, net, ring, epsilon=0.5)
    for _ in range(8):
        ro.step()
    b = ring.sample()
    b["targets"] = S.masked_target(net(b["next_states"]), b["mask"], b["rewards"], b["dones"])
    return b


def same(x, y):
    return x.shape == y.shape and torch.equal(x.reshape(-1).view(torch.uint8), y.reshape(-1).view(torch.uint8))


def main():
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    S = graft.load_package()
    layers = S.qnet.glorot_layers(7)
    b = transitions(S, dev, 40 + 23 * rank, 100 + rank)
    net = S.qnet.QNet(layers, dev)
    group = S.qnet.DistributedLearnerGroup(net)
    opt = S.qnet.RMSProp()
    res = []
    for _ in range(UPDATES):
        loss, g = group.train_step(b["states"], b["actions"], b["targets"], opt, want_grad=True)
        res.append((loss.cpu(), g.cpu()))
    torch.cuda.synchronize(dev)
    group.check()
    mine = {k: b[k].cpu() for k in ("states", "actions", "targets")}
    mine.update(theta=net.theta_device.cpu(), acc=opt.acc.cpu(), res=res)
    every = [None] * world
    dist.all_gather_object(every, mine)
    if rank == 0:
        ref = S.qnet.QNet(layers, dev)
        opt_ref = S.qnet.RMSProp()
        cat = {k: torch.cat([e[k] for e in every]).to(dev).contiguous() for k in ("states", "actions", "targets")}
        ok = True
        for k in range(UPDATES):
            loss, g = ref.train_step(cat["states"], cat["actions"], cat["targets"], opt_ref, want_grad=True)
            ok &= all(same(e["res"][k][0], loss.cpu()) and same(e["res"][k][1], g.cpu()) for e in every)
        ok &= all(same(e["theta"], ref.theta_device.cpu()) and same(e["acc"], opt_ref.acc.cpu()) for e in every)
        print(json.dumps({"world": world, "updates": UPDATES, "B_per_rank": [int(e["actions"].numel()) for e in every],
                          "same_bits_as_one_gpu": bool(ok),
                          "theta_equal_on_all_ranks": all(same(e["theta"], every[0]["theta"]) for e in every)}))
    dist.barrier()                       # nobody still reads a peer's published sums
    group.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
