#!/usr/bin/env python3
"""train! (utils.jl:420-494) on the device: fill the replay ring, then play, sample 64, target, RMSProp update, target sync
every 1,000 updates, epsilon decay — train.Trainer over the library.  Prints the loss and the moving average of the
episode returns every --report updates.  Needs a B200.

One play advances every one of --envs games by one step (the reference plays one whole episode of one game per update);
--updates-per-step sets how many updates follow each play.  --save PATH writes a checkpoint at the end (save_trainer,
utils.jl:408-412); --resume PATH continues a saved run bit for bit (load_trainer, utils.jl:413-418) up to --batches updates in all.

Started under torchrun (one process per GPU: python -m torch.distributed.run --nproc-per-node 8 examples/dqn_train.py) it
trains one Q-net data-parallel (DESIGN §5f): every rank plays its own --envs games into its own replay ring and samples 64
transitions from it, and every update is the update of all ranks' minibatches together.  With --shared-replay the ranks'
minibatches are instead drawn together, uniformly without replacement from the union of all rings (DESIGN §5g), as the
reference samples its one buffer.  Rank 0 reports; --save and --resume take one file per rank (PATH.rank<r>).
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as graft  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--batches", type=int, default=20000, help="updates in all (the reference's n_batches)")
    ap.add_argument("--updates-per-step", type=int, default=1)
    ap.add_argument("--precision", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--report", type=int, default=1000)
    ap.add_argument("--window", type=int, default=1000, help="episodes in the moving average of the returns")
    ap.add_argument("--capacity", type=int, default=50000, help="replay ring capacity per rank (the reference's 50,000)")
    ap.add_argument("--shared-replay", action="store_true",
                    help="under torchrun: draw each update's minibatch uniformly from the union of every rank's ring instead of "
                         "64 from each rank's own; with R ranks, --capacity C/R per rank keeps the reference's C transitions in "
                         "the union")
    ap.add_argument("--save", metavar="PATH", help="write a checkpoint of the run here at the end")
    ap.add_argument("--resume", metavar="PATH", help="continue the run saved here (its --envs, --capacity, --precision and --shared-replay are the checkpoint's)")
    args = ap.parse_args()
    S = graft.load_package()
    world, rank, dev = 1, 0, 0
    if "WORLD_SIZE" in os.environ:                       # torchrun: one rank per GPU
        import torch.distributed as dist
        dist.init_process_group("gloo")
        world, rank, dev = dist.get_world_size(), dist.get_rank(), int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(dev)
    suffix = ".rank%d" % rank if world > 1 else ""
    say = print if rank == 0 else (lambda *a: None)
    if args.resume:
        tr = S.train.Trainer.load(args.resume + suffix, device=dev, world=world, rank=rank)
        say("resumed %s: %d updates, %d transitions stored" % (args.resume, tr.n_updates, tr.stored))
    else:
        tr = S.train.Trainer(n_envs=args.envs, device=dev, precision=args.precision, capacity=args.capacity,
                             updates_per_step=args.updates_per_step, world=world, rank=rank, shared_replay=args.shared_replay)
    if world > 1:
        handles = [None] * world
        dist.all_gather_object(handles, tr.handle())
        tr.connect(handles)
    tr.fill_buffer()
    say("filled: %d transitions stored, replay %d/%d (per rank, %d ranks)" % (tr.stored, len(tr.replay), tr.replay.capacity, world)
        if world > 1 else "filled: %d transitions stored, replay %d/%d" % (tr.stored, len(tr.replay), tr.replay.capacity))
    while tr.n_updates < args.batches:
        tr.iteration()
        if tr.n_updates % args.report < args.updates_per_step:
            rets = tr.episode_returns()
            avg = float(rets[-args.window:].mean()) if rets.numel() else float("nan")
            loss = float(torch.stack(tr.losses[-args.report:]).mean())
            say("batch %7d  loss %.5f  episodes %8d  avg return (last %d) %.3f  epsilon %.4f"
                  % (tr.n_updates, loss, rets.numel(), args.window, avg, tr.epsilon))
    say("env errors %d" % tr.env.count_errors())
    if args.save:
        tr.save(args.save + suffix)
        say("saved %s" % (args.save + suffix))
    if world > 1:
        dist.barrier()                                   # no rank still waits on a peer's published sums or reads its ring
        tr.learner.check()
        if tr.sampler is not None:
            tr.sampler.check()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
