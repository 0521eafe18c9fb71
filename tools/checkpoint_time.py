#!/usr/bin/env python3
"""Checkpoints of a device run, timed: SnakeGame.state_dict / load_state_dict at 65,536 and 2^20 envs, ReplayBuffer
state_dict / load_state_dict of a full 50,000-record ring, the two validation kernels alone (k_env_validate,
k_replay_validate: device time from a torch.profiler run of the loads), and Trainer.save / Trainer.load at 65,536 envs.
Save and load times are host wall clock around calls that end in a synchronise, median of the repetitions.  Prints one JSON
object naming the card and its power limit, and writes it to the path given.

    python tools/checkpoint_time.py [out.json]
"""
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g  # noqa: E402

S = g.load_package()
dev = torch.device("cuda", 0)


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], text=True).strip()
        return dict(zip(q.split(","), [v.strip() for v in line.split(",")]))
    except (OSError, subprocess.CalledProcessError):
        return {"name": torch.cuda.get_device_name(0), "power.limit": "unknown"}


def wall_ms(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return round(statistics.median(ts), 3)


def kernel_us(fn, name, reps):
    """device time per call of the kernels whose name contains `name`, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = sum((getattr(ev, "self_device_time_total", 0) or getattr(ev, "device_time_total", 0))
              for ev in prof.key_averages() if ev.device_type.name == "CUDA" and name in ev.key)
    return round(tot / reps, 2)


def play(env, steps):
    q = torch.rand(env.n, 3, device=dev)
    out = env.alloc_outputs(obs="f32", ep_stats=True, act=True, compressible=False)
    for _ in range(steps):
        env.step_fused(q=q, eps=0.3, out=out)


def env_case(n):
    env, twin = S.SnakeGame(n), S.SnakeGame(n)
    play(env, 50)
    d = env.state_dict()
    return {"envs": n, "blob_bytes": d["blob"].numel(),
            "save_ms": wall_ms(env.state_dict, 10), "load_ms": wall_ms(lambda: twin.load_state_dict(d), 10),
            "k_env_validate_us": kernel_us(lambda: twin.load_state_dict(d), "k_env_validate", 10)}


def ring_case():
    env = S.SnakeGame(65536)
    rb, rb2 = S.ReplayBuffer(50000, 0), S.ReplayBuffer(50000, 0)
    env.step_fused(q=torch.rand(65536, 3, device=dev), eps=0.3, obs=None, replay=rb)
    d = rb.state_dict()
    assert len(rb) == 50000
    return {"records": len(rb), "blob_bytes": d["blob"].numel(),
            "save_ms": wall_ms(rb.state_dict, 10), "load_ms": wall_ms(lambda: rb2.load_state_dict(d), 10),
            "k_replay_validate_us": kernel_us(lambda: rb2.load_state_dict(d), "k_replay_validate", 10)}


def trainer_case():
    tr = S.train.Trainer(n_envs=65536, fill=50000, target_sync=7, seed=1)
    tr.fill_buffer()
    for _ in range(20):
        tr.iteration()
    torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "run.pt")
        save = wall_ms(lambda: tr.save(path), 3)
        size = os.path.getsize(path)
        load = wall_ms(lambda: S.train.Trainer.load(path), 3)
    return {"envs": 65536, "file_bytes": size, "save_ms": save, "load_ms": load}


def main():
    res = {"card": card(), "env": [env_case(65536), env_case(1 << 20)], "ring": ring_case(), "trainer": trainer_case()}
    res["card_after"] = card()
    txt = json.dumps(res, indent=1)
    print(txt)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
