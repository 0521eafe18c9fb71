#!/usr/bin/env python3
"""A/B of k_step<F32, SELECT> at 2^20 envs writing its outputs into plain device memory (torch.empty) or into memory with
generic L2 compression (SnakeGame.alloc_outputs(compressible=True): snk_device_alloc, cuMemCreate with
CU_MEM_ALLOCATION_COMP_GENERIC).

  python tools/compress_ab.py [--envs E] [--pairs P] [--steps K] [--warmup W]

The inputs are bench.py's (q, u, ridx ring of 4 draw sets seeded 42, eps = 0.05).  Every run restarts the envs from the
initial state, so all runs compute the same outputs; the outputs of each plain / compressible pair are compared bit for bit.
The runs alternate plain, compressible, plain, ... so that drift of the machine shows up in both arms.  One line per run
and a JSON summary (median and range of each arm) on stdout.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import __graft_entry__ as graft  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    S = graft.load_package()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    E = args.envs
    env = S.SnakeGame(E, device=0, auto_reset=True)
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    R = 4
    qs = [torch.rand(E, 3, device=dev, generator=g) * 2 - 1 for _ in range(R)]
    us = [torch.rand(E, device=dev, generator=g) for _ in range(R)]
    rs = [torch.randint(0, 3, (E,), device=dev, generator=g, dtype=torch.uint8) for _ in range(R)]

    plain = env.alloc_outputs(obs="f32", mask=True, act=True, compressible=False)
    compressed = env.alloc_outputs(obs="f32", mask=True, act=True, compressible=True)
    all_comp = all(S.is_compressible(v) for v in compressed.values() if torch.is_tensor(v))
    print("compressible allocations:", all_comp, file=sys.stderr)

    def run(out):
        env.reset()
        for i in range(args.warmup):
            env.step_fused(q=qs[i % R], eps=0.05, u=us[i % R], ridx=rs[i % R], out=out)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            j = (args.warmup + i) % R
            env.step_fused(q=qs[j], eps=0.05, u=us[j], ridx=rs[j], out=out)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / args.steps

    res = {"plain": [], "compressible": []}
    identical = True
    for p in range(args.pairs):
        for name, out in (("plain", plain), ("compressible", compressed)):
            us_step = run(out)
            res[name].append(us_step)
            print("pair %d %-12s %.2f us/step  %.4g env-steps/s" % (p, name, us_step, E / (us_step * 1e-6)), file=sys.stderr)
        same = all(torch.equal(plain[k].view(torch.uint8), compressed[k].view(torch.uint8))
                   for k, v in plain.items() if torch.is_tensor(v))
        identical &= same
        print("pair %d outputs bit-identical: %s" % (p, same), file=sys.stderr)
    med = {k: statistics.median(v) for k, v in res.items()}
    summary = {"envs": E, "steps": args.steps, "pairs": args.pairs, "device": torch.cuda.get_device_name(dev),
               "us_per_step": res, "median_us": med, "speedup": med["plain"] / med["compressible"],
               "ranges_overlap": max(res["compressible"]) >= min(res["plain"]),
               "all_compressible": all_comp, "outputs_bit_identical": identical}
    print(json.dumps(summary))
    env.close()
    return 0 if identical else 1


if __name__ == "__main__":
    sys.exit(main())
