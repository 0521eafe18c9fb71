#!/usr/bin/env python3
"""The learner on the device, timed: snk_qnet_train_step at B = 64 and B = 6,250 split into the gradient kernel
(k_sample_grads), the reduce + RMSProp + repack kernel (k_qnet_train_apply) and the host wait of the next forward (conv1's
weights are kernel parameters, so that forward waits for the update's copy of them); one Trainer iteration at 4,096 and 65,536
envs; and torch (tools/torch_qnet.py + autograd + torch.optim.RMSprop(lr=5e-4, alpha=0.9, eps=1e-8), the same formula in
Float32) on the same GPU.  Prints one JSON object naming the card and its power limit.

    python tools/train_time.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g  # noqa: E402
from tools.torch_qnet import TorchQNet  # noqa: E402

S = g.load_package()
dev = torch.device("cuda", 0)


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm,clocks_event_reasons.sw_power_cap,clocks_event_reasons.hw_slowdown"
    try:
        line = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], text=True).strip()
        return dict(zip(q.split(","), [v.strip() for v in line.split(",")]))
    except (OSError, subprocess.CalledProcessError):
        return {"name": torch.cuda.get_device_name(0), "power.limit": "unknown"}


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


def kernel_us(fn, reps):
    """per-call device time of each kernel / copy fn launches, from torch.profiler (a separate, profiled run)"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count:
            key = "k_sample_grads" if "k_sample_grads" in ev.key else "k_qnet_train_apply" if "k_qnet_train_apply" in ev.key \
                else "memcpy_dtoh" if "DtoH" in ev.key or "Device -> Pageable" in ev.key or "Device -> Pinned" in ev.key else ev.key
            out[key] = out.get(key, 0.0) + (getattr(ev, "self_device_time_total", 0) or getattr(ev, "device_time_total", 0)) / reps
    return {k: round(v, 2) for k, v in out.items()}


def minibatch(ring, net, B):
    b = ring.stack_exp(ring.sample_indices(B))
    b["targets"] = S.masked_target(net(b["next_states"]), b["mask"], b["rewards"], b["dones"])
    return b


def learner(ring, B, reps):
    net = S.qnet.QNet(S.qnet.glorot_layers(0), dev, "f32")
    opt = S.qnet.RMSProp()
    b = minibatch(ring, net, B)
    step = lambda: net.train_step(b["states"], b["actions"], b["targets"], opt)
    res = {"B": B, "train_step_ms": round(events_ms(step, reps), 4), "kernels_us_per_step": kernel_us(step, reps)}
    # host wait: how long a forward right after an update blocks the host (it waits for the update to finish on the device),
    # against the same forward with nothing pending
    obs = b["states"][:64].contiguous()
    waits, plain = [], []
    for _ in range(reps):
        torch.cuda.synchronize()
        step()
        t0 = time.perf_counter()
        net(obs)
        waits.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        net(obs)
        plain.append(time.perf_counter() - t0)
    waits.sort(), plain.sort()
    res["forward_after_update_host_us_median"] = round(1e6 * waits[len(waits) // 2], 1)
    res["forward_no_update_host_us_median"] = round(1e6 * plain[len(plain) // 2], 1)
    # an update and one acting forward in a loop, as the Trainer runs them: the host waits every time
    res["train_step_plus_forward_loop_ms"] = round(events_ms(lambda: (step(), net(obs)), reps), 4)
    return res


def torch_baseline(ring, B, reps):
    layers = S.qnet.glorot_layers(0)
    tq = TorchQNet(layers, dev, dtype=torch.float32)
    params = []
    for p in tq.params:
        p[1].requires_grad_()
        p[2].requires_grad_()
        params += [p[1], p[2]]
    opt = torch.optim.RMSprop(params, lr=5e-4, alpha=0.9, eps=1e-8)
    net = S.qnet.QNet(layers, dev, "f32")
    b = minibatch(ring, net, B)
    a = b["actions"].long()[:, None]
    y = b["targets"].float()

    def step():
        opt.zero_grad(set_to_none=True)
        q = tq(b["states"]).gather(1, a)[:, 0]
        F.huber_loss(q, y, delta=1.0).backward()
        opt.step()
    return {"B": B, "torch_fp32_autograd_rmsprop_ms": round(events_ms(step, reps), 4)}


def trainer_iteration(n_envs, iters):
    tr = S.train.Trainer(n_envs=n_envs, seed=0)
    tr.fill_buffer()
    for _ in range(3):
        tr.iteration()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        tr.iteration()
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / iters
    return {"n_envs": n_envs, "updates_per_step": tr.updates_per_step, "iteration_ms": round(ms, 4),
            "env_steps_per_s": round(n_envs / (ms * 1e-3), 1), "final_loss": float(tr.losses[-1])}


def main():
    info = card()
    env = S.SnakeGame(16384, auto_reset=True)
    ring = S.ReplayBuffer(capacity=50000)
    net = S.qnet.QNet(S.qnet.glorot_layers(0), dev, "f32")
    ro = S.rollout.Rollout(env, net, net, ring, epsilon=0.3)
    for _ in range(4):
        ro.step()
    res = {"card": info, "learner": [learner(ring, 64, 200), learner(ring, 6250, 10)],
           "torch": [torch_baseline(ring, 64, 200), torch_baseline(ring, 6250, 10)],
           "trainer": [trainer_iteration(4096, 200), trainer_iteration(65536, 50)]}
    info2 = card()
    res["card_after"] = {k: info2.get(k) for k in ("clocks.sm", "clocks_event_reasons.sw_power_cap", "clocks_event_reasons.hw_slowdown")}
    line = json.dumps(res)
    print(line)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
