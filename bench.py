#!/usr/bin/env python3
"""bench.py — Snake env-steps/sec on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--envs E] [--dump-outputs DIR]

Workload (config.workload): BASELINE config 3 — E = 1,048,576 batched envs PER GPU (weak scaling: envs are
independent, each rank owns its own shard, no collective on the step path), every step = ONE fused kernel
doing epsilon-greedy selection (eps = 0.05, injected Q (3,E) f32 + u f32 + ridx u8) + step! + losing mask +
Float32 two-frame observation.  Inputs are synthetic, generated on the device before the timed region.
`value` times that kernel with everything resident in HBM; `e2e` times one iteration of a HOST trainer's data path
(utils.jl:436-443) through the host-buffer C-ABI entry points with pinned host tensors, H2D + D2H inside the timed region:
snk_step_fused_store_host (q, u, ridx up; lossless 2-bit packed next_state, reward, done, mask, action down; every transition
store!d into the device replay ring) + snk_replay_gather_host (stack_exp of 64 sampled transitions expanded to Float32 — where
the reference casts, utils.jl:361-362).  The full-Float32 and int8 observation forms of the same call are secondary keys.
`config2_4096_envs` reports BASELINE config 2 (4,096 envs, given actions) as a CUDA-graph of steps.

--impl reference: the reference's CPU implementation of the same path.  Julia is not in the image, so this is
the C restatement in oracle/ run in its reference-shaped mode (dense Int64 boards, a board copy per step,
three whole-game deep copies per step for the losing mask), all host threads, on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)

BYTES_PER_STEP_CONFIG3 = 876   # SURVEY.md §8(d): 50 state + 1 action + 4 reward + 1 done + 3 mask + 800 obs + 12 q + 4 u + 1 ridx
BYTES_PER_STEP_CONFIG2 = 859
REF_SAMPLE_ENVS = 32768        # env count of the CPU arm's bounded sample (independent of the host's thread count)
DUMP_MAX_ENVS = 65536          # --dump-outputs: 824 bytes of float32 per env
METRIC = "snake_env_steps_per_sec"
UNIT = "env-steps/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bf16_peak_tflops():
    """dense bf16 TFLOP/s of this pool's B200 (burst figure: the kernels it is used for are timed alone)"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return float(json.load(open(p))["bf16_tflops"]) if os.path.exists(p) else 1590.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_run(n_envs, n_steps, threads, keep_history=True, seed=42):
    """env-steps/s of the oracle (reference-shaped by default) over `threads` host threads."""
    from oracle import oracle_lib as O
    b = O.OracleBatch(n_envs, auto_reset=True, keep_history=keep_history)
    per = (n_envs + threads - 1) // threads
    ts = [threading.Thread(target=b.run_random, args=(i * per, min(n_envs, (i + 1) * per), n_steps, seed))
          for i in range(threads) if i * per < n_envs]
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    return n_envs * n_steps / dt, dt


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = host_threads()
    n_envs, n_steps = REF_SAMPLE_ENVS, 200                       # fixed sample: comparable across boxes
    cpu_reference_run(min(n_envs, 1024), 20, threads)            # warm the allocator / page in the library
    vals = []
    for _ in range(max(1, args.warmup)):
        cpu_reference_run(n_envs, 20, threads)
    t_all = 0.0
    for _ in range(max(1, args.steps)):
        v, dt = cpu_reference_run(n_envs, n_steps, threads)
        vals.append(v)
        t_all += dt
        if t_all > 120:
            break
    v = n_envs * n_steps * len(vals) / t_all
    sample = "%d envs x %d steps per bench step, uniform random actions, auto-reset, f32 obs + mask built per step" % (n_envs, n_steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
        "warmup": args.warmup, "ms_per_step": 1e3 * t_all / len(vals), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": "config3: batched envs, step! + losing mask + f32 two-frame obs per env-step (CPU arm: bounded sample)",
                   "envs_per_bench_step": n_envs, "steps_per_bench_step": n_steps, "host_threads": threads,
                   "differences_from_the_gpu_arm": ["%d envs instead of 1,048,576 per GPU (bounded sample)" % n_envs,
                                                    "given uniform random actions: no epsilon-greedy select from Q",
                                                    "reference-shaped oracle (keep_history: board copy per step, 3 whole-game deep copies per step)"]},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "note": "C restatement of the Julia reference (Julia is not installed); reference-shaped mode: "
                                 "Int64 boards, board copy per step, 3 whole-game deep copies per step"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    import __graft_entry__ as graft
    S = graft.load_package()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: keep this rank's pinned host buffers and copy threads on the GPU's own NUMA node
    affinity = {"bound": False, "reason": "--no-numa-bind"} if args.no_numa_bind else S.shard.bind_host_near_gpu(local)
    if world > 1:
        # NCCL prints its version banner to stdout from C when the communicator is created; stdout must carry only
        # the one JSON line, so fd 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier(device_ids=[local])
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    strong = args.total_envs > 0                             # BASELINE config 3 as literally stated: 1M envs env-sharded
    E = (args.total_envs + world - 1) // world if strong else args.envs
    K, W = args.steps, max(3, args.warmup)
    env = S.SnakeGame(E, device=local, auto_reset=True)      # adopts torch's current stream
    out = env.alloc_outputs(obs="f32", mask=True, act=True)
    # synthetic inputs: a ring of pre-generated draw sets (counter-seeded per rank), resident in HBM
    g = torch.Generator(device=dev)
    g.manual_seed(42 + rank)
    R = 4
    qs = [torch.rand(E, 3, device=dev, generator=g) * 2 - 1 for _ in range(R)]
    us = [torch.rand(E, device=dev, generator=g) for _ in range(R)]
    rs = [torch.randint(0, 3, (E,), device=dev, generator=g, dtype=torch.uint8) for _ in range(R)]
    eps = 0.05                                               # structs.jl:165 epsilon_end

    def one_step(i):
        j = i % R
        env.step_fused(q=qs[j], eps=eps, u=us[j], ridx=rs[j], out=out)

    # clocks are sampled from BEFORE the warm-up to the end of the timed region (a 20-step region lasts 3 ms, one
    # nvidia-smi period is 20 ms): the warm-up is preceded by extra untimed steps until the sampler has delivered.
    # Their number depends on how soon it delivers, so the envs restart from the initial state after them: with the same
    # arguments, every run's timed steps compute the same outputs from the same inputs.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    extra, t_w = 0, time.perf_counter()
    while rank == 0 and len(sampler.rows) < 8 and time.perf_counter() - t_w < 1.5 and sampler.proc is not None:
        for i in range(50):
            one_step(extra + i)
        torch.cuda.synchronize()
        extra += 50
    env.reset()
    for i in range(W):
        one_step(i)
    barrier()
    use_graph = E < 400_000       # a shard this small takes < 60 us per step: launch through a CUDA graph of R steps
    if not use_graph:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        ev[0].record()
        for i in range(K):
            one_step(W + i)
            ev[i + 1].record()
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        total_ms = ev[0].elapsed_time(ev[K])
        kern_ms = sum(ev[i].elapsed_time(ev[i + 1]) for i in range(K)) / K
    else:
        st = torch.cuda.Stream(dev)
        env.use_stream(st)
        with torch.cuda.stream(st):
            one_step(0)
            st.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=st):
                for i in range(R):
                    one_step(i)
            graph.replay()
            st.synchronize()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(K // R):
                graph.replay()
            for i in range(K % R):                       # EXACTLY K steps: the remainder as plain launches
                one_step(i)
            e1.record(st)
            st.synchronize()
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        total_ms = e0.elapsed_time(e1)
        kern_ms = total_ms / K
        env.use_stream(torch.cuda.current_stream(dev))
    total_ms = max_over_ranks(total_ms)
    kern_ms = max_over_ranks(kern_ms)
    value = world * E * K / (total_ms * 1e-3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    n_err = env.count_errors()

    # ---- the same fused step with the other observation formats (SURVEY 8(d): report all three byte counts)
    variants = {}
    if rank == 0 and not use_graph and not args.skip_variants:
        for name, fmt, nbytes in (("int8_obs", "i8", BYTES_PER_STEP_CONFIG3 - 800 + 200), ("bit_records", "bits", BYTES_PER_STEP_CONFIG3 - 800 + 24),
                                  ("no_obs", None, BYTES_PER_STEP_CONFIG3 - 800)):
            out_v = env.alloc_outputs(obs=fmt, mask=True)
            Kv = min(K, 400)
            for i in range(5):
                env.step_fused(q=qs[i % R], eps=eps, u=us[i % R], ridx=rs[i % R], out=out_v)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for i in range(Kv):
                env.step_fused(q=qs[i % R], eps=eps, u=us[i % R], ridx=rs[i % R], out=out_v)
            a1.record()
            torch.cuda.synchronize()
            ms_v = a0.elapsed_time(a1) / Kv
            variants[name] = {"value": E / (ms_v * 1e-3), "unit": UNIT, "ms_per_step": ms_v, "bytes_per_env_step": nbytes,
                              "hbm_frac": E * nbytes / (ms_v * 1e-3) / 1e9 / peaks()[0]}
            del out_v
        variants["note"] = ("single GPU, device-timed like `value`; int8 observations (the reference's game.state is an integer array), "
                            "24-byte bit records (SNK_OBS_BITS: the state as two bit-boards, no table expansion) and no observation at all "
                            "(reward / done / mask only): the smaller the output, the more the kernel is bound by its per-env arithmetic "
                            "and latency instead of HBM")

    # ---- e2e: one iteration of a host trainer's data path through the host-buffer C ABI, copies inside the timed region
    Ke = max(2, min(K, args.e2e_steps))
    ring = S.ReplayBuffer(capacity=50000, device=local, batch_size=64)
    host = {"q": S.pinned_empty((E, 3), torch.float32), "u": S.pinned_empty((E,), torch.float32),
            "ridx": S.pinned_empty((E,), torch.uint8), "act_idx": S.pinned_empty((E,), torch.uint8),
            "reward": S.pinned_empty((E,), torch.float32), "done": S.pinned_empty((E,), torch.uint8),
            "mask": S.pinned_empty((E, 3), torch.uint8)}
    host["q"].copy_(qs[0]); host["u"].copy_(us[0]); host["ridx"].copy_(rs[0])
    batch_host = {"states": S.pinned_empty((64, 2, 10, 10), torch.float32), "next_states": S.pinned_empty((64, 2, 10, 10), torch.float32),
                  "actions": S.pinned_empty((64,), torch.uint8), "rewards": S.pinned_empty((64,), torch.float32),
                  "dones": S.pinned_empty((64,), torch.uint8), "mask": S.pinned_empty((64, 3), torch.uint8)}
    idx_rng = torch.Generator().manual_seed(7 + rank)

    def e2e_run(fmt, dtype, per_env, store):
        host["obs"] = S.pinned_empty((E, 2, 10, 10) if per_env == 200 else (E, per_env), dtype)
        host["obs_fmt"] = fmt
        # SNK_OBS_BITS carries reward / done / mask / action inside its 24-byte record: no separate output arrays
        h = {k: v for k, v in host.items() if k in ("q", "u", "ridx", "obs", "obs_fmt")} if fmt == "bits" else host

        def it():
            env.step_fused_host(h, q=True, eps=eps, replay=ring if store else None)
            if store:                                             # sample(rpb) + stack_exp (utils.jl:442-443): 64 transitions as Float32;
                idx = torch.randint(0, len(ring), (64,), generator=idx_rng, dtype=torch.int64)     # ordered behind the step's kernels,
                ring.stack_exp_host(idx, out=batch_host)                                          # beside its device->host copies
            env.sync()                                            # every output of the step is in host memory

        for _ in range(2):
            it()
        barrier()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(Ke):
            it()
        t1.record()
        env.sync()
        barrier()
        return max_over_ranks(t0.elapsed_time(t1))

    e2e_ms = e2e_run("bits", torch.uint8, 24, True)
    e2e_value = world * E * Ke / (e2e_ms * 1e-3)
    h2d = E * (12 + 4 + 1) + 64 * 8
    d2h = E * 24 + 64 * 1613
    e2e_f32_ms = e2e_i8_ms = e2e_p2_ms = None
    if not args.skip_variants:
        e2e_p2_ms = e2e_run("packed2", torch.uint8, 50, True)
        e2e_f32_ms = e2e_run("f32", torch.float32, 200, False)
        e2e_i8_ms = e2e_run("i8", torch.int8, 200, False)
    del host["obs"]
    ring.close()

    # ---- BASELINE config 2 (4,096 envs, given actions) as a CUDA graph of steps: launch-latency regime
    cfg2 = None
    if rank == 0 and not args.skip_config2:
        n2, T = 4096, 200
        env2 = S.SnakeGame(n2, device=local, auto_reset=True)
        out2 = env2.alloc_outputs(obs="f32", mask=True)
        acts = torch.randint(0, 3, (T, n2), device=dev, dtype=torch.uint8)
        st = torch.cuda.Stream(dev)
        env2.use_stream(st)
        with torch.cuda.stream(st):
            for t in range(3):
                env2.step_fused(act_idx=acts[t], out=out2)
            st.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=st):
                for t in range(T):
                    env2.step_fused(act_idx=acts[t], out=out2)
            for _ in range(3):
                graph.replay()
            st.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(st)
            reps = 10
            for _ in range(reps):
                graph.replay()
            a1.record(st)
            st.synchronize()
        ms2 = a0.elapsed_time(a1) / (reps * T)
        # the same T steps as ONE launch of the multi-step rollout kernel (env state stays in registers)
        ro = env2.rollout(acts, obs="f32", mask=True)
        st.synchronize(); torch.cuda.synchronize()
        with torch.cuda.stream(st):
            for _ in range(3):
                env2.rollout(acts, out=ro)
            st.synchronize()
            a0.record(st)
            for _ in range(reps):
                env2.rollout(acts, out=ro)
            a1.record(st)
            st.synchronize()
        ms3 = a0.elapsed_time(a1) / (reps * T)
        cfg2 = {"workload": "config2: 4,096 envs, given uniform random actions, f32 obs + mask, %d steps" % T,
                "value": n2 / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3,
                "hbm_frac": n2 * BYTES_PER_STEP_CONFIG2 / (ms3 * 1e-3) / 1e9 / peaks()[0],
                "api": "snk_rollout_fused: all %d steps in one launch, outputs for every step kept (%.0f MB)" % (T, T * n2 * 807 / 1e6),
                "per_step_launches_in_a_cuda_graph": {"value": n2 / (ms2 * 1e-3), "ms_per_step": ms2},
                "note": "3.5 MB per step: latency bound by construction, not an HBM-roofline case"}
        env2.close()

    # ---- BASELINE config 4: 65,536 envs acting from the Q-net, masked max-Q targets, 50k replay ring
    cfg4 = None
    if rank == 0 and not args.skip_config4:
        cfg4 = bench_config4(S, dev, local)

    # ---- BASELINE config 5a: Gram of the deviation matrix (K=1000 snapshots x P=181,395 weights), tcgen05
    gram = None
    if rank == 0 and not args.skip_gram:
        gram = bench_gram(S, dev, cpu_too=(world == 1 and not args.skip_cpu))

    # ---- BASELINE config 5b shape: row-sharded Gram across the ranks (6,250 rows of J per GPU, P = 181,395)
    gram_sh = None
    if world > 1 and not args.skip_gram:
        gram_sh = bench_gram_sharded(S, dev, rank, world, local, max_over_ranks, R=args.gram_rows)

    # ---- CPU baseline beside it (rank 0, N=1 only): bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        threads = host_threads()
        n_c = REF_SAMPLE_ENVS
        cpu_reference_run(1024, 20, threads)
        v_mt, dt_mt = cpu_reference_run(n_c, 200, threads)
        v_1t, dt_1t = cpu_reference_run(4096, 100, 1)
        cpu = {"value": v_mt, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "%d envs x 200 steps over %d threads (%.1f s); single thread: 4096 envs x 100 steps = %.3g env-steps/s (%.1f s)"
                         % (n_c, threads, dt_mt, v_1t, dt_1t),
               "single_thread_value": v_1t,
               "note": "C restatement of the Julia reference in reference-shaped mode (Julia is not installed on the box)"}

    if rank == 0:
        peak, peak_src = peaks()
        achieved = BYTES_PER_STEP_CONFIG3 * E / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "u64 bitboards -> f32 obs", "data": "synthetic",
            "config": {"workload": "config3: %d envs per GPU, eps-greedy(0.05) select from injected Q + step! + losing mask + f32 two-frame obs, one fused kernel per step" % E,
                       "envs_per_gpu": E, "global_envs": E * world, "parallelism": "env-sharded x%d, no collective" % world,
                       "launch": "CUDA graph of %d steps" % R if use_graph else "one launch per step",
                       "l2": "per-step working set %.2f GB per GPU > 126 MB L2 (no flush needed)" % (E * 930 / 1e9),
                       "env_errors": n_err},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src, "kernel": "k_step<F32,select>",
                         "bytes_per_env_step": BYTES_PER_STEP_CONFIG3, "kernel_ms": kern_ms},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": Ke, "ms_per_step": e2e_ms / Ke,
                    "api": "snk_step_fused_store_host (pinned host buffers: q/u/ridx up; one 24-byte record per env down = next_state as "
                           "two bit-boards + reward / done / next_is_suicidal / action, lossless; every transition store!d into the device "
                           "replay ring) + snk_sync + snk_replay_gather_host (stack_exp of 64 sampled transitions as Float32, "
                           "utils.jl:343-383) per step",
                    "obs_format": "bits (SNK_OBS_BITS, include/snake_b200.h; decoded by unpack_bits, bit-identical to the int8 state: "
                                  "tests/test_env_parity_gpu.py); Float32 only for the 64 sampled transitions, as the reference casts "
                                  "(utils.jl:361-362)",
                    "host_affinity_rank0": affinity},
            "gpu_launches": K * world,
            "clocks": clocks,
            "warmup_extra_untimed_steps": extra,
        }
        if e2e_p2_ms is not None:
            line["e2e"]["packed2_obs_variant"] = {"value": world * E * Ke / (e2e_p2_ms * 1e-3), "d2h_bytes_per_step": E * 59 + 64 * 1613,
                                                  "api": "the same call with 2-bit packed next_state (50 B/env) + separate reward / done / mask / "
                                                         "action arrays (the headline form earlier in round 2)"}
        if e2e_f32_ms is not None:
            line["e2e"]["full_f32_obs_variant"] = {"value": world * E * Ke / (e2e_f32_ms * 1e-3), "d2h_bytes_per_step": E * 809,
                                                   "api": "snk_step_fused_host, Float32 next_state for every env (round-1 headline form)"}
            line["e2e"]["int8_obs_variant"] = {"value": world * E * Ke / (e2e_i8_ms * 1e-3), "d2h_bytes_per_step": E * 209,
                                               "api": "snk_step_fused_host, int8 next_state for every env"}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if variants:
            line["obs_format_variants"] = variants
        if cfg2 is not None:
            line["config2_4096_envs"] = cfg2
        if cfg4 is not None:
            line["config4_65536_envs"] = cfg4
        if gram is not None:
            line["gram_5a"] = gram
        if gram_sh is not None:
            line["gram_5b_sharded"] = gram_sh
        line["roofline"]["traffic"] = ncu_traffic_bytes()
        print(json.dumps(line))
    env.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def dump_outputs(path, out, max_envs=DUMP_MAX_ENVS):
    """Writes what the last timed step returned to its caller as float32 `path`/<name>.npy: act_idx (E,), reward (E,),
    done (E,), mask (E, 3), obs (E, 2, 10, 10).  Above max_envs envs only a fixed seeded sample of envs is written, the
    same for every run with the same --envs; env_index.npy (float64) lists the envs written."""
    import numpy as np
    import torch
    E = out["reward"].numel()
    idx = np.arange(E) if E <= max_envs else np.sort(np.random.default_rng(0).choice(E, max_envs, replace=False))
    sel = torch.from_numpy(idx).to(out["reward"].device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))
    for name in ("act_idx", "reward", "done", "mask", "obs"):
        np.save(os.path.join(path, name + ".npy"), out[name].index_select(0, sel).float().cpu().numpy())


def bench_config4(S, dev, local, n=65536, steps=20):
    """One rollout step = q_net(state) -> fused eps-greedy/step!/virtual_step/obs/store! -> t_net(next_state) ->
    masked max-Q target (utils.jl:203-208, 448-451).  Q-net = seeded Glorot init of structs.jl:127-139 (the
    two-frame checkpoints BASELINE names are missing from the reference mount).  Native kernels in both precisions
    ("f32" = Float32-faithful, the like-for-like number; "bf16" = fast mode); the torch/cuDNN timings are LIBRARY baselines."""
    import torch
    from tools.torch_qnet import TorchQNet
    env = S.SnakeGame(n, device=local, auto_reset=True)
    rb = S.ReplayBuffer(capacity=50000, device=local)
    layers = S.qnet.glorot_layers(seed=0)
    out = {"workload": "config4: %d envs, eps=0.05, Glorot-init Q-net (synthetic weights), 50k replay ring" % n}
    peak = bf16_peak_tflops()
    nets = [("native_f32", S.qnet.QNet(layers, dev, "f32"), S.qnet.PRECISION_NOTES["f32"]),
            ("native_bf16", S.qnet.QNet(layers, dev, "bf16"), S.qnet.PRECISION_NOTES["bf16"])]
    if not os.environ.get("SNK_BENCH_SKIP_LIBRARY"):
        nets += [("library_cudnn_fp32", TorchQNet(layers, dev, dtype=torch.float32), "LIBRARY baseline: torch conv2d/linear, fp32 with TF32 off"),
                 ("library_cudnn_tf32", TorchQNet(layers, dev, dtype=torch.float32, allow_tf32=True), "LIBRARY baseline: torch default (TF32 convolutions)"),
                 ("library_cudnn_bf16", TorchQNet(layers, dev, dtype=torch.bfloat16, channels_last=True), "LIBRARY baseline: torch bf16 channels_last")]
    ref64 = TorchQNet(layers, dev, dtype=torch.float64)
    for name, qn, note in nets:
        ro = S.rollout.Rollout(env, qn, qn, rb, epsilon=0.05)
        for _ in range(3):
            ro.step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            ro.step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        x = ro.state                                              # the network forward alone
        for _ in range(2):
            qn(x)
        e0.record()
        for _ in range(steps):
            qn(x)
        e1.record()
        torch.cuda.synchronize()
        fwd = e0.elapsed_time(e1) / steps
        want = ref64(x[:4096].double())
        err = float(((qn(x[:4096]).double() - want).abs().max() / want.abs().max()).item())
        tflops = 4870784.0 * n / (fwd * 1e-3) / 1e12            # SURVEY 8(a) row Q: 4,870,784 FLOP per sample (useful)
        out[name] = {"env_steps_per_s": n / (ms * 1e-3), "ms_per_step": ms, "qnet_forward_ms": fwd, "qnet_useful_tflops": tflops,
                     "max_err_vs_float64_of_maxQ": err, "note": note}
        if name.startswith("native"):
            mma_x = 4.0 if name == "native_f32" else 1.0        # the split issues every MMA for (hi, lo) x (hi, lo)
            out[name]["roofline"] = {
                "bound": "tensor", "achieved": tflops, "peak": peak, "unit": "TFLOP/s", "frac": tflops / peak,
                "achieved_executed": tflops * mma_x, "frac_executed": tflops * mma_x / peak, "traffic": None,
                "note": "achieved = useful FLOP (4,870,784 per sample, SURVEY 8a row Q) / time of snk_qnet_forward; executed = the MMAs issued "
                        "(useful x %.0f); ncu tensor-pipe %% in profiles/r02_ncu_qnet_*.csv" % mma_x}
    out["like_for_like"] = "native_f32 (the reference network is Float32; bf16 and TF32 give different greedy actions)"
    out["replay_len"] = len(rb)
    env.close()
    rb.close()
    return out


def ncu_csv_traffic(pattern, kernel_prefix):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of kernels whose name starts with kernel_prefix, from the newest
    committed ncu --set full capture profiles/r??_<pattern>.csv (raw page export); (bytes, file) or (None, None)."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r??_" + pattern + ".csv")))
    for path in reversed(files):
        rows = list(csv.reader(open(path)))
        if not rows or "dram__bytes_read.sum" not in rows[0]:
            continue
        hdr, units = rows[0], rows[1]
        r, w = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        name_col = hdr.index("Kernel Name") if "Kernel Name" in hdr else 0
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        vals = [float(x[r]) * scale.get(units[r], 1e6) + float(x[w]) * scale.get(units[w], 1e6)
                for x in rows[2:] if len(x) > max(r, w) and kernel_prefix in x[name_col]]
        if vals:
            return sum(vals) / len(vals), os.path.relpath(path, ROOT)
    return None, None


def ncu_traffic_bytes():
    """per k_step launch, from the newest committed capture of this same workload (profiles/r??_ncu_k_step_full.csv)"""
    return ncu_csv_traffic("ncu_k_step_full", "k_step")[0]


def gram_block_flops(S, rows_a, rows_b, P, terms, symmetric):
    """what the tensor pipe executes for one block (the library's own tile plan: computed tiles, padded, x products)"""
    import ctypes as C
    v = C.c_double(0)
    S._check(S.lib().snk_gram_block_flops(int(rows_a), int(rows_b), int(P), int(terms), 1 if symmetric else 0, C.byref(v)))
    return v.value


def bench_gram_sharded(S, dev, rank, world, local, max_over_ranks, R=6250, P=181395, iters=3):
    """BASELINE config 5b: the Gram of per-sample gradients of the DQN loss over the replay buffer, row-sharded.
    Every rank fills its own device replay ring by acting with the Float32-faithful Q-net, draws R transitions, and
      timed: snk_qnet_sample_grads (rows of J straight into this rank's bf16 planes) + snk_gram_shard_run (planes ring over
             NVLink peer memory under the tcgen05 main loop, device-side barriers, peer-read mirror) -> G[rows_rank, :].
    Verified on EVERY rank against Float64 dot products of Float32 J rows (>= 1000 off-diagonal entries), and against the
    NCCL all-gather + all-to-all form of the same Gram (bit-identical)."""
    import torch
    import torch.distributed as dist
    from snake_b200 import gram_sharded as GS
    n_env = 16384
    env = S.SnakeGame(n_env, device=local, auto_reset=True)
    ring = S.ReplayBuffer(capacity=50000, device=local, seed=1000 + rank)
    q_net = S.qnet.QNet(S.qnet.glorot_layers(seed=0), dev, "f32")
    t_net = S.qnet.QNet(S.qnet.glorot_layers(seed=1), dev, "f32")
    ro = S.rollout.Rollout(env, q_net, t_net, ring, epsilon=0.3)
    g = torch.Generator(device=dev)
    g.manual_seed(100 + rank)
    for _ in range(30):                                          # 491,520 transitions through a 50,000-slot ring (mid-game boards)
        ro.step(u=torch.rand(n_env, device=dev, generator=g), ridx=torch.randint(0, 3, (n_env,), device=dev, generator=g, dtype=torch.uint8))
    batch = ring.stack_exp(ring.sample_indices(R))               # sample(rpb) + stack_exp, R distinct transitions
    y = S.masked_target(t_net(batch["next_states"]), batch["mask"], batch["rewards"], batch["dones"])
    dg = GS.DistributedGram([R] * world, P, dev)
    planes = dg.shard.planes()
    times, t_prod = [], []
    for it in range(iters + 1):
        torch.cuda.synchronize()
        dist.barrier(device_ids=[local])
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        q_net.sample_grads(batch["states"], batch["actions"], y, planes=planes, want_loss=False)
        e1.record()
        G = dg.run(None, terms=3)
        e2.record()
        torch.cuda.synchronize()
        t = max_over_ranks(e0.elapsed_time(e2))
        tp = max_over_ranks(e0.elapsed_time(e1))
        if it > 0:
            times.append(t)
            t_prod.append(tp)
    dg.shard.check()
    # ---- verification on every rank: 128 random local rows x (8 probe rows of every rank), Float64 dot products of FP32 J rows
    gi = torch.Generator(device="cpu").manual_seed(5 + rank)
    rows_i = torch.randperm(R, generator=gi)[:128].to(dev)
    sub = torch.cat([rows_i, torch.arange(8, device=dev)])
    Jsub = q_net.sample_grads(batch["states"][sub].contiguous(), batch["actions"][sub].contiguous(), y[sub].contiguous(),
                              want_J=True, want_loss=False)["J"]
    probes = [torch.empty(8, P, dtype=torch.float32, device=dev) for _ in range(world)]
    dist.all_gather(probes, Jsub[128:].contiguous())
    Jp = torch.cat(probes, 0).double()                           # (8 world, P): rows 0..7 of every rank
    want = Jsub[:128].double() @ Jp.T                            # (128, 8 world)
    cols = torch.tensor([r * R + k for r in range(world) for k in range(8)], device=dev)
    got = G[rows_i][:, cols].double()
    offdiag = (rows_i[:, None] + rank * R) != cols[None, :]
    scale = torch.sqrt(torch.diagonal(Jsub[:128].double() @ Jsub[:128].double().T))[:, None] * torch.sqrt((Jp * Jp).sum(1))[None, :]
    err = float(((got - want).abs() / scale)[offdiag].max().item())
    errs = [None] * world
    dist.all_gather_object(errs, err)
    fingerprints = [None] * world                                # the ranks hold DIFFERENT transitions: norm of each rank's first J row
    dist.all_gather_object(fingerprints, float(Jsub[0].double().norm().item()))
    n_checked = int(offdiag.sum().item())
    Gring = G.clone()
    dg.close()
    # ---- baseline: the same block Grams behind library collectives (NCCL all-gather of the planes, all-to-all of the blocks to mirror)
    J = q_net.sample_grads(batch["states"], batch["actions"], y, want_J=True, want_loss=False)["J"]
    ag = GS.AllGatherGram([R] * world, P, dev)
    times_ag = []
    for it in range(iters + 1):
        torch.cuda.synchronize()
        dist.barrier(device_ids=[local])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        Ga = ag.run(J, terms=3)
        e1.record()
        torch.cuda.synchronize()
        t = max_over_ranks(e0.elapsed_time(e1))
        if it > 0:
            times_ag.append(t)
    same = bool(torch.equal(Ga, Gring))
    ag.close()
    del J
    env.close()
    ring.close()
    ms = sorted(times)[len(times) // 2]
    ms_prod = sorted(t_prod)[len(t_prod) // 2]
    Kt = R * world
    useful = 2.0 * Kt * Kt * P
    executed = 0.0                                               # what the busiest rank's tensor pipe executes: its blocks' computed tiles x 3 products
    for r in range(world):
        tot = 0.0
        for i, (_, a0, a1, b0, b1) in enumerate(GS.ring_schedule([R] * world, r)):
            if a1 > a0 and b1 > b0:
                tot += gram_block_flops(S, a1 - a0, b1 - b0, P, 3, i == 0)
        executed = max(executed, tot)
    gram_s = (ms - ms_prod) * 1e-3
    mma = executed / gram_s / 1e12
    alg = float(Kt) * (Kt + 1) * P / world / gram_s / 1e12       # SURVEY 8(d): a symmetric-half implementation reports M(M+1)P
    peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained", 1421.8)) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1421.8
    return {"workload": "config5b: Gram of per-sample DQN-loss gradients J (%d transitions per GPU out of each rank's 50,000-slot replay ring "
                        "x %d parameters), row-sharded over %d GPUs, hi/lo bf16 split" % (R, P, world),
            "data": "real J: rollout with the Float32-faithful Q-net (Glorot-init synthetic weights) -> replay ring -> sample -> "
                    "masked max-Q targets -> per-sample gradients",
            "K_total": Kt, "ms": ms, "producer_ms": ms_prod, "gram_ms": ms - ms_prod,
            "useful_tflops_total": useful / gram_s / 1e12, "mma_tflops_per_gpu": mma,
            "roofline": {"bound": "tensor", "achieved": alg, "peak": peak, "unit": "TFLOP/s", "frac": alg / peak,
                         "achieved_executed": mma, "frac_executed": mma / peak, "executed_over_algorithmic": executed / (useful / world), "traffic": None,
                         "note": "per GPU, Gram phase only; peak = sustained bf16 (a %.0f ms region); achieved = SURVEY 8(d)'s count for a symmetric-half "
                                 "implementation, K(K+1)P / GPUs / time (useful_tflops_total keeps the full-square 2 K^2 P of the earlier lines); "
                                 "executed = the tiles the busiest rank computes (own block: upper-triangle tiles; half the ring) x 3 products of the "
                                 "hi/lo split, padding included" % ms},
            "verify_per_rank": {"entries_per_rank": n_checked, "max_err_over_sqrt_GiiGjj": errs, "first_checked_row_norm_per_rank": fingerprints,
                                "how": "128 random local rows x rows 0..7 of every rank (off-diagonal), Float64 dot products of FP32 J rows"},
            "nccl_allgather_baseline_ms": sorted(times_ag)[len(times_ag) // 2], "nccl_allgather_same_bits_rank0": same,
            "exchange": "snk_gram_shard_run: cudaMemcpyAsync from peer-mapped (cudaIpc) memory on a copy stream under the MMA main loop; "
                        "device-side barriers over peer memory; transpose exchange by peer loads inside the mirror kernel; "
                        "torch.distributed only carries the IPC handles at set-up",
            "timed": "per-sample gradients into the planes + one snk_gram_shard_run per rank; buffers and IPC mappings set up once"}


def bench_gram(S, dev, K=1000, P=181395, iters=10, cpu_too=False):
    """G = A A^T for A = D^T (K x P), synthetic N(0,1) snapshots cast through Float32 (the reference stores
    Float64.(theta::Float32)); L2 flushed between timed iterations; accuracy against torch Float64."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    A = torch.randn(K, P, device=dev, dtype=torch.float32, generator=g).double()
    ref = A @ A.T
    plan = S.GramPlan(K, P, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    peak = bf16_peak_tflops()
    out = {"workload": "config5a: Gram G = D'D of K=%d snapshots x P=%d weights (compute_D.jl D, plot_traj.jl spectrum)" % (K, P),
           "flop_useful": 2.0 * K * K * P, "peak_bf16_tflops_burst": peak}

    def timed(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2]

    out["pack_ms"] = timed(lambda: plan.pack(A))
    out["pack_hbm_frac"] = 12.0 * K * P / (out["pack_ms"] * 1e-3) / 1e9 / peaks()[0]
    A32 = A.float()
    out["pack_f32_ms"] = timed(lambda: plan.pack(A32))
    out["pack_f32_hbm_frac"] = 8.0 * K * P / (out["pack_f32_ms"] * 1e-3) / 1e9 / peaks()[0]
    plan.pack(A)
    Dc = A.clone()
    out["center_ms"] = timed(lambda: S.center_columns(Dc))       # Welford + centring of the Float64 D (3 passes over 1.45 GB)
    out["center_hbm_frac"] = 3 * 8.0 * K * P / (out["center_ms"] * 1e-3) / 1e9 / peaks()[0]
    del Dc
    G = torch.empty(K, K, dtype=torch.float32, device=dev)
    for terms in (3, 1):
        ms = timed(lambda: plan.gram(terms, 0, out=G))
        err = float((G.double() - ref).norm() / ref.norm())
        mma = gram_block_flops(S, K, K, P, terms, True) / (ms * 1e-3) / 1e12
        useful = 2.0 * K * K * P / (ms * 1e-3) / 1e12            # full-square equivalent (what the earlier rounds' lines called useful)
        alg = float(K) * (K + 1) * P / (ms * 1e-3) / 1e12        # SURVEY 8(d): a symmetric-half implementation reports K(K+1)P
        traffic, src = ncu_csv_traffic("ncu_gram_5a_terms%d_full" % terms, "k_gram")
        out["terms%d" % terms] = {"ms": ms, "useful_tflops": useful, "mma_tflops": mma,
                                  "frac_of_measured_bf16_peak": mma / peak, "rel_fro_err_vs_fp64": err,
                                  "roofline": {"bound": "tensor", "achieved": alg, "peak": peak, "unit": "TFLOP/s",
                                               "frac": alg / peak, "achieved_executed": mma, "frac_executed": mma / peak, "traffic": traffic,
                                               "algorithmic_bytes": (2 if terms == 3 else 1) * 2.0 * K * ((P + 63) // 64 * 64),
                                               "traffic_source": src,
                                               "note": "achieved = SURVEY 8(d)'s count for a symmetric-half implementation, K(K+1)P / time (useful_tflops keeps the "
                                                       "full-square 2 K^2 P); executed = the tiles actually computed (upper-triangle tiles of the "
                                                       "padded problem) x products per k-step (3 for the hi/lo split); time covers the tile kernel + the "
                                                       "split-K/mirror pass; traffic = ncu dram bytes of the tile kernel actually run, algorithmic_bytes = the "
                                                       "bf16 planes read once"}}
    Ab = A.to(torch.bfloat16)
    ms = timed(lambda: torch.matmul(Ab, Ab.T))
    out["cublas_bf16_same_shape_ms"] = ms
    if cpu_too:
        # BASELINE.md section 3: the reference-sized Gram in Float64 on the host cores (what LinearAlgebra/OpenBLAS does for the
        # reference's svd(D) path); one run, ~2-10 s
        Ah = A.cpu()
        t0 = time.perf_counter()
        Gh = Ah @ Ah.T
        dt = time.perf_counter() - t0
        out["cpu_fp64_baseline"] = {"ms": 1e3 * dt, "gflops": 2.0 * K * K * P / dt / 1e9, "cores": torch.get_num_threads(),
                                    "kind": "library (torch CPU matmul, Float64)",
                                    "rel_fro_err_of_gpu_split_vs_this": float(((plan.gram(3, 0).cpu().double() - Gh).norm() / Gh.norm()).item())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU (weak scaling)")
    ap.add_argument("--total-envs", type=int, default=0, help="strong scaling: this many envs in total, sharded over the ranks")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the CPUs next to its GPU")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-config2", action="store_true")
    ap.add_argument("--skip-gram", action="store_true")
    ap.add_argument("--gram-rows", type=int, default=6250, help="rows of J per GPU in the row-sharded Gram (config 5b: 6,250)")
    ap.add_argument("--skip-config4", action="store_true")
    ap.add_argument("--skip-variants", action="store_true", help="skip the int8-observation / no-observation timings")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32, at most %d envs: "
                         "about 54 MB)" % DUMP_MAX_ENVS)
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
