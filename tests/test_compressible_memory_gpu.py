"""Outputs of the fused step in device memory with generic L2 compression (alloc_outputs(compressible=True), the default):
the same bytes as in torch.empty buffers, ordinary torch tensors, and memory that is given back when they die."""
import ctypes

import pytest
import torch

from tests.util import pkg

pytestmark = pytest.mark.gpu

FORMATS = ("f32", "i8", "i64", "packed2", "bits", None)


@pytest.fixture(scope="module")
def S():
    S = pkg()
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return S


def bench_inputs(E, dev, R=4):
    """bench.py's synthetic inputs: a ring of R (q, u, ridx) draw sets seeded 42"""
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    qs = [torch.rand(E, 3, device=dev, generator=g) * 2 - 1 for _ in range(R)]
    us = [torch.rand(E, device=dev, generator=g) for _ in range(R)]
    rs = [torch.randint(0, 3, (E,), device=dev, generator=g, dtype=torch.uint8) for _ in range(R)]
    return qs, us, rs


def tensors(out):
    return {k: v for k, v in out.items() if torch.is_tensor(v)}


def assert_same_bytes(a, b, what):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, (what, k)
        assert torch.equal(a[k].reshape(-1).view(torch.uint8), b[k].reshape(-1).view(torch.uint8)), (what, k)


def test_device_supports_compression(S):
    yes = ctypes.c_int(-1)
    assert S.lib().snk_compression_supported(0, ctypes.byref(yes)) == 0
    assert yes.value == 1           # a B200: if this fails, every other test here only checks the plain fallback


def test_bench_workload_is_bit_identical_over_50_select_steps(S):
    E, dev = 1 << 20, torch.device("cuda", 0)
    qs, us, rs = bench_inputs(E, dev)
    res = []
    for comp in (False, True):
        env = S.SnakeGame(E, device=0, auto_reset=True)
        out = env.alloc_outputs(obs="f32", mask=True, act=True, compressible=comp)
        assert all(S.is_compressible(v) == comp for v in tensors(out).values())
        snaps = []
        for i in range(50):
            env.step_fused(q=qs[i % 4], eps=0.05, u=us[i % 4], ridx=rs[i % 4], out=out)
            if i % 10 == 9:
                snaps.append({k: v.clone() for k, v in tensors(out).items()})
        res.append(snaps)
        assert env.count_errors() == 0
        env.close()
    for i, (a, b) in enumerate(zip(*res)):
        assert_same_bytes(a, b, "snapshot %d" % i)


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("n", [1, 255, 70001])
def test_every_format_at_ragged_sizes(S, fmt, n):
    dev = torch.device("cuda", 0)
    acts = torch.randint(0, 3, (12, n), device=dev, dtype=torch.uint8, generator=torch.Generator(device=dev).manual_seed(n))
    res = []
    for comp in (False, True):
        env = S.SnakeGame(n, device=0, auto_reset=True)
        out = env.alloc_outputs(obs=fmt, mask=True, ep_stats=True, compressible=comp)
        for t in range(12):
            env.step_fused(act_idx=acts[t], out=out)
        res.append({k: v.clone() for k, v in tensors(out).items()})
        env.close()
    assert_same_bytes(res[0], res[1], "fmt %s n %d" % (fmt, n))


def test_outputs_behave_like_torch_tensors_and_outlive_the_env(S):
    n, dev = 5000, torch.device("cuda", 0)
    env = S.SnakeGame(n, device=0, auto_reset=True)
    ref = S.SnakeGame(n, device=0, auto_reset=True)
    out = env.alloc_outputs(obs="f32", mask=True, ep_stats=True)
    plain = ref.alloc_outputs(obs="f32", mask=True, ep_stats=True, compressible=False)
    assert S.is_compressible(out["obs"]) and not S.is_compressible(plain["obs"])
    assert out["obs"].device == dev and out["obs"].is_contiguous() and out["obs"].shape == (n, 2, 10, 10)
    acts = [torch.randint(0, 3, (n,), device=dev, dtype=torch.uint8) for _ in range(4)]
    for e, o in ((env, out), (ref, plain)):
        for a in acts:
            e.step_fused(act_idx=a, out=o)
    idx = torch.tensor([0, 17, n - 1], device=dev)
    assert torch.equal(out["obs"].index_select(0, idx), plain["obs"].index_select(0, idx))
    assert torch.equal(out["obs"].cpu(), plain["obs"].cpu())
    kept = out["obs"].clone()
    assert not S.is_compressible(kept) and torch.equal(kept, plain["obs"])

    # inside a CUDA graph: the env's kernels and torch ops on the compressible tensors, replayed
    st = torch.cuda.Stream(dev)
    st.wait_stream(torch.cuda.current_stream(dev))
    for e in (env, ref):
        e.use_stream(st)
    with torch.cuda.stream(st):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=st):
            env.step_fused(act_idx=acts[0], out=out)
            s_comp = out["obs"].sum(dim=(1, 2, 3)) + out["reward"]
        graph.replay()
        ref.step_fused(act_idx=acts[0], out=plain)
        s_plain = plain["obs"].sum(dim=(1, 2, 3)) + plain["reward"]
        st.synchronize()
    torch.cuda.synchronize()
    assert torch.equal(s_comp, s_plain)
    assert_same_bytes(tensors(out), tensors(plain), "after graph replay")

    snapshot = {k: v.clone() for k, v in tensors(out).items()}
    env.close()
    ref.close()
    torch.cuda.synchronize()
    assert_same_bytes(tensors(out), snapshot, "after close")
    assert float(out["obs"].abs().sum()) > 0


def test_allocating_and_freeing_1gb_twenty_times_gives_the_memory_back(S):
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(dev)
    for _ in range(20):
        t = S.compressible_empty((1 << 28,), torch.float32, dev)
        assert S.is_compressible(t)
        t.fill_(1.0)
        del t
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info(dev)
    assert abs(free1 - free0) < (64 << 20), (free0, free1)


def test_free_rejects_memory_it_did_not_allocate(S):
    t = torch.empty(16, device="cuda")
    assert S.lib().snk_device_free(ctypes.c_void_p(t.data_ptr())) == -1          # SNK_ERR_INVALID
    assert b"snk_device_alloc" in S.lib().snk_last_error()


def test_a_buffer_that_dies_during_a_graph_capture_is_freed_after_it(S):
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(dev)
    x = torch.arange(1024, dtype=torch.float32, device=dev)
    t = S.compressible_empty((1 << 26,), torch.float32, dev)
    assert S.is_compressible(t)
    st = torch.cuda.Stream(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        y = x * 2
        del t                                   # freeing now would synchronise the device inside the capture
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y, torch.arange(1024, dtype=torch.float32, device=dev) * 2)
    S.compressible_empty((1,), torch.uint8, dev)   # the next allocation outside the capture frees what was left over
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info(dev)
    assert abs(free1 - free0) < (64 << 20), (free0, free1)
