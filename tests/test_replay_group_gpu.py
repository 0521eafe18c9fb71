"""The replay group (snk_replay_group_*, csrc/snake_env.cu; ReplayGroup / Trainer(shared_replay=True); DESIGN §5g).

R ranks draw one minibatch uniformly without replacement from the union of their rings.  The ranks' outputs concatenated in
rank order must be, bit for bit, ReplayBuffer.sample_indices + stack_exp of ONE full ring holding the ranks' filled records
concatenated (capacity Σn, draw counter e), built here from the ranks' checkpoint blobs and loaded with snk_replay_load_host.
The virtual-rank tests run R groups on one GPU, each driven from its own stream; the two-GPU test runs
tools/replay_group_check.py under torchrun.  No test makes a peer miss a wait.  The CPU test at the end checks arguments."""
import ctypes as C
import json
import os
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.util import ROOT, pkg, synth_actions

gpu = pytest.mark.gpu
SPLITS = [[64], [64, 1], [300, 5, 129], [16] * 4]
N_ENVS = 64
# (capacity, steps of N_ENVS stores): partly filled, exactly full, wrapped
FILLS = [(1000, 10), (512, 8), (700, 15)]
OUT_KEYS = ("states", "next_states", "actions", "rewards", "dones", "mask", "ep_return", "score")


def same_bits(x, y):
    return x.shape == y.shape and torch.equal(x.reshape(-1).view(torch.uint8), y.reshape(-1).view(torch.uint8))


def _records(rb):
    """(filled records as bytes, n) of a ring, after the work enqueued so far"""
    blob = rb.state_dict()["blob"].numpy().tobytes()
    return blob[40:], (len(blob) - 40) // 128


def union_ring(rings, draws, seed, sum_B):
    """ONE full ring of capacity Σn holding the rings' filled records concatenated in rank order, with draw counter `draws`"""
    S = pkg()
    recs = [_records(rb) for rb in rings]
    n = sum(k for _, k in recs)
    header = b"snk-rpl\0" + struct.pack("<IIqqQ", 1, 128, n, n, draws)
    blob = torch.frombuffer(bytearray(header + b"".join(r for r, _ in recs)), dtype=torch.uint8)
    ref = S.ReplayBuffer(n, rings[0].device.index, sum_B, seed)
    ref.load_state_dict({"blob": blob, "seed": seed, "batch_size": sum_B})
    return ref


def _fill(S, rank, cap, steps, stream):
    """a ring of capacity `cap` after `steps` fused steps of N_ENVS games; the games run on `stream`"""
    with torch.cuda.stream(stream):
        rb = S.ReplayBuffer(cap, 0, 64, 0)
        env = S.SnakeGame(N_ENVS, device=0, seed=100 + rank)
        for t in range(steps):
            env.step_fused(act_idx=torch.from_numpy(synth_actions(N_ENVS, t, 7 + rank)).cuda(), replay=rb)
    return rb, env


def _check_call(ref, outs, split):
    idx = ref.sample_indices(sum(split))
    want = ref.stack_exp(idx, ep_stats=True)
    torch.cuda.synchronize()
    off = 0
    for r, b in enumerate(split):
        assert torch.equal(outs[r]["idx"], idx[off:off + b]), r
        for k in OUT_KEYS:
            assert same_bits(outs[r][k], want[k][off:off + b]), (r, k)
        off += b


def _run(split, order=None, store_between=False, calls=5):
    S = pkg()
    R = len(split)
    seed = 1000 + 7 * R
    streams = [torch.cuda.Stream(0) for _ in range(R)]
    made = [_fill(S, r, *FILLS[r % len(FILLS)], streams[r]) for r in range(R)]
    rings, envs = [m[0] for m in made], [m[1] for m in made]
    torch.cuda.synchronize()
    groups = [S.ReplayGroup(rb, R, r, split, seed) for r, rb in enumerate(rings)]
    S.connect_local_replay(groups)
    # the actions of the stores between calls, on the device up front: a copy from pageable memory would make the host wait
    # for the rank's stream, whose sample call waits for ranks the host has not enqueued yet
    acts = [[torch.from_numpy(synth_actions(N_ENVS, 50 + e, r)).cuda() for r in range(R)] for e in range(calls)]
    torch.cuda.synchronize()
    for e in range(calls):
        ref = union_ring(rings, e, seed, sum(split))          # the rings as the calls of round e see them (synchronises)
        outs = [None] * R
        for r in (range(R) if order is None else order):
            with torch.cuda.stream(streams[r]):
                outs[r] = groups[r].sample(want_idx=True, ep_stats=True)
                if store_between:                             # enqueued before the lower ranks' sample calls
                    envs[r].step_fused(act_idx=acts[e][r], replay=rings[r])
        torch.cuda.synchronize()
        _check_call(ref, outs, split)
    for g in groups:
        g.check()
        assert g.draws == calls
    return groups, rings


# ---- 1. the union sample is the sample of one ring holding the union --------------------------------------------------------
@gpu
@pytest.mark.parametrize("split", SPLITS, ids=lambda s: "x".join(map(str, s)))
def test_union_sample_equals_the_sample_of_one_ring(split):
    _run(split)


@gpu
def test_one_rank_group_is_replay_buffer_sample():
    S = pkg()
    rb, _ = _fill(S, 0, 700, 15, torch.cuda.current_stream())
    mirror, _ = _fill(S, 0, 700, 15, torch.cuda.current_stream())       # the same ring, sampled the ordinary way
    mirror.seed = 99
    g = S.ReplayGroup(rb, 1, 0, [64], 99)
    for _ in range(5):
        got, want = g.sample(), mirror.sample()
        torch.cuda.synchronize()
        for k in want:
            assert same_bits(got[k], want[k]), k
    g.check()


# ---- 2. the ranks order themselves on the device, also while they keep storing --------------------------------------------
@gpu
@pytest.mark.parametrize("split", SPLITS[1:], ids=lambda s: "x".join(map(str, s)))
def test_reverse_order_with_stores_between_calls(split):
    _run(split, order=list(range(len(split)))[::-1], store_between=True)


# ---- ΣB > n: reported, nothing written ----------------------------------------------------------------------------------------
@gpu
def test_a_sample_larger_than_the_union_is_refused_and_writes_nothing():
    S = pkg()
    rb, _ = _fill(S, 0, 512, 1, torch.cuda.current_stream())           # 64 transitions
    g = S.ReplayGroup(rb, 1, 0, [65], 5)
    dev = rb.device
    out = {k: torch.full((65, 2, 10, 10) if "states" in k else (65,), 7, dtype=torch.float32, device=dev) for k in ("states", "next_states")}
    idx = torch.full((65,), -7, dtype=torch.int64, device=dev)
    acts = torch.full((65,), 9, dtype=torch.uint8, device=dev)
    L = S.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert L.snk_replay_group_sample(g._g, C.c_void_p(idx.data_ptr()), C.c_void_p(out["states"].data_ptr()),
                                     C.c_void_p(out["next_states"].data_ptr()), C.c_void_p(acts.data_ptr()), None, None, None,
                                     None, None, st) == 0
    t, f = C.c_int(0), C.c_int(0)
    assert L.snk_replay_group_status_host(g._g, C.byref(t), C.byref(f)) == -1
    assert f.value == 1 and t.value == 0
    assert bool((idx == -7).all()) and bool((acts == 9).all())
    assert all(bool((v == 7).all()) for v in out.values())
    with pytest.raises(S.SnakeB200Error, match="more transitions"):
        g.check()


# ---- 3. Trainer(shared_replay=True) --------------------------------------------------------------------------------------------
KW = dict(n_envs=4096, batch_size=32, target_sync=10, fill=8192, seed=3)


@gpu
def test_world_one_shared_replay_trainer_is_the_plain_trainer():
    S = pkg()
    a, b = S.train.Trainer(**KW), S.train.Trainer(shared_replay=True, **KW)
    for tr in (a, b):
        tr.train(30)
    torch.cuda.synchronize()
    b.sampler.check()
    assert a.n_updates == b.n_updates == 30
    assert same_bits(torch.stack(a.losses), torch.stack(b.losses))
    for name in ("q_net", "t_net"):
        assert same_bits(getattr(a, name).theta_device, getattr(b, name).theta_device), name
    assert same_bits(a.opt.acc, b.opt.acc)
    ba, bb = a.replay.state_dict()["blob"], b.replay.state_dict()["blob"]
    assert torch.equal(ba[40:], bb[40:]) and torch.equal(ba[:32], bb[:32])      # records, capacity and count
    assert struct.unpack("<Q", ba[32:40].numpy().tobytes())[0] == 30               # the draw counter: the ring's ...
    assert struct.unpack("<Q", bb[32:40].numpy().tobytes())[0] == 0
    assert b.sampler.draws == 30                                                   # ... or the group's


def _trainers(S, streams, **kw):
    trs = []
    for r, s in enumerate(streams):
        with torch.cuda.stream(s):
            trs.append(S.train.Trainer(world=len(streams), rank=r, shared_replay=True, **kw))
    S.train.Trainer.connect_local(trs)
    return trs


def _iterate(trs, streams, n):
    for _ in range(n):
        for tr, s in zip(trs, streams):
            with torch.cuda.stream(s):
                tr.iteration()


@gpu
def test_two_rank_shared_replay_updates_are_the_update_of_the_union_minibatch(tmp_path):
    S = pkg()
    streams = [torch.cuda.Stream(0) for _ in range(2)]
    a = _trainers(S, streams, **KW)
    for tr, s in zip(a, streams):
        with torch.cuda.stream(s):
            tr.fill_buffer()
    bs = KW["batch_size"]
    for _ in range(3):                        # each update against QNet.train_step on the reference ring's minibatch
        for tr, s in zip(a, streams):
            with torch.cuda.stream(s):
                tr._play(tr.epsilon)
        torch.cuda.synchronize()
        t0 = a[0]
        ref = union_ring([tr.replay for tr in a], t0.sampler.draws, KW["seed"], 2 * bs)
        net = S.qnet.QNet(S.qnet.glorot_layers(0), t0.q_net.device)
        net.load_params(t0.q_net.theta_device.clone())
        tnet = S.qnet.QNet(S.qnet.glorot_layers(0), t0.q_net.device)
        tnet.load_params(t0.t_net.theta_device.clone())
        opt = S.qnet.RMSProp(acc=None if t0.opt.acc is None else t0.opt.acc.clone())
        b = ref.stack_exp(ref.sample_indices(2 * bs))
        # the targets as each rank computes them: its t_net forward over its own slice of the minibatch
        y = torch.cat([S.masked_target(tnet(b["next_states"][s].contiguous()), b["mask"][s].contiguous(), b["rewards"][s],
                                       b["dones"][s], gamma=t0.gamma) for s in (slice(0, bs), slice(bs, 2 * bs))])
        loss, _ = net.train_step(b["states"], b["actions"], y, opt)
        for tr, s in zip(a, streams):
            with torch.cuda.stream(s):
                tr.update()
        torch.cuda.synchronize()
        for tr in a:
            assert same_bits(tr.q_net.theta_device, net.theta_device)
            assert same_bits(tr.opt.acc, opt.acc)
            assert same_bits(tr.losses[-1], loss)
    _iterate(a, streams, 7)
    paths = [str(tmp_path / ("rank%d.pt" % r)) for r in range(2)]
    for tr, s, path in zip(a, streams, paths):
        with torch.cuda.stream(s):
            tr.save(path)
    _iterate(a, streams, 20)
    torch.cuda.synchronize()
    for tr in a:
        tr.learner.check()
        tr.sampler.check()
    assert a[0].n_updates == a[1].n_updates == 30
    assert same_bits(torch.stack(a[0].losses), torch.stack(a[1].losses))
    for name in ("q_net", "t_net"):
        assert same_bits(getattr(a[0], name).theta_device, getattr(a[1], name).theta_device), name
    assert same_bits(a[0].opt.acc, a[1].opt.acc)

    b = []
    for r, (s, path) in enumerate(zip(streams, paths)):
        with torch.cuda.stream(s):
            b.append(S.train.Trainer.load(path, device=0, world=2, rank=r, shared_replay=True))
    S.train.Trainer.connect_local(b)
    assert b[0].n_updates == 10 and b[0].sampler.draws == 10
    _iterate(b, streams, 20)
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        y.learner.check()
        y.sampler.check()
        assert same_bits(x.q_net.theta_device, y.q_net.theta_device)
        assert same_bits(x.t_net.theta_device, y.t_net.theta_device)
        assert same_bits(x.opt.acc, y.opt.acc)
        assert same_bits(torch.stack(x.losses), torch.stack(y.losses))
        assert torch.equal(x.env.state_dict()["blob"], y.env.state_dict()["blob"])
        assert torch.equal(x.replay.state_dict()["blob"], y.replay.state_dict()["blob"])
        assert x.sampler.draws == y.sampler.draws == 30

    # a checkpoint of the other setting is refused
    with pytest.raises(ValueError, match="shared_replay"):
        S.train.Trainer.load(paths[0], world=2, rank=0, shared_replay=False)
    plain = S.train.Trainer(n_envs=4096, batch_size=32, world=2, rank=0)
    with pytest.raises(ValueError, match="shared_replay"):
        plain.load_state_dict(torch.load(paths[0], weights_only=True))
    d = plain.state_dict()
    assert d["shared_replay"] is False and "replay_group" not in d
    with pytest.raises(ValueError, match="shared_replay"):
        b[0].load_state_dict(d)
    d.pop("shared_replay")                                      # an older checkpoint: no key = False
    with pytest.raises(ValueError, match="shared_replay"):
        b[0].load_state_dict(d)


# ---- 4. two real GPUs -----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_two_gpu_union_sample_equals_one_ring():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29583", os.path.join(ROOT, "tools", "replay_group_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["world"] == 2 and d["calls"] == 5
    assert d["same_bits_as_one_ring"] is True


# ---- 5. argument checks ----------------------------------------------------------------------------------------------------------
def test_group_entry_points_check_their_arguments():
    L = pkg().lib()
    g = C.c_void_p(7)
    ok = (C.c_int64 * 16)(*([64] * 16))
    for world, rank in ((0, 0), (17, 0), (2, -1), (2, 2), (1, 1)):
        assert L.snk_replay_group_create(C.byref(g), C.c_void_p(8), world, rank, ok, 0) == -1
        assert g.value is None                                     # *out cleared
    assert L.snk_replay_group_create(None, C.c_void_p(8), 1, 0, ok, 0) == -1
    assert L.snk_replay_group_create(C.byref(g), None, 1, 0, ok, 0) == -1
    assert L.snk_replay_group_create(C.byref(g), C.c_void_p(8), 1, 0, None, 0) == -1
    for bad in ([0, 64], [64, -3]):
        arr = (C.c_int64 * 2)(*bad)
        assert L.snk_replay_group_create(C.byref(g), C.c_void_p(8), 2, 0, arr, 0) == -1
        assert b"batch_all" in L.snk_last_error()
    buf = (C.c_uint8 * 256)()
    assert L.snk_replay_group_export_host(None, buf) == -1
    assert L.snk_replay_group_connect_host(None, buf, 2) == -1
    assert L.snk_replay_group_connect_local(None, None, 0) == -1
    assert L.snk_replay_group_sample(None, None, None, None, None, None, None, None, None, None, None) == -1
    d = C.c_uint64(0)
    assert L.snk_replay_group_draws(None, C.byref(d)) == -1
    assert L.snk_replay_group_set_draws(None, 3) == -1
    assert L.snk_replay_group_status_host(None, C.byref(C.c_int(0)), C.byref(C.c_int(0))) == -1
    assert L.snk_replay_group_destroy(None) == 0


@gpu
def test_a_group_refuses_a_wrong_handle_count_and_a_sample_before_connect():
    S = pkg()
    rings = [_fill(S, r, 512, 2, torch.cuda.current_stream())[0] for r in range(2)]
    g0, g1 = S.ReplayGroup(rings[0], 2, 0, [8, 8], 1), S.ReplayGroup(rings[1], 2, 1, [8, 8], 1)
    with pytest.raises(S.SnakeB200Error, match="not connected"):
        g0.sample()
    h = [g0.handle(), g1.handle()]
    assert len(h[0]) == 128
    with pytest.raises(S.SnakeB200Error, match="one handle per rank"):
        g0.connect(h[:1])
    with pytest.raises(S.SnakeB200Error, match="one handle per rank"):
        g0.connect(h + h[:1])
    arr = (C.c_void_p * 2)(g0._g.value, g1._g.value)
    assert S.lib().snk_replay_group_connect_local(g0._g, arr, 3) == -1
    arr_swapped = (C.c_void_p * 2)(g1._g.value, g0._g.value)
    assert S.lib().snk_replay_group_connect_local(g0._g, arr_swapped, 2) == -1
    other = S.ReplayGroup(rings[1], 2, 1, [8, 9], 1)            # another batch_all
    arr_other = (C.c_void_p * 2)(g0._g.value, other._g.value)
    assert S.lib().snk_replay_group_connect_local(g0._g, arr_other, 2) == -1
    with pytest.raises(ValueError, match="one entry per rank"):
        S.ReplayGroup(rings[0], 2, 0, [8], 1)
    g0.check()
    g1.check()
    for g in (g0, g1, other):
        g.close()
