"""The data-parallel learner (snk_qnet_group_*, csrc/qnet.cu; LearnerGroup / Trainer(world, rank); DESIGN §5f).

A group update of R ranks with local minibatches B_0 .. B_{R-1} must be, on every rank, bit for bit the single-GPU
QNet.train_step of the minibatches concatenated in rank order: θ, the RMSProp state, g and the loss.  The virtual-rank tests
run R groups on one GPU, each driven from its own stream; the two-GPU test runs tools/dp_learner_check.py under torchrun.
No test makes a peer miss a wait: the timeout path is only read, never provoked.  The CPU tests at the end check arguments."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.test_learner_gpu import _boards, _targets
from tests.test_sample_grads_gpu import _layers, _transitions
from tests.util import ROOT, pkg

gpu = pytest.mark.gpu
P = 181395
SPLITS = [[37], [64, 1], [300, 5, 129], [16] * 4]         # [300, ...]: one rank spans more than 2 x 148 samples


def same_bits(x, y):
    return x.shape == y.shape and torch.equal(x.reshape(-1).view(torch.uint8), y.reshape(-1).view(torch.uint8))


def _run(split, precision, fresh_acc, order=None, updates=5):
    S = pkg()
    R, B = len(split), sum(split)
    seed = 10 * R + len(str(split))
    batch = _transitions(512, 12, B, seed)
    dev = batch["states"].device
    layers = _layers(seed)
    ref = S.qnet.QNet(layers, dev, precision)
    y = _targets(ref, batch, seed)
    acc0 = None if fresh_acc else torch.from_numpy(np.abs(np.random.default_rng(seed).normal(0, 1e-4, P)).astype(np.float32)).cuda()
    opt_ref = S.qnet.RMSProp(acc=None if acc0 is None else acc0.clone())
    nets = [S.qnet.QNet(layers, dev, precision) for _ in split]
    opts = [S.qnet.RMSProp(acc=None if acc0 is None else acc0.clone()) for _ in split]
    group = S.qnet.LocalLearnerGroup(nets)
    off = np.concatenate([[0], np.cumsum(split)])
    batches = [(batch["states"][a:b], batch["actions"][a:b], y[a:b]) for a, b in zip(off[:-1], off[1:])]
    theta0 = ref.theta_device.clone()
    for _ in range(updates):
        loss, g = ref.train_step(batch["states"], batch["actions"], y, opt_ref, want_grad=True)
        out = group.train_step(batches, opts, want_grad=True, order=order)
        torch.cuda.synchronize()
        for r in range(R):
            assert same_bits(nets[r].theta_device, ref.theta_device), r
            assert same_bits(opts[r].acc, opt_ref.acc), r
            assert same_bits(out[r][1], g), r
            assert same_bits(out[r][0], loss), r
    group.check()
    assert not torch.equal(ref.theta_device, theta0)
    obs = _boards(1000, 20, seed)
    want = ref(obs)
    for net in nets:
        assert same_bits(net(obs), want)
    group.close()


# ---- 1. virtual ranks: the group update is the update of the concatenated minibatch -----------------------------------
@gpu
@pytest.mark.parametrize("precision", ["f32", "bf16"])
@pytest.mark.parametrize("split", SPLITS, ids=lambda s: "x".join(map(str, s)))
def test_group_update_is_the_update_of_the_concatenated_batch(split, precision):
    for fresh_acc in (True, False):
        _run(split, precision, fresh_acc)


# ---- 2. the ranks order themselves on the device --------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("split", SPLITS[1:], ids=lambda s: "x".join(map(str, s)))
def test_ranks_enqueued_in_reverse_order_give_the_same_bits(split):
    _run(split, "f32", False, order=list(range(len(split)))[::-1])


# ---- 3. Trainer: two virtual ranks, identical on both, and a saved group run continues bit for bit ------------------------
def _trainers(S, streams, **kw):
    trs = []
    for r, s in enumerate(streams):
        with torch.cuda.stream(s):
            trs.append(S.train.Trainer(world=len(streams), rank=r, **kw))
    S.train.Trainer.connect_local(trs)
    return trs


def _iterate(trs, streams, n):
    """one iteration per rank per round, ranks in order: no rank's host waits on its stream before every rank has enqueued
    the update that stream waits for"""
    for _ in range(n):
        for tr, s in zip(trs, streams):
            with torch.cuda.stream(s):
                tr.iteration()


@gpu
def test_two_virtual_rank_trainers_agree_and_continue_bit_for_bit(tmp_path):
    S = pkg()
    streams = [torch.cuda.Stream(0) for _ in range(2)]
    kw = dict(n_envs=4096, batch_size=32, target_sync=10, fill=8192, seed=3)
    a = _trainers(S, streams, **kw)
    for tr, s in zip(a, streams):
        with torch.cuda.stream(s):
            tr.fill_buffer()
    _iterate(a, streams, 10)
    paths = [str(tmp_path / ("rank%d.pt" % r)) for r in range(2)]
    for tr, s, path in zip(a, streams, paths):
        with torch.cuda.stream(s):
            tr.save(path)
    _iterate(a, streams, 20)
    torch.cuda.synchronize()
    for tr in a:
        tr.learner.check()
    assert a[0].n_updates == a[1].n_updates == 30
    assert same_bits(torch.stack(a[0].losses), torch.stack(a[1].losses))
    for name in ("q_net", "t_net"):
        assert same_bits(getattr(a[0], name).theta_device, getattr(a[1], name).theta_device), name
    assert same_bits(a[0].opt.acc, a[1].opt.acc)
    assert not torch.equal(a[0].replay.state_dict()["blob"], a[1].replay.state_dict()["blob"])   # each rank its own ring

    b = []
    for r, (s, path) in enumerate(zip(streams, paths)):
        with torch.cuda.stream(s):
            b.append(S.train.Trainer.load(path, device=0, world=2, rank=r))
    S.train.Trainer.connect_local(b)
    assert b[0].n_updates == 10
    _iterate(b, streams, 20)
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        y.learner.check()
        assert same_bits(x.q_net.theta_device, y.q_net.theta_device)
        assert same_bits(x.t_net.theta_device, y.t_net.theta_device)
        assert same_bits(x.opt.acc, y.opt.acc)
        assert same_bits(torch.stack(x.losses), torch.stack(y.losses))
        assert torch.equal(x.env.state_dict()["blob"], y.env.state_dict()["blob"])
        assert torch.equal(x.replay.state_dict()["blob"], y.replay.state_dict()["blob"])
    with pytest.raises(ValueError, match="rank"):
        S.train.Trainer.load(paths[0], rank=1)
    with pytest.raises(ValueError, match="world"):
        S.train.Trainer.load(paths[0], world=1)


# ---- 4. two real GPUs ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_two_gpu_group_matches_one_gpu_train_step():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29581", os.path.join(ROOT, "tools", "dp_learner_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["world"] == 2 and d["updates"] == 5
    assert d["same_bits_as_one_gpu"] is True and d["theta_equal_on_all_ranks"] is True


# ---- 5. argument checks ---------------------------------------------------------------------------------------------------
def test_group_entry_points_check_their_arguments():
    L = pkg().lib()
    g = C.c_void_p(7)
    for world, rank in ((0, 0), (17, 0), (2, -1), (2, 2), (1, 1)):
        assert L.snk_qnet_group_create(C.byref(g), None, world, rank) == -1
        assert g.value is None                                     # *out cleared
    assert L.snk_qnet_group_create(None, None, 1, 0) == -1
    buf = (C.c_uint8 * 128)()
    assert L.snk_qnet_group_export_host(None, buf) == -1
    assert L.snk_qnet_group_connect_host(None, buf, 2) == -1
    assert L.snk_qnet_group_connect_local(None, None, 0) == -1
    assert L.snk_qnet_group_train_step(None, None, None, None, 1, None, 5e-4, 0.9, 1e-8, None, None, None) == -1
    assert L.snk_qnet_group_status_host(None, C.byref(C.c_int(0))) == -1
    assert L.snk_qnet_group_destroy(None) == 0


@gpu
def test_a_group_refuses_a_wrong_handle_count_and_an_update_before_connect():
    S = pkg()
    batch = _transitions(256, 4, 8, 5)
    dev = batch["states"].device
    nets = [S.qnet.QNet(_layers(5), dev) for _ in range(2)]
    g0, g1 = S.qnet.LearnerGroup(nets[0], 2, 0), S.qnet.LearnerGroup(nets[1], 2, 1)
    y = torch.zeros(8, dtype=torch.float64, device=dev)
    theta0 = nets[0].theta_device.clone()
    with pytest.raises(S.SnakeB200Error, match="not connected"):
        g0.train_step(batch["states"], batch["actions"], y, S.qnet.RMSProp())
    h = [g0.handle(), g1.handle()]
    with pytest.raises(S.SnakeB200Error, match="one handle per rank"):
        g0.connect(h[:1])
    with pytest.raises(S.SnakeB200Error, match="one handle per rank"):
        g0.connect(h + h[:1])
    arr = (C.c_void_p * 2)(g0._g.value, g1._g.value)
    assert S.lib().snk_qnet_group_connect_local(g0._g, arr, 3) == -1
    arr_swapped = (C.c_void_p * 2)(g1._g.value, g0._g.value)
    assert S.lib().snk_qnet_group_connect_local(g0._g, arr_swapped, 2) == -1
    torch.cuda.synchronize()
    assert same_bits(nets[0].theta_device, theta0)
    g0.check()
    g1.check()
    g0.close()
    g1.close()
