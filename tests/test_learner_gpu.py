"""The learner on the device (snk_qnet_train_step / snk_qnet_set_params, csrc/qnet.cu) against oracle/learner_oracle.py.

Reference: utils.jl:452-472 — Flux.gradient of mean(huber(q_net(s)[a], y)), update!(RMSProp(5e-4), ...), update_target_net!.
Stated tolerances: the mean gradient within 2e-5 relative Frobenius error of the Float64 oracle and 2e-5 of its largest entry
elementwise (the per-sample rows are FP32, as in test_sample_grads_gpu.py); the reduction, the RMSProp step and every
re-derived device layout are bit-exact.  Parity unpinned by the reference (Flux / Zygote unpinned)."""
import numpy as np
import pytest
import torch

from oracle import learner_oracle as LO
from tests.test_sample_grads_gpu import _layers, _transitions
from tests.util import bits, pkg, synth_actions

pytestmark = pytest.mark.gpu

P = 181395


def _targets(net, batch, seed):
    """targets on both branches of the Huber loss"""
    B = batch["states"].shape[0]
    rng = np.random.default_rng(seed)
    q = net(batch["states"])
    q_sel = q.gather(1, batch["actions"].long()[:, None])[:, 0].double().cpu().numpy()
    delta = np.where(rng.random(B) < 0.25, rng.choice([-1, 1], B) * rng.uniform(1.2, 3.0, B), rng.uniform(-0.9, 0.9, B))
    return torch.from_numpy(q_sel - delta).cuda()


def _restructure(like, theta):
    """layers of the shapes of `like` holding Flux.destructure-ordered theta"""
    out, off = [], 0
    for kind, p in like:
        if kind in ("conv", "dense"):
            d = dict(p)
            for k in ("W", "b"):
                n = p[k].size
                d[k] = np.asarray(theta[off:off + n], dtype=np.float32).reshape(p[k].shape, order="F")
                off += n
            out.append((kind, d))
        else:
            out.append((kind, p))
    assert off == P
    return out


def _boards(n, steps, seed):
    S = pkg()
    env = S.SnakeGame(n, auto_reset=True)
    for t in range(steps):
        env.step(torch.from_numpy(synth_actions(n, t, seed=seed)).cuda())
    return env.assemble_state("f32")


@pytest.mark.parametrize("B,seed", [(64, 1), (37, 2)])
def test_mean_gradient_and_loss_match_float64_oracle(B, seed):
    S = pkg()
    layers = _layers(seed)
    batch = _transitions(512, 12, B, seed)
    net = S.qnet.QNet(layers, batch["states"].device, precision="f32")
    y = _targets(net, batch, seed)
    opt = S.qnet.RMSProp()
    loss, g = net.train_step(batch["states"], batch["actions"], y, opt, want_grad=True)
    want, want_loss = LO.mean_grad(layers, batch["states"].cpu().numpy(), batch["actions"].cpu().numpy(), y.cpu().numpy())
    g = g.cpu().numpy().astype(np.float64)
    assert np.linalg.norm(g - want) / np.linalg.norm(want) < 2e-5
    assert np.abs(g - want).max() < 2e-5 * np.abs(want).max()
    assert abs(float(loss) - want_loss) < 2e-5 * want_loss


@pytest.mark.parametrize("B", [64, 700])
def test_reduction_is_the_float64_running_sum_of_the_rows(B):
    """g = Float32((sum_i J_i in Float64, in sample order) / B) exactly, also when the minibatch spans several chunks of the
    row scratch (700 > 2 x 148 samples)"""
    S = pkg()
    batch = _transitions(512, 12, B, 3)
    net = S.qnet.QNet(_layers(3), batch["states"].device, precision="f32")
    y = _targets(net, batch, 3)
    rows = net.sample_grads(batch["states"], batch["actions"], y, want_J=True, want_loss=True)
    J, losses = rows["J"].cpu().numpy(), rows["loss"].cpu().numpy()
    s = np.zeros(P)
    for r in J:
        s += r.astype(np.float64)
    loss, g = net.train_step(batch["states"], batch["actions"], y, S.qnet.RMSProp(), want_grad=True)
    sl = 0.0
    for v in losses:
        sl += float(v)
    assert np.array_equal(bits(g.cpu().numpy()), bits((s / B).astype(np.float32)))
    assert np.array_equal(bits(loss.cpu().numpy()), bits(np.float32(sl / B)))


@pytest.mark.parametrize("fresh_acc", [True, False])
def test_five_updates_are_bit_exact_rmsprop(fresh_acc):
    S = pkg()
    batch = _transitions(512, 12, 64, 4)
    net = S.qnet.QNet(_layers(4), batch["states"].device, precision="f32")
    y = _targets(net, batch, 4)
    acc0 = None
    if not fresh_acc:
        acc0 = torch.from_numpy(np.abs(np.random.default_rng(4).normal(0, 1e-4, P)).astype(np.float32)).cuda()
    opt = S.qnet.RMSProp(acc=acc0)
    theta = net.theta.copy()
    acc = np.zeros(P, np.float32) if fresh_acc else acc0.cpu().numpy()
    for _ in range(5):
        _, g = net.train_step(batch["states"], batch["actions"], y, opt, want_grad=True)
        theta, acc = LO.rmsprop(theta, acc, g.cpu().numpy())
        assert np.array_equal(bits(net.theta), bits(theta))
        assert np.array_equal(bits(opt.acc.cpu().numpy()), bits(acc))
    assert not np.array_equal(net.theta, S.bson_io.destructure(_layers(4)))


@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_every_layout_follows_theta(precision):
    """a trained handle computes exactly what a handle created from its downloaded theta computes"""
    S = pkg()
    layers = _layers(6)
    batch = _transitions(512, 12, 64, 6)
    net = S.qnet.QNet(layers, batch["states"].device, precision=precision)
    y = _targets(net, batch, 6)
    opt = S.qnet.RMSProp()
    for _ in range(3):
        net.train_step(batch["states"], batch["actions"], y, opt)
    fresh = S.qnet.QNet(_restructure(layers, net.theta), net.device, precision=precision)
    for n in (1000, 65536):
        obs = _boards(n, 20, 6)
        assert torch.equal(net(obs).view(torch.int32), fresh(obs).view(torch.int32)), n
    a = net.sample_grads(batch["states"], batch["actions"], y, want_J=True)
    b = fresh.sample_grads(batch["states"], batch["actions"], y, want_J=True)
    assert torch.equal(a["J"].view(torch.int32), b["J"].view(torch.int32))
    assert torch.equal(a["loss"].view(torch.int32), b["loss"].view(torch.int32))
    assert not net.overflow()


def test_target_sync_copies_and_then_stays():
    S = pkg()
    batch = _transitions(512, 12, 64, 7)
    dev = batch["states"].device
    q = S.qnet.QNet(_layers(7), dev)
    t = S.qnet.QNet(_layers(8), dev)
    y = _targets(q, batch, 7)
    opt = S.qnet.RMSProp()
    q.train_step(batch["states"], batch["actions"], y, opt)
    obs = _boards(4096, 10, 7)
    assert not torch.equal(q(obs), t(obs))
    t.load_params_from(q)
    assert np.array_equal(bits(t.theta), bits(q.theta))
    q_before = t(obs)
    assert torch.equal(q_before.view(torch.int32), q(obs).view(torch.int32))
    q.train_step(batch["states"], batch["actions"], y, opt)
    assert not torch.equal(q(obs), q_before)
    assert torch.equal(t(obs).view(torch.int32), q_before.view(torch.int32))


def test_same_step_from_same_state_is_deterministic():
    S = pkg()
    batch = _transitions(512, 12, 64, 9)
    dev = batch["states"].device
    acc0 = torch.from_numpy(np.abs(np.random.default_rng(9).normal(0, 1e-4, P)).astype(np.float32)).cuda()
    res = []
    for _ in range(2):
        net = S.qnet.QNet(_layers(9), dev)
        y = _targets(net, batch, 9)
        opt = S.qnet.RMSProp(acc=acc0.clone())
        loss, g = net.train_step(batch["states"], batch["actions"], y, opt, want_grad=True)
        res.append([bits(x) for x in (net.theta, opt.acc.cpu().numpy(), g.cpu().numpy(), loss.cpu().numpy())])
    for a, b in zip(*res):
        assert np.array_equal(a, b)


def test_two_hundred_updates_fit_one_minibatch():
    S = pkg()
    batch = _transitions(512, 12, 64, 10)
    dev = batch["states"].device
    net = S.qnet.QNet(_layers(10), dev)
    t = S.qnet.QNet(_layers(11), dev)
    y = S.masked_target(t(batch["next_states"]), batch["mask"], batch["rewards"], batch["dones"])

    def batch_loss():
        return float(net.sample_grads(batch["states"], batch["actions"], y)["loss"].double().mean())

    opt = S.qnet.RMSProp()
    before = batch_loss()
    for _ in range(200):
        net.train_step(batch["states"], batch["actions"], y, opt)
    after = batch_loss()
    assert after * 10 <= before, (before, after)


def test_forward_after_an_update_refuses_a_stream_capture():
    """conv1's kernel parameters come to the host after an update; a forward that would have to wait for them inside a
    capture fails with a clear error instead of breaking the capture, and the next forward outside it works"""
    S = pkg()
    batch = _transitions(256, 6, 64, 12)
    net = S.qnet.QNet(_layers(12), batch["states"].device)
    y = _targets(net, batch, 12)
    obs = batch["states"]
    net.train_step(batch["states"], batch["actions"], y, S.qnet.RMSProp())
    out = torch.empty(64, 3, device=obs.device)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        with pytest.raises(S.SnakeB200Error, match="outside the stream capture"):
            net(obs, out=out)
    q1 = net(obs)
    fresh = S.qnet.QNet(_restructure(_layers(12), net.theta), obs.device)
    assert torch.equal(q1.view(torch.int32), fresh(obs).view(torch.int32))


def test_trainer_runs_the_loop():
    S = pkg()
    tr = S.train.Trainer(n_envs=1024, fill=4096, target_sync=5, updates_per_step=2, seed=1)
    tr.train(10)
    assert tr.n_updates == 10 and tr.stored == 10 * 1024
    assert np.array_equal(bits(tr.t_net.theta), bits(tr.q_net.theta))          # synced after update 10
    tr.iteration()
    assert tr.n_updates == 12 and len(tr.losses) == 12 and len(tr.replay) == 11 * 1024
    assert not np.array_equal(tr.t_net.theta, tr.q_net.theta)
    assert abs(tr.epsilon - (1.0 - 12e-6)) < 1e-12
    losses = torch.stack(tr.losses).cpu().numpy()
    assert np.isfinite(losses).all() and (losses >= 0).all()
    assert tr.episode_returns().numel() > 0
    assert tr.env.count_errors() == 0
