"""Checkpoints of a device run (snk_env_* / snk_replay_* save and load, Trainer.save / Trainer.load; DESIGN §5e).

A run saved after K steps and continued must compute exactly the bits of the run that never stopped, and a load must refuse
every state the step kernel cannot have stored, leaving the handle as it was.  The CPU tests at the end check arguments only."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.util import G2_ACTIONS, pkg, synth_actions

gpu = pytest.mark.gpu
DEV = torch.device("cuda", 0)
ENV_HEADER, REPLAY_HEADER = 176, 40
# misc field offsets (csrc/snake_env.cu)
M_HR, M_HC, M_TR, M_TC, M_FR, M_FC, M_PFR, M_PFC, M_PD, M_LEN, M_T, M_DONE = 0, 4, 8, 12, 16, 20, 24, 28, 32, 34, 41, 51
DELTA = {0: (-1, 0), 1: (1, 0), 2: (0, -1), 3: (0, 1)}


@pytest.fixture(scope="module")
def S():
    import __graft_entry__ as g
    g.build()
    return pkg()


def same_bits(x, y):
    return x.shape == y.shape and torch.equal(x.contiguous().view(torch.uint8), y.contiguous().view(torch.uint8))


def lockstep(a, b, steps, t0, eps=0.3):
    """step a and b with the same Q-values and internal ε-greedy draws; every output of every step must agree bit for bit.
    The observation format rotates over Float32, int8 and the bit records."""
    fmts = ("f32", "i8", "bits")
    outs = {f: (a.alloc_outputs(obs=f, ep_stats=True, act=True, compressible=False),
                b.alloc_outputs(obs=f, ep_stats=True, act=True, compressible=False)) for f in fmts}
    g = torch.Generator(device=DEV)
    for t in range(steps):
        g.manual_seed(t0 + t)
        q = torch.rand(a.n, 3, generator=g, device=DEV)
        oa, ob = outs[fmts[t % 3]]
        a.step_fused(q=q, eps=eps, out=oa)
        b.step_fused(q=q, eps=eps, out=ob)
        for k, v in oa.items():
            if isinstance(v, torch.Tensor):
                assert same_bits(v, ob[k]), (t, k)


def play(env, steps, t0, eps=0.3):
    """steps fused steps of env alone; returns (apples eaten, episodes ended)"""
    out = env.alloc_outputs(obs="f32", ep_stats=True, act=True, compressible=False)
    g = torch.Generator(device=DEV)
    eaten = ended = 0
    for t in range(steps):
        g.manual_seed(t0 + t)
        env.step_fused(q=torch.rand(env.n, 3, generator=g, device=DEV), eps=eps, out=out)
        eaten += int((out["reward"] == 1.0).sum())
        ended += int(out["done"].sum())
    return eaten, ended


def blob_equal(x, y):
    return torch.equal(x["blob"], y["blob"])


# ---- 1. a loaded handle continues bit for bit ------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("case", ["auto_reset", "frozen", "food_exhausted"])
def test_env_continues_bit_for_bit(S, case):
    n = 70001
    kw = {"auto_reset": case != "frozen"}
    a = S.SnakeGame(n, seed=7, food_list=[(7, 3)] if case == "food_exhausted" else None, **kw)
    eaten, ended = play(a, 300, 0)
    assert eaten > 0 and ended > 0
    if case == "frozen":
        heads = a.assemble_state("bits")[:, 18].cpu()
        r, c = heads & 15, heads >> 4
        on_wall = (r == 0) | (r == 9) | (c == 0) | (c == 9)
        assert bool((on_wall & (a.lost.cpu() == 1)).any())                  # frozen wall deaths are in the blob
    if case == "food_exhausted":
        assert a.count_errors() > 0 and bool(((a.error_flags & S.ENV_ERR_FOOD) != 0).any())
    saved = a.state_dict()
    b = S.SnakeGame(n, **kw)                                                # default seed and food list: the blob brings both
    b.load_state_dict(saved)
    assert blob_equal(b.state_dict(), saved)
    lockstep(a, b, 500, 300)
    assert blob_equal(a.state_dict(), b.state_dict())


# ---- 2. no false rejects ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["random_idx", "step_cap", "random_abs", "random_abs_frozen"])
def test_every_reachable_state_loads(S, mode):
    """4,096 envs x 2,000 steps; every checkpoint taken every 100 steps loads into a twin"""
    n = 4096
    auto = mode != "random_abs_frozen" and mode != "step_cap"
    env, twin = S.SnakeGame(n, auto_reset=auto), S.SnakeGame(n, auto_reset=auto)
    loop = torch.tensor([0, 3, 1, 2], dtype=torch.uint8, device=DEV)        # U R D L: a 2x2 circle, never eats, hits the 500-step cap
    seen_cap = False
    for c in range(20):
        T = 100
        rnd = torch.stack([torch.from_numpy(synth_actions(n, 100 * c + t, seed=5)) for t in range(T)]).to(DEV)
        if mode == "random_idx":
            env.rollout(rnd, obs=None, mask=False)
        elif mode == "step_cap":
            circle = loop[(torch.arange(T, device=DEV) + 100 * c) % 4][:, None].expand(T, n)
            acts = torch.where(torch.arange(n, device=DEV) < n // 2, circle, (rnd + torch.arange(n, device=DEV) % 2).to(torch.uint8))
            env.rollout(acts.contiguous(), obs=None, mask=False, is_abs=True)
            seen_cap |= bool((env.steps == 500).any())
        else:
            for t in range(T):
                env.step_abs((rnd[t] + (torch.arange(n, device=DEV) + t) % 2).to(torch.uint8))   # directions 0..3, reverses lose
        twin.load_state_dict(env.state_dict())
    if mode == "step_cap":
        assert seen_cap


@gpu
def test_the_reference_best_game_loads_at_every_step(S):
    """tests/util.G2_ACTIONS: 33 apples (a 35-segment snake, the second chain word live) and a wall death; the state after
    every step loads"""
    n = 256
    env, twin = S.SnakeGame(n, auto_reset=False), S.SnakeGame(n, auto_reset=False)
    code = {"U": 0, "D": 1, "L": 2, "R": 3}
    for ch in G2_ACTIONS:
        env.step_abs(torch.full((n,), code[ch], dtype=torch.uint8, device=DEV))
        twin.load_state_dict(env.state_dict())
    assert int(env.score[0]) == 33 and int(env.lost[0]) == 1


# ---- 3. corrupted blobs are refused, the handle left as it was -------------------------------------------------------------
def make_env(head, dirs, t=20, done=0, food=(2, 2), pfood=(2, 2), err=0):
    """the seven state words of one env built from a head and its direction chain (entry j: the move that took segment j+1 to
    segment j), consistent by construction"""
    r, c = head
    occ, clo, chi = 0, 0, 0
    if 1 <= r <= 8 and 1 <= c <= 8:
        occ |= 1 << ((r - 1) + 8 * (c - 1))
    for j, d in enumerate(dirs):
        r, c = r - DELTA[d][0], c - DELTA[d][1]
        if 1 <= r <= 8 and 1 <= c <= 8:
            occ |= 1 << ((r - 1) + 8 * (c - 1))
        if j < 32:
            clo |= d << (2 * j)
        else:
            chi |= d << (2 * (j - 32))
    misc = (head[0] << M_HR) | (head[1] << M_HC) | (r << M_TR) | (c << M_TC) | (food[0] << M_FR) | (food[1] << M_FC) | \
           (pfood[0] << M_PFR) | (pfood[1] << M_PFC) | (dirs[0] << M_PD) | ((len(dirs) + 1) << M_LEN) | (t << M_T) | \
           (done << M_DONE) | (err << 52)
    return {"occ": occ, "pocc": occ, "clo": clo, "chi": chi, "cons": 0, "misc": misc}


def put_env(blob, n, k, st):
    """blob (uint8 CPU tensor) with env k replaced by the state words st"""
    blob = blob.clone()
    u = blob[ENV_HEADER:ENV_HEADER + 48 * n].numpy().view(np.uint64).reshape(6, n)
    for row, key in enumerate(("occ", "pocc", "clo", "chi", "cons", "misc")):
        u[row, k] = np.uint64(st[key] & (2 ** 64 - 1))
    return blob


def field(st, shift, width, value):
    st = dict(st)
    st["misc"] = (st["misc"] & ~(((1 << width) - 1) << shift)) | (value << shift)
    return st


BASE = make_env((4, 4), [0, 0, 2])             # head (4,4), body (5,4) (6,4), tail (6,5): moved up last
CORRUPT = [                                    # (name, state, words of the expected message)
    ("head r 12", field(BASE, M_HR, 4, 12), "head"),
    ("live head on the wall", make_env((0, 4), [0, 0, 2]), "head"),
    ("corner head of a lost env", make_env((0, 0), [0, 0], done=1), "head"),
    ("tail r 0", field(BASE, M_TR, 4, 0), "tail not an interior"),
    ("tail off the chain", field(BASE, M_TC, 4, 7), "does not end on the tail"),
    ("food r 12", field(BASE, M_FR, 4, 12), "food neither"),
    ("food half the no-food code", field(field(BASE, M_FR, 4, 0), M_FC, 4, 5), "food neither"),
    ("previous food on the wall", field(BASE, M_PFR, 4, 9), "previous food"),
    ("len 1", field(BASE, M_LEN, 7, 1), "length"),
    ("len 65", field(BASE, M_LEN, 7, 65), "length"),
    ("step count 600", field(BASE, M_T, 10, 600), "step count"),
    ("live env at step 500", field(BASE, M_T, 10, 500), "step count"),
    ("error bit 2", field(BASE, 52, 4, 4), "unused bits"),
    ("bit 60 of misc", dict(BASE, misc=BASE["misc"] | (1 << 60)), "unused bits"),
    ("cons outside the 50-entry list", dict(BASE, cons=1 << 55), "consumed food"),
    ("prev_dir not the last move", field(BASE, M_PD, 2, 3), "previous direction"),
    ("chain leaves the board", make_env((1, 4), [1, 0]), "leaves the board"),
    ("chain crosses itself", make_env((4, 4), [0, 2, 1, 3, 0]), "crosses itself"),
    ("live head on its body", make_env((4, 4), [0, 2, 1, 3]), "crosses itself"),
    ("occ misses a segment", dict(BASE, occ=BASE["occ"] & ~(1 << (4 + 8 * 3))), "occupancy"),
    ("occ has an extra cell", dict(BASE, occ=BASE["occ"] | 1), "occupancy"),
]
ACCEPT = [                                     # states the kernels do produce, next to the refused ones
    ("base", BASE),
    ("lost on the wall", make_env((0, 4), [0, 0, 2], done=1)),
    ("lost at step 500", field(field(BASE, M_T, 10, 500), M_DONE, 1, 1)),
    ("lost head on its body", make_env((4, 4), [0, 2, 1, 3], done=1)),
    ("no food, both error bits", make_env((4, 4), [0, 0, 2], food=(0, 0), err=3)),
    # a 40-segment snake (the second chain word live): up column 1, down column 2, ... (D in the chain = the body goes up)
    ("long snake", make_env((8, 1), [1] * 7 + [2] + [0] * 7 + [2] + [1] * 7 + [2] + [0] * 7 + [2] + [1] * 7, food=(0, 0))),
]


@gpu
def test_corrupted_env_blobs_are_refused_and_leave_the_handle_untouched(S):
    n, k = 4096, 1234
    env, twin = S.SnakeGame(n), S.SnakeGame(n)
    play(env, 40, 1000)
    good = env.state_dict()
    twin.load_state_dict(good)
    for name, st in ACCEPT:
        env.load_state_dict({"blob": put_env(good["blob"], n, k, st)})
    env.load_state_dict(good)
    for name, st, words in CORRUPT:
        with pytest.raises(S.SnakeB200Error) as ei:
            env.load_state_dict({"blob": put_env(good["blob"], n, k, st)})
        assert "error -1" in str(ei.value) and words in str(ei.value), (name, str(ei.value))
        assert ei.value.first_bad == k, name
        assert blob_equal(env.state_dict(), good), name
    # the lowest failing env is reported
    two = put_env(put_env(good["blob"], n, k + 1000, CORRUPT[0][1]), n, k, CORRUPT[-1][1])
    with pytest.raises(S.SnakeB200Error) as ei:
        env.load_state_dict({"blob": two})
    assert ei.value.first_bad == k
    # refusals of the blob as a whole
    bad_magic, bad_version, food65 = good["blob"].clone(), good["blob"].clone(), good["blob"].clone()
    bad_magic[0] ^= 1
    bad_version[8] += 1
    food65[40:44] = torch.tensor([65, 0, 0, 0], dtype=torch.uint8)
    for blob, words in ((bad_magic, "magic"), (bad_version, "version"), (good["blob"][:100], "truncated"),
                        (good["blob"][:-1], "blob of"), (food65, "food list")):
        with pytest.raises(S.SnakeB200Error) as ei:
            env.load_state_dict({"blob": blob})
        assert "error -1" in str(ei.value) and words in str(ei.value) and ei.value.first_bad == -1, words
    with pytest.raises(S.SnakeB200Error, match="envs"):
        S.SnakeGame(n + 1).load_state_dict(good)
    with pytest.raises(S.SnakeB200Error, match="SNK_AUTO_RESET"):
        S.SnakeGame(n, auto_reset=False).load_state_dict(good)
    # after all of it the handle steps exactly like its untouched twin
    assert blob_equal(env.state_dict(), good)
    lockstep(env, twin, 30, 2000)


# ---- 4. the replay ring ----------------------------------------------------------------------------------------------------
def fill_ring(S, env, rb, steps, t0):
    for t in range(steps):
        env.step_fused(act_idx=torch.from_numpy(synth_actions(env.n, t0 + t, seed=11)).to(DEV), obs=None, replay=rb)


@gpu
@pytest.mark.parametrize("capacity", [1000, 50000])          # wrapped, partly filled
def test_ring_continues_bit_for_bit(S, capacity):
    n = 4096
    env, env2 = S.SnakeGame(n), S.SnakeGame(n)
    rb = S.ReplayBuffer(capacity, 0, batch_size=64, seed=3)
    fill_ring(S, env, rb, 3, 0)
    rb.sample_indices()                                       # the sampler's counter is part of the state
    saved = rb.state_dict()
    rb2 = S.ReplayBuffer(capacity, 0, batch_size=32, seed=99)
    rb2.load_state_dict(saved)
    assert (rb2.seed, rb2.batch_size) == (3, 64)
    assert (len(rb2), rb2.position) == (len(rb), rb.position)
    assert blob_equal(rb2.state_dict(), saved)
    for _ in range(5):
        i1, i2 = rb.sample_indices(), rb2.sample_indices()
        assert torch.equal(i1, i2)
        e1, e2 = rb.stack_exp(i1, ep_stats=True), rb2.stack_exp(i2, ep_stats=True)
        for key in e1:
            assert same_bits(e1[key], e2[key]), key
    env2.load_state_dict(env.state_dict())
    fill_ring(S, env, rb, 2, 3)
    fill_ring(S, env2, rb2, 2, 3)
    assert (len(rb2), rb2.position) == (len(rb), rb.position)
    assert blob_equal(rb.state_dict(), rb2.state_dict())


@gpu
def test_corrupted_ring_blobs_are_refused(S):
    n = 4096
    env = S.SnakeGame(n)
    rb = S.ReplayBuffer(1000, 0)
    fill_ring(S, env, rb, 3, 0)
    good = rb.state_dict()
    slot = 321
    for byte, value, words in ((0, 3, "action index"), (1, 2, "done"), (2, 8, "mask bits"), (3, 4, "previous direction")):
        blob = good["blob"].clone()
        blob[REPLAY_HEADER + 128 * slot + 100 + byte] = value
        blob[REPLAY_HEADER + 128 * (slot + 500) + 100] = 3    # a later bad record: the lowest is reported
        with pytest.raises(S.SnakeB200Error) as ei:
            rb.load_state_dict(dict(good, blob=blob))
        assert "error -1" in str(ei.value) and words in str(ei.value) and ei.value.first_bad == slot, words
        assert blob_equal(rb.state_dict(), good)
    bad_magic = good["blob"].clone()
    bad_magic[3] ^= 1
    for blob, words in ((bad_magic, "magic"), (good["blob"][:39], "truncated"), (good["blob"][:-128], "blob of")):
        with pytest.raises(S.SnakeB200Error, match=words):
            rb.load_state_dict(dict(good, blob=blob))
    with pytest.raises(S.SnakeB200Error, match="ring of 1000"):
        S.ReplayBuffer(2000, 0).load_state_dict(good)
    assert blob_equal(rb.state_dict(), good)


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_a_blob_saved_on_one_device_loads_on_another(S):
    a, b = S.SnakeGame(1000, device=0), S.SnakeGame(1000, device=1)
    play(a, 50, 0)
    b.load_state_dict(a.state_dict())
    assert blob_equal(a.state_dict(), b.state_dict())


# ---- 5. a Trainer saved and loaded continues bit for bit -------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_trainer_continues_bit_for_bit(S, precision, tmp_path):
    K, M = 20, 30
    tr = S.train.Trainer(n_envs=4096, precision=precision, fill=8192, target_sync=7, seed=1)
    tr.fill_buffer()
    for _ in range(K):
        tr.iteration()
    path = str(tmp_path / "run.pt")
    tr.save(path)
    for _ in range(M):
        tr.iteration()
    tr2 = S.train.Trainer.load(path, device=0, n_envs=4096, capacity=50000, batch_size=64, precision=precision)
    assert tr2.n_updates == K
    for _ in range(M):
        tr2.iteration()
    assert tr2.n_updates == K + M                             # crosses target syncs at 21 and 28 ...
    assert same_bits(tr.q_net.theta_device, tr2.q_net.theta_device)
    assert same_bits(tr.t_net.theta_device, tr2.t_net.theta_device)
    assert same_bits(tr.opt.acc, tr2.opt.acc)
    assert same_bits(torch.stack(tr.losses), torch.stack(tr2.losses))
    assert same_bits(tr.episode_returns(), tr2.episode_returns())
    assert tr.epsilon == tr2.epsilon and tr.stored == tr2.stored
    assert blob_equal(tr.env.state_dict(), tr2.env.state_dict())
    assert blob_equal(tr.replay.state_dict(), tr2.replay.state_dict())
    with pytest.raises(ValueError, match="n_envs"):
        S.train.Trainer.load(path, n_envs=1024)


# ---- 6. without a GPU: argument checks ------------------------------------------------------------------------------------
def test_checkpoint_entry_points_check_their_arguments(S):
    L = S.lib()
    size, bad = C.c_size_t(7), C.c_int64(5)
    buf = (C.c_uint8 * 64)()
    for fn in (L.snk_env_checkpoint_bytes, L.snk_replay_checkpoint_bytes):
        assert fn(None, C.byref(size)) == -1 and fn(None, None) == -1
    for fn in (L.snk_env_save_host, L.snk_replay_save_host):
        assert fn(None, None, 0) == -1 and fn(None, buf, 64) == -1
    for fn in (L.snk_env_load_host, L.snk_replay_load_host):
        bad.value = 5
        assert fn(None, buf, 64, C.byref(bad)) == -1 and bad.value == -1
        assert fn(None, None, 0, None) == -1
    assert L.snk_version() == 200


def test_malformed_state_dicts_are_refused_before_the_library(S):
    env = object.__new__(S.SnakeGame)
    env._h = C.c_void_p()
    for d in (None, {}, {"blob": torch.zeros(8)}, {"blob": torch.zeros(2, 4, dtype=torch.uint8)}, {"blob": [1, 2]}):
        with pytest.raises(ValueError):
            env.load_state_dict(d)
    with pytest.raises(S.SnakeB200Error, match="null handle") as ei:     # well formed: the library refuses the null handle
        env.load_state_dict({"blob": torch.zeros(176, dtype=torch.uint8)})
    assert ei.value.first_bad == -1
    rb = object.__new__(S.ReplayBuffer)
    rb._r, rb.capacity = C.c_void_p(), 1000
    for d in ({"blob": torch.zeros(40, dtype=torch.uint8)}, {"blob": torch.zeros(40, dtype=torch.uint8), "seed": 0, "batch_size": 2000}):
        with pytest.raises(ValueError):
            rb.load_state_dict(d)
    opt = S.qnet.RMSProp()
    for d in ({}, {"eta": 1, "rho": 0.9, "epsilon": 1e-8, "acc": None},
              {"eta": 5e-4, "rho": 0.9, "epsilon": 1e-8, "acc": torch.zeros(10)}):
        with pytest.raises(ValueError):
            opt.load_state_dict(d, "cpu")
    opt.load_state_dict({"eta": 1e-3, "rho": 0.5, "epsilon": 1e-6, "acc": torch.ones(S.qnet.N_PARAMS)}, "cpu")
    assert opt.state_dict()["eta"] == 1e-3 and torch.equal(opt.acc, torch.ones(S.qnet.N_PARAMS))
    net = object.__new__(S.qnet.QNet)
    net.precision = "f32"
    with pytest.raises(ValueError):
        net.load_state_dict({"theta": torch.zeros(S.qnet.N_PARAMS), "precision": "bf16"})
    with pytest.raises(ValueError):
        net.load_params(np.zeros(10, np.float32))
    with pytest.raises(ValueError):
        net.load_params(np.zeros(S.qnet.N_PARAMS, np.float64))
    tr = object.__new__(S.train.Trainer)
    with pytest.raises(ValueError, match="missing"):
        tr.load_state_dict({"n_envs": 4096})


def test_trainer_load_refuses_other_shapes_before_building(S, tmp_path):
    path = str(tmp_path / "t.pt")
    torch.save({"n_envs": 4096, "capacity": 50000, "batch_size": 64, "precision": "f32"}, path)
    for kw, key in (({"n_envs": 1024}, "n_envs"), ({"capacity": 1000}, "capacity"), ({"batch_size": 32}, "batch_size"),
                    ({"precision": "bf16"}, "precision")):
        with pytest.raises(ValueError, match=key):
            S.train.Trainer.load(path, **kw)
    torch.save({"something": 1}, path)
    with pytest.raises(ValueError, match="not a Trainer checkpoint"):
        S.train.Trainer.load(path)
