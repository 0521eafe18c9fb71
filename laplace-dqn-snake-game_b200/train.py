"""train! (utils.jl:420-494) with every array on the device.

    fill_buffer!(tr)                        (:389-402)  Rollout.step() with fill_epsilon until more than `fill` transitions
    loop                                    (:434-482)  play, then `updates_per_step` times:
        sample + stack_exp                  (:442-443)  ReplayBuffer.sample()
        t_net(next_states), masked target   (:448-451)  masked_target(...)  (gamma 0.97)
        Flux.gradient + update!(RMSProp)    (:452-466)  QNet.train_step(..., RMSProp(5e-4, 0.9, 1e-8))
        update_target_net! every 1,000      (:469-472)  t_net.load_params_from(q_net)
        epsilon decay                       (:480)      epsilon = max(0.05, epsilon - 1e-6) per batch
    save_trainer / load_trainer             (:408-418)  Trainer.save(path) / Trainer.load(path): a run continued from a
                                                        checkpoint computes the bits of the run that never stopped

Data parallelism (DESIGN §5f): Trainer(world=R, rank=r) is rank r of R trainers, one per GPU.  Each plays its own n_envs
games into its own replay ring (the ring's and the games' seeds are derived from (seed, rank)) and samples batch_size
transitions from it; the update goes through a LearnerGroup, so every rank applies the same update: QNet.train_step of the
R minibatches concatenated in rank order.  epsilon, the target-sync counter and the target net stay per rank and agree
everywhere because θ does.  Deviation: the global minibatch is stratified over the ranks' rings, not uniform over their
union.  Before the first update the ranks are connected: connect(every rank's handle()) or Trainer.connect_local.

Deviation from the reference: it plays one whole episode of one game per update; here one play is one Rollout.step(), which
advances each of the N games by one step (and stores N transitions), followed by `updates_per_step` updates.  The ratio of
transitions to updates is therefore N / updates_per_step per play instead of one episode's length.
"""
import ctypes as C

import torch

from . import ReplayBuffer, SnakeGame, _check, lib, masked_target
from .qnet import LearnerGroup, QNet, RMSProp, glorot_layers
from .rollout import Rollout

ENV_SEED = 42                          # SnakeGame's default seed


def rank_seed(seed, rank):
    """the seed rank `rank` of a data-parallel run uses where a single-process run uses `seed` (rank 0: `seed` itself)"""
    return int(seed) if rank == 0 else (int(seed) + 0x9E3779B97F4A7C15 * int(rank)) % 2 ** 64


class Trainer:
    def __init__(self, n_envs=4096, device=0, layers=None, precision="f32", capacity=50000, batch_size=64, gamma=0.97,
                 eta=5e-4, rho=0.9, opt_epsilon=1e-8, epsilon=1.0, epsilon_min=0.05, epsilon_decay=1e-6,
                 target_sync=1000, fill=50000, fill_epsilon=1.0, updates_per_step=1, seed=0, world=1, rank=0):
        dev = torch.device("cuda", device)
        self.precision = precision
        self.world, self.rank = int(world), int(rank)
        if layers is None:
            layers = glorot_layers(seed)                       # Flux's default init (structs.jl:127-139)
        self.q_net = QNet(layers, dev, precision)
        self.t_net = QNet(layers, dev, precision)
        # a single-process run has no group: QNet.train_step is the same update
        self.learner = LearnerGroup(self.q_net, self.world, self.rank) if self.world > 1 else None
        self.env = SnakeGame(n_envs, device=device, auto_reset=True, seed=rank_seed(ENV_SEED, self.rank))
        self.replay = ReplayBuffer(capacity, device, batch_size, rank_seed(seed, self.rank))
        self.opt = RMSProp(eta, rho, opt_epsilon)
        self.rollout = Rollout(self.env, self.q_net, self.t_net, self.replay, epsilon=fill_epsilon)
        self.gamma, self.epsilon, self.epsilon_min, self.epsilon_decay = float(gamma), float(epsilon), float(epsilon_min), float(epsilon_decay)
        self.target_sync, self.fill, self.fill_epsilon = int(target_sync), int(fill), float(fill_epsilon)
        self.updates_per_step = int(updates_per_step)
        self.n_updates = 0
        self.stored = 0                # transitions stored into the replay ring so far
        self.losses = []               # one 0-d f32 device tensor per update: the minibatch's mean Huber loss
        self.returns = []              # per play: the returns (f32, device) of the episodes that finished in it

    def handle(self):
        """this rank's learner-group handle (64 bytes), for connect() on every rank"""
        return self.learner.handle()

    def connect(self, handles):
        """every rank's handle() in rank order"""
        self.learner.connect(handles)

    @staticmethod
    def connect_local(trainers):
        """wire the trainers of ONE process together as virtual ranks 0 .. R-1 on one GPU.  Each must be built and run with
        its own stream current, and the host must not wait on one rank's stream before every rank has enqueued its update
        (e.g. all ranks play, then all ranks update)."""
        arr = (C.c_void_p * len(trainers))(*[t.learner._g.value for t in trainers])
        for t in trainers:
            _check(lib().snk_qnet_group_connect_local(t.learner._g, arr, len(trainers)))

    def _play(self, epsilon):
        self.rollout.epsilon = epsilon
        res = self.rollout.step()
        self.stored += self.env.n
        self.returns.append(res["ep_return"][res["done"].bool()])
        return res

    def fill_buffer(self):
        """fill_buffer! (utils.jl:389-402): play until more than `fill` transitions were stored"""
        while self.stored <= self.fill:
            self._play(self.fill_epsilon)

    def update(self):
        """one minibatch update (utils.jl:442-480)"""
        b = self.replay.sample()
        y = masked_target(self.t_net(b["next_states"]), b["mask"], b["rewards"], b["dones"], gamma=self.gamma)
        learner = self.learner if self.learner is not None else self.q_net
        loss, _ = learner.train_step(b["states"], b["actions"], y, self.opt)
        self.losses.append(loss)
        self.n_updates += 1
        if self.n_updates % self.target_sync == 0:
            self.t_net.load_params_from(self.q_net)
        self.epsilon = max(self.epsilon_min, self.epsilon - self.epsilon_decay)
        return loss

    def iteration(self):
        """one play followed by updates_per_step updates"""
        self._play(self.epsilon)
        for _ in range(self.updates_per_step):
            self.update()

    def train(self, n_batches):
        """train! until n_batches updates in all (fills the buffer first if it was not filled yet)"""
        self.fill_buffer()
        while self.n_updates < n_batches:
            self.iteration()

    def episode_returns(self):
        """the returns of every episode finished so far, in order (f32, device)"""
        return torch.cat(self.returns) if self.returns else torch.empty(0, dtype=torch.float32, device=self.q_net.device)

    # -- checkpoints (save_trainer / load_trainer, utils.jl:408-418) ------------------------------------------------------
    _HYPER = ("gamma", "epsilon_min", "epsilon_decay", "target_sync", "fill", "fill_epsilon", "updates_per_step")
    _SHAPE = ("n_envs", "capacity", "batch_size", "precision")
    _RANK = (("world", 1), ("rank", 0))          # a checkpoint without them is a single-process run's

    def state_dict(self):
        """Everything train() depends on, as CPU tensors and plain numbers: the hyper-parameters, the counters, the loss and
        return histories (concatenated), both nets, the optimiser, the games and the replay ring."""
        dev = self.q_net.device
        return {
            "n_envs": self.env.n, "capacity": self.replay.capacity, "batch_size": self.replay.batch_size, "precision": self.precision,
            "world": self.world, "rank": self.rank,
            **{k: getattr(self, k) for k in self._HYPER},
            "n_updates": self.n_updates, "stored": self.stored, "epsilon": self.epsilon,
            "losses": (torch.stack(self.losses) if self.losses else torch.empty(0, dtype=torch.float32, device=dev)).cpu(),
            "returns": self.episode_returns().cpu(),
            "q_net": self.q_net.state_dict(), "t_net": self.t_net.state_dict(), "opt": self.opt.state_dict(),
            "env": self.env.state_dict(), "replay": self.replay.state_dict(),
        }

    def load_state_dict(self, d):
        """Continue the run a state_dict() was taken of; it must have this trainer's N, capacity, batch size, precision, world
        and rank."""
        keys = self._SHAPE + self._HYPER + ("n_updates", "stored", "epsilon", "losses", "returns", "q_net", "t_net", "opt", "env", "replay")
        if not isinstance(d, dict) or any(k not in d for k in keys):
            raise ValueError("not a Trainer state_dict: missing %s" % [k for k in keys if not isinstance(d, dict) or k not in d])
        mine = (self.env.n, self.replay.capacity, self.replay.batch_size, self.precision)
        for k, v in zip(self._SHAPE, mine):
            if d[k] != v:
                raise ValueError("checkpoint has %s = %r, this trainer %r" % (k, d[k], v))
        for k, default in self._RANK:
            if d.get(k, default) != getattr(self, k):
                raise ValueError("checkpoint has %s = %r, this trainer %r" % (k, d.get(k, default), getattr(self, k)))
        for k in ("losses", "returns"):
            if not isinstance(d[k], torch.Tensor) or d[k].dtype != torch.float32 or d[k].dim() != 1:
                raise ValueError("%s must be a 1-d float32 tensor" % k)
        dev = self.q_net.device
        self.env.load_state_dict(d["env"])
        self.replay.load_state_dict(d["replay"])
        self.q_net.load_state_dict(d["q_net"])
        self.t_net.load_state_dict(d["t_net"])
        self.opt.load_state_dict(d["opt"], dev)
        for k in self._HYPER:
            setattr(self, k, type(getattr(self, k))(d[k]))
        self.n_updates, self.stored, self.epsilon = int(d["n_updates"]), int(d["stored"]), float(d["epsilon"])
        self.losses = list(d["losses"].to(dev).unbind())
        self.returns = [d["returns"].to(dev)] if d["returns"].numel() else []
        # the acting state of the next play: snk_state equals the patched next_state the uninterrupted run acts on (DESIGN §4)
        self.env.assemble_state("f32", out=self.rollout.out["obs"])
        self.rollout._patch = False

    def save(self, path):
        torch.save(self.state_dict(), path)

    @classmethod
    def load(cls, path, device=0, n_envs=None, capacity=None, batch_size=None, precision=None, world=None, rank=None):
        """A Trainer continuing the run saved at path (torch.load with weights_only=True).  n_envs, capacity, batch_size,
        precision, world, rank: when given, a checkpoint with other values is refused (ValueError).  A rank of a group run
        must then be connected again before its next update."""
        d = torch.load(path, map_location="cpu", weights_only=True)
        if not isinstance(d, dict) or any(k not in d for k in cls._SHAPE):
            raise ValueError("%s is not a Trainer checkpoint" % path)
        got = {k: d[k] for k in cls._SHAPE}
        got.update({k: d.get(k, default) for k, default in cls._RANK})
        for k, want in zip(cls._SHAPE + ("world", "rank"), (n_envs, capacity, batch_size, precision, world, rank)):
            if want is not None and got[k] != want:
                raise ValueError("checkpoint has %s = %r, %r was asked for" % (k, got[k], want))
        tr = cls(n_envs=d["n_envs"], device=device, precision=d["precision"], capacity=d["capacity"], batch_size=d["batch_size"],
                 world=got["world"], rank=got["rank"])
        tr.load_state_dict(d)
        return tr
