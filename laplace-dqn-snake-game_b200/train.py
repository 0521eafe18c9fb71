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

Deviation from the reference: it plays one whole episode of one game per update; here one play is one Rollout.step(), which
advances each of the N games by one step (and stores N transitions), followed by `updates_per_step` updates.  The ratio of
transitions to updates is therefore N / updates_per_step per play instead of one episode's length.
"""
import torch

from . import ReplayBuffer, SnakeGame, masked_target
from .qnet import QNet, RMSProp, glorot_layers
from .rollout import Rollout


class Trainer:
    def __init__(self, n_envs=4096, device=0, layers=None, precision="f32", capacity=50000, batch_size=64, gamma=0.97,
                 eta=5e-4, rho=0.9, opt_epsilon=1e-8, epsilon=1.0, epsilon_min=0.05, epsilon_decay=1e-6,
                 target_sync=1000, fill=50000, fill_epsilon=1.0, updates_per_step=1, seed=0):
        dev = torch.device("cuda", device)
        self.precision = precision
        if layers is None:
            layers = glorot_layers(seed)                       # Flux's default init (structs.jl:127-139)
        self.q_net = QNet(layers, dev, precision)
        self.t_net = QNet(layers, dev, precision)
        self.env = SnakeGame(n_envs, device=device, auto_reset=True)
        self.replay = ReplayBuffer(capacity, device, batch_size, seed)
        self.opt = RMSProp(eta, rho, opt_epsilon)
        self.rollout = Rollout(self.env, self.q_net, self.t_net, self.replay, epsilon=fill_epsilon)
        self.gamma, self.epsilon, self.epsilon_min, self.epsilon_decay = float(gamma), float(epsilon), float(epsilon_min), float(epsilon_decay)
        self.target_sync, self.fill, self.fill_epsilon = int(target_sync), int(fill), float(fill_epsilon)
        self.updates_per_step = int(updates_per_step)
        self.n_updates = 0
        self.stored = 0                # transitions stored into the replay ring so far
        self.losses = []               # one 0-d f32 device tensor per update: the minibatch's mean Huber loss
        self.returns = []              # per play: the returns (f32, device) of the episodes that finished in it

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
        loss, _ = self.q_net.train_step(b["states"], b["actions"], y, self.opt)
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

    def state_dict(self):
        """Everything train() depends on, as CPU tensors and plain numbers: the hyper-parameters, the counters, the loss and
        return histories (concatenated), both nets, the optimiser, the games and the replay ring."""
        dev = self.q_net.device
        return {
            "n_envs": self.env.n, "capacity": self.replay.capacity, "batch_size": self.replay.batch_size, "precision": self.precision,
            **{k: getattr(self, k) for k in self._HYPER},
            "n_updates": self.n_updates, "stored": self.stored, "epsilon": self.epsilon,
            "losses": (torch.stack(self.losses) if self.losses else torch.empty(0, dtype=torch.float32, device=dev)).cpu(),
            "returns": self.episode_returns().cpu(),
            "q_net": self.q_net.state_dict(), "t_net": self.t_net.state_dict(), "opt": self.opt.state_dict(),
            "env": self.env.state_dict(), "replay": self.replay.state_dict(),
        }

    def load_state_dict(self, d):
        """Continue the run a state_dict() was taken of; it must have this trainer's N, capacity, batch size and precision."""
        keys = self._SHAPE + self._HYPER + ("n_updates", "stored", "epsilon", "losses", "returns", "q_net", "t_net", "opt", "env", "replay")
        if not isinstance(d, dict) or any(k not in d for k in keys):
            raise ValueError("not a Trainer state_dict: missing %s" % [k for k in keys if not isinstance(d, dict) or k not in d])
        mine = (self.env.n, self.replay.capacity, self.replay.batch_size, self.precision)
        for k, v in zip(self._SHAPE, mine):
            if d[k] != v:
                raise ValueError("checkpoint has %s = %r, this trainer %r" % (k, d[k], v))
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
    def load(cls, path, device=0, n_envs=None, capacity=None, batch_size=None, precision=None):
        """A Trainer continuing the run saved at path (torch.load with weights_only=True).  n_envs, capacity, batch_size,
        precision: when given, a checkpoint with other values is refused (ValueError)."""
        d = torch.load(path, map_location="cpu", weights_only=True)
        if not isinstance(d, dict) or any(k not in d for k in cls._SHAPE):
            raise ValueError("%s is not a Trainer checkpoint" % path)
        for k, want in zip(cls._SHAPE, (n_envs, capacity, batch_size, precision)):
            if want is not None and d[k] != want:
                raise ValueError("checkpoint has %s = %r, %r was asked for" % (k, d[k], want))
        tr = cls(n_envs=d["n_envs"], device=device, precision=d["precision"], capacity=d["capacity"], batch_size=d["batch_size"])
        tr.load_state_dict(d)
        return tr
