"""The reference's Q-network (structs.jl:127-139) on the device — native kernels only.

    Conv((3,3), 2=>16, relu; pad=1) -> Conv((3,3), 16=>32, relu; pad=1) -> Conv((6,6), 32=>64, relu) ->
    Flux.flatten -> Dense(1600, 64, relu) -> Dense(64, 3)

`QNet` hands Flux.destructure(q_net) to snk_qnet_create and runs snk_qnet_forward (tcgen05 implicit-GEMM convolutions,
csrc/qnet.cu).  precision="f32" (default) is the Float32-faithful mode the reference's Float32 network needs for
identical greedy actions; precision="bf16" is the fast, lower-precision mode.  QNet.train_step with an RMSProp is the learner of train!
(utils.jl:452-466) on the device; load_params_from is update_target_net!.  There is no library (cuDNN) path in the
product: the torch restatement used as a timing baseline and cross-check lives in tools/torch_qnet.py.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import bson_io

SHAPES = [("conv", (3, 3, 2, 16), 1), ("conv", (3, 3, 16, 32), 1), ("conv", (6, 6, 32, 64), 0),
          ("dense", (64, 1600), None), ("dense", (3, 64), None)]
N_PARAMS = 181395
PRECISIONS = {"bf16": 0, "f32": 1}            # SNK_QNET_BF16, SNK_QNET_F32 (include/snake_b200.h)
PRECISION_NOTES = {
    "f32": "Float32-faithful: fp16 (hi, lo) split operands, four partial products on tcgen05, FP32 accumulation",
    "bf16": "bf16 operands on tcgen05, FP32 accumulation: ~1.5e-2 of max|Q|, NOT the reference's Float32 fidelity",
}


def glorot_layers(seed=0, in_frames=2):
    """Flux's default init: Glorot-uniform weights, zero bias (seeded, synthetic: the two-frame checkpoints named
    by BASELINE config 4 are missing from the reference mount)."""
    rng = np.random.default_rng(seed)
    layers = []
    for kind, shp, pad in SHAPES:
        if kind == "conv":
            k1, k2, cin, cout = shp
            if cin == 2:
                cin = in_frames
            fan_in, fan_out = k1 * k2 * cin, k1 * k2 * cout
            lim = math.sqrt(6.0 / (fan_in + fan_out))
            layers.append(("conv", {"W": rng.uniform(-lim, lim, (k1, k2, cin, cout)).astype(np.float32),
                                    "b": np.zeros(cout, np.float32), "pad": [pad, pad], "stride": [1, 1]}))
            if shp[0] == 6:
                layers.append(("flatten", {}))
        else:
            out, inn = shp
            lim = math.sqrt(6.0 / (inn + out))
            layers.append(("dense", {"W": rng.uniform(-lim, lim, (out, inn)).astype(np.float32),
                                     "b": np.zeros(out, np.float32)}))
    return layers


class QNet:
    """q_net / t_net of DQNModel (structs.jl:120-147) as a callable: obs (N,2,10,10) f32 [= Julia (10,10,2,N)] -> Q (N,3)."""

    def __init__(self, layers, device, precision="f32"):
        from . import _check, lib
        if precision not in PRECISIONS:
            raise ValueError("precision must be 'f32' or 'bf16'")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("QNet runs on a CUDA device only (no CPU fallback)")
        self.precision = precision
        self._theta = np.ascontiguousarray(bson_io.destructure(layers), dtype=np.float32)
        if self._theta.size != N_PARAMS:
            raise ValueError("the native Q-net is the two-frame network of structs.jl:127-139 (%d parameters), got %d"
                             % (N_PARAMS, self._theta.size))
        self.n_params = int(self._theta.size)
        self._updated = False          # theta changed on the device since create (train_step / load_params_from)
        self._q = C.c_void_p()
        _check(lib().snk_qnet_create(C.byref(self._q), self._theta.ctypes.data_as(C.c_void_p), self._theta.size,
                                     self.device.index or 0, PRECISIONS[precision]))

    def close(self):
        if getattr(self, "_q", None):
            try:
                from . import lib
                lib().snk_qnet_destroy(self._q)
            except Exception:          # interpreter shutdown: module globals may already be gone
                pass
            self._q = None

    __del__ = close

    @classmethod
    def from_trainer_bson(cls, path, device, which="q_net", precision="f32"):
        """q_net / t_net of ./trainers/<name>.bson (load_trainer, utils.jl:413-418)"""
        q, t = bson_io.load_trainer_nets(path)
        return cls(q if which == "q_net" else t, device, precision)

    def forward(self, obs, out=None):
        """snk_qnet_forward: obs (N,2,10,10) float32 contiguous -> Q (N,3) float32 [= Julia (3,N)]"""
        from . import _check, _ptr, lib
        n = obs.shape[0]
        if out is None:
            out = torch.empty(n, 3, dtype=torch.float32, device=self.device)
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _check(lib().snk_qnet_forward(self._q, _ptr(obs, torch.float32, n * 200, self.device), n,
                                      _ptr(out, torch.float32, 3 * n, self.device), st))
        return out

    __call__ = forward

    def sample_grads(self, states, actions, targets, planes=None, want_J=False, want_loss=True):
        """Per-sample gradients of huber(q_net(s_i)[a_i], y_i) (utils.jl:452-466), FP32, Flux.destructure order.
        states (B,2,10,10) f32, actions (B) u8 (0-based), targets (B) f64 — as ReplayBuffer.stack_exp / masked_target give.
        planes: (hi_ptr, lo_ptr, pitch) of bf16 Gram planes to fill (GramShard.planes(), GramPlan.planes()) or None.
        Returns dict(J (B, 181395) f32 if want_J, loss (B) f32 if want_loss)."""
        from . import _check, _ptr, lib
        B = states.shape[0]
        dev = self.device
        out = {}
        if want_J:
            out["J"] = torch.empty(B, N_PARAMS, dtype=torch.float32, device=dev)
        if want_loss:
            out["loss"] = torch.empty(B, dtype=torch.float32, device=dev)
        hi, lo, pitch = (C.c_void_p(planes[0]), C.c_void_p(planes[1]), int(planes[2])) if planes is not None else (None, None, 0)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _check(lib().snk_qnet_sample_grads(self._q, _ptr(states, torch.float32, B * 200, dev), _ptr(actions, torch.uint8, B, dev),
                                           _ptr(targets, torch.float64, B, dev), B, hi, lo, pitch, _ptr(out.get("J")), N_PARAMS,
                                           _ptr(out.get("loss")), st))
        return out

    @property
    def theta(self):
        """Flux.destructure(q_net): (181,395) float32 numpy array of the current parameters (downloaded after an update)."""
        if self._updated:
            return self.theta_device.cpu().numpy()
        return self._theta

    @property
    def theta_device(self):
        """The net's own parameters on the device, (181,395) float32 in Flux.destructure order: a view, read-only, that changes
        with every train_step / load_params_from."""
        from . import _check, lib
        p = C.c_void_p()
        _check(lib().snk_qnet_params(self._q, C.byref(p)))
        return torch.as_tensor(_ParamsView(self, p.value), device=self.device)

    def train_step(self, states, actions, targets, opt, want_grad=False):
        """One minibatch update (utils.jl:452-466): Flux.gradient of mean(huber(q_net(s)[a], y)) and update!(opt, theta, g),
        on the device; every layout of this net (both forward precisions, sample_grads) follows the new theta.
        states (B,2,10,10) f32, actions (B) u8 (0-based), targets (B) f64 as for sample_grads; opt an RMSProp.
        Returns (loss, g): loss a 0-d f32 tensor (the batch mean), g (181,395) f32 if want_grad else None.  Enqueued on the
        current stream."""
        from . import _check, _ptr, lib
        B = states.shape[0]
        dev = self.device
        acc = opt.state(dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        g = torch.empty(N_PARAMS, dtype=torch.float32, device=dev) if want_grad else None
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _check(lib().snk_qnet_train_step(self._q, _ptr(states, torch.float32, B * 200, dev), _ptr(actions, torch.uint8, B, dev),
                                         _ptr(targets, torch.float64, B, dev), B, _ptr(acc, torch.float32, N_PARAMS, dev),
                                         opt.eta, opt.rho, opt.epsilon, _ptr(g), _ptr(loss), st))
        self._updated = True
        return loss, g

    def load_params_from(self, other):
        """update_target_net! (utils.jl:469-472): this net's parameters become a copy of `other`'s (a QNet on the same device,
        either precision), on the device, enqueued on the current stream."""
        from . import _check, lib
        if other.device != self.device:
            raise ValueError("load_params_from: nets on %s and %s" % (other.device, self.device))
        p = C.c_void_p()
        _check(lib().snk_qnet_params(other._q, C.byref(p)))
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _check(lib().snk_qnet_set_params(self._q, p, st))
        self._updated = True

    def load_params(self, theta):
        """θ = theta: (181,395) float32, a tensor on any device or a numpy array, in Flux.destructure order; every layout
        re-derived on the device (snk_qnet_set_params), enqueued on the current stream."""
        from . import _check, _ptr, lib
        t = torch.as_tensor(theta)
        if t.dtype != torch.float32 or t.numel() != N_PARAMS:
            raise ValueError("load_params: theta must be %d float32 values, got %d %s" % (N_PARAMS, t.numel(), t.dtype))
        t = t.reshape(-1).to(self.device).contiguous()
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _check(lib().snk_qnet_set_params(self._q, _ptr(t, torch.float32, N_PARAMS, self.device), st))
        self._updated = True

    def state_dict(self):
        """{'theta': (181,395) f32 CPU tensor, 'precision'}"""
        return {"theta": self.theta_device.cpu(), "precision": self.precision}

    def load_state_dict(self, d):
        """θ of a state_dict(); the precision must be this net's"""
        if not isinstance(d, dict) or "theta" not in d or d.get("precision") != self.precision:
            raise ValueError("a QNet state_dict of precision %r with 'theta' is required" % self.precision)
        self.load_params(d["theta"])

    def overflow(self):
        """f32 mode: True if an activation left the fp16 range of the split operands since the last call (synchronises)."""
        from . import _check, lib
        f = C.c_int(0)
        _check(lib().snk_qnet_overflow_host(self._q, C.byref(f)))
        return bool(f.value)


GROUP_HANDLE_BYTES = 64          # SNK_QNET_GROUP_HANDLE_BYTES


class LearnerGroup:
    """One rank of a data-parallel learner (snk_qnet_group, DESIGN §5f): R ranks, each with its own QNet holding the same θ and
    its own local minibatch.  train_step continues the Float64 running sum of the gradient rows that rank - 1 published and
    every rank applies the sum of rank R - 1, so after each update every rank holds the same θ, acc, g and loss, equal bit for
    bit to QNet.train_step on the ranks' minibatches concatenated in rank order.  The ranks wait for each other on the
    device.  Set-up: handle() on every rank, then connect(every rank's handle, in rank order)."""

    def __init__(self, net, world, rank):
        from . import _check, lib
        self.net, self.world, self.rank = net, int(world), int(rank)
        self._g = C.c_void_p()
        _check(lib().snk_qnet_group_create(C.byref(self._g), net._q, self.world, self.rank))

    def handle(self):
        """this rank's 64-byte handle (bytes), to be sent to every other rank"""
        from . import _check, lib
        h = (C.c_uint8 * GROUP_HANDLE_BYTES)()
        _check(lib().snk_qnet_group_export_host(self._g, h))
        return bytes(h)

    def connect(self, handles):
        """handles: every rank's handle() in rank order (this rank's own entry is ignored)"""
        from . import _check, lib
        blob = b"".join(bytes(h) for h in handles)
        _check(lib().snk_qnet_group_connect_host(self._g, (C.c_uint8 * len(blob)).from_buffer_copy(blob),
                                                 len(handles)))

    def train_step(self, states, actions, targets, opt, want_grad=False):
        """QNet.train_step of this rank's B_r transitions as part of the group's update; (loss, g) are the whole update's
        (the same on every rank).  Enqueued on the current stream; every rank must call it the same number of times."""
        from . import _check, _ptr, lib
        net, dev = self.net, self.net.device
        B = states.shape[0]
        acc = opt.state(dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        g = torch.empty(N_PARAMS, dtype=torch.float32, device=dev) if want_grad else None
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _check(lib().snk_qnet_group_train_step(self._g, _ptr(states, torch.float32, B * 200, dev), _ptr(actions, torch.uint8, B, dev),
                                               _ptr(targets, torch.float64, B, dev), B, _ptr(acc, torch.float32, N_PARAMS, dev),
                                               opt.eta, opt.rho, opt.epsilon, _ptr(g), _ptr(loss), st))
        net._updated = True
        return loss, g

    def check(self):
        """raises if a wait of this rank gave up on a peer (synchronises)"""
        from . import _check, lib
        t = C.c_int(0)
        _check(lib().snk_qnet_group_status_host(self._g, C.byref(t)))

    def close(self):
        if getattr(self, "_g", None):
            try:
                from . import lib
                lib().snk_qnet_group_destroy(self._g)
            except Exception:          # interpreter shutdown
                pass
            self._g = None

    __del__ = close


class LocalLearnerGroup:
    """R virtual ranks of a LearnerGroup in ONE process on ONE GPU (connect_local), each driven from its own stream: the
    ranks order themselves on the device, so the host may enqueue them in any order.  For tests on a single B200."""

    def __init__(self, nets):
        from . import _check, lib
        world = len(nets)
        self.groups = [LearnerGroup(n, world, r) for r, n in enumerate(nets)]
        self.streams = [torch.cuda.Stream(n.device) for n in nets]
        arr = (C.c_void_p * world)(*[g._g.value for g in self.groups])
        for g in self.groups:
            _check(lib().snk_qnet_group_connect_local(g._g, arr, world))

    def train_step(self, batches, opts, want_grad=False, order=None):
        """batches[r] = (states, actions, targets) of rank r, opts[r] its RMSProp; the ranks are enqueued in `order` (default
        0 .. R-1).  Returns [(loss, g)] per rank; the current stream waits for all of them."""
        cur = torch.cuda.current_stream(self.groups[0].net.device)
        out = [None] * len(self.groups)
        for r in (range(len(self.groups)) if order is None else order):
            s = self.streams[r]
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                out[r] = self.groups[r].train_step(*batches[r], opts[r], want_grad)
        for s in self.streams:
            cur.wait_stream(s)
        return out

    def check(self):
        for g in self.groups:
            g.check()

    def close(self):
        for g in self.groups:
            g.close()


class DistributedLearnerGroup(LearnerGroup):
    """This process's rank of a LearnerGroup over torch.distributed (one process per GPU): the 64-byte handles travel through
    all_gather_object once, the only thing torch.distributed is used for; updates need no communicator."""

    def __init__(self, net, group=None):
        import torch.distributed as dist
        super().__init__(net, dist.get_world_size(group), dist.get_rank(group))
        handles = [None] * self.world
        dist.all_gather_object(handles, self.handle(), group=group)
        self.connect(handles)


class _ParamsView:
    """__cuda_array_interface__ of a QNet's device theta; keeps the net alive as long as a tensor views it."""

    def __init__(self, net, ptr):
        self.net = net
        self.__cuda_array_interface__ = {"shape": (N_PARAMS,), "typestr": "<f4", "data": (ptr, False), "version": 3,
                                         "strides": None, "stream": None}


class RMSProp:
    """Flux.Optimise.RMSProp(eta, rho, epsilon) of the reference's trainer (structs.jl:137: RMSProp(5e-4), stored as
    (0.0005, 0.9, 1e-8)).  `acc` is its state for theta: (181,395) f32 on the net's device, zero on the first update (a fresh
    optimiser); an ordinary tensor, so it can be saved and restored with the parameters."""

    def __init__(self, eta=5e-4, rho=0.9, epsilon=1e-8, acc=None):
        self.eta, self.rho, self.epsilon = float(eta), float(rho), float(epsilon)
        self.acc = acc

    def state(self, device):
        if self.acc is None:
            self.acc = torch.zeros(N_PARAMS, dtype=torch.float32, device=device)
        return self.acc

    def state_dict(self):
        """{'eta', 'rho', 'epsilon', 'acc': (181,395) f32 CPU tensor, or None before the first update}"""
        return {"eta": self.eta, "rho": self.rho, "epsilon": self.epsilon, "acc": None if self.acc is None else self.acc.cpu()}

    def load_state_dict(self, d, device):
        """the hyper-parameters and `acc` of a state_dict(); acc goes to `device` (the net's)"""
        if not isinstance(d, dict) or not all(isinstance(d.get(k), float) for k in ("eta", "rho", "epsilon")) or "acc" not in d:
            raise ValueError("an RMSProp state_dict holds the floats 'eta', 'rho', 'epsilon' and 'acc'")
        acc = d["acc"]
        if acc is not None and (not isinstance(acc, torch.Tensor) or acc.dtype != torch.float32 or acc.numel() != N_PARAMS):
            raise ValueError("RMSProp acc must be None or %d float32 values" % N_PARAMS)
        self.eta, self.rho, self.epsilon = d["eta"], d["rho"], d["epsilon"]
        self.acc = None if acc is None else acc.reshape(-1).to(device, copy=True).contiguous()
