"""snake_b200 — host-side mirror of the reference's environment API over libsnake_b200.so.

The directory is called ``laplace-dqn-snake-game_b200`` (not an importable name); load it with
``__graft_entry__.load_package()`` which registers it as the module ``snake_b200``.

Julia is not available in this image, so this ctypes layer plays the role the shipped
``julia/SnakeB200.jl`` wrapper plays for a Julia host: the same function names and argument
meaning as the reference (`structs.jl`, `utils.jl`), batched over N envs, calling the identical
C symbols declared in ``include/snake_b200.h``.  torch is used only to own device memory and
streams.  There is NO CPU fallback: if the CUDA library is missing or no B200 is present every
entry point raises.
"""
import ctypes as C
import os
import warnings

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SNAKE_B200_LIB", os.path.join(_HERE, "libsnake_b200.so"))   # same override as julia/SnakeB200.jl

OBS_NONE, OBS_F32, OBS_I8, OBS_I64, OBS_PACKED2, OBS_BITS = 0, 1, 2, 3, 4, 5
AUTO_RESET = 1
ENV_ERR_FOOD, ENV_ERR_ACTION = 1, 2
_OBS = {
    "f32": (OBS_F32, torch.float32, 200), "i8": (OBS_I8, torch.int8, 200),
    "i64": (OBS_I64, torch.int64, 200), "packed2": (OBS_PACKED2, torch.uint8, 50),
    "bits": (OBS_BITS, torch.uint8, 24),          # bit-boards + the step's scalars in one 24-byte record: unpack_bits()
}


def _obs_shape(fmt, lead):
    """shape of the observations in format fmt for the leading dims `lead`: (*lead, 2, 10, 10) when one element is one cell"""
    per = _OBS[fmt][2]
    return (*lead, 2, 10, 10) if per == 200 else (*lead, per)


def _fmt_code(out):
    """obs_fmt code of an output dict: OBS_NONE when it holds no 'obs'"""
    return _OBS[out["obs_fmt"]][0] if out.get("obs") is not None else OBS_NONE


def _outputs(new, lead, obs, mask, ep_stats, act=False):
    """the output dict of a step (lead = (N,)) or a rollout (lead = (T, N)); new(shape, dtype) allocates"""
    out = {"reward": new(lead, torch.float32), "done": new(lead, torch.uint8)}
    if obs:
        out["obs"] = new(_obs_shape(obs, lead), _OBS[obs][1])
        out["obs_fmt"] = obs
    if mask:
        out["mask"] = new((*lead, 3), torch.uint8)
    if ep_stats:
        out["ep_return"] = new(lead, torch.float32)
        out["ep_score"] = new(lead, torch.int32)
    if act:
        out["act_idx"] = new(lead, torch.uint8)
    return out


def unpack_bits(rec):
    """Decodes SNK_OBS_BITS records (include/snake_b200.h): rec (N, 24) uint8, CPU or CUDA ->
    dict(state (N,2,10,10) int8 [= Julia (10,10,2,N): state[n, f, c, r]], reward (N,) f32, done (N,) u8, mask (N,3) u8 =
    next_is_suicidal, action (N,) u8).  Lossless: state equals the 'i8' observation of the same step bit for bit."""
    rec = rec.reshape(-1, 24)
    n, dev = rec.shape[0], rec.device
    shifts = torch.arange(8, device=dev, dtype=torch.uint8)
    idx = torch.arange(n, device=dev)

    def board(occ_bytes, food, head=None):
        # bitmap bit (r-1) + 8 (c-1): byte j of the little-endian u64 is column c = j + 1, its bit i is row r = i + 1
        b = torch.zeros(n, 10, 10, dtype=torch.int8, device=dev)              # [c][r]
        b[:, 0, :] = -1
        b[:, 9, :] = -1
        b[:, :, 0] = -1
        b[:, :, 9] = -1
        b[:, 1:9, 1:9] = ((occ_bytes[:, :, None] >> shifts) & 1).to(torch.int8)
        fr, fc = (food & 15).long(), (food >> 4).long()
        cur = b[idx, fc, fr]
        b[idx, fc, fr] = torch.where((food != 0) & (cur == 0), torch.full_like(cur, 2), cur)     # the snake hides the food
        if head is not None:
            b[idx, (head >> 4).long(), (head & 15).long()] = 1               # drawn last: overwrites the wall on a wall death
        return b

    state = torch.stack([board(rec[:, 0:8], rec[:, 16]), board(rec[:, 8:16], rec[:, 17], rec[:, 18])], dim=1)
    flags = rec[:, 19]
    return {"state": state, "reward": rec[:, 20:24].contiguous().view(torch.float32).reshape(n),
            "done": (flags >> 3) & 1, "mask": torch.stack([(flags >> k) & 1 for k in range(3)], dim=1),
            "action": (flags >> 4) & 3}

# direction codes in the order of utils.jl:8
U, D, L, R = 0, 1, 2, 3
DIRS = ((-1, 0), (1, 0), (0, -1), (0, 1))


class SnakeB200Error(RuntimeError):
    pass


_lib = None


def lib():
    """Loads libsnake_b200.so (built by __graft_entry__.build()); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SnakeB200Error(
            "%s not found: run `python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
            "There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i64, u32, i32, f32, f64 = C.c_void_p, C.c_int64, C.c_uint32, C.c_int, C.c_float, C.c_double
    sig = {
        "snk_create": [C.POINTER(vp), i64, i32, u32],
        "snk_destroy": [vp], "snk_reset": [vp], "snk_sync": [vp],
        "snk_set_food_list_host": [vp, vp, i32],
        "snk_default_food_list_host": [vp, C.POINTER(i32)],
        "snk_set_stream": [vp, vp], "snk_use_own_stream": [vp], "snk_get_stream": [vp, C.POINTER(vp)],
        "snk_set_seed": [vp, C.c_uint64],
        "snk_available_actions": [vp, vp],
        "snk_step": [vp, vp, vp, vp], "snk_step_abs": [vp, vp, vp, vp],
        "snk_step_fused": [vp, vp, f32, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp],
        "snk_step_fused_host": [vp, vp, f32, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp],
        "snk_rollout_fused": [vp, vp, i64, i32, vp, vp, vp, i32, vp, vp, vp],
        "snk_host_alloc": [C.POINTER(vp), C.c_size_t], "snk_host_free": [vp],
        "snk_device_alloc": [C.POINTER(vp), C.c_size_t, i32, u32, C.POINTER(i32)], "snk_device_free": [vp],
        "snk_compression_supported": [i32, C.POINTER(i32)],
        "snk_state": [vp, vp, i32], "snk_losing_mask": [vp, vp],
        "snk_state_host": [vp, vp, i32], "snk_losing_mask_host": [vp, vp], "snk_available_actions_host": [vp, vp],
        "snk_patch_reset_obs": [vp, vp, vp, i32],
        "snk_get_score_host": [vp, vp], "snk_get_done_host": [vp, vp], "snk_get_error_flags_host": [vp, vp],
        "snk_get_steps_host": [vp, vp],
        "snk_step_fused_store_host": [vp, vp, vp, f32, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp],
        "snk_replay_gather_host": [vp, vp, i64, vp, vp, vp, vp, vp, vp, vp],
        "snk_select_action": [vp, vp, f32, vp, vp, vp],
        "snk_masked_target": [vp, vp, vp, vp, f64, f32, vp, vp, i64, vp],
        "snk_get_score": [vp, vp], "snk_get_done": [vp, vp], "snk_get_error_flags": [vp, vp],
        "snk_get_steps": [vp, vp], "snk_count_errors_host": [vp, C.POINTER(i64)],
        "snk_env_checkpoint_bytes": [vp, C.POINTER(C.c_size_t)], "snk_env_save_host": [vp, vp, C.c_size_t],
        "snk_env_load_host": [vp, vp, C.c_size_t, C.POINTER(i64)],
        "snk_replay_checkpoint_bytes": [vp, C.POINTER(C.c_size_t)], "snk_replay_save_host": [vp, vp, C.c_size_t],
        "snk_replay_load_host": [vp, vp, C.c_size_t, C.POINTER(i64)],
        "snk_center_columns": [vp, i64, i64, vp, vp, vp],
        "snk_d_store_snapshot": [vp, i64, i64, i64, vp, vp],
        "snk_laplace_sample_weights": [vp, vp, vp, i64, i64, vp, vp, vp, vp],
        "snk_replay_create": [C.POINTER(vp), i64, i32], "snk_replay_destroy": [vp], "snk_replay_clear": [vp],
        "snk_replay_length": [vp, C.POINTER(i64), C.POINTER(i64)],
        "snk_step_fused_store": [vp, vp, vp, f32, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp],
        "snk_replay_gather": [vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp],
        "snk_replay_sample_indices": [vp, C.c_uint64, i64, vp, vp],
        "snk_replay_bad_index_host": [vp, C.POINTER(i32)],
        "snk_qnet_create": [C.POINTER(vp), vp, i64, i32, i32], "snk_qnet_destroy": [vp],
        "snk_qnet_forward": [vp, vp, i64, vp, vp], "snk_qnet_precision": [vp, C.POINTER(i32)],
        "snk_qnet_overflow_host": [vp, C.POINTER(i32)], "snk_qnet_debug_timing": [vp, vp],
        "snk_qnet_sample_grads": [vp, vp, vp, vp, i64, vp, vp, i64, vp, i64, vp, vp],
        "snk_qnet_train_step": [vp, vp, vp, vp, i64, vp, f64, f64, f64, vp, vp, vp],
        "snk_qnet_set_params": [vp, vp, vp], "snk_qnet_params": [vp, C.POINTER(vp)],
        "snk_qnet_group_create": [C.POINTER(vp), vp, i32, i32], "snk_qnet_group_destroy": [vp],
        "snk_qnet_group_export_host": [vp, vp], "snk_qnet_group_connect_host": [vp, vp, i32],
        "snk_qnet_group_connect_local": [vp, vp, i32],
        "snk_qnet_group_train_step": [vp, vp, vp, vp, i64, vp, f64, f64, f64, vp, vp, vp],
        "snk_qnet_group_status_host": [vp, C.POINTER(i32)],
        "snk_gram_workspace_bytes": [i64, i64, i32, C.POINTER(C.c_size_t)],
        "snk_gram_pack": [vp, i32, i64, i64, vp, vp],
        "snk_gram": [vp, i64, i64, i32, i32, i32, vp, vp],
        "snk_gram_config": [i32],
        "snk_gram_planes_layout": [i64, i64, C.POINTER(C.c_size_t), C.POINTER(i64)],
        "snk_gram_pack_planes": [vp, i32, i64, i64, vp, vp, vp],
        "snk_gram_block_scratch_bytes": [i64, i64, i64, i32, C.POINTER(C.c_size_t)],
        "snk_gram_block": [vp, vp, i64, vp, vp, i64, i64, i32, i32, i32, i32, vp, vp, i64, vp],
        "snk_gram_block_flops": [i64, i64, i64, i32, i32, C.POINTER(C.c_double)],
        "snk_gram_transpose_block": [vp, i64, i64, i64, vp, i64, vp],
        "snk_gram_shard_create": [C.POINTER(vp), vp, i32, i32, i64, i32, i32], "snk_gram_shard_destroy": [vp],
        "snk_gram_shard_export_host": [vp, vp], "snk_gram_shard_connect_host": [vp, vp],
        "snk_gram_shard_connect_local": [vp, vp],
        "snk_gram_shard_run": [vp, vp, i32, i32, i32, vp, i64, vp],
        "snk_gram_shard_pack": [vp, vp, i32, vp], "snk_gram_shard_ring": [vp, i32, i32, vp],
        "snk_gram_shard_mirror": [vp, vp, i64, vp], "snk_gram_shard_barrier": [vp, vp],
        "snk_gram_shard_schedule": [vp, i32, i32, C.POINTER(i32), vp, vp, vp, vp],
        "snk_gram_shard_planes": [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(i64)],
        "snk_gram_shard_status_host": [vp, C.POINTER(i32)],
        "snk_ipc_alloc": [C.POINTER(vp), C.c_size_t], "snk_ipc_free": [vp],
        "snk_ipc_export": [vp, vp], "snk_ipc_import": [vp, C.POINTER(vp)], "snk_ipc_close": [vp],
        "snk_copy_async": [vp, vp, C.c_size_t, vp],
    }
    for name, argtypes in sig.items():
        fn = getattr(L, name)
        fn.argtypes = argtypes
        fn.restype = i32
    L.snk_num_envs.argtypes = [vp]
    L.snk_num_envs.restype = i64
    L.snk_last_error.restype = C.c_char_p
    L.snk_version.restype = i32
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise SnakeB200Error("libsnake_b200 error %d: %s" % (rc, lib().snk_last_error().decode()))


def _save_blob(size_fn, save_fn, handle):
    """a checkpoint blob of the library (snk_*_save_host) as a uint8 CPU tensor"""
    n = C.c_size_t(0)
    _check(size_fn(handle, C.byref(n)))
    blob = torch.empty(n.value, dtype=torch.uint8)
    _check(save_fn(handle, C.c_void_p(blob.data_ptr()), n.value))
    return blob


def _load_blob(load_fn, handle, d):
    """snk_*_load_host of d['blob']; a refusal raises SnakeB200Error with the library's message and `first_bad`, the index of
    the lowest record that failed validation (-1 when the blob was refused for another reason)"""
    blob = d.get("blob") if isinstance(d, dict) else None
    if not isinstance(blob, torch.Tensor) or blob.dtype != torch.uint8 or blob.dim() != 1:
        raise ValueError("a state_dict with 'blob': a 1-d uint8 tensor (from state_dict()) is required")
    blob = blob.cpu().contiguous()
    bad = C.c_int64(-1)
    rc = load_fn(handle, C.c_void_p(blob.data_ptr()), blob.numel(), C.byref(bad))
    if rc != 0:
        err = SnakeB200Error("libsnake_b200 error %d: %s" % (rc, lib().snk_last_error().decode()))
        err.first_bad = bad.value
        raise err


def _ptr(t, dtype=None, numel=None, device=None):
    if t is None:
        return None
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise TypeError("expected %s, got %s" % (dtype, t.dtype))
    if numel is not None and t.numel() != numel:
        raise ValueError("expected %d elements, got %d" % (numel, t.numel()))
    if device is not None and t.device != device:
        raise ValueError("tensor on %s, env on %s" % (t.device, device))
    return C.c_void_p(t.data_ptr())


ALLOC_COMPRESSIBLE = 1
_compression = {}            # device index -> snk_compression_supported
_compressible = set()        # base pointers of the live compressible allocations
_deferred = []               # pointers whose free had to wait: freed by the next allocation or free outside a graph capture


def _free_deferred():
    while _deferred and not torch.cuda.is_current_stream_capturing():
        p = _deferred[-1]
        if lib().snk_device_free(C.c_void_p(p)) != 0:
            warnings.warn("snk_device_free: %s" % lib().snk_last_error().decode())
            return
        _deferred.pop()
        _compressible.discard(p)


class _DeviceBuffer:
    """Owns one snk_device_alloc allocation; torch.as_tensor() views it through __cuda_array_interface__ and keeps this
    object alive as long as any tensor sharing the memory lives.  The memory is freed with it."""

    def __init__(self, nbytes, device):
        p, comp = C.c_void_p(), C.c_int(0)
        _check(lib().snk_device_alloc(C.byref(p), nbytes, device, ALLOC_COMPRESSIBLE, C.byref(comp)))
        self.ptr = p.value
        if comp.value:
            _compressible.add(self.ptr)
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 3,
                                         "strides": None, "stream": None}

    def __del__(self):
        # freeing synchronises the device, which a CUDA graph capture does not allow: a buffer that dies while one runs on
        # this thread's current stream is freed later; a free that fails stays queued with a warning
        try:
            _deferred.append(self.ptr)
            _free_deferred()
        except Exception:              # interpreter shutdown: module globals may already be gone
            pass


def compressible_empty(shape, dtype, device):
    """torch.empty(shape, dtype, device) in device memory with generic L2 compression (snk_device_alloc): lossless, but
    data of few distinct words crosses the DRAM bus compressed.  Plain torch.empty where the device has no compression."""
    device = torch.device(device)
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _compression:
        yes = C.c_int(0)
        _check(lib().snk_compression_supported(idx, C.byref(yes)))
        _compression[idx] = bool(yes.value)
    if not _compression[idx]:
        return torch.empty(shape, dtype=dtype, device=device)
    _free_deferred()
    n = torch.Size(shape).numel() * torch.empty((), dtype=dtype).element_size()
    raw = torch.as_tensor(_DeviceBuffer(max(n, 1), idx), device=torch.device("cuda", idx))
    return raw[:n].view(dtype).view(shape)


def is_compressible(t):
    """True when tensor t lives in compressible device memory (compressible_empty / alloc_outputs)."""
    return t.untyped_storage().data_ptr() in _compressible


def default_food_list():
    """The 50 cells a fresh Xoshiro(42) yields (structs.jl:70), 1-based (row, col)."""
    buf = (C.c_uint8 * 100)()
    n = C.c_int(0)
    _check(lib().snk_default_food_list_host(buf, C.byref(n)))
    return [(buf[2 * i], buf[2 * i + 1]) for i in range(n.value)]


class SnakeGame:
    """N batched reference games (structs.jl:6-100) living in the HBM of one B200.

    Method names follow utils.jl; every array is batched with N as the LAST Julia dimension,
    i.e. the leading torch dimension: obs (N, 2, 10, 10) torch-contiguous is byte-identical to
    Julia's (10, 10, 2, N) column-major array.
    """

    def __init__(self, n_envs, device=0, auto_reset=True, board_size=10, n_frames=2, food_list=None, seed=42):
        if board_size != 10 or n_frames != 2:
            raise ValueError("only board_size=10, n_frames=2 (the reference defaults, structs.jl:33) are supported")
        self.n = int(n_envs)
        self.device = torch.device("cuda", device)
        self._h = C.c_void_p()
        _check(lib().snk_create(C.byref(self._h), self.n, int(device), AUTO_RESET if auto_reset else 0))
        self.auto_reset = bool(auto_reset)
        self.use_stream(torch.cuda.current_stream(self.device))
        if food_list is not None:
            self.set_food_list(food_list)
            self.reset()
        if seed != 42:
            _check(lib().snk_set_seed(self._h, int(seed)))

    def close(self):
        try:
            if getattr(self, "_h", None) and self._h.value:
                lib().snk_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:              # interpreter shutdown: module globals may already be gone
            pass

    __del__ = close

    # -- plumbing -------------------------------------------------------------------------------
    def use_stream(self, stream):
        """Run on a torch stream (so torch ops and env kernels are ordered)."""
        _check(lib().snk_set_stream(self._h, C.c_void_p(stream.cuda_stream)))

    def sync(self):
        _check(lib().snk_sync(self._h))

    def _new(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    # -- structs.jl:33-99 -----------------------------------------------------------------------
    def reset(self):
        _check(lib().snk_reset(self._h))

    def set_food_list(self, cells_rc):
        """Inject the food_list (structs.jl:70): 1-based (row, col) pairs in 2..9, at most 64."""
        flat = bytes(int(v) for rc in cells_rc for v in rc)
        buf = (C.c_uint8 * max(len(flat), 1)).from_buffer_copy(flat or b"\0")
        _check(lib().snk_set_food_list_host(self._h, buf, len(flat) // 2))

    # -- utils.jl:7-10 --------------------------------------------------------------------------
    def available_actions(self):
        out = self._new((self.n, 3), torch.uint8)
        _check(lib().snk_available_actions(self._h, _ptr(out)))
        return out

    # -- utils.jl:100-109 -----------------------------------------------------------------------
    def step(self, act_idx):
        """step!(game, available_actions(game)[act_idx]) -> (reward f32, done u8)"""
        r, d = self._new((self.n,), torch.float32), self._new((self.n,), torch.uint8)
        _check(lib().snk_step(self._h, _ptr(act_idx, torch.uint8, self.n, self.device), _ptr(r), _ptr(d)))
        return r, d

    def step_abs(self, dirs):
        """step!(game, DIRS[dir]) with absolute directions (play_snake.jl:96-111)"""
        r, d = self._new((self.n,), torch.float32), self._new((self.n,), torch.uint8)
        _check(lib().snk_step_abs(self._h, _ptr(dirs, torch.uint8, self.n, self.device), _ptr(r), _ptr(d)))
        return r, d

    # -- the fused rollout step -----------------------------------------------------------------
    def alloc_outputs(self, obs="f32", mask=True, ep_stats=False, act=False, compressible=True):
        """Output buffers of step_fused, to be reused step after step.  compressible: in device memory with generic L2
        compression (compressible_empty) - the same values, but the Float32 step writes fewer DRAM bytes and runs faster.
        Allocate them outside CUDA graph captures: allocating and freeing such memory synchronises the device.  (A buffer
        that is garbage-collected during a capture on the current stream is freed after it.)"""
        new = (lambda shape, dt: compressible_empty(shape, dt, self.device)) if compressible else self._new
        return _outputs(new, (self.n,), obs, mask, ep_stats, act)

    def step_fused(self, act_idx=None, q=None, eps=0.0, u=None, ridx=None, out=None, obs="f32", replay=None):
        """One kernel: [epsilon_greedy] + step! + virtual_step + next_state (+ Float32 cast).

        Either act_idx (N) u8 or q (N,3) f32 must be given.  Returns the `out` dict
        (reward, done, obs, mask, ...); pass a dict from alloc_outputs() to reuse buffers.
        replay: a ReplayBuffer — every env's transition is store!d (utils.jl:267-277) by the same kernel.
        """
        if out is None:            # buffers for one call: torch's caching allocator hands them out without a driver call
            out = self.alloc_outputs(obs=obs, act=q is not None, compressible=False)
        dev = self.device
        if q is not None:
            act_p = _ptr(out.get("act_idx"), torch.uint8, self.n, dev)
        else:
            if act_idx is None:
                raise ValueError("need act_idx or q")
            act_p = _ptr(act_idx, torch.uint8, self.n, dev)
        args = (_ptr(q, torch.float32, 3 * self.n, dev) if q is not None else None, float(eps),
                _ptr(u, torch.float32, self.n, dev), _ptr(ridx, torch.uint8, self.n, dev), act_p,
                _ptr(out.get("reward")), _ptr(out.get("done")), _ptr(out.get("obs")), _fmt_code(out), _ptr(out.get("mask")),
                _ptr(out.get("ep_return")), _ptr(out.get("ep_score")))
        if replay is None:
            _check(lib().snk_step_fused(self._h, *args))
        else:                      # also store! every env's Experience into the device replay ring
            _check(lib().snk_step_fused_store(self._h, replay._r, *args))
        return out

    def rollout(self, actions, obs="f32", mask=True, ep_stats=False, is_abs=False, out=None):
        """T steps in ONE launch for a known action stream (play_episode's actions_list mode, utils.jl:209-219).
        actions: (T, N) u8.  Returns step-major arrays: reward (T,N), done (T,N), obs (T,N,2,10,10), mask (T,N,3)."""
        T = actions.shape[0]
        dev = self.device
        if out is None:
            out = _outputs(self._new, (T, self.n), obs, mask, ep_stats)
        _check(lib().snk_rollout_fused(self._h, _ptr(actions, torch.uint8, T * self.n, dev), T, int(is_abs),
                                       _ptr(out.get("reward")), _ptr(out.get("done")), _ptr(out.get("obs")), _fmt_code(out),
                                       _ptr(out.get("mask")), _ptr(out.get("ep_return")), _ptr(out.get("ep_score"))))
        return out

    def step_fused_host(self, host, q=False, eps=0.0, replay=None):
        """Same through HOST (pinned) tensors: `host` is a dict of CPU tensors with the keys of
        alloc_outputs() plus the inputs ('act_idx', or 'q' [+ 'u', 'ridx']).  ASYNCHRONOUS: call sync() before
        reading an output or overwriting an input.  replay: also store! every transition into the device ring."""
        g = lambda k: _ptr(host.get(k))
        args = (g("q") if q else None, float(eps), g("u") if q else None, g("ridx") if q else None,
                g("act_idx"), g("reward"), g("done"), g("obs"), _fmt_code(host), g("mask"), g("ep_return"), g("ep_score"))
        if replay is None:
            _check(lib().snk_step_fused_host(self._h, *args))
        else:
            _check(lib().snk_step_fused_store_host(self._h, replay._r, *args))
        return host

    # -- utils.jl:135-149 -----------------------------------------------------------------------
    def assemble_state(self, fmt="f32", out=None):
        """(board_{t-1}, board_t) of every env: (N,2,10,10) [= Julia (10,10,2,N)]"""
        code, dt, per = _OBS[fmt]
        if out is None:
            out = self._new(_obs_shape(fmt, (self.n,)), dt)
        _check(lib().snk_state(self._h, _ptr(out, dt, self.n * per, self.device), code))
        return out

    def patch_reset_obs(self, done, obs, fmt="f32"):
        """rows of `obs` (a step's next_state output) of the envs that step re-initialised become (init, init): obs then is
        the acting state of the next step (snk_patch_reset_obs)"""
        code, dt, per = _OBS[fmt]
        _check(lib().snk_patch_reset_obs(self._h, _ptr(done, torch.uint8, self.n, self.device),
                                         _ptr(obs, dt, self.n * per, self.device), code))
        return obs

    # host-array forms of the per-call API (what a Julia host calls where the reference reads a field of `game`)
    def _host(self, fn, shape, dtype, *extra):
        out = torch.empty(shape, dtype=dtype)
        _check(fn(self._h, C.c_void_p(out.data_ptr()), *extra))
        return out

    def assemble_state_host(self, fmt="f32"):
        code, dt, _ = _OBS[fmt]
        return self._host(lib().snk_state_host, _obs_shape(fmt, (self.n,)), dt, code)

    def virtual_step_host(self):
        return self._host(lib().snk_losing_mask_host, (self.n, 3), torch.uint8)

    def available_actions_host(self):
        return self._host(lib().snk_available_actions_host, (self.n, 3), torch.uint8)

    def score_host(self):
        return self._host(lib().snk_get_score_host, (self.n,), torch.int32)

    def lost_host(self):
        return self._host(lib().snk_get_done_host, (self.n,), torch.uint8)

    # -- utils.jl:112-132 -----------------------------------------------------------------------
    def virtual_step(self):
        """next_is_suicidal (N,3) u8 for the current state"""
        out = self._new((self.n, 3), torch.uint8)
        _check(lib().snk_losing_mask(self._h, _ptr(out)))
        return out

    # -- utils.jl:153-172 -----------------------------------------------------------------------
    def epsilon_greedy(self, q, eps, u=None, ridx=None):
        """action index (N) u8: ridx where u < eps else argmax(q).  u/ridx None -> internal draws."""
        out = self._new((self.n,), torch.uint8)
        _check(lib().snk_select_action(self._h, _ptr(q, torch.float32, 3 * self.n, self.device), float(eps),
                                       _ptr(u, torch.float32, self.n, self.device),
                                       _ptr(ridx, torch.uint8, self.n, self.device), _ptr(out)))
        return out

    # -- fields ---------------------------------------------------------------------------------
    def _scalar(self, fn, dtype):
        out = self._new((self.n,), dtype)
        _check(fn(self._h, _ptr(out)))
        return out

    @property
    def score(self):
        return self._scalar(lib().snk_get_score, torch.int32)

    @property
    def lost(self):
        return self._scalar(lib().snk_get_done, torch.uint8)

    @property
    def error_flags(self):
        return self._scalar(lib().snk_get_error_flags, torch.uint8)

    @property
    def steps(self):
        return self._scalar(lib().snk_get_steps, torch.int32)

    def count_errors(self):
        c = C.c_int64(0)
        _check(lib().snk_count_errors_host(self._h, C.byref(c)))
        return c.value

    # -- checkpoints (save_trainer / load_trainer, utils.jl:408-418) ---------------------------------------------------
    def state_dict(self):
        """{'blob': uint8 CPU tensor}: the N games, the generator's seed and call count and the food list (snk_env_save_host),
        after the work enqueued so far"""
        return {"blob": _save_blob(lib().snk_env_checkpoint_bytes, lib().snk_env_save_host, self._h)}

    def load_state_dict(self, d):
        """The games continue bit for bit from where state_dict() left them.  Needs the same N and auto_reset; a blob the
        library refuses raises SnakeB200Error and leaves the games as they were."""
        _load_blob(lib().snk_env_load_host, self._h, d)


def masked_target(q_next, mask, rewards, dones, gamma=0.97, fill=-100.0, out_dtype=torch.float64):
    """utils.jl:448-451: q_next[mask] .= -100; y = r + 0.97 * max_a q_next * (1 - done).

    q_next (B,3) f32, mask (B,3) u8, rewards (B) f32, dones (B) u8 on one CUDA device.
    Float64 result like the reference's broadcast (out_dtype=torch.float32 rounds it once).
    """
    B = rewards.numel()
    dev = rewards.device
    y = torch.empty(B, dtype=out_dtype, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    with torch.cuda.device(dev):
        _check(lib().snk_masked_target(
            _ptr(q_next, torch.float32, 3 * B, dev), _ptr(mask, torch.uint8, 3 * B, dev),
            _ptr(rewards, torch.float32, B, dev), _ptr(dones, torch.uint8, B, dev), float(gamma), float(fill),
            _ptr(y) if out_dtype == torch.float64 else None, _ptr(y) if out_dtype == torch.float32 else None, B, st))
    return y


def center_columns(Dt):
    """compute_D.jl:76-81 / la_utils.jl:163-169 on device.

    Dt: (K, P) float64 torch-contiguous CUDA tensor = Julia's P x K column-major deviation_matrix
    (row k of Dt is snapshot k).  Centred in place; returns (mean (P), var (P)).
    """
    K, P = Dt.shape
    dev = Dt.device
    mean = torch.empty(P, dtype=torch.float64, device=dev)
    var = torch.empty(P, dtype=torch.float64, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    with torch.cuda.device(dev):
        _check(lib().snk_center_columns(_ptr(Dt, torch.float64), P, K, _ptr(mean), _ptr(var), st))
    return mean, var




def pinned_empty(shape, dtype):
    return torch.empty(shape, dtype=dtype, pin_memory=True)


DTYPE_F32, DTYPE_F64 = 1, 2


class GramPlan:
    """Gram G = A A^T of the snapshot matrix on tcgen05 tensor cores (plot_traj.jl:10-16: the K x K matrix
    whose eigenvalues / (K-1) are S.^2/(K-1) of svd(D)).

    A: (K, P) float64 or float32 CUDA tensor, torch-contiguous = Julia's P x K column-major D.
    pack() splits it into bf16 planes once; gram() can then be run for terms = 1 or 3.
    """

    def __init__(self, K, P, device, splits=0):
        self.K, self.P, self.splits = int(K), int(P), int(splits)
        self.device = torch.device(device)
        nbytes = C.c_size_t(0)
        _check(lib().snk_gram_workspace_bytes(self.K, self.P, self.splits, C.byref(nbytes)))
        self.ws = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def pack(self, A):
        if tuple(A.shape) != (self.K, self.P):
            raise ValueError("A must be (K, P) = (%d, %d)" % (self.K, self.P))
        dt = {torch.float64: DTYPE_F64, torch.float32: DTYPE_F32}[A.dtype]
        with torch.cuda.device(self.device):
            _check(lib().snk_gram_pack(_ptr(A, device=self.device), dt, self.P, self.K, _ptr(self.ws), self._stream()))
        return self

    def planes(self):
        """(hi pointer, lo pointer, pitch in elements) of the bf16 planes inside the workspace: a producer
        (QNet.sample_grads) can write them instead of pack()"""
        pb, pitch = C.c_size_t(0), C.c_int64(0)
        _check(lib().snk_gram_planes_layout(self.K, self.P, C.byref(pb), C.byref(pitch)))
        return self.ws.data_ptr(), self.ws.data_ptr() + pb.value, pitch.value

    def gram(self, terms=3, block_k=0, out=None):
        G = out if out is not None else torch.empty(self.K, self.K, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _check(lib().snk_gram(_ptr(self.ws), self.P, self.K, int(terms), int(block_k), self.splits,
                                  _ptr(G, torch.float32, self.K * self.K, self.device), self._stream()))
        return G


def gram(A, terms=3, block_k=0, splits=0):
    """One-shot G = A A^T (see GramPlan)."""
    return GramPlan(A.shape[0], A.shape[1], A.device, splits).pack(A).gram(terms, block_k)


class ReplayBuffer:
    """ReplayBuffer (structs.jl:104-116) on the device: capacity 50,000, batch_size 64 by default.

    store! happens inside SnakeGame.step_fused(..., replay=rb); sample()/stack_exp() mirror utils.jl:280-287 and
    utils.jl:343-383.  Indices are 0-based slots."""

    def __init__(self, capacity=50000, device=0, batch_size=64, seed=0):
        if batch_size > capacity:
            raise ValueError("batch_size cannot be greater than the capacity of the buffer.")     # structs.jl:113
        self.capacity, self.batch_size, self.seed = int(capacity), int(batch_size), int(seed)
        self.device = torch.device("cuda", device)
        self._r = C.c_void_p()
        _check(lib().snk_replay_create(C.byref(self._r), self.capacity, int(device)))

    def close(self):
        try:
            if getattr(self, "_r", None) and self._r.value:
                lib().snk_replay_destroy(self._r)
                self._r = C.c_void_p()
        except Exception:
            pass

    __del__ = close

    def _len_pos(self):
        n, p = C.c_int64(0), C.c_int64(0)
        _check(lib().snk_replay_length(self._r, C.byref(n), C.byref(p)))
        return n.value, p.value

    def __len__(self):
        return self._len_pos()[0]

    @property
    def position(self):                 # 1-based like the Julia field
        return self._len_pos()[1]

    def isfull(self):                   # utils.jl:289-291 (sic: position == capacity)
        return self.position == self.capacity

    def isready(self):                  # utils.jl:293-296
        return len(self) >= self.batch_size

    def empty_buffer(self):             # utils.jl:311-314
        _check(lib().snk_replay_clear(self._r))

    def sample_indices(self, B=None):
        """min(batch_size, length) distinct slots (utils.jl:280-287), (B,) int64 on the device"""
        B = min(self.batch_size, len(self)) if B is None else int(B)
        idx = torch.empty(B, dtype=torch.int64, device=self.device)
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _check(lib().snk_replay_sample_indices(self._r, self.seed, B, _ptr(idx), st))
        return idx

    def stack_exp(self, idx, ep_stats=False):
        """utils.jl:343-383 for the transitions at idx: dict(states, actions, rewards, next_states, dones, mask)"""
        B = idx.numel()
        dev = self.device
        out = {"states": torch.empty(B, 2, 10, 10, dtype=torch.float32, device=dev),
               "next_states": torch.empty(B, 2, 10, 10, dtype=torch.float32, device=dev),
               "actions": torch.empty(B, dtype=torch.uint8, device=dev),
               "rewards": torch.empty(B, dtype=torch.float32, device=dev),
               "dones": torch.empty(B, dtype=torch.uint8, device=dev),
               "mask": torch.empty(B, 3, dtype=torch.uint8, device=dev)}
        if ep_stats:
            out["ep_return"] = torch.empty(B, dtype=torch.float32, device=dev)
            out["score"] = torch.empty(B, dtype=torch.int32, device=dev)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _check(lib().snk_replay_gather(self._r, _ptr(idx, torch.int64, B, dev), B, _ptr(out["states"]),
                                       _ptr(out["next_states"]), _ptr(out["actions"]), _ptr(out["rewards"]),
                                       _ptr(out["dones"]), _ptr(out["mask"]), _ptr(out.get("ep_return")),
                                       _ptr(out.get("score")), st))
        return out

    def sample(self):
        return self.stack_exp(self.sample_indices())

    def stack_exp_host(self, idx_host, out=None):
        """stack_exp for 0-based slots given as a CPU int64 tensor, into HOST tensors (pinned if `out` holds pinned
        tensors): what a host-side trainer receives per minibatch (utils.jl:442-443).  Returns when the data is there."""
        B = idx_host.numel()
        if out is None:
            out = {"states": torch.empty(B, 2, 10, 10, dtype=torch.float32), "next_states": torch.empty(B, 2, 10, 10, dtype=torch.float32),
                   "actions": torch.empty(B, dtype=torch.uint8), "rewards": torch.empty(B, dtype=torch.float32),
                   "dones": torch.empty(B, dtype=torch.uint8), "mask": torch.empty(B, 3, dtype=torch.uint8)}
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        p = lambda k: C.c_void_p(out[k].data_ptr())
        _check(lib().snk_replay_gather_host(self._r, C.c_void_p(idx_host.data_ptr()), B, p("states"), p("next_states"),
                                            p("actions"), p("rewards"), p("dones"), p("mask"), st))
        return out

    def bad_index(self):
        f = C.c_int(0)
        _check(lib().snk_replay_bad_index_host(self._r, C.byref(f)))
        return bool(f.value)

    # -- checkpoints (save_buffer / load_buffer, utils.jl:316-340) -----------------------------------------------------
    def state_dict(self):
        """{'blob': uint8 CPU tensor (the filled records, the stored count, the sampler's call count), 'seed', 'batch_size'}"""
        return {"blob": _save_blob(lib().snk_replay_checkpoint_bytes, lib().snk_replay_save_host, self._r),
                "seed": self.seed, "batch_size": self.batch_size}

    def load_state_dict(self, d):
        """The ring continues bit for bit (the same samples, the same slots filled next).  Needs the same capacity; a blob the
        library refuses raises SnakeB200Error and leaves the ring as it was."""
        if not isinstance(d, dict) or not isinstance(d.get("seed"), int) or not isinstance(d.get("batch_size"), int):
            raise ValueError("a ReplayBuffer state_dict holds 'blob', 'seed' and 'batch_size'")
        if not 0 < d["batch_size"] <= self.capacity:
            raise ValueError("batch_size cannot be greater than the capacity of the buffer.")
        _load_blob(lib().snk_replay_load_host, self._r, d)
        self.seed, self.batch_size = d["seed"], d["batch_size"]


from . import shard  # noqa: E402,F401
from . import bson_io, laplace, qnet, rollout, train  # noqa: E402,F401
