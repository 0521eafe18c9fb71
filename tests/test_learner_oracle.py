"""CPU checks of the learner: the RMSProp restatement of oracle/learner_oracle.py (Flux.Optimise, utils.jl:466) against values
computed by hand, and the argument checks of snk_qnet_train_step / snk_qnet_set_params / snk_qnet_params."""
import ctypes as C
import math
import struct

import numpy as np
import pytest
import torch

from oracle import learner_oracle as LO
from tests.util import graft, pkg


def f32(x):
    return struct.unpack("f", struct.pack("f", x))[0]


def test_rmsprop_first_step_by_hand():
    # g = 1, acc = 0: acc = Float32(0.1 * 1 * 1), delta = Float32(1 * (5e-4 / (sqrt_f32(acc) + 1e-8)))
    theta, acc = LO.rmsprop(np.float32([1.0]), np.float32([0.0]), np.float32([1.0]))
    a = f32((1.0 - 0.9) * 1.0 * 1.0)
    assert acc[0] == a == np.float32(0.1)
    d = f32(1.0 * (5e-4 / (f32(math.sqrt(a)) + 1e-8)))
    assert theta[0] == np.float32(np.float32(1.0) - np.float32(d))
    assert abs(float(theta[0]) - (1.0 - 5e-4 / math.sqrt(0.1))) < 1e-7


def test_rmsprop_by_hand_with_state_and_zero_gradient():
    theta, acc = LO.rmsprop(np.float32([0.25, -3.0]), np.float32([4.0, 2.5e-3]), np.float32([0.0, -0.02]), eta=1e-3, rho=0.5,
                            epsilon=0.0)
    assert theta[0] == np.float32(0.25) and acc[0] == np.float32(2.0)                    # g = 0: theta stays, acc decays by rho
    g = float(np.float32(-0.02))
    a = f32(0.5 * float(np.float32(2.5e-3)) + (0.5 * g) * g)
    assert acc[1] == np.float32(a)
    d = f32(g * (1e-3 / f32(math.sqrt(a))))
    assert theta[1] == np.float32(np.float32(-3.0) - np.float32(d))
    assert d < 0 and theta[1] > -3.0                                                     # a step against the gradient


def test_rmsprop_follows_torch_rmsprop_to_float32_rounding():
    """torch.optim.RMSprop(lr, alpha, eps) is the same formula evaluated in Float32: over a few steps the two differ only by
    rounding"""
    rng = np.random.default_rng(0)
    th0 = rng.normal(0, 0.1, 4096).astype(np.float32)
    p = torch.nn.Parameter(torch.from_numpy(th0.copy()))
    opt = torch.optim.RMSprop([p], lr=5e-4, alpha=0.9, eps=1e-8)
    th, acc = th0, np.zeros_like(th0)
    for _ in range(5):
        g = rng.normal(0, 1e-2, th0.size).astype(np.float32)
        p.grad = torch.from_numpy(g.copy())
        opt.step()
        th, acc = LO.rmsprop(th, acc, g)
    assert np.allclose(p.detach().numpy(), th, rtol=0, atol=1e-6)
    assert not np.array_equal(th, th0)


def test_float32_evaluation_rounds_differently():
    """the Optimisers.jl form evaluates the same expression in Float32; the Flux.Optimise form (Float64 hyper-parameters)
    is what the oracle and the library restate, and the two differ in the last bits"""
    rng = np.random.default_rng(1)
    th = rng.normal(0, 0.1, 100000).astype(np.float32)
    acc = np.abs(rng.normal(0, 1e-4, th.size)).astype(np.float32)
    g = rng.normal(0, 1e-2, th.size).astype(np.float32)
    th64, acc64 = LO.rmsprop(th, acc, g)
    r, e, eps = np.float32(0.9), np.float32(5e-4), np.float32(1e-8)
    acc32 = r * acc + (np.float32(1) - r) * g * g
    th32 = th - g * (e / (np.sqrt(acc32) + eps))
    assert not np.array_equal(acc32, acc64) and not np.array_equal(th32, th64)
    assert np.allclose(th32, th64, rtol=0, atol=1e-6)


@pytest.fixture(scope="module")
def L():
    graft.build()
    return pkg().lib()


def test_train_step_argument_validation(L):
    a = (None, None, None, None)
    assert L.snk_qnet_train_step(*a, 0, None, 5e-4, 0.9, 1e-8, None, None, None) == -1
    assert b"B must be >= 1" in L.snk_last_error()
    for eta, rho, eps in ((0.0, 0.9, 1e-8), (-1e-3, 0.9, 1e-8), (5e-4, 1.0, 1e-8), (5e-4, -0.1, 1e-8), (5e-4, 0.9, -1.0),
                          (float("nan"), 0.9, 1e-8)):
        assert L.snk_qnet_train_step(*a, 64, None, eta, rho, eps, None, None, None) == -1
        assert b"RMSProp needs" in L.snk_last_error(), (eta, rho, eps)
    assert L.snk_qnet_train_step(*a, 64, None, 5e-4, 0.0, 0.0, None, None, None) == -1
    assert b"null argument" in L.snk_last_error()


def test_set_params_and_params_argument_validation(L):
    assert L.snk_qnet_set_params(None, None, None) == -1
    assert b"null argument" in L.snk_last_error()
    p = C.c_void_p()
    assert L.snk_qnet_params(None, C.byref(p)) == -1
    assert b"null argument" in L.snk_last_error()
