"""Oracle (test infrastructure): the learner of train! (utils.jl:452-466) in numpy.

mean_grad: Flux.gradient of mean(huber(q_net(s)[a], y)) = (1/B) sum_i J_i, from the Float64 per-sample rows of
qgrad_oracle, and the batch-mean loss.

rmsprop: Flux.Optimise's RMSProp apply! + update! (structs.jl:137, utils.jl:466) with Julia's type promotion: the
hyper-parameters are Float64, acc / g / theta Float32, so every broadcast is evaluated in Float64 and stored back as Float32:

    acc   = Float32(rho * Float64(acc) + ((1 - rho) * Float64(g)) * Float64(g))      @. acc = ρ*acc + (1-ρ)*Δ*conj(Δ)
    delta = Float32(Float64(g) * (eta / (Float64(sqrt_f32(acc)) + epsilon)))         @. Δ *= η / (√acc + ϵ)
    theta = theta - delta                                                            Float32

numpy evaluates each float64 operation correctly rounded and without fused multiply-adds, like Julia's broadcast.  Flux and
Optimisers.jl are unpinned third-party code: parity unpinned by the reference.
"""
import numpy as np

from oracle import qgrad_oracle as QG


def mean_grad(layers, states, actions, targets):
    """(g (P,) float64, mean loss float64): the Float64 mean of the per-sample gradient rows and losses"""
    J, loss, _ = QG.per_sample_grads(layers, states, actions, targets)
    return J.mean(axis=0), float(np.mean(loss))


def rmsprop(theta, acc, g, eta=5e-4, rho=0.9, epsilon=1e-8):
    """one RMSProp step; theta, acc, g Float32 arrays.  Returns (theta', acc') as new Float32 arrays."""
    theta, acc, g = (np.asarray(a, dtype=np.float32) for a in (theta, acc, g))
    gd = g.astype(np.float64)
    acc_new = (rho * acc.astype(np.float64) + ((1.0 - rho) * gd) * gd).astype(np.float32)
    delta = (gd * (eta / (np.sqrt(acc_new).astype(np.float64) + epsilon))).astype(np.float32)
    return (theta - delta).astype(np.float32), acc_new
