# SnakeB200.jl — thin `ccall` wrapper over libsnake_b200.so (include/snake_b200.h).
#
# NOT EXECUTED IN THE BUILD IMAGE (Julia is not installed there); the tests drive the identical C symbols
# through ctypes.  It is the binding a maintainer of lucagiorgetti/Laplace-DQN-Snake-game adds so that
# `utils.jl` / `main.jl` keep their entry points: the same names (`available_actions`, `step!`,
# `virtual_step`, `assemble_state!`, `epsilon_greedy`), the same 3-action relative control, the same
# (10,10,2,N) two-frame state — now for N games at once on a B200.
#
# Host-array methods use the `_host` entry points (pinned or plain Julia Arrays); if CUDA.jl is loaded the
# device entry points can be called with `pointer(::CuArray)` the same way.
module SnakeB200

export BatchedSnakeGame, available_actions, step!, step_fused!, virtual_step, assemble_state!,
       epsilon_greedy, masked_target, center_columns!, reset!, set_food_list!, score, lost,
       DeviceReplayBuffer, store_step!, store_step_host!, store_step_host_bits!, stack_exp, sample_indices, DeviceQNet, forward!, overflowed,
       sample_grads!, RMSPropState, train_step!, update_target_net!, params_device, store_snapshot!, gram!, sample_model_weights!, empty_buffer!, patch_reset_obs!,
       GramShard, export_handle, connect!, run!, planes, LearnerGroup, check_peers, ReplayGroup, sample!,
       step_device!, step_abs_device!, step_fused_device!, rollout_device!, state_device!, losing_mask_device!,
       lost_device!, steps_device!, error_flags_device!, count_errors, seed!, set_stream!, num_envs, library_version,
       default_food_list, device_alloc, device_free, compression_supported, checkpoint, restore!

const lib = get(ENV, "SNAKE_B200_LIB", joinpath(@__DIR__, "..", "libsnake_b200.so"))

const OBS_F32, OBS_I8, OBS_I64, OBS_PACKED2, OBS_BITS = Cint(1), Cint(2), Cint(3), Cint(4), Cint(5)
const AUTO_RESET = UInt32(1)
const QNET_BF16, QNET_F32 = Cint(0), Cint(1)
# utils.jl:8 order
const DIRS = (CartesianIndex(-1, 0), CartesianIndex(1, 0), CartesianIndex(0, -1), CartesianIndex(0, 1))

struct SnakeB200Error <: Exception
    code::Int
    msg::String
end
function check(rc::Cint)
    rc == 0 && return nothing
    throw(SnakeB200Error(rc, unsafe_string(ccall((:snk_last_error, lib), Cstring, ()))))
end

"""N batched `SnakeGame`s (structs.jl:6-100) resident on one GPU."""
mutable struct BatchedSnakeGame
    handle::Ptr{Cvoid}
    n::Int
    # host staging, laid out exactly like `stack_exp` (utils.jl:343-383)
    state::Array{Float32,4}        # (10,10,2,N): next_state of the last step
    reward::Vector{Float32}
    lost::Vector{UInt8}
    next_is_suicidal::Matrix{UInt8}   # (3,N)
    actions::Vector{UInt8}
    function BatchedSnakeGame(n::Integer; device::Integer = 0, auto_reset::Bool = true,
                              board_size::Integer = 10, n_frames::Integer = 2)
        (board_size == 10 && n_frames == 2) || throw("only board_size = 10, n_frames = 2 are supported")
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:snk_create, lib), Cint, (Ref{Ptr{Cvoid}}, Int64, Cint, UInt32),
                    h, n, device, auto_reset ? AUTO_RESET : UInt32(0)))
        g = new(h[], n, zeros(Float32, 10, 10, 2, n), zeros(Float32, n), zeros(UInt8, n), ones(UInt8, 3, n),
                zeros(UInt8, n))
        finalizer(x -> ccall((:snk_destroy, lib), Cint, (Ptr{Cvoid},), x.handle), g)
        virtual_step(g)            # both mirrors come from the library, also for the constructor state
        assemble_state!(g)
        return g
    end
end

"""every game back to `SnakeGame()` (structs.jl:33-99); the host mirrors are refreshed from the device"""
function reset!(g::BatchedSnakeGame)
    check(ccall((:snk_reset, lib), Cint, (Ptr{Cvoid},), g.handle))
    fill!(g.reward, 0f0); fill!(g.lost, 0x00)
    virtual_step(g)
    assemble_state!(g)
    return g
end

"""food_list injection (structs.jl:70): vector of CartesianIndex{2} in 2:9 × 2:9."""
function set_food_list!(g::BatchedSnakeGame, cells::Vector{CartesianIndex{2}})
    rc = UInt8[x for c in cells for x in (c[1], c[2])]
    check(ccall((:snk_set_food_list_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Cint), g.handle, rc, length(cells)))
    reset!(g)
end

sync(g::BatchedSnakeGame) = check(ccall((:snk_sync, lib), Cint, (Ptr{Cvoid},), g.handle))

# utils.jl:448-451 (device pointers; use with CUDA.jl CuArrays)
function masked_target(q_next::Ptr{Float32}, mask::Ptr{UInt8}, r::Ptr{Float32}, done::Ptr{UInt8},
                       y::Ptr{Float64}, B::Integer; gamma::Float64 = 0.97, fill::Float32 = -100f0)
    check(ccall((:snk_masked_target, lib), Cint,
                (Ptr{Float32}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8}, Cdouble, Cfloat, Ptr{Float64}, Ptr{Float32}, Int64, Ptr{Cvoid}),
                q_next, mask, r, done, gamma, fill, y, C_NULL, B, C_NULL))
end

"""
    step_fused!(g, actions)            # action indices 1:3 into available_actions, as the Q-net's argmax gives
    step_fused!(g, q, ε; u, ridx)      # epsilon_greedy + step! + virtual_step + next state, one kernel

Fills `g.state` (Float32 (10,10,2,N) next_state), `g.reward`, `g.lost`, `g.next_is_suicidal` — the fields
`play_episode` (utils.jl:198-259) collects per step — and returns `g`.
"""
function step_fused!(g::BatchedSnakeGame, actions::AbstractVector{<:Integer})
    g.actions .= UInt8.(actions .- 1)                       # Julia 1-based index -> 0-based
    check(ccall((:snk_step_fused_host, lib), Cint,
                (Ptr{Cvoid}, Ptr{Float32}, Cfloat, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8},
                 Ptr{Cvoid}, Cint, Ptr{UInt8}, Ptr{Float32}, Ptr{Int32}),
                g.handle, C_NULL, 0f0, C_NULL, C_NULL, g.actions, g.reward, g.lost, g.state, OBS_F32,
                g.next_is_suicidal, C_NULL, C_NULL))
    sync(g)
    return g
end
function step_fused!(g::BatchedSnakeGame, q::Matrix{Float32}, epsilon::Float32;
                     u::Vector{Float32} = rand(Float32, g.n), ridx::Vector{UInt8} = rand(UInt8(0):UInt8(2), g.n))
    size(q) == (3, g.n) || throw(DimensionMismatch("q must be (3, N)"))
    check(ccall((:snk_step_fused_host, lib), Cint,
                (Ptr{Cvoid}, Ptr{Float32}, Cfloat, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8},
                 Ptr{Cvoid}, Cint, Ptr{UInt8}, Ptr{Float32}, Ptr{Int32}),
                g.handle, q, epsilon, u, ridx, g.actions, g.reward, g.lost, g.state, OBS_F32,
                g.next_is_suicidal, C_NULL, C_NULL))
    sync(g)
    return g
end

# The reference's per-call API on HOST arrays: every function asks the library (the `_host` entry points copy the
# answer down and return when it has arrived), nothing is reconstructed on the Julia side -------------------------------

"""utils.jl:100-109 for all N games; `actions` are indices 1:3 into available_actions(g)."""
step!(g::BatchedSnakeGame, actions::AbstractVector{<:Integer}) = step_fused!(g, actions)

"""utils.jl:112-132: `next_is_suicidal` (3,N) of the CURRENT states, `trues(3)` for a lost game."""
function virtual_step(g::BatchedSnakeGame)
    check(ccall((:snk_losing_mask_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, g.next_is_suicidal))
    return g.next_is_suicidal .!= 0
end

"""utils.jl:135-139: the (10,10,2,N) Float32 two-frame state of every game as it is NOW (also right after `reset!`)."""
function assemble_state!(g::BatchedSnakeGame)
    check(ccall((:snk_state_host, lib), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Cint), g.handle, g.state, OBS_F32))
    return g.state
end

"""utils.jl:7-10 for all N games: (3,N) direction codes 0:3 in the order U, D, L, R (`DIRS[code + 1]` is the CartesianIndex)."""
function available_actions(g::BatchedSnakeGame)
    out = Matrix{UInt8}(undef, 3, g.n)
    check(ccall((:snk_available_actions_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, out))
    return out
end

"""`game.score` (structs.jl:21) of every game"""
function score(g::BatchedSnakeGame)
    out = Vector{Int32}(undef, g.n)
    check(ccall((:snk_get_score_host, lib), Cint, (Ptr{Cvoid}, Ptr{Int32}), g.handle, out))
    return out
end
"""`game.lost` (structs.jl:28) of every game"""
function lost(g::BatchedSnakeGame)
    check(ccall((:snk_get_done_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, g.lost))
    return g.lost .!= 0
end

# device-pointer forms of the same getters
score(g::BatchedSnakeGame, d_score::Ptr{Int32}) = check(ccall((:snk_get_score, lib), Cint, (Ptr{Cvoid}, Ptr{Int32}), g.handle, d_score))

"""utils.jl:7-10 on device: fills a (3,N) UInt8 device array with direction codes 0:3 (U,D,L,R)."""
available_actions(g::BatchedSnakeGame, d_out::Ptr{UInt8}) =
    check(ccall((:snk_available_actions, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, d_out))

"""rows of `d_obs` (a fused step's next_state output) of the games that step re-initialised become (init, init): the
acting state of the next step without a second expansion of all N states"""
patch_reset_obs!(g::BatchedSnakeGame, d_done::Ptr{UInt8}, d_obs::Ptr{Cvoid}, obs_fmt::Integer = OBS_F32) =
    check(ccall((:snk_patch_reset_obs, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Ptr{Cvoid}, Cint), g.handle, d_done, d_obs, obs_fmt))

"""utils.jl:153-172 on device pointers: out[i] = ridx[i] if u[i] < ε else argmax(q[:, i]) - 1."""
epsilon_greedy(g::BatchedSnakeGame, d_q::Ptr{Float32}, epsilon::Float32, d_u::Ptr{Float32}, d_ridx::Ptr{UInt8},
               d_out::Ptr{UInt8}) =
    check(ccall((:snk_select_action, lib), Cint, (Ptr{Cvoid}, Ptr{Float32}, Cfloat, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}),
                g.handle, d_q, epsilon, d_u, d_ridx, d_out))

"""compute_D.jl:76-81 on a device-resident P×K Float64 deviation_matrix (column-major, as Julia stores it)."""
center_columns!(d_D::Ptr{Float64}, P::Integer, K::Integer, d_mean::Ptr{Float64}, d_var::Ptr{Float64}) =
    check(ccall((:snk_center_columns, lib), Cint, (Ptr{Float64}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Cvoid}),
                d_D, P, K, d_mean, d_var, C_NULL))

# ---- ReplayBuffer on the device (structs.jl:104-116; store! / sample / stack_exp, utils.jl:265-383) -----------
mutable struct DeviceReplayBuffer
    handle::Ptr{Cvoid}
    capacity::Int
    batch_size::Int
    function DeviceReplayBuffer(capacity::Integer = 50000; device::Integer = 0, batch_size::Integer = 64)
        batch_size > capacity && throw("batch_size cannot be greater than the capacity of the buffer.")   # structs.jl:113
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:snk_replay_create, lib), Cint, (Ref{Ptr{Cvoid}}, Int64, Cint), h, capacity, device))
        r = new(h[], capacity, batch_size)
        finalizer(x -> ccall((:snk_replay_destroy, lib), Cint, (Ptr{Cvoid},), x.handle), r)
        return r
    end
end
"""empty_buffer! (utils.jl:311): forget every stored Experience."""
empty_buffer!(r::DeviceReplayBuffer) = check(ccall((:snk_replay_clear, lib), Cint, (Ptr{Cvoid},), r.handle))
function Base.length(r::DeviceReplayBuffer)
    n = Ref{Int64}(0); p = Ref{Int64}(0)
    check(ccall((:snk_replay_length, lib), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}), r.handle, n, p))
    return Int(n[])
end

"""One fused step that also `store!`s every env's Experience (device pointers: q, u, ridx, outputs)."""
store_step!(g::BatchedSnakeGame, r::DeviceReplayBuffer, d_q::Ptr{Float32}, epsilon::Float32, d_u::Ptr{Float32},
            d_ridx::Ptr{UInt8}, d_act::Ptr{UInt8}, d_reward::Ptr{Float32}, d_done::Ptr{UInt8}, d_obs::Ptr{Float32},
            d_mask::Ptr{UInt8}) =
    check(ccall((:snk_step_fused_store, lib), Cint,
                (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}, Cfloat, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8},
                 Ptr{Cvoid}, Cint, Ptr{UInt8}, Ptr{Float32}, Ptr{Int32}),
                g.handle, r.handle, d_q, epsilon, d_u, d_ridx, d_act, d_reward, d_done, d_obs, OBS_F32, d_mask, C_NULL, C_NULL))

"""One iteration's play step for a HOST trainer (utils.jl:436-440): epsilon_greedy + step! + virtual_step, every game's
Experience store!d into the device ring; down come reward / lost / next_is_suicidal / actions and the lossless 2-bit packed
next states (50 B per game; Float32 states are produced for the sampled minibatch only, `stack_exp`)."""
function store_step_host!(g::BatchedSnakeGame, r::DeviceReplayBuffer, q::Matrix{Float32}, epsilon::Float32, packed::Matrix{UInt8};
                          u::Vector{Float32} = rand(Float32, g.n), ridx::Vector{UInt8} = rand(UInt8(0):UInt8(2), g.n))
    size(q) == (3, g.n) && size(packed) == (50, g.n) || throw(DimensionMismatch("q must be (3, N), packed (50, N)"))
    check(ccall((:snk_step_fused_store_host, lib), Cint,
                (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}, Cfloat, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8},
                 Ptr{Cvoid}, Cint, Ptr{UInt8}, Ptr{Float32}, Ptr{Int32}),
                g.handle, r.handle, q, epsilon, u, ridx, g.actions, g.reward, g.lost, packed, OBS_PACKED2,
                g.next_is_suicidal, C_NULL, C_NULL))
    sync(g)
    return g
end

"""The same step with ONE 24-byte record per game coming down (`SNK_OBS_BITS`, include/snake_b200.h: the next state as two
bit-boards, next_is_suicidal, lost, the action taken and the reward) — less than half the bytes of the packed form; `records` is
(24, N) UInt8 and `unpack_bits(records)` turns it into the reference's arrays."""
function store_step_host_bits!(g::BatchedSnakeGame, r::DeviceReplayBuffer, q::Matrix{Float32}, epsilon::Float32, records::Matrix{UInt8};
                               u::Vector{Float32} = rand(Float32, g.n), ridx::Vector{UInt8} = rand(UInt8(0):UInt8(2), g.n))
    size(q) == (3, g.n) && size(records) == (24, g.n) || throw(DimensionMismatch("q must be (3, N), records (24, N)"))
    check(ccall((:snk_step_fused_store_host, lib), Cint,
                (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}, Cfloat, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8},
                 Ptr{Cvoid}, Cint, Ptr{UInt8}, Ptr{Float32}, Ptr{Int32}),
                g.handle, r.handle, q, epsilon, u, ridx, C_NULL, C_NULL, C_NULL, records, OBS_BITS, C_NULL, C_NULL, C_NULL))
    sync(g)
    return records
end

"""Decodes `SNK_OBS_BITS` records (24, N): (state::Array{Int,4} (10,10,2,N) as `game.state`, reward, lost, next_is_suicidal
(3, N), action 1:3).  Pure Julia, no library call."""
function unpack_bits(records::Matrix{UInt8})
    N = size(records, 2)
    state = zeros(Int, 10, 10, 2, N)
    reward = Vector{Float32}(undef, N); lost = Vector{Bool}(undef, N)
    suicidal = Matrix{Bool}(undef, 3, N); action = Vector{Int}(undef, N)
    for n in 1:N
        rec = @view records[:, n]
        for f in 1:2
            b = @view state[:, :, f, n]
            b[1, :] .= -1; b[10, :] .= -1; b[:, 1] .= -1; b[:, 10] .= -1
            for c in 1:8, r in 1:8                       # bit (r-1) + 8 (c-1) of the little-endian u64: byte c, bit r-1
                (rec[8 * (f - 1) + c] >> (r - 1)) & 0x01 == 0x01 && (b[r + 1, c + 1] = 1)
            end
            food = rec[16 + f]
            if food != 0x00
                fr, fc = Int(food & 0x0f) + 1, Int(food >> 4) + 1
                b[fr, fc] == 0 && (b[fr, fc] = 2)        # the snake hides the food
            end
        end
        head = rec[19]
        state[Int(head & 0x0f) + 1, Int(head >> 4) + 1, 2, n] = 1      # drawn last: overwrites the wall on a wall death
        flags = rec[20]
        for k in 1:3
            suicidal[k, n] = (flags >> (k - 1)) & 0x01 == 0x01
        end
        lost[n] = (flags >> 3) & 0x01 == 0x01
        action[n] = Int((flags >> 4) & 0x03) + 1
        reward[n] = reinterpret(Float32, UInt32(rec[21]) | UInt32(rec[22]) << 8 | UInt32(rec[23]) << 16 | UInt32(rec[24]) << 24)
    end
    return state, reward, lost, suicidal, action
end

"""`stack_exp(sample(rpb))` (utils.jl:343-383) into HOST arrays for the 0-based slots `idx`: (states, actions 1:3, rewards,
next_states, dones, suicidal_mask) in the reference's order and shapes."""
function stack_exp(r::DeviceReplayBuffer, idx::Vector{Int64})
    B = length(idx)
    states = Array{Float32,4}(undef, 10, 10, 2, B); next_states = similar(states)
    actions = Vector{UInt8}(undef, B); rewards = Vector{Float32}(undef, B); dones = Vector{UInt8}(undef, B)
    mask = Matrix{UInt8}(undef, 3, B)
    check(ccall((:snk_replay_gather_host, lib), Cint,
                (Ptr{Cvoid}, Ptr{Int64}, Int64, Ptr{Float32}, Ptr{Float32}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Cvoid}),
                r.handle, idx, B, states, next_states, actions, rewards, dones, mask, C_NULL))
    return states, Int.(actions) .+ 1, rewards, next_states, dones .!= 0, mask .!= 0
end

"""`sample(rpb)` indices (0-based slots, distinct) into a device Int64 buffer."""
sample_indices(r::DeviceReplayBuffer, d_idx::Ptr{Int64}, B::Integer; seed::Integer = 0) =
    check(ccall((:snk_replay_sample_indices, lib), Cint, (Ptr{Cvoid}, UInt64, Int64, Ptr{Int64}, Ptr{Cvoid}),
                r.handle, seed, B, d_idx, C_NULL))

"""`stack_exp(batch)` on the device: states/next_states (10,10,2,B) Float32, actions (0-based), rewards, dones, mask (3,B)."""
stack_exp(r::DeviceReplayBuffer, d_idx::Ptr{Int64}, B::Integer, d_states::Ptr{Float32}, d_next::Ptr{Float32},
          d_actions::Ptr{UInt8}, d_rewards::Ptr{Float32}, d_dones::Ptr{UInt8}, d_mask::Ptr{UInt8}) =
    check(ccall((:snk_replay_gather, lib), Cint,
                (Ptr{Cvoid}, Ptr{Int64}, Int64, Ptr{Float32}, Ptr{Float32}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8},
                 Ptr{Float32}, Ptr{Int32}, Ptr{Cvoid}),
                r.handle, d_idx, B, d_states, d_next, d_actions, d_rewards, d_dones, d_mask, C_NULL, C_NULL, C_NULL))

# ---- checkpoints: save_trainer / load_trainer (utils.jl:408-418), save_buffer / load_buffer (utils.jl:316-340) -----------
"""The library's checkpoint of the games (seed, generator counter, food list, every game's state) as bytes: write them
anywhere; `restore!` continues bit for bit."""
function checkpoint(g::BatchedSnakeGame)
    n = Ref{Csize_t}(0)
    check(ccall((:snk_env_checkpoint_bytes, lib), Cint, (Ptr{Cvoid}, Ref{Csize_t}), g.handle, n))
    blob = Vector{UInt8}(undef, n[])
    check(ccall((:snk_env_save_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Csize_t), g.handle, blob, length(blob)))
    return blob
end
"""Load a `checkpoint(g)` of games with the same N and auto-reset flag; a refused blob (SnakeB200Error naming the cause and
the first failing game) leaves `g` as it was.  The host mirrors are refreshed from the device."""
function restore!(g::BatchedSnakeGame, blob::Vector{UInt8})
    bad = Ref{Int64}(-1)
    check(ccall((:snk_env_load_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Csize_t, Ref{Int64}), g.handle, blob, length(blob), bad))
    virtual_step(g)
    assemble_state!(g)
    return g
end
"""The ring's checkpoint (the filled records, the stored count, the sampler's call count) as bytes."""
function checkpoint(r::DeviceReplayBuffer)
    n = Ref{Csize_t}(0)
    check(ccall((:snk_replay_checkpoint_bytes, lib), Cint, (Ptr{Cvoid}, Ref{Csize_t}), r.handle, n))
    blob = Vector{UInt8}(undef, n[])
    check(ccall((:snk_replay_save_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Csize_t), r.handle, blob, length(blob)))
    return blob
end
"""Load a `checkpoint(r)` of a ring of the same capacity; a refused blob leaves `r` as it was."""
function restore!(r::DeviceReplayBuffer, blob::Vector{UInt8})
    bad = Ref{Int64}(-1)
    check(ccall((:snk_replay_load_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Csize_t, Ref{Int64}), r.handle, blob, length(blob), bad))
    return r
end

# ---- Q-net forward (structs.jl:127-139) from Flux.destructure(q_net) ------------------------------------------
mutable struct DeviceQNet
    handle::Ptr{Cvoid}
    # theta, _ = Flux.destructure(model.q_net); precision = :f32 (Float32-faithful, the default) or :bf16 (fast, ~1e-2)
    function DeviceQNet(theta::Vector{Float32}; device::Integer = 0, precision::Symbol = :f32)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:snk_qnet_create, lib), Cint, (Ref{Ptr{Cvoid}}, Ptr{Float32}, Int64, Cint, Cint), h, theta, length(theta), device,
                    precision == :bf16 ? QNET_BF16 : QNET_F32))
        q = new(h[])
        finalizer(x -> ccall((:snk_qnet_destroy, lib), Cint, (Ptr{Cvoid},), x.handle), q)
        return q
    end
end
"""q_net(states): d_obs (10,10,2,N) Float32 -> d_q (3,N) Float32, both on the device."""
forward!(q::DeviceQNet, d_obs::Ptr{Float32}, N::Integer, d_q::Ptr{Float32}) =
    check(ccall((:snk_qnet_forward, lib), Cint, (Ptr{Cvoid}, Ptr{Float32}, Int64, Ptr{Float32}, Ptr{Cvoid}), q.handle, d_obs, N, d_q, C_NULL))

"""`true` if a forward since the last call left the fp16 range of the Float32-faithful mode's split operands"""
function overflowed(q::DeviceQNet)
    f = Ref{Cint}(0)
    check(ccall((:snk_qnet_overflow_host, lib), Cint, (Ptr{Cvoid}, Ref{Cint}), q.handle, f))
    return f[] != 0
end

"""Per-sample gradients of `Flux.huber_loss(q_net(s)[a], y)` (utils.jl:452-466), rows in Flux.destructure order, written as
the bf16 planes a Gram consumes (`planes(::GramShard)`) and / or as Float32 rows; device pointers."""
sample_grads!(q::DeviceQNet, d_states::Ptr{Float32}, d_actions::Ptr{UInt8}, d_targets::Ptr{Float64}, B::Integer,
              d_hi::Ptr{Cvoid}, d_lo::Ptr{Cvoid}, pitch::Integer, d_J::Ptr{Float32}, ldJ::Integer, d_loss::Ptr{Float32}) =
    check(ccall((:snk_qnet_sample_grads, lib), Cint,
                (Ptr{Cvoid}, Ptr{Float32}, Ptr{UInt8}, Ptr{Float64}, Int64, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float32}, Int64,
                 Ptr{Float32}, Ptr{Cvoid}),
                q.handle, d_states, d_actions, d_targets, B, d_hi, d_lo, pitch, d_J, ldJ, d_loss, C_NULL))

# ---- the learner (utils.jl:452-472) --------------------------------------------------------------------------------
"""Flux.Optimise.RMSProp(eta, rho, epsilon) (structs.jl:137: RMSProp(5e-4) = (0.0005, 0.9, 1e-8)) and its state for θ:
181,395 Float32 on `device`, zero-initialised here (a fresh optimiser), freed with the object."""
mutable struct RMSPropState
    d_acc::Ptr{Float32}
    eta::Float64
    rho::Float64
    epsilon::Float64
    function RMSPropState(; eta::Real = 5e-4, rho::Real = 0.9, epsilon::Real = 1e-8, device::Integer = 0)
        p, _ = device_alloc(181395 * 4, device; compressible = false)
        zero = zeros(Float32, 181395)
        check(ccall((:snk_copy_async, lib), Cint, (Ptr{Cvoid}, Ptr{Float32}, Csize_t, Ptr{Cvoid}), p, zero, sizeof(zero), C_NULL))
        o = new(Ptr{Float32}(p), eta, rho, epsilon)
        finalizer(x -> device_free(Ptr{Cvoid}(x.d_acc)), o)
        return o
    end
end

"""One minibatch update of `q` on the device (utils.jl:452-466): Flux.gradient of mean(huber(q_net(s)[a], y)) and
update!(opt, θ, g).  Device pointers as for `sample_grads!`; d_grad (181,395 Float32) and d_loss (1 Float32, the batch mean)
optional.  Enqueued on the default stream; order it with any forward of `q` (the same stream does)."""
train_step!(q::DeviceQNet, opt::RMSPropState, d_states::Ptr{Float32}, d_actions::Ptr{UInt8}, d_targets::Ptr{Float64}, B::Integer;
            d_grad::Ptr{Float32} = Ptr{Float32}(C_NULL), d_loss::Ptr{Float32} = Ptr{Float32}(C_NULL)) =
    check(ccall((:snk_qnet_train_step, lib), Cint,
                (Ptr{Cvoid}, Ptr{Float32}, Ptr{UInt8}, Ptr{Float64}, Int64, Ptr{Float32}, Cdouble, Cdouble, Cdouble, Ptr{Float32},
                 Ptr{Float32}, Ptr{Cvoid}),
                q.handle, d_states, d_actions, d_targets, B, opt.d_acc, opt.eta, opt.rho, opt.epsilon, d_grad, d_loss, C_NULL))

"""θ of `q` on the device (Flux.destructure order, 181,395 Float32): read-only, changes with every update"""
function params_device(q::DeviceQNet)
    p = Ref{Ptr{Float32}}(C_NULL)
    check(ccall((:snk_qnet_params, lib), Cint, (Ptr{Cvoid}, Ref{Ptr{Float32}}), q.handle, p))
    return p[]
end

"""update_target_net! (utils.jl:469-472): t's parameters become a copy of q's, on the device"""
update_target_net!(t::DeviceQNet, q::DeviceQNet) =
    check(ccall((:snk_qnet_set_params, lib), Cint, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Cvoid}), t.handle, params_device(q), C_NULL))

# ---- Laplace deviation matrix (compute_D.jl, plot_traj.jl, la_utils.jl) ----------------------------------------
"""deviation_matrix[:, position] = Float64.(theta) (compute_D.jl:67-71); position is 1-based like Julia's."""
store_snapshot!(d_D::Ptr{Float64}, P::Integer, K::Integer, position::Integer, d_theta::Ptr{Float32}) =
    check(ccall((:snk_d_store_snapshot, lib), Cint, (Ptr{Float64}, Int64, Int64, Int64, Ptr{Float32}, Ptr{Cvoid}),
                d_D, P, K, position - 1, d_theta, C_NULL))

"""G = D'D (K x K Float32) of a centred device-resident D; eigen(G).values ./ (K-1) == svd(D).S .^ 2 ./ (K-1)."""
function gram!(d_D::Ptr{Float64}, P::Integer, K::Integer, d_workspace::Ptr{Cvoid}, d_G::Ptr{Float32}; terms::Integer = 3)
    check(ccall((:snk_gram_pack, lib), Cint, (Ptr{Cvoid}, Cint, Int64, Int64, Ptr{Cvoid}, Ptr{Cvoid}), d_D, 2, P, K, d_workspace, C_NULL))
    check(ccall((:snk_gram, lib), Cint, (Ptr{Cvoid}, Int64, Int64, Cint, Cint, Cint, Ptr{Float32}, Ptr{Cvoid}),
                d_workspace, P, K, terms, 0, 0, d_G, C_NULL))
end
function gram_workspace_bytes(P::Integer, K::Integer)
    n = Ref{Csize_t}(0)
    check(ccall((:snk_gram_workspace_bytes, lib), Cint, (Int64, Int64, Cint, Ref{Csize_t}), K, P, 0, n))
    return Int(n[])
end

"""sample_model (la_utils.jl:83-95) with injected z1 (P), z2 (K) on the device."""
sample_model_weights!(d_mean::Ptr{Float64}, d_var::Ptr{Float64}, d_D::Ptr{Float64}, P::Integer, K::Integer,
                      d_z1::Ptr{Float64}, d_z2::Ptr{Float64}, d_w::Ptr{Float64}) =
    check(ccall((:snk_laplace_sample_weights, lib), Cint,
                (Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cvoid}),
                d_mean, d_var, d_D, P, K, d_z1, d_z2, d_w, C_NULL))

# ---- device-pointer forms of the per-call API (for CUDA.jl users: pass `pointer(cuarray)`) ----------------------------
# Everything below takes device pointers, enqueues on the handle's stream and returns; call sync(g) before reading.

"""step!(game, action) for N games (utils.jl:100-109): d_act holds 0-based indices into available_actions."""
step_device!(g::BatchedSnakeGame, d_act::Ptr{UInt8}, d_reward::Ptr{Float32}, d_done::Ptr{UInt8}) =
    check(ccall((:snk_step, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8}), g.handle, d_act, d_reward, d_done))

"""play_snake.jl:96-111 control: d_dir holds absolute directions 0:3 (U,D,L,R); the reverse of prev_dir loses (utils.jl:57)."""
step_abs_device!(g::BatchedSnakeGame, d_dir::Ptr{UInt8}, d_reward::Ptr{Float32}, d_done::Ptr{UInt8}) =
    check(ccall((:snk_step_abs, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8}), g.handle, d_dir, d_reward, d_done))

"""One fused launch on device buffers: epsilon_greedy (when d_q != C_NULL; d_u / d_ridx = injected draws or C_NULL) ->
step! -> virtual_step -> assemble_state!.  Any output pointer may be C_NULL.  obs_fmt: OBS_F32 / OBS_I8 / OBS_I64 / OBS_PACKED2."""
step_fused_device!(g::BatchedSnakeGame, d_q::Ptr{Float32}, epsilon::Real, d_u::Ptr{Float32}, d_ridx::Ptr{UInt8},
                   d_act::Ptr{UInt8}, d_reward::Ptr{Float32}, d_done::Ptr{UInt8}, d_obs::Ptr{Cvoid}, obs_fmt::Integer,
                   d_mask::Ptr{UInt8}, d_ep_return::Ptr{Float32}, d_ep_score::Ptr{Int32}) =
    check(ccall((:snk_step_fused, lib), Cint,
                (Ptr{Cvoid}, Ptr{Float32}, Cfloat, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8},
                 Ptr{Cvoid}, Cint, Ptr{UInt8}, Ptr{Float32}, Ptr{Int32}),
                g.handle, d_q, epsilon, d_u, d_ridx, d_act, d_reward, d_done, d_obs, obs_fmt, d_mask, d_ep_return, d_ep_score))

"""play_episode(...; actions_list = ...) (utils.jl:209-219) for N games: T scripted steps in ONE launch; d_act is (N,T)
column-major = step-major; outputs are step-major too ((N,T), (3,N,T), (10,10,2,N,T)); any output may be C_NULL."""
rollout_device!(g::BatchedSnakeGame, d_act::Ptr{UInt8}, T::Integer, is_abs::Bool, d_reward::Ptr{Float32}, d_done::Ptr{UInt8},
                d_obs::Ptr{Cvoid}, obs_fmt::Integer, d_mask::Ptr{UInt8}, d_ep_return::Ptr{Float32}, d_ep_score::Ptr{Int32}) =
    check(ccall((:snk_rollout_fused, lib), Cint,
                (Ptr{Cvoid}, Ptr{UInt8}, Int64, Cint, Ptr{Float32}, Ptr{UInt8}, Ptr{Cvoid}, Cint, Ptr{UInt8}, Ptr{Float32}, Ptr{Int32}),
                g.handle, d_act, T, is_abs ? 1 : 0, d_reward, d_done, d_obs, obs_fmt, d_mask, d_ep_return, d_ep_score))

"""assemble_state! (utils.jl:135-149) into a device buffer in the chosen format."""
state_device!(g::BatchedSnakeGame, d_obs::Ptr{Cvoid}, obs_fmt::Integer = OBS_F32) =
    check(ccall((:snk_state, lib), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Cint), g.handle, d_obs, obs_fmt))

"""virtual_step (utils.jl:112-132) of the current states: (3,N) UInt8, 1 = that action loses."""
losing_mask_device!(g::BatchedSnakeGame, d_mask::Ptr{UInt8}) =
    check(ccall((:snk_losing_mask, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, d_mask))

lost_device!(g::BatchedSnakeGame, d_done::Ptr{UInt8}) = check(ccall((:snk_get_done, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, d_done))
steps_device!(g::BatchedSnakeGame, d_steps::Ptr{Int32}) = check(ccall((:snk_get_steps, lib), Cint, (Ptr{Cvoid}, Ptr{Int32}), g.handle, d_steps))
"""per-env sticky error bits (ERR_FOOD where the reference would throw BoundsError, utils.jl:23,37; ERR_ACTION for an index > 2)."""
error_flags_device!(g::BatchedSnakeGame, d_flags::Ptr{UInt8}) =
    check(ccall((:snk_get_error_flags, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, d_flags))
function count_errors(g::BatchedSnakeGame)
    n = Ref{Int64}(0)
    check(ccall((:snk_count_errors_host, lib), Cint, (Ptr{Cvoid}, Ref{Int64}), g.handle, n))
    return n[]
end

"""seed of the internal counter-based draws used when epsilon_greedy gets no injected u / ridx (the reference uses the global RNG)."""
seed!(g::BatchedSnakeGame, seed::Integer) = check(ccall((:snk_set_seed, lib), Cint, (Ptr{Cvoid}, UInt64), g.handle, UInt64(seed)))
"""run the handle's work on a caller-owned CUDA stream (e.g. CUDA.stream().handle); C_NULL = the legacy default stream."""
set_stream!(g::BatchedSnakeGame, stream::Ptr{Cvoid}) = check(ccall((:snk_set_stream, lib), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), g.handle, stream))
num_envs(g::BatchedSnakeGame) = Int(ccall((:snk_num_envs, lib), Int64, (Ptr{Cvoid},), g.handle))
library_version() = Int(ccall((:snk_version, lib), Cint, ()))

"""the 50 food cells of Xoshiro(42) (structs.jl:33,70) as the library holds them: vector of (row, col), 1-based."""
function default_food_list()
    cells = zeros(UInt8, 2, 64)
    n = Ref{Cint}(0)
    check(ccall((:snk_default_food_list_host, lib), Cint, (Ptr{UInt8}, Ref{Cint}), cells, n))
    return [(Int(cells[1, i]), Int(cells[2, i])) for i in 1:n[]]
end

# ---- row-sharded Gram: one process (Distributed.jl worker / MPI rank) per GPU, ONE call per rank and Gram ----------------
"""This rank's share of G = A A' for A row-sharded over `length(rows_all)` GPUs of one box (BASELINE config 5b)."""
mutable struct GramShard
    handle::Ptr{Cvoid}
    rows::Int
    K::Int
    function GramShard(rows_all::Vector{Int64}, rank::Integer, P::Integer; device::Integer = rank, splits::Integer = 0)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:snk_gram_shard_create, lib), Cint, (Ref{Ptr{Cvoid}}, Ptr{Int64}, Cint, Cint, Int64, Cint, Cint),
                    h, rows_all, length(rows_all), rank, P, splits, device))
        g = new(h[], rows_all[rank + 1], sum(rows_all))
        finalizer(x -> ccall((:snk_gram_shard_destroy, lib), Cint, (Ptr{Cvoid},), x.handle), g)
        return g
    end
end
"""192 bytes to send to every other rank (e.g. `MPI.Allgather`, or `fetch` from each Distributed.jl worker)"""
function export_handle(g::GramShard)
    h = Vector{UInt8}(undef, 192)
    check(ccall((:snk_gram_shard_export_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, h))
    return h
end
"""`handles` = the 192-byte handles of ALL ranks, concatenated in rank order"""
connect!(g::GramShard, handles::Vector{UInt8}) =
    check(ccall((:snk_gram_shard_connect_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, handles))
"""G[rows of this rank, :] into the device buffer d_G (rows x K Float32).  d_A: this rank's rows of A on the device (Float64:
dtype 2, Float32: dtype 1) or C_NULL when the planes were filled by `sample_grads!`.  Enqueued; every rank must call it."""
run!(g::GramShard, d_A::Ptr{Cvoid}, dtype::Integer, d_G::Ptr{Float32}; terms::Integer = 3) =
    check(ccall((:snk_gram_shard_run, lib), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float32}, Int64, Ptr{Cvoid}),
                g.handle, d_A, dtype, terms, 0, d_G, g.K, C_NULL))
"""(hi, lo, pitch): the bf16 planes of this rank's rows, for a producer that writes them directly"""
function planes(g::GramShard)
    hi = Ref{Ptr{Cvoid}}(C_NULL); lo = Ref{Ptr{Cvoid}}(C_NULL); pitch = Ref{Int64}(0)
    check(ccall((:snk_gram_shard_planes, lib), Cint, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}, Ref{Ptr{Cvoid}}, Ref{Int64}), g.handle, hi, lo, pitch))
    return hi[], lo[], Int(pitch[])
end

# ---- data-parallel learner: one process (Distributed.jl worker / MPI rank) per GPU, one Q-net trained on all of them ---------
"""Rank `rank` of a learner group of `world` ranks around `q` (DESIGN §5f).  Every rank's `q` holds the same θ; after each
`train_step!` every rank holds θ, acc, g and loss of `train_step!(q, ...)` on the ranks' minibatches concatenated in rank
order, bit for bit.  `q` must outlive the group."""
mutable struct LearnerGroup
    handle::Ptr{Cvoid}
    world::Int
    q::DeviceQNet
    function LearnerGroup(q::DeviceQNet, world::Integer, rank::Integer)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:snk_qnet_group_create, lib), Cint, (Ref{Ptr{Cvoid}}, Ptr{Cvoid}, Cint, Cint), h, q.handle, world, rank))
        g = new(h[], world, q)
        finalizer(x -> ccall((:snk_qnet_group_destroy, lib), Cint, (Ptr{Cvoid},), x.handle), g)
        return g
    end
end
"""64 bytes to send to every other rank"""
function export_handle(g::LearnerGroup)
    h = Vector{UInt8}(undef, 64)
    check(ccall((:snk_qnet_group_export_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, h))
    return h
end
"""`handles` = the 64-byte handles of ALL ranks, concatenated in rank order"""
connect!(g::LearnerGroup, handles::Vector{UInt8}) =
    check(ccall((:snk_qnet_group_connect_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Cint), g.handle, handles, length(handles) ÷ 64))
"""This rank's part of one group update: its own B_local transitions (device pointers as for `train_step!`).  Enqueued on
the default stream; every rank must call it the same number of times."""
train_step!(g::LearnerGroup, opt::RMSPropState, d_states::Ptr{Float32}, d_actions::Ptr{UInt8}, d_targets::Ptr{Float64},
            B_local::Integer; d_grad::Ptr{Float32} = Ptr{Float32}(C_NULL), d_loss::Ptr{Float32} = Ptr{Float32}(C_NULL)) =
    check(ccall((:snk_qnet_group_train_step, lib), Cint,
                (Ptr{Cvoid}, Ptr{Float32}, Ptr{UInt8}, Ptr{Float64}, Int64, Ptr{Float32}, Cdouble, Cdouble, Cdouble, Ptr{Float32},
                 Ptr{Float32}, Ptr{Cvoid}),
                g.handle, d_states, d_actions, d_targets, B_local, opt.d_acc, opt.eta, opt.rho, opt.epsilon, d_grad, d_loss, C_NULL))
"""throws if a wait of this rank gave up on a peer (synchronises)"""
function check_peers(g::LearnerGroup)
    t = Ref{Cint}(0)
    check(ccall((:snk_qnet_group_status_host, lib), Cint, (Ptr{Cvoid}, Ref{Cint}), g.handle, t))
end

# ---- replay group: one minibatch drawn uniformly from the union of every rank's ring (DESIGN §5g) -------------------------
"""Rank `rank` of a replay group of `world` ranks around the ring `r`.  `batch_all` (one share B_q >= 1 per rank) and `seed` are
the same on every rank.  The ranks' `sample!` outputs concatenated in rank order are `sample_indices` + `stack_exp` of one
full ring holding every rank's filled records, bit for bit.  `r` must outlive the group."""
mutable struct ReplayGroup
    handle::Ptr{Cvoid}
    world::Int
    r::DeviceReplayBuffer
    function ReplayGroup(r::DeviceReplayBuffer, world::Integer, rank::Integer, batch_all::Vector{Int64}, seed::Integer)
        length(batch_all) == world || throw(ArgumentError("batch_all needs one entry per rank"))
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:snk_replay_group_create, lib), Cint, (Ref{Ptr{Cvoid}}, Ptr{Cvoid}, Cint, Cint, Ptr{Int64}, UInt64),
                    h, r.handle, world, rank, batch_all, UInt64(seed)))
        g = new(h[], world, r)
        finalizer(x -> ccall((:snk_replay_group_destroy, lib), Cint, (Ptr{Cvoid},), x.handle), g)
        return g
    end
end
"""128 bytes to send to every other rank"""
function export_handle(g::ReplayGroup)
    h = Vector{UInt8}(undef, 128)
    check(ccall((:snk_replay_group_export_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}), g.handle, h))
    return h
end
"""`handles` = the 128-byte handles of ALL ranks, concatenated in rank order"""
connect!(g::ReplayGroup, handles::Vector{UInt8}) =
    check(ccall((:snk_replay_group_connect_host, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Cint), g.handle, handles, length(handles) ÷ 128))
"""This rank's share of one group minibatch into device buffers in `stack_exp`'s layout (states / next_states (10,10,2,B)
Float32, actions B UInt8 0-based, rewards B Float32, dones B UInt8, mask (3,B) UInt8; d_idx: the union indices, Int64).  Any
may be C_NULL.  Enqueued on the default stream; every rank must call it the same number of times."""
sample!(g::ReplayGroup, d_states::Ptr{Float32}, d_next_states::Ptr{Float32}, d_actions::Ptr{UInt8}, d_rewards::Ptr{Float32},
        d_dones::Ptr{UInt8}, d_mask::Ptr{UInt8}; d_idx::Ptr{Int64} = Ptr{Int64}(C_NULL)) =
    check(ccall((:snk_replay_group_sample, lib), Cint,
                (Ptr{Cvoid}, Ptr{Int64}, Ptr{Float32}, Ptr{Float32}, Ptr{UInt8}, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32},
                 Ptr{Int32}, Ptr{Cvoid}),
                g.handle, d_idx, d_states, d_next_states, d_actions, d_rewards, d_dones, d_mask, Ptr{Float32}(C_NULL),
                Ptr{Int32}(C_NULL), C_NULL))
"""throws if a wait of this rank gave up on a peer, or a call asked for more transitions than the rings held (synchronises)"""
function check_peers(g::ReplayGroup)
    t = Ref{Cint}(0); f = Ref{Cint}(0)
    check(ccall((:snk_replay_group_status_host, lib), Cint, (Ptr{Cvoid}, Ref{Cint}, Ref{Cint}), g.handle, t, f))
end

"""`bytes` of device memory on `device` for the outputs of the fused step; with `compressible`, memory with generic L2
compression where the device supports it (lossless; the Float32 step writes fewer DRAM bytes).  Returns (pointer, compressible)."""
function device_alloc(bytes::Integer, device::Integer = 0; compressible::Bool = true)
    p = Ref{Ptr{Cvoid}}(C_NULL); got = Ref{Cint}(0)
    check(ccall((:snk_device_alloc, lib), Cint, (Ref{Ptr{Cvoid}}, Csize_t, Cint, UInt32, Ref{Cint}),
                p, bytes, device, compressible ? UInt32(1) : UInt32(0), got))
    return p[], got[] != 0
end
"""frees memory from `device_alloc` (synchronises the device first)"""
device_free(p::Ptr{Cvoid}) = check(ccall((:snk_device_free, lib), Cint, (Ptr{Cvoid},), p))
function compression_supported(device::Integer = 0)
    yes = Ref{Cint}(0)
    check(ccall((:snk_compression_supported, lib), Cint, (Cint, Ref{Cint}), device, yes))
    return yes[] != 0
end

end # module
