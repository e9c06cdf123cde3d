# DRiLB200.jl — Julia host shim over libdril_b200.so (include/dril_b200.h).
#
# UNVERIFIED IN THIS REPO: the build image has no Julia toolchain (SURVEY.md §8c), so this file is
# the binding a DRiL.jl maintainer would add, kept thin and mechanical: every method is one or two
# `ccall`s.  The same ABI is exercised end-to-end from Python (dril.jl_b200/_lib.py, tests/).
#
# What it provides (dispatch contract of the reference, paths relative to DRiL.jl):
#   CudaBatchedEnv <: AbstractParallelEnv      src/interfaces/environments.jl:39-157
#   train!(agent, env::CudaBatchedEnv, alg::PPO, max_steps; callbacks)   src/algorithms/ppo.jl:100-325
#   collect_rollout!(buf::DeviceRolloutBuffer, agent, alg, env::CudaBatchedEnv)  src/buffers/rollout_buffer.jl:46-90
#   evaluate_agent(agent, env::CudaBatchedEnv; ...)                              src/evaluation.jl:54-143
#   save_normalization_stats / load_normalization_stats! / sync_normalization_stats!   src/environment_wrappers/normalizeWrapperEnv.jl:261-309
#   extract_policy(agent, norm_env::CudaBatchedEnv)                              src/deployment/deployment_policy.jl:50-71
# Agent.train_state.parameters stays the source of truth: parameters are flattened in
# ComponentVector order on the way in and copied back after train! so extract_policy,
# predict_actions and save_policy_params_and_state keep working unchanged.
module DRiLB200

using DRiL
using DRiL: AbstractParallelEnv, AbstractCallback, Agent, PPO, Box, Discrete
using ComponentArrays: ComponentVector, getaxes
using Random

const LIB = get(ENV, "DRIL_B200_LIB", joinpath(@__DIR__, "..", "dril.jl_b200", "libdril_b200.so"))

struct DrilError <: Exception
    msg::String
end
last_error() = unsafe_string(ccall((:dril_last_error, LIB), Cstring, ()))
check(status::Int32) = status == 0 ? nothing : throw(DrilError(last_error()))

# ---- mirrors of the C structs ------------------------------------------------------------------
struct NormCfg
    training::Int32; norm_obs::Int32; norm_reward::Int32
    clip_obs::Float32; clip_reward::Float32; gamma::Float32; epsilon::Float32
end
struct PPOHyper
    gamma::Float32; gae_lambda::Float32; clip_range::Float32; clip_range_vf::Float32
    ent_coef::Float32; vf_coef::Float32; max_grad_norm::Float32; target_kl::Float32
    normalize_advantage::Int32; learning_rate::Float32
    adam_beta1::Float32; adam_beta2::Float32; adam_eps::Float32
end
struct IterStats
    entropy_loss::Float32; policy_loss::Float32; value_loss::Float32; approx_kl_div::Float32
    clip_fraction::Float32; loss::Float32; explained_variance::Float32; grad_norm::Float32
    learning_rate::Float32; entropy::Float32; ratio::Float32; rollout_ms::Float32; update_ms::Float32
    n_minibatch_steps::Int32; kl_stopped::Int32; episodes::Int64
    episode_return_sum::Float64; episode_length_sum::Float64
    ep_rew_mean::Float32; ep_len_mean::Float32; episodes_in_window::Int64
end
neg(x) = isnothing(x) ? -1.0f0 : Float32(x)
PPOHyper(alg::PPO) = PPOHyper(alg.gamma, alg.gae_lambda, alg.clip_range, neg(alg.clip_range_vf), alg.ent_coef,
    alg.vf_coef, neg(alg.max_grad_norm), neg(alg.target_kl), Int32(alg.normalize_advantage), alg.learning_rate,
    0.9f0, 0.999f0, 1.0f-5)   # Optimisers.Adam(eta, (0.9, 0.999), 1e-5): src/algorithms/ppo.jl:64-66

# ---- context -----------------------------------------------------------------------------------
mutable struct Context
    h::Ptr{Cvoid}
    function Context(device::Integer = 0; seed::Integer = 0)
        out = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:dril_ctx_create, LIB), Int32, (Int32, UInt64, Ref{Ptr{Cvoid}}), device, seed, out))
        ctx = new(out[])
        finalizer(c -> ccall((:dril_ctx_destroy, LIB), Int32, (Ptr{Cvoid},), c.h), ctx)
    end
end
const DEFAULT_CTX = Ref{Union{Nothing, Context}}(nothing)
default_ctx() = (isnothing(DEFAULT_CTX[]) && (DEFAULT_CTX[] = Context()); DEFAULT_CTX[])

# ---- batched env -------------------------------------------------------------------------------
const ENV_KINDS = Dict(:cartpole => 0, :pendulum => 1, :synthetic => 2, :mountaincar => 3, :mountaincar_continuous => 4, :acrobot => 5)
# per-env physical parameters (dril_b200.h): name => default, in the order of the C arrays
const ENV_PARAMS = Dict(
    :cartpole => (:gravity => 9.8, :masscart => 1.0, :masspole => 0.1, :length => 0.5, :force_mag => 10.0, :tau => 0.02),
    :pendulum => (:g => 10.0, :m => 1.0, :l => 1.0, :dt => 0.05),
    :synthetic => (),
    :mountaincar => (:force => 0.001, :gravity => 0.0025),
    :mountaincar_continuous => (:power => 0.0015, :gravity => 0.0025),
    :acrobot => (:link_length_1 => 1.0, :link_mass_1 => 1.0, :link_mass_2 => 1.0, :link_com_pos_1 => 0.5, :link_com_pos_2 => 0.5, :link_moi => 1.0),
)

# the non-velocity components (1-based) of each kind's observation: the frame of an env with mask_velocities = true
const VELOCITY_FREE = Dict(:cartpole => [1, 3], :pendulum => [1, 2], :mountaincar => [1], :mountaincar_continuous => [1],
                           :acrobot => [1, 2, 3, 4])

"""
    CudaBatchedEnv(kind, n_envs; max_steps, act_start, monitor_window, normalize, env_params, observe_params, history_len,
                   mask_velocities, obs_noise, action_delay)

Device-resident replacement of `NormalizeWrapperEnv(MonitorWrapperEnv(MultiThreadedParallelEnv(envs)))`
for `kind in (:cartpole, :pendulum, :synthetic, :mountaincar, :mountaincar_continuous, :acrobot)`.
`env_params = Dict(:length => (0.25, 1.0), ...)`: per-env physical parameters, see `set_env_params!`.
`observe_params = true`: every observation is `[base observation | the running episode's parameter values]` in the order of
`ENV_PARAMS[kind]`, raw (Scaling maps the base components only); `observation_space` is widened by `[0, Inf)` per parameter.
`history_len = k` (1 to 4): every observation is the last k frames `[f_{t-k+1} | ... | f_t]`, oldest first;
`mask_velocities = true` keeps only each frame's non-velocity components (`VELOCITY_FREE[kind]`); `observation_space` is the
(scaled) bounds of the kept components tiled k times.  `reset!` restarts the history from the current frame.
`obs_noise`, `action_delay`: sensor noise and actuation delay, see `set_obs_noise!` and `set_action_delay!`.
"""
mutable struct CudaBatchedEnv <: AbstractParallelEnv
    ctx::Context
    h::Ptr{Cvoid}
    kind::Symbol
    n_envs::Int
    obs_space::Box{Float32}
    act_space::Union{Box{Float32}, Discrete{Int}}
    monitor_window::Int
    normalize::Union{Nothing, NormCfg}
    terminated::Vector{Bool}
    truncated::Vector{Bool}
end

function CudaBatchedEnv(kind::Symbol, n_envs::Integer; ctx = default_ctx(), max_steps = 0, obs_dim = 0, act_start = 1,
        monitor_window = 0, normalize::Union{Nothing, NormCfg} = nothing, gid_offset = 0, scaling::Bool = false,
        env_params = nothing, observe_params::Bool = false, history_len::Integer = 1, mask_velocities::Bool = false,
        obs_noise = nothing, action_delay = 0)
    obs_space, act_space = if kind == :cartpole
        hi = Float32[4.8, Inf32, 0.41887903, Inf32]
        Box(-hi, hi), Discrete(2, act_start)
    elseif kind == :pendulum
        Box(Float32[-1, -1, -8], Float32[1, 1, 8]), Box(Float32[-2], Float32[2])
    elseif kind == :mountaincar
        Box(Float32[-1.2, -0.07], Float32[0.6, 0.07]), Discrete(3, act_start)
    elseif kind == :mountaincar_continuous
        Box(Float32[-1.2, -0.07], Float32[0.6, 0.07]), Box(Float32[-1], Float32[1])
    elseif kind == :acrobot
        hi = Float32[1, 1, 1, 1, 4pi, 9pi]
        Box(-hi, hi), Discrete(3, act_start)
    else
        Box(-ones(Float32, obs_dim), ones(Float32, obs_dim)), Discrete(2, act_start)
    end
    out = Ref{Ptr{Cvoid}}(C_NULL)
    normptr = isnothing(normalize) ? C_NULL : Ref(normalize)
    GC.@preserve normptr check(ccall((:dril_env_create, LIB), Int32,
        (Ptr{Cvoid}, Int32, Int64, Int32, Int32, Int32, Int64, Ptr{NormCfg}, Int32, Ref{Ptr{Cvoid}}),
        ctx.h, ENV_KINDS[kind], n_envs, max_steps, size(obs_space)[1], act_start, gid_offset,
        isnothing(normalize) ? C_NULL : Base.unsafe_convert(Ptr{NormCfg}, normptr), monitor_window, out))
    observe_params && check(ccall((:dril_env_set_observe_params, LIB), Int32, (Ptr{Cvoid}, Int32), out[], 1))
    if scaling
        # ScalingWrapperEnv around every env of the batch (scalingWrapperEnv.jl:14-49): Box/Box envs only; the device maps
        # observations to [-1, 1] and actions back from [-1, 1], so the spaces the agent sees are the scaled ones
        obs_space isa Box && act_space isa Box || error("ScalingWrapperEnv needs Box observation and action spaces")
        check(ccall((:dril_env_set_scaling, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}),
            out[], 1, vec(obs_space.low), vec(obs_space.high), vec(act_space.low), vec(act_space.high)))
        obs_space = Box(-ones(Float32, size(obs_space.low)), ones(Float32, size(obs_space.high)))
        act_space = Box(-ones(Float32, size(act_space.low)), ones(Float32, size(act_space.high)))
    end
    if history_len != 1 || mask_velocities
        check(ccall((:dril_env_set_obs_history, LIB), Int32, (Ptr{Cvoid}, Int32, Int32), out[], history_len, mask_velocities))
        keep = mask_velocities ? VELOCITY_FREE[kind] : collect(1:length(obs_space.low))
        obs_space = Box(repeat(vec(obs_space.low)[keep], history_len), repeat(vec(obs_space.high)[keep], history_len))
    end
    if observe_params
        P = length(ENV_PARAMS[kind])
        obs_space = Box(vcat(vec(obs_space.low), zeros(Float32, P)), vcat(vec(obs_space.high), fill(Inf32, P)))
    end
    if observe_params || history_len != 1 || mask_velocities
        d = Ref{Int32}(0)
        check(ccall((:dril_env_obs_dim, LIB), Int32, (Ptr{Cvoid}, Ref{Int32}), out[], d))
        d[] == size(obs_space)[1] || error("observation width $(d[]) != $(size(obs_space)[1])")
    end
    env = CudaBatchedEnv(ctx, out[], kind, n_envs, obs_space, act_space, monitor_window, normalize,
        falses(n_envs), falses(n_envs))
    finalizer(e -> ccall((:dril_env_destroy, LIB), Int32, (Ptr{Cvoid},), e.h), env)
    isnothing(env_params) || isempty(env_params) || set_env_params!(env; env_params...)
    isnothing(obs_noise) || set_obs_noise!(env, obs_noise)
    all(iszero, action_delay) || set_action_delay!(env, action_delay)
    env
end

# components of each kind's base observation: the rows of an observation-noise array
const BASE_OBS_DIM = Dict(:cartpole => 4, :pendulum => 3, :mountaincar => 2, :mountaincar_continuous => 2, :acrobot => 6)
const MAX_ACTION_DELAY = 4

"""
    set_obs_noise!(env, std)

Per-env observation (sensor) noise: `std` is a number, a vector of `F0 = BASE_OBS_DIM[kind]` deviations (one per component of
the base observation) or an `F0 x n_envs` matrix; `nothing` turns it off.  Component j of every observation gets
`std[j, n] * z` added to its raw value (before Scaling, the velocity mask and the history), `z ~ N(0, 1)` a pure function of
(seed, env, episode, step, j).  Takes effect at the next observation.
"""
function set_obs_noise!(env::CudaBatchedEnv, std)
    if isnothing(std)
        check(ccall((:dril_env_set_obs_noise, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}), env.h, 0, C_NULL))
        return env
    end
    F0 = get(BASE_OBS_DIM, env.kind, 0)
    s = std isa Number ? fill(Float32(std), F0, env.n_envs) : std isa AbstractVector ? repeat(Float32.(std), 1, env.n_envs) : Float32.(std)
    size(s, 2) == env.n_envs || error("obs_noise of size $(size(s)): need ($F0, $(env.n_envs))")
    m = Matrix{Float32}(permutedims(s))   # column j = component j: the C layout [n_comp][n_envs]
    check(ccall((:dril_env_set_obs_noise, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}), env.h, size(s, 1), m))
    env
end

"""
    set_action_delay!(env, delay)

Per-env action (actuation) delay: a number or a vector of `n_envs` delays d in `0:MAX_ACTION_DELAY`; env n applies the
action chosen d steps earlier in its episode (the first action after a reset fills its queue); `nothing` turns it off.
Restarts every env's queue.
"""
function set_action_delay!(env::CudaBatchedEnv, delay)
    if isnothing(delay)
        check(ccall((:dril_env_set_action_delay, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}), env.h, C_NULL))
        return env
    end
    d = delay isa Number ? fill(Int32(delay), env.n_envs) : Int32.(collect(delay))
    check(ccall((:dril_env_set_action_delay, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}), env.h, d))
    env
end

# dril_adr_param
struct AdrParam
    index::Int32
    init_lo::Float32
    init_hi::Float32
    limit_lo::Float32
    limit_hi::Float32
    delta::Float32
end

"""
    set_adr!(env, params; thresholds, p_boundary = 0.2, buffer_size = 64)
    set_adr!(env, nothing)

Automatic domain randomisation (include/dril_b200.h has the rules): `params = [:length => (init = (0.5, 0.5),
limits = (0.1, 2.0), step = 0.05), ...]` (any iterable of `name => (init, limits, step)` pairs: its iteration order is the
order of `adr_state`; a `Dict` iterates in no fixed order), `thresholds = (t_low, t_high)` in episode-return units (required).
After every collected rollout a boundary whose last `buffer_size` episodes average `>= t_high` moves outwards by its step,
`<= t_low` inwards (never inside the initial range).  `nothing` turns ADR off and leaves every env at the ranges it reached.
Needs a Monitor.
"""
function set_adr!(env::CudaBatchedEnv, ::Nothing)
    check(ccall((:dril_env_set_adr, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{AdrParam}, Float32, Int64, Float32, Float32),
        env.h, 0, C_NULL, 0, 1, 0, 1))
    env
end
function set_adr!(env::CudaBatchedEnv, params; thresholds, p_boundary = 0.2, buffer_size = 64)
    names = [first(p) for p in ENV_PARAMS[env.kind]]
    ps = [AdrParam(findfirst(==(k), names) - 1, q.init[1], q.init[2], q.limits[1], q.limits[2], q.step) for (k, q) in params]
    check(ccall((:dril_env_set_adr, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{AdrParam}, Float32, Int64, Float32, Float32),
        env.h, length(ps), ps, p_boundary, buffer_size, thresholds[1], thresholds[2]))
    env
end

"""
    adr_state(env, n) -> (lo, hi, sums, counts, round)

The ADR state of an env with `n` parameters under ADR (in the iteration order of the `params` given to `set_adr!`): the ranges, the per-slot return
sums and episode counts buffered since each slot's last decision (slot `2i - 1` the low and `2i` the high side of parameter i),
and the number of rounds so far.
"""
function adr_state(env::CudaBatchedEnv, n::Integer)
    lo, hi = zeros(Float32, n), zeros(Float32, n)
    sums, counts = zeros(Float64, 2n), zeros(Int64, 2n)
    r = Ref{Int64}(0)
    check(ccall((:dril_env_get_adr, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Ptr{Float64}, Ptr{Int64}, Ref{Int64}),
        env.h, lo, hi, sums, counts, r))
    (lo, hi, sums, counts, r[])
end

"""
    set_env_params!(env; length = (0.25, 1.0), masspole = 0.2, ...)

Per-env physical parameters (names and defaults: `ENV_PARAMS[kind]`).  Each value is a number, a vector of `n_envs`, or a
tuple `(lo, hi)` of either: every reset draws a value per env from `[lo, hi]`.  Unnamed parameters keep their defaults; with
no keyword the env returns to the built-in constants.
"""
function set_env_params!(env::CudaBatchedEnv; kw...)
    spec = ENV_PARAMS[env.kind]
    names = Symbol[first(p) for p in spec]
    for k in keys(kw)
        k in names || error("$(env.kind) has no parameter $k; it has $names")
    end
    if isempty(kw)
        isempty(names) || check(ccall((:dril_env_set_params, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}, Ptr{Float32}),
            env.h, length(names), C_NULL, C_NULL))
        return env
    end
    n = env.n_envs
    lo = Matrix{Float32}(undef, n, length(names))   # column k = parameter k: the C layout [n_params][n_envs]
    hi = similar(lo)
    for (k, (name, default)) in enumerate(spec)
        v = get(kw, name, default)
        a, b = v isa Tuple ? v : (v, v)
        lo[:, k] .= Float32.(a)
        hi[:, k] .= Float32.(b)
    end
    check(ccall((:dril_env_set_params, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}, Ptr{Float32}), env.h, length(names), lo, hi))
    env
end

"""
    env_params(env) -> Dict(name => Vector{Float32}(n_envs))

Each env's parameter values for its running episode.
"""
function env_params(env::CudaBatchedEnv)
    spec = ENV_PARAMS[env.kind]
    v = Matrix{Float32}(undef, env.n_envs, length(spec))
    isempty(spec) || check(ccall((:dril_env_get_params, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}), env.h, length(spec), v))
    Dict(first(p) => v[:, k] for (k, p) in enumerate(spec))
end

DRiL.number_of_envs(env::CudaBatchedEnv) = env.n_envs
DRiL.observation_space(env::CudaBatchedEnv) = env.obs_space
DRiL.action_space(env::CudaBatchedEnv) = env.act_space
DRiL.terminated(env::CudaBatchedEnv) = copy(env.terminated)
DRiL.truncated(env::CudaBatchedEnv) = copy(env.truncated)
DRiL.get_info(env::CudaBatchedEnv) = [Dict{String, Any}() for _ in 1:env.n_envs]
DRiL.is_monitored(env::CudaBatchedEnv) = env.monitor_window > 0
Random.seed!(env::CudaBatchedEnv, seed::Integer) =
    (check(ccall((:dril_env_seed, LIB), Int32, (Ptr{Cvoid}, UInt64), env.h, seed)); env)

function DRiL.reset!(env::CudaBatchedEnv)
    check(ccall((:dril_env_reset, LIB), Int32, (Ptr{Cvoid},), env.h))
    fill!(env.terminated, false); fill!(env.truncated, false)
    return nothing
end

function DRiL.observe(env::CudaBatchedEnv)
    D = size(env.obs_space)[1]
    obs = Matrix{Float32}(undef, D, env.n_envs)          # C layout [n][D] == Julia (D, n) column-major
    check(ccall((:dril_env_observe, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}), env.h, obs))
    return [obs[:, i] for i in 1:env.n_envs]
end

function DRiL.act!(env::CudaBatchedEnv, actions::AbstractVector)
    n, D = env.n_envs, size(env.obs_space)[1]
    acts = env.act_space isa Discrete ? Int64.(actions) : reduce(hcat, [Float32.(vec(a)) for a in actions])
    rewards = Vector{Float32}(undef, n); term = Vector{UInt8}(undef, n); trunc = Vector{UInt8}(undef, n)
    tobs = Matrix{Float32}(undef, D, n); epr = Vector{Float32}(undef, n); epl = Vector{Int64}(undef, n)
    check(ccall((:dril_env_step, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}, Ptr{UInt8}, Ptr{UInt8}, Ptr{Float32}, Ptr{Float32}, Ptr{Int64}),
        env.h, acts, rewards, term, trunc, tobs, epr, epl))
    env.terminated .= term .!= 0; env.truncated .= trunc .!= 0
    infos = Vector{Dict{String, Any}}(undef, n)
    for i in 1:n
        d = Dict{String, Any}()
        env.truncated[i] && (d["terminal_observation"] = tobs[:, i])
        if env.monitor_window > 0 && (env.terminated[i] || env.truncated[i])
            d["episode"] = Dict("r" => epr[i], "l" => Int(epl[i]))
        end
        infos[i] = d
    end
    return rewards, copy(env.terminated), copy(env.truncated), infos
end

function DRiL.log_stats(env::CudaBatchedEnv, logger::DRiL.AbstractTrainingLogger)
    env.monitor_window > 0 || return nothing
    r = Ref{Float32}(0); l = Ref{Float32}(0); nw = Ref{Int64}(0); tot = Ref{Int64}(0)
    check(ccall((:dril_env_monitor_stats, LIB), Int32, (Ptr{Cvoid}, Ref{Float32}, Ref{Float32}, Ref{Int64}, Ref{Int64}),
        env.h, r, l, nw, tot))
    if nw[] > 0
        DRiL.log_scalar!(logger, "env/ep_rew_mean", r[])
        DRiL.log_scalar!(logger, "env/ep_len_mean", l[])
    end
    return nothing
end

# ---- device policy (one per Agent, cached in agent.aux-like side table) -------------------------
mutable struct DevicePolicy
    h::Ptr{Cvoid}
    n_params::Int
end
const POLICIES = IdDict{Any, DevicePolicy}()

function device_policy(agent::Agent, ctx::Context)
    get!(POLICIES, agent) do
        layer = agent.layer
        as = DRiL.action_space(layer)
        hidden = Int32[size(l.weight, 1) for l in values(agent.train_state.parameters.critic_head)][1:end-1]
        obs_dim = prod(size(DRiL.observation_space(layer)))
        out = Ref{Ptr{Cvoid}}(C_NULL)
        if as isa Discrete
            check(ccall((:dril_policy_create, LIB), Int32,
                (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Int32, Int32, Int32, Ptr{Float32}, Ptr{Float32}, Ref{Ptr{Cvoid}}),
                ctx.h, obs_dim, length(hidden), hidden, 0, as.n, as.start, C_NULL, C_NULL, out))
        else
            lo, hi = Float32.(vec(as.low)), Float32.(vec(as.high))
            check(ccall((:dril_policy_create, LIB), Int32,
                (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Int32, Int32, Int32, Ptr{Float32}, Ptr{Float32}, Ref{Ptr{Cvoid}}),
                ctx.h, obs_dim, length(hidden), hidden, 1, length(lo), 0, lo, hi, out))
        end
        n = Ref{Int64}(0)
        check(ccall((:dril_policy_num_params, LIB), Int32, (Ptr{Cvoid}, Ref{Int64}), out[], n))
        DevicePolicy(out[], n[])
    end
end

"Flatten Lux parameters in ComponentVector order (== layers/layer_lux.jl:4-52 NamedTuple order)."
flat_params(agent::Agent) = Vector{Float32}(ComponentVector(agent.train_state.parameters))
function push_params!(p::DevicePolicy, agent::Agent)
    flat = flat_params(agent)
    @assert length(flat) == p.n_params
    check(ccall((:dril_policy_set_params, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}, Int64), p.h, flat, length(flat)))
end
function pull_params!(agent::Agent, p::DevicePolicy)
    flat = Vector{Float32}(undef, p.n_params)
    check(ccall((:dril_policy_get_params, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}, Int64), p.h, flat, length(flat)))
    ax = getaxes(ComponentVector(agent.train_state.parameters))
    ps = NamedTuple(ComponentVector(flat, ax))
    agent.train_state = DRiL.Accessors.@set agent.train_state.parameters = ps
    return agent
end

# ---- rollout buffer ------------------------------------------------------------------------------
mutable struct DeviceRolloutBuffer
    h::Ptr{Cvoid}
    n_steps::Int
    n_envs::Int
end
function DeviceRolloutBuffer(ctx::Context, env::CudaBatchedEnv, n_steps::Integer)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    as = env.act_space
    check(ccall((:dril_buffer_create, LIB), Int32, (Ptr{Cvoid}, Int64, Int64, Int32, Int32, Int32, Ref{Ptr{Cvoid}}),
        ctx.h, n_steps, env.n_envs, size(env.obs_space)[1], as isa Discrete ? 0 : 1, as isa Discrete ? 1 : prod(size(as)), out))
    b = DeviceRolloutBuffer(out[], n_steps, env.n_envs)
    finalizer(x -> ccall((:dril_buffer_destroy, LIB), Int32, (Ptr{Cvoid},), x.h), b)
end
Base.length(b::DeviceRolloutBuffer) = b.n_steps * b.n_envs

"Callbacks that override `on_step` (src/buffers/trajectory.jl:34-39); the others keep the fused rollout."
on_step_callbacks(callbacks) = isnothing(callbacks) ? AbstractCallback[] :
    [c for c in callbacks if which(DRiL.on_step, (typeof(c), Dict)) != which(DRiL.on_step, (AbstractCallback, Dict))]

"""
collect_rollout!(buffer, agent, alg, env) -> (fps, success)  (src/buffers/rollout_buffer.jl:46-90).
When a callback overrides `on_step` the rollout runs in chunks of one step (`dril_rollout_collect_steps`): the observe()
before the loop (trajectory.jl:32) precedes the first hook, hook i sees the env after i - 1 steps, and a `false` stops the
collection there; otherwise one fused launch.
"""
function DRiL.collect_rollout!(buf::DeviceRolloutBuffer, agent::Agent, alg::PPO, env::CudaBatchedEnv; callbacks = nothing,
        push = true)
    p = device_policy(agent, env.ctx)
    push && push_params!(p, agent)
    active = on_step_callbacks(callbacks)
    if !isempty(active)
        n_steps, n_envs = buf.n_steps, buf.n_envs
        t0 = time()
        check(ccall((:dril_rollout_collect_steps, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Int32, Ptr{Cvoid}),
            env.h, p.h, buf.h, 0, 0, 1, C_NULL))
        for i in 1:n_steps
            all(c -> DRiL.on_step(c, Base.@locals), active) || return 0.0f0, false
            check(ccall((:dril_rollout_collect_steps, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Int32, Ptr{Cvoid}),
                env.h, p.h, buf.h, i - 1, 1, 0, C_NULL))
        end
        check(ccall((:dril_gae, LIB), Int32, (Ptr{Cvoid}, Float32, Float32), buf.h, alg.gamma, alg.gae_lambda))
        return Float32(n_steps * n_envs / max(time() - t0, 1e-12)), true
    end
    fps = Ref{Float32}(0)
    check(ccall((:dril_rollout_collect, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Float32}),
        env.h, p.h, buf.h, C_NULL, fps))
    check(ccall((:dril_gae, LIB), Int32, (Ptr{Cvoid}, Float32, Float32), buf.h, alg.gamma, alg.gae_lambda))
    return fps[], true
end

"""
    train!(agent, env::CudaBatchedEnv, alg::PPO, max_steps; callbacks) -> (learn_stats, to)

Same contract as src/algorithms/ppo.jl:100-325: returns the 10-field `learn_stats` NamedTuple and a
TimerOutput; callbacks get a `Dict{Symbol,Any}` with the keys pinned by test/test_callbacks.jl:24-38;
a callback returning `false` aborts and `train!` returns `nothing`; `add_step!` once per rollout.
"""
const BUFFERS = IdDict{Any, DeviceRolloutBuffer}()      # one device buffer per agent, reused while its shape fits (allocation is the expensive part)
function cached_buffer(agent::Agent, env::CudaBatchedEnv, n_steps::Integer)
    b = get(BUFFERS, agent, nothing)
    if b === nothing || b.n_steps != n_steps || b.n_envs != env.n_envs
        b = DeviceRolloutBuffer(env.ctx, env, n_steps)
        BUFFERS[agent] = b
    end
    return b
end

function DRiL.train!(agent::Agent, env::CudaBatchedEnv, alg::PPO{T}, max_steps::Int;
        ad_type = nothing, callbacks::Union{Vector{<:AbstractCallback}, Nothing} = nothing) where {T}
    to = DRiL.TimerOutput()
    n_steps, n_envs = alg.n_steps, env.n_envs
    roll_buffer = cached_buffer(agent, env, n_steps)
    iterations = max_steps ÷ (n_steps * n_envs)
    total_steps = iterations * n_steps * n_envs
    p = device_policy(agent, env.ctx)
    push_params!(p, agent)
    keys10 = (:entropy_losses, :policy_losses, :value_losses, :approx_kl_divs, :clip_fractions, :losses,
        :explained_variances, :fps, :grad_norms, :learning_rates)
    stats = Dict(k => Float32[] for k in keys10)
    total_fps = stats[:fps]
    shuffle_seed = rand(agent.rng, UInt64)
    epoch_counter = UInt64(0)
    hook(f, loc) = isnothing(callbacks) || all(c -> f(c, loc), callbacks)
    # all lazily made allocations up front (data-parallel hosts synchronise their ranks after this, e.g. in on_training_start)
    check(ccall((:dril_iteration_prepare, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int64),
        env.h, p.h, roll_buffer.h, alg.epochs, alg.batch_size))
    hook(DRiL.on_training_start, Base.@locals) || return nothing
    # without callbacks nothing on the host can influence the next iteration: iteration i + 1 is enqueued before the record of
    # iteration i is read (FIFO of 4 slots in the library), so the device never waits for the host
    pipelined = isnothing(callbacks)
    enqueue() = begin
        hyper = Ref(PPOHyper(alg))
        check(ccall((:dril_ppo_iteration_async, LIB), Int32,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{PPOHyper}, Int32, Int64, UInt64, UInt64),
            env.h, p.h, roll_buffer.h, hyper, alg.epochs, alg.batch_size, shuffle_seed, epoch_counter))
        epoch_counter += alg.epochs
    end
    completed = false
    try
        for i in 1:iterations
            learning_rate = alg.learning_rate
            hook(DRiL.on_rollout_start, Base.@locals) || return nothing
            st = Ref{IterStats}()
            local fps::Float32
            if pipelined
                i == 1 && enqueue()
                i < iterations && enqueue()
                check(ccall((:dril_iteration_result, LIB), Int32, (Ptr{Cvoid}, Ref{IterStats}), p.h, st))
                fps = Float32(n_steps * n_envs / (st[].rollout_ms * 1.0f-3))
            else
                # split like src/algorithms/ppo.jl:160-186: collect_rollout! (on_step hooks inside), bookkeeping, on_rollout_end,
                # then the update: a hook returning false skips the update, every hook sees the rollout's parameters
                fps, ok = DRiL.collect_rollout!(roll_buffer, agent, alg, env; callbacks, push = false)
                ok || return nothing
            end
            push!(total_fps, fps)
            DRiL.add_step!(agent, n_steps * n_envs)
            DRiL.increment_step!(agent.logger, n_steps * n_envs)
            DRiL.log_scalar!(agent.logger, "env/fps", fps)
            DRiL.log_stats(env, agent.logger)
            hook(DRiL.on_rollout_end, Base.@locals) || return nothing
            if !pipelined
                hyper = Ref(PPOHyper(alg))
                check(ccall((:dril_ppo_update, LIB), Int32,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{PPOHyper}, Int32, Int64, UInt64, UInt64, Ref{IterStats}),
                    p.h, roll_buffer.h, hyper, alg.epochs, alg.batch_size, shuffle_seed, epoch_counter, st))
                epoch_counter += alg.epochs
            end
            s = st[]
            push!(stats[:learning_rates], learning_rate); push!(stats[:explained_variances], s.explained_variance)
            push!(stats[:entropy_losses], s.entropy_loss); push!(stats[:policy_losses], s.policy_loss)
            push!(stats[:value_losses], s.value_loss); push!(stats[:approx_kl_divs], s.approx_kl_div)
            push!(stats[:clip_fractions], s.clip_fraction); push!(stats[:losses], s.loss); push!(stats[:grad_norms], s.grad_norm)
            for (k, v) in ("train/entropy_loss" => s.entropy_loss, "train/explained_variance" => s.explained_variance,
                "train/policy_loss" => s.policy_loss, "train/value_loss" => s.value_loss, "train/approx_kl_div" => s.approx_kl_div,
                "train/clip_fraction" => s.clip_fraction, "train/loss" => s.loss, "train/grad_norm" => s.grad_norm,
                "train/learning_rate" => learning_rate)
                DRiL.log_scalar!(agent.logger, k, v)
            end
        end
        completed = true
    finally
        if !completed          # drain unread pipelined results
            st = Ref{IterStats}()
            while ccall((:dril_iteration_result, LIB), Int32, (Ptr{Cvoid}, Ref{IterStats}), p.h, st) == 0 end
        end
        pull_params!(agent, p)  # an aborted train! keeps the parameters it updated in place (ppo.jl:179-186)
    end
    learn_stats = NamedTuple{keys10}(Tuple(stats[k] for k in keys10))
    hook(DRiL.on_training_end, Base.@locals) || return nothing
    return learn_stats, to
end

# ---- evaluation on the device (src/evaluation.jl:54-143) -------------------------------------------------------------------------
"""
    evaluate_agent(agent, env::CudaBatchedEnv; n_eval_episodes, deterministic, reward_threshold, return_stats)

Same contract as src/evaluation.jl:54-143; the episode loop runs on the device (`dril_evaluate`: fused policy + env steps in
chunks, one device -> host copy of the episode records per chunk, episodes appended in (step, env) order).
"""
function DRiL.evaluate_agent(agent::Agent, env::CudaBatchedEnv; n_eval_episodes::Int = 10, deterministic::Bool = true,
        reward_threshold = nothing, return_stats::Bool = true, warn::Bool = true, rng = agent.rng, show_progress::Bool = false,
        chunk_steps::Integer = 64)
    p = device_policy(agent, env.ctx)
    push_params!(p, agent)
    er = Vector{Float32}(undef, n_eval_episodes); el = Vector{Int64}(undef, n_eval_episodes)
    got = Ref{Int64}(0); steps = Ref{Int64}(0)
    check(ccall((:dril_evaluate, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int32, Int32, Ptr{Float32}, Ptr{Int64}, Ref{Int64}, Ref{Int64}),
        env.h, p.h, n_eval_episodes, Int32(deterministic), Int32(chunk_steps), er, el, got, steps))
    mean_reward = DRiL.mean(er)
    if reward_threshold !== nothing && mean_reward < reward_threshold
        error("Mean reward below threshold: $(round(mean_reward, digits = 2)) < $(reward_threshold)")
    end
    return_stats || return er, Int.(el)
    return (; mean_reward, std_reward = DRiL.std(er), mean_length = DRiL.mean(el), std_length = DRiL.std(el))
end

# ---- normaliser statistics (src/environment_wrappers/normalizeWrapperEnv.jl:261-309) and deployment ------------------------------
function norm_stats(env::CudaBatchedEnv)
    D = size(env.obs_space)[1]
    m = Vector{Float32}(undef, D); v = Vector{Float32}(undef, D)
    oc = Ref{Int64}(0); rc = Ref{Int64}(0); rm = Ref{Float32}(0); rv = Ref{Float32}(0)
    check(ccall((:dril_env_get_norm_stats, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Ref{Int64}, Ref{Float32}, Ref{Float32}, Ref{Int64}), env.h, m, v, oc, rm, rv, rc))
    return (; obs_mean = m, obs_var = v, obs_count = oc[], ret_mean = rm[], ret_var = rv[], ret_count = rc[])
end
set_norm_stats!(env::CudaBatchedEnv, s) = check(ccall((:dril_env_set_norm_stats, LIB), Int32,
    (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int64, Float32, Float32, Int64),
    env.h, Float32.(s.obs_mean), Float32.(s.obs_var), s.obs_count, s.ret_mean, s.ret_var, s.ret_count))

"save_normalization_stats(env, filepath): the ten keys of normalizeWrapperEnv.jl:261-277, through DRiL's own JLD2 `save`."
function DRiL.save_normalization_stats(env::CudaBatchedEnv, filepath::String)
    s, c = norm_stats(env), env.normalize
    return DRiL.save(filepath, Dict("obs_mean" => s.obs_mean, "obs_var" => s.obs_var, "obs_count" => s.obs_count,
        "ret_mean" => [s.ret_mean], "ret_var" => [s.ret_var], "ret_count" => s.ret_count, "clip_obs" => c.clip_obs,
        "clip_reward" => c.clip_reward, "gamma" => c.gamma, "epsilon" => c.epsilon))
end
function DRiL.load_normalization_stats!(env::CudaBatchedEnv, filepath::String)
    d = DRiL.load(filepath)
    set_norm_stats!(env, (; obs_mean = d["obs_mean"], obs_var = d["obs_var"], obs_count = d["obs_count"],
        ret_mean = first(d["ret_mean"]), ret_var = first(d["ret_var"]), ret_count = d["ret_count"]))
    return env
end
"sync_normalization_stats!(eval_env, train_env): statistics copied, the eval env's discounted returns zeroed (normalizeWrapperEnv.jl:299-309)"
function DRiL.sync_normalization_stats!(eval_env::CudaBatchedEnv, train_env::CudaBatchedEnv)
    set_norm_stats!(eval_env, norm_stats(train_env))
    check(ccall((:dril_env_zero_returns, LIB), Int32, (Ptr{Cvoid},), eval_env.h))
    return nothing
end
"extract_policy(agent, norm_env) -> NormWrapperPolicy (src/deployment/deployment_policy.jl:50-71) with the device env's obs statistics"
function DRiL.extract_policy(agent::Agent, norm_env::CudaBatchedEnv)
    s = norm_stats(norm_env)
    rms = DRiL.RunningMeanStd{Float32}(s.obs_mean, s.obs_var, s.obs_count)
    return DRiL.NormWrapperPolicy(DRiL.extract_policy(agent), rms, norm_env.normalize.epsilon, norm_env.normalize.clip_obs)
end

# ---- kernel-path switches and data-parallel setup (include/dril_b200.h) --------------------------------------------
"`set_option(\"tc\" | \"ft\" | \"ftg\" | \"fused_tail\" | \"tc_rollout\" | \"single_net\" | \"mma\", 0/1)`: process-wide kernel-path switches (all default on;\nthe last two apply to policies created afterwards)."
set_option(key::AbstractString, value::Integer) =
    check(ccall((:dril_set_option, LIB), Int32, (Cstring, Int32), key, value))

"`:tensor`: the update of this policy runs a tcgen05 loss/grad kernel (update_ft.cuh / update_ftg.cuh / update_tc.cuh); `:mma`: the general-shape kernel with its
wide layers on mma.sync 3xTF32 tiles; `:fp32`: the general-shape kernel on FMA tiles only."
function update_path(p::DevicePolicy)
    out = Ref{Int32}(0)
    check(ccall((:dril_policy_update_path, LIB), Int32, (Ptr{Cvoid}, Ref{Int32}), p.h, out))
    return out[] == 1 ? :tensor : (out[] == 2 ? :mma : :fp32)
end

"""
    comm_init!(ctx, rank, nranks, unique_id; exchange_handles)

One process (or task) per GPU.  `unique_id` is the 128-byte id of `comm_unique_id()` created on rank 0 and broadcast by
the host program (MPI.jl, a file, sockets).  When `exchange_handles(my_handle::Vector{UInt8})::Vector{Vector{UInt8}}`
is given (an all-gather of the 64-byte CUDA IPC handles in rank order) the gradient / moment exchanges run over NVLink
peer memory inside the update kernel instead of NCCL.  Envs are sharded by `gid_offset = rank * n_envs`.
"""
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:dril_comm_unique_id, LIB), Int32, (Ptr{UInt8},), id))
    return id
end
function comm_init!(ctx::Context, rank::Integer, nranks::Integer, unique_id::Vector{UInt8}; exchange_handles = nothing,
        n_params::Integer = 0)
    check(ccall((:dril_comm_init, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{UInt8}), ctx.h, rank, nranks, unique_id))
    if exchange_handles !== nothing
        mine = Vector{UInt8}(undef, 64)
        check(ccall((:dril_comm_p2p_export, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{UInt8}), ctx.h, n_params + 8, mine))
        all = reduce(vcat, exchange_handles(mine))
        check(ccall((:dril_comm_p2p_import, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}), ctx.h, all))
    end
    return nothing
end

end # module
