# MuZeroB200.jl -- drop-in replacement for the hot path of deveshjawla/MuZero.jl: the same function names and
# signatures as src/SelfPlay.jl, src/ReplayBuffer.jl and src/Learning.jl, with bodies that `ccall` into
# libmuzero_b200.so (include/muzero_b200.h).  Include it INSTEAD of those three files, after Constructors.jl,
# game.jl and params.jl (so that `conf`, `hyper`, `GameHistory`, `Config`, `FeedForwardHP` exist).
#
# STATUS: source only.  Julia is not installed in the build image, so this file has never been executed; the
# identical call sequence is exercised through the Python mirror (muzero.jl_b200/api.py) by the test-suite.
module MuZeroB200

import Serialization   # stdlib: checkpoint files of the reference (src/Learning.jl:431-433)

const LIB = get(ENV, "MUZERO_B200_LIB", joinpath(@__DIR__, "..", "libmuzero_b200.so"))
const MZ_MAX_A = 16

# POD mirror of mz_config (field order is the ABI)
mutable struct MzConfig
    game::Int32; W::Int32; H::Int32; C::Int32; A::Int32; num_players::Int32; stacked_observations::Int32; max_moves::Int32
    num_iters::Int32; num_unroll_steps::Int32; td_steps::Int32; batch_size::Int32; replay_buffer_size::Int32; pb_c_base::Int32
    intermediate_rewards::Int32; tie_mode::Int32
    pb_c_init::Float32; discount::Float32; dirichlet_alpha::Float32; exploration_eps::Float32
    seed::UInt64
    child_order::NTuple{MZ_MAX_A,Int32}
    width_hidden::Int32; depth_representation::Int32; depth_prediction::Int32; depth_dynamics::Int32
    depth_policy::Int32; depth_value::Int32; depth_reward::Int32; depth_state_head::Int32
    hidden_state_size::Int32; reward_activation_tanh::Int32
    num_slots::Int32; nn_mode::Int32
    net_type::Int32; rn_num_blocks::Int32; rn_num_filters::Int32; rn_kernel::Int32; rn_first_head_filters::Int32; rn_second_head_filters::Int32
    per::Int32; per_alpha::Int32
    temperature_threshold::Int32
    use_batch_norm::Int32
    MzConfig() = new()
end

struct MzError <: Exception
    code::Int32
    msg::String
end

mutable struct Engine          # one mz_ctx = one GPU; replaces the RemoteChannels of games/tictactoe/main.jl:15-21
    ctx::Ptr{Cvoid}
    cfg::MzConfig
    training_step::Int
    next_game::Int
    mcts_calls::Int            # keys the random streams of the reference-signature run_mcts (the reference draws from a global RNG)
    nn_token::UInt             # objectid of the Flux NNs last uploaded by sync_networks!
end

check(e::Engine, rc) = rc == 0 ? nothing : throw(MzError(rc, unsafe_string(ccall((:mz_last_error, LIB), Cstring, (Ptr{Cvoid},), e.ctx))))

"Build the engine from the reference's `conf::Config` and `hyper::FeedForwardHP` or `hyper::ResNetHP` (src/Constructors.jl:18-90)."
# nn_mode: 0 = exact fp32 (bit-identical to the CPU restatement of the reference), 2 = tensor cores at near-Float32 accuracy (bf16 hi + lo
# operands; > 99 % of the Float32 search decisions at twice the throughput, learner on the tensor cores too), 1 = plain bf16 tensor cores
function Engine(conf, hyper; device::Integer=0, num_slots::Integer=4096, nn_mode::Integer=0)
    c = MzConfig()
    ccall((:mz_default_config, LIB), Cint, (Ref{MzConfig},), c)
    c.W, c.H, c.C = conf.observation_shape
    c.A = length(conf.action_space); c.num_players = length(conf.players)
    c.stacked_observations = conf.stacked_observations; c.max_moves = conf.max_moves; c.num_iters = conf.num_iters
    c.num_unroll_steps = conf.num_unroll_steps; c.td_steps = conf.td_steps; c.batch_size = conf.batch_size
    conf.replay_buffer_size < num_slots && @warn "replay_buffer_size raised to num_slots (a wave saves up to num_slots games at once)" conf.replay_buffer_size num_slots
    c.replay_buffer_size = max(conf.replay_buffer_size, num_slots); c.pb_c_base = conf.pb_c_base
    c.intermediate_rewards = conf.intermediate_rewards; c.pb_c_init = conf.pb_c_init; c.discount = conf.discount
    c.dirichlet_alpha = conf.dirichlet_α; c.exploration_eps = conf.exploration_ϵ; c.seed = conf.seed
    c.per = conf.PER; c.per_alpha = conf.PER_alpha
    c.temperature_threshold = isnothing(conf.temperature_threshold) ? -1 : conf.temperature_threshold   # src/SelfPlay.jl:344-346
    c.use_batch_norm = hasproperty(hyper, :use_batch_norm) && hyper.use_batch_norm ? 1 : 0             # src/Learning.jl:70-79 (exact fp32 and split-precision paths)
    order = zeros(Int32, MZ_MAX_A)
    ccall((:mz_julia_dict_order, LIB), Cint, (Cint, Ptr{Int32}), c.A, order)   # or: collect(keys(Dict(a => 0 for a in conf.action_space)))
    c.child_order = Tuple(order)
    if hasproperty(hyper, :num_blocks)      # ResNetHP (src/Constructors.jl:77-90): the repaired residual networks, bf16 on the tensor cores
        c.net_type = 1; c.nn_mode = 1
        c.rn_num_blocks = hyper.num_blocks; c.rn_num_filters = hyper.num_filters; c.rn_kernel = hyper.conv_kernel_size[1]
        c.rn_first_head_filters = hyper.num_first_head_filters; c.rn_second_head_filters = hyper.num_second_head_filters
        c.depth_value = hyper.depth_value; c.width_hidden = hyper.hidden_state_size   # width of the heads' dense layers (Learning.jl:205-222)
        c.hidden_state_size = c.W * c.H * c.rn_num_filters
    else                                    # FeedForwardHP (src/Constructors.jl:62-75)
        c.width_hidden = hyper.width_hidden; c.depth_representation = hyper.depth_representation
        c.depth_prediction = hyper.depth_prediction; c.depth_dynamics = hyper.depth_dynamics; c.depth_policy = hyper.depth_policy
        c.depth_value = hyper.depth_value; c.depth_reward = hyper.depth_reward; c.depth_state_head = hyper.depth_state_head
        c.hidden_state_size = hyper.hidden_state_size; c.reward_activation_tanh = hyper.reward_activation === tanh
        c.nn_mode = nn_mode
    end
    c.num_slots = num_slots
    ctx = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:mz_create, LIB), Cint, (Ref{MzConfig}, Cint, Ref{Ptr{Cvoid}}), c, device, ctx)
    rc == 0 || throw(MzError(rc, unsafe_string(ccall((:mz_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL))))
    e = Engine(ctx[], c, 0, 0, 0, UInt(0))
    finalizer(x -> ccall((:mz_destroy, LIB), Cint, (Ptr{Cvoid},), x.ctx), e)
    return e
end

# ---- networks: init_representation / init_prediction / init_dynamics (src/Learning.jl:87,100,118) ----------------
# Flux is the reference's dependency, not this module's: its scripts load it into Main (src/Learning.jl:1-20), and it is looked up there
# only when a Flux model is actually converted.
_flux() = getfield(Main, :Flux)
"Flatten a Flux Chain of Dense layers into the blob order of the ABI: per Dense `vec(W)` (column-major (out,in)) then `b`."
flux_blob(model) = reduce(vcat, [vec(Float32.(p)) for p in _flux().params(model)])
"""
Blob of a (repaired) `ResNetHP` network (DESIGN.md §2.4): walks the Flux model in construction order; `Conv` -> `vec(weight)` (Flux's
`(k,k,cin,cout)` column-major, flipped-kernel convention), `bias`; `BatchNorm` -> `β, γ, μ, σ²` (the running statistics are not in
`Flux.params`); `Dense` -> `vec(weight)`, `bias`. Containers (`Chain`, `SkipConnection`, `Parallel`, the reference's `Split`) are walked
field by field.
"""
function flux_blob_resnet(model)
    F = _flux(); out = Float32[]
    function walk(l)
        if l isa F.Conv
            append!(out, vec(Float32.(l.weight))); append!(out, Float32.(l.bias))
        elseif l isa F.BatchNorm
            append!(out, Float32.(l.β)); append!(out, Float32.(l.γ)); append!(out, Float32.(l.μ)); append!(out, Float32.(l.σ²))
        elseif l isa F.Dense
            append!(out, vec(Float32.(l.weight))); append!(out, Float32.(l.bias))
        elseif l isa Function || l isa Number || l isa AbstractArray{<:Number} || l isa Nothing
            nothing
        elseif l isa Tuple || l isa AbstractVector
            foreach(walk, l)
        else
            foreach(f -> walk(getfield(l, f)), fieldnames(typeof(l)))
        end
    end
    walk(model)
    return out
end
"Inverse of `flux_blob` for Dense chains: copies a blob into the parameters of a Flux model of the same architecture."
function load_blob!(model, blob::Vector{Float32})
    off = 0
    for p in _flux().params(model)
        n = length(p); copyto!(p, reshape(view(blob, off+1:off+n), size(p))); off += n
    end
    off == length(blob) || error("blob has $(length(blob)) floats, the model takes $off")
    return model
end
"""
Checkpoint I/O in the reference's own format (src/Learning.jl:426-434 writes `\$(step)_representation.bin` etc. with `Serialization`;
games/tictactoe/play.jl:12-14 reads them): `load_networks!` feeds Julia-trained Flux chains to the kernels, `save_networks` writes the
engine's weights as Flux chains built by the reference's `init_*(hyper)` so that play.jl can `deserialize` them.
"""
function load_networks!(e::Engine, networks_path::String, step::Integer; blob=flux_blob)
    for (net, name) in enumerate(("representation", "prediction", "dynamics"))
        model = Serialization.deserialize(joinpath(networks_path, "$(step)_$(name).bin"))
        set_weights!(e, net - 1, blob(model))
    end
    return e
end
function save_networks(e::Engine, networks_path::String, step::Integer, inits::NamedTuple, hyper)
    for (net, name) in enumerate((:representation, :prediction, :dynamics))
        model = load_blob!(getfield(inits, name)(hyper), get_weights(e, net - 1))
        Serialization.serialize(joinpath(networks_path, "$(step)_$(name).bin"), model)
    end
end
set_weights!(e::Engine, net::Integer, blob::Vector{Float32}) =
    check(e, ccall((:mz_set_weights, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float32}, Int64), e.ctx, net, blob, length(blob)))
function get_weights(e::Engine, net::Integer=3)
    n = ccall((:mz_num_params, LIB), Cint, (Ref{MzConfig}, Cint), e.cfg, net)
    blob = Vector{Float32}(undef, n)
    check(e, ccall((:mz_get_weights, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float32}, Int64), e.ctx, net, blob, n))
    return blob
end
"NNs = (representation=…, prediction=…, dynamics=…): callables with the shapes of the Flux chains, batched on the GPU."
function init_networks(e::Engine; seed=e.cfg.seed)
    check(e, ccall((:mz_init_weights, LIB), Cint, (Ptr{Cvoid}, UInt64), e.ctx, seed))
    hs, A = Int(e.cfg.hidden_state_size), Int(e.cfg.A)
    representation = x -> (B = size(x)[end]; h = Matrix{Float32}(undef, hs, B);
        check(e, ccall((:mz_representation, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float32}, Ptr{Float32}), e.ctx, B, x, h)); h)
    prediction = h -> (B = size(h)[end]; v = Matrix{Float32}(undef, 1, B); p = Matrix{Float32}(undef, A, B);
        check(e, ccall((:mz_prediction, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}), e.ctx, B, h, v, p)); (v, p))
    dynamics = sa -> (B = size(sa)[end]; h = Matrix{Float32}(undef, hs, B); r = Matrix{Float32}(undef, 1, B);
        check(e, ccall((:mz_dynamics, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}), e.ctx, B, sa, h, r)); (h, r))
    return (representation=representation, prediction=prediction, dynamics=dynamics)
end

# ---- run_mcts (src/SelfPlay.jl:230) ----------------------------------------------------------------------
struct Node                    # what callers read from the returned root (SelfPlay.jl:62-70, 115-122, 293-306)
    visit_counts::Vector{Int32}
    priors::Vector{Float32}
    value::Float32
    legal_actions::Vector{Int}
end
legal_mask(actions) = UInt32(reduce(|, (1 << (a - 1) for a in actions)))
function run_mcts(e::Engine, observation::Array{Float32,3}, legal_actions::Vector{Int}, to_play::Int, exploration::Bool; game_id=0, move_idx=1)::Node
    @assert !isempty(legal_actions) "Legal actions should not be an empty array. Got $(legal_actions)"
    A = Int(e.cfg.A); vc = zeros(Int32, A); rv = zeros(Float32, 1); pri = zeros(Float32, A)
    check(e, ccall((:mz_run_mcts, LIB), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Float32}, Ptr{UInt32}, Ptr{Int32}, Cint, Ptr{UInt64}, Ptr{Int32}, Ptr{Int32}, Ptr{Float32}, Ptr{Float32}),
        e.ctx, 1, observation, UInt32[legal_mask(legal_actions)], Int32[to_play], exploration, UInt64[game_id], Int32[move_idx], vc, rv, pri))
    return Node(vc, pri, rv[1], legal_actions)
end
function select_action(e::Engine, node::Node, temperature::Float32; game_id=0, move_idx=1)::Int
    act = zeros(Int32, 1)
    check(e, ccall((:mz_select_action, LIB), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Int32}, Ptr{UInt32}, Cfloat, Ptr{UInt64}, Ptr{Int32}, Ptr{Int32}),
        e.ctx, 1, node.visit_counts, UInt32[legal_mask(node.legal_actions)], temperature, UInt64[game_id], Int32[move_idx], act))
    return act[1]
end

# ---- self_play! / play_game / save_game (src/SelfPlay.jl:330-419, src/ReplayBuffer.jl:133-161) -----------------
visit_softmax_temperature_fn(trained_steps::Int)::Float32 = trained_steps < 500e3 ? 1.0 : trained_steps < 750e3 ? 0.5 : 0.25
"Plays `n_games` games on the GPU's game slots and save_game()s each into the device replay buffer."
function self_play!(e::Engine, n_games::Integer; temperature=visit_softmax_temperature_fn(e.training_step))
    sims = Ref{Int64}(0); moves = Ref{Int64}(0)
    check(e, ccall((:mz_self_play, LIB), Cint, (Ptr{Cvoid}, UInt64, Int64, Cfloat, Ref{Int64}, Ref{Int64}), e.ctx, e.next_game, n_games, temperature, sims, moves))
    e.next_game += n_games
    return sims[], moves[]
end
# ---- competitive_play! (src/SelfPlay.jl:421-435), batched ------------------------------------------------------
const OPPONENTS = Dict("self" => 0, "random" => 1, "expert" => 2, "network" => 3)
"The networks `competitive_play!(e; opponent=\"network\")` plays against: one network (`net` 0..2, after a full set) or all of them (3)."
set_opponent_networks!(e::Engine, blob::Vector{Float32}, net::Integer=3) =
    check(e, ccall((:mz_set_opponent_weights, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float32}, Int64), e.ctx, net, blob, length(blob)))
"The opponent networks become a copy of the engine's current networks (on the device): snapshot, train, then evaluate against it."
snapshot_opponent!(e::Engine) = check(e, ccall((:mz_snapshot_opponent, LIB), Cint, (Ptr{Cvoid},), e.ctx))
"""
`n_games` games of `play_game(env, 0.0f0, render, conf.opponent, conf.muzero_player, NNs)` at once. The reference renders one game and
returns nothing; this returns `(wins, draws, losses, simulations)` for MuZero. "expert" is a one-ply lookahead (the reference's
`expert_agent()` is undefined); "human" stays with the reference's own loop. The games are saved to the engine's replay buffer like
self-play games: evaluate on an `Engine` of its own. "network": the other side is a second MuZero searching with the opponent networks
(`set_opponent_networks!`, `snapshot_opponent!`).
"""
function competitive_play!(e::Engine, n_games::Integer=1; opponent::String="random", muzero_player::Integer=1, temperature=0.0f0)
    haskey(OPPONENTS, opponent) || error("Wrong argument: opponent argument should be self, human, expert, random or network")
    w = Ref{Int64}(0); d = Ref{Int64}(0); l = Ref{Int64}(0); sims = Ref{Int64}(0)
    check(e, ccall((:mz_arena, LIB), Cint, (Ptr{Cvoid}, UInt64, Int64, Cint, Cint, Cfloat, Ref{Int64}, Ref{Int64}, Ref{Int64}, Ref{Int64}),
                   e.ctx, e.next_game, n_games, OPPONENTS[opponent], muzero_player, temperature, w, d, l, sims))
    e.next_game += n_games
    return (wins=w[], draws=d[], losses=l[], simulations=sims[])
end
"GameHistory for replay key `key` (fields and shapes of src/Constructors.jl:6-16)."
function history(e::Engine, key::Integer, GameHistory)
    Tm = Int(e.cfg.max_moves) + 1; A = Int(e.cfg.A); W, H, C = Int(e.cfg.W), Int(e.cfg.H), Int(e.cfg.C)
    gid = zeros(Int64, 1); T = zeros(Int32, 1); obs = zeros(Float32, W, H, C, Tm); act = zeros(Int32, Tm); rew = zeros(Float32, Tm)
    tp = zeros(Int32, Tm); cv = zeros(Float32, A, Tm); rv = zeros(Float32, Tm)
    check(e, ccall((:mz_history_export, LIB), Cint,
        (Ptr{Cvoid}, Int64, Cint, Ptr{Int64}, Ptr{Int32}, Ptr{Float32}, Ptr{Int32}, Ptr{Float32}, Ptr{Int32}, Ptr{Float32}, Ptr{Float32}),
        e.ctx, key, 1, gid, T, obs, act, rew, tp, cv, rv))
    t = T[1]
    return GameHistory(obs[:, :, :, 1:t], Int.(act[1:t]), rew[1:t], Int.(tp[1:t]), cv[:, 1:t], rv[1:t], nothing, nothing, nothing)
end
function play_game(e::Engine, temperature, render::Bool, opponent::String, muzero_player::Int, GameHistory)
    opponent == "self" || error("only opponent == \"self\" is on the accelerated path")
    self_play!(e, 1; temperature=Float32(temperature))
    n = Ref{Int64}(0); k = Ref{Int64}(0); s = Ref{Int64}(0)
    check(e, ccall((:mz_replay_info, LIB), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}, Ref{Int64}), e.ctx, n, k, s))
    return history(e, k[] + n[] - 1, GameHistory)
end

# ---- get_batch (src/ReplayBuffer.jl:188-217) --------------------------------------------------------------------
function get_batch(e::Engine; step=e.training_step + 1)
    B = Int(e.cfg.batch_size); K1 = Int(e.cfg.num_unroll_steps) + 1; A = Int(e.cfg.A)
    planes = Int(e.cfg.C) * (Int(e.cfg.stacked_observations) + 1) + Int(e.cfg.stacked_observations)
    index = zeros(Int32, 2, B); obs = zeros(Float32, Int(e.cfg.W), Int(e.cfg.H), planes, B)
    actions = zeros(Float32, K1, B); values = zeros(Float32, K1, B); rewards = zeros(Float32, K1, B)
    policies = zeros(Float32, A, K1, B); gscale = zeros(Float32, B)
    check(e, ccall((:mz_get_batch, LIB), Cint,
        (Ptr{Cvoid}, UInt64, Ptr{Int32}, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}, Ptr{Float32}),
        e.ctx, step, index, obs, actions, values, rewards, policies, gscale))
    index_batch = [(Int(index[1, b]), Float32(index[2, b])) for b in 1:B]
    return index_batch, (obs, actions, values, rewards, policies, nothing, gscale)
end

# ---- learning! (src/Learning.jl:306-438) ------------------------------------------------------------------------
"Fill `reanalysed_predicted_root_values` (Constructors.jl:13) of games `key0 .. key0+n-1` from the current networks; `get_batch` then bootstraps from them (ReplayBuffer.jl:8)."
reanalyse!(e::Engine, key0::Integer, n::Integer) = check(e, ccall((:mz_reanalyse, LIB), Cint, (Ptr{Cvoid}, Int64, Cint), e.ctx, key0, n))

"""MuZero Reanalyze: `run_mcts` again at every stored position of games `key0 .. key0+n-1` with the current networks (root, game id and
move index as self-play had them); refreshes `child_visits` and `reanalysed_predicted_root_values`.  Returns the simulations run."""
function reanalyse_search!(e::Engine, key0::Integer, n::Integer; exploration::Bool=false)
    sims = Ref{Int64}(0)
    check(e, ccall((:mz_reanalyse_search, LIB), Cint, (Ptr{Cvoid}, Int64, Cint, Cint, Ptr{Int64}), e.ctx, key0, n, exploration ? 1 : 0, sims))
    return sims[]
end

"`steps` iterations of get_batch -> unroll -> loss -> gradients -> ADAM(Cos schedule); returns the last three losses."
function learning!(e::Engine, steps::Integer; grad_mode::Integer=0)
    losses = zeros(Float32, 3)
    check(e, ccall((:mz_learn_steps, LIB), Cint, (Ptr{Cvoid}, Int64, Cint, Cint, Ptr{Float32}), e.ctx, e.training_step + 1, steps, grad_mode, losses))
    e.training_step += steps
    return (l_representation=losses[1], l_prediction=losses[2], l_dynamics=losses[3])
end

# =====================================================================================================================================
# The reference's own signatures (SURVEY.md 8b), bound to a module-global engine exactly as the reference binds the globals `conf` and
# `hyper` (games/tictactoe/params.jl:2,18).  After `bind!(Engine(conf, hyper), conf, GameHistory)` the driver script
# games/tictactoe/main.jl:14-41 runs unchanged: the RemoteChannel arguments are kept and carry the counters; networks, replay buffer and
# games live on the GPU.  self_play! plays one wave of `num_slots` concurrent games per iteration (the reference's lock-step
# take!(training_step), SelfPlay.jl:396 / Learning.jl:411, is the ceiling this path removes).  Run the two actors as tasks of one process
# (`@async self_play!(...)`, `@async learning!(...)`): a context is used by one host thread at a time.
# =====================================================================================================================================
const ENGINE = Ref{Union{Nothing,Engine}}(nothing)
const CONF = Ref{Any}(nothing)
const GAME_HISTORY = Ref{Any}(nothing)      # the reference's GameHistory type (src/Constructors.jl:6-16)
function bind!(e::Engine, conf, GameHistory)
    ENGINE[] = e; CONF[] = conf; GAME_HISTORY[] = GameHistory
    return e
end
engine() = ENGINE[] === nothing ? error("no engine bound: MuZeroB200.bind!(Engine(conf, hyper), conf, GameHistory) first") : ENGINE[]

"NNs from `init_networks` are closures over the device weights (nothing to do); Flux models are flattened and uploaded when they change."
function sync_networks!(e::Engine, NNs)
    NNs.representation isa Function && return e
    id = objectid(NNs.representation) ⊻ objectid(NNs.prediction) ⊻ objectid(NNs.dynamics)
    if id != e.nn_token
        blob = e.cfg.net_type == 1 ? flux_blob_resnet : flux_blob
        set_weights!(e, 0, blob(NNs.representation)); set_weights!(e, 1, blob(NNs.prediction)); set_weights!(e, 2, blob(NNs.dynamics))
        e.nn_token = id
    end
    return e
end
"init_representation / init_prediction / init_dynamics (src/Learning.jl:87,100,118): the three callables of `init_networks`, initialised once per engine."
const NETWORKS = Ref{Any}(nothing)
_nets() = (NETWORKS[] === nothing && (NETWORKS[] = init_networks(engine())); NETWORKS[])
init_representation(hyper) = _nets().representation
init_prediction(hyper) = _nets().prediction
init_dynamics(hyper) = _nets().dynamics

# src/SelfPlay.jl:230
function run_mcts(observation::Array{Float32,3}, legal_actions::Vector{Int}, to_play::Int, exploration::Bool, NNs)::Node
    e = sync_networks!(engine(), NNs)
    e.mcts_calls += 1
    return run_mcts(e, observation, legal_actions, to_play, exploration; game_id=(1 << 31) + e.mcts_calls, move_idx=1)
end
# src/SelfPlay.jl:293
select_action(node::Node, temperature) = (e = engine(); select_action(e, node, Float32(temperature); game_id=(1 << 31) + e.mcts_calls, move_idx=1))

"n games of play_game through mz_play_games: GameHistory objects in game-id order; nothing is saved."
function play_games(e::Engine, n::Integer, temperature, opponent::String, muzero_player::Integer)
    haskey(OPPONENTS, opponent) || error("Wrong argument: opponent argument should be self, human, expert, random or network")   # SelfPlay.jl:323
    Tm = Int(e.cfg.max_moves) + 1; A = Int(e.cfg.A); W, H, C = Int(e.cfg.W), Int(e.cfg.H), Int(e.cfg.C)
    gid = zeros(Int64, n); T = zeros(Int32, n); obs = zeros(Float32, W, H, C, Tm, n); act = zeros(Int32, Tm, n); rew = zeros(Float32, Tm, n)
    tp = zeros(Int32, Tm, n); cv = zeros(Float32, A, Tm, n); rv = zeros(Float32, Tm, n); sims = Ref{Int64}(0)
    check(e, ccall((:mz_play_games, LIB), Cint,
        (Ptr{Cvoid}, UInt64, Cint, Cfloat, Cint, Cint, Ptr{Int64}, Ptr{Int32}, Ptr{Float32}, Ptr{Int32}, Ptr{Float32}, Ptr{Int32}, Ptr{Float32}, Ptr{Float32}, Ref{Int64}),
        e.ctx, e.next_game, n, temperature, OPPONENTS[opponent], muzero_player, gid, T, obs, act, rew, tp, cv, rv, sims))
    e.next_game += n
    GH = GAME_HISTORY[]
    return [(t = T[j]; GH(obs[:, :, :, 1:t, j], Int.(act[1:t, j]), rew[1:t, j], Int.(tp[1:t, j]), cv[:, 1:t, j], rv[1:t, j], nothing, nothing, nothing)) for j in sortperm(gid)]
end
# src/SelfPlay.jl:330
function play_game(env, temperature, render::Bool, opponent::String, muzero_player::Int, NNs)
    e = sync_networks!(engine(), NNs)
    return play_games(e, 1, Float32(temperature), opponent, muzero_player)[1]
end

_bump!(ch, delta) = put!(ch, take!(ch) + delta)      # src/Constructors.jl:55-59
function _counters(e::Engine)
    c = zeros(Int64, 3)
    check(e, ccall((:mz_replay_counters, LIB), Cint, (Ptr{Cvoid}, Ptr{Int64}), e.ctx, c))
    return c
end
# src/ReplayBuffer.jl:133-135
function save_game(history, remote_buffer, num_played_games, num_played_steps, total_samples)
    e = engine(); before = _counters(e)
    Tm = Int(e.cfg.max_moves) + 1; A = Int(e.cfg.A); W, H, C = Int(e.cfg.W), Int(e.cfg.H), Int(e.cfg.C)
    t = length(history.action_history)
    obs = zeros(Float32, W, H, C, Tm); obs[:, :, :, 1:t] .= history.observation_history[:, :, :, 1:t]
    pad(v, T) = (o = zeros(T, Tm); o[1:t] .= v[1:t]; o)
    cv = zeros(Float32, A, Tm); cv[:, 1:t] .= history.child_visits[:, 1:t]
    check(e, ccall((:mz_history_import, LIB), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Int64}, Ptr{Int32}, Ptr{Float32}, Ptr{Int32}, Ptr{Float32}, Ptr{Int32}, Ptr{Float32}, Ptr{Float32}),
        e.ctx, 1, Int64[before[1]], Int32[t], obs, pad(history.action_history, Int32), pad(history.reward_history, Float32),
        pad(history.to_play_history, Int32), cv, pad(history.root_values, Float32)))
    after = _counters(e)
    _bump!(num_played_games, after[1] - before[1]); _bump!(num_played_steps, after[2] - before[2])   # :149-151
    take!(total_samples); put!(total_samples, after[3])                                              # :152, evictions included (:156-160)
    return nothing
end
# src/SelfPlay.jl:384-390
function self_play!(env, training_step, num_played_games, num_played_steps, total_samples, remote_NNs, remote_buffer)::Bool
    e = sync_networks!(engine(), fetch(remote_NNs))                          # :392
    conf = CONF[]; training_step_ = 0
    while training_step_ ≤ conf.training_steps                               # :394
        training_step_ = fetch(training_step)                                # :396, without the lock-step take!
        e.training_step = training_step_
        before = _counters(e)
        self_play!(e, Int(e.cfg.num_slots))                                  # play_game + save_game for a wave of games (:405-417)
        after = _counters(e)
        _bump!(num_played_games, after[1] - before[1]); _bump!(num_played_steps, after[2] - before[2])
        take!(total_samples); put!(total_samples, after[3])
        yield()
    end
    return true
end
# src/ReplayBuffer.jl:188
function get_batch(buffer)
    return get_batch(engine())
end
# src/Learning.jl:306-309
function learning!(num_played_games, training_step, remote_NNs, remote_buffer)::Bool
    e = engine(); conf = CONF[]
    while fetch(num_played_games) < 1                                        # :311-314
        yield()
    end
    training_step_ = fetch(training_step)
    while training_step_ ≤ conf.training_steps                               # :327
        n = min(conf.checkpoint_interval, conf.training_steps - training_step_ + 1)
        e.training_step = training_step_
        losses = learning!(e, n)                                             # :329-404, n iterations queued back to back
        training_step_ += n
        take!(training_step); put!(training_step, training_step_)            # :411
        @info "Training Progress" training_step_ losses...                   # :421-424
        yield()
    end
    return true
end

end # module
