/*
 * muzero_b200.h -- C ABI of the B200-native self-play / learner hot path (libmuzero_b200.so).
 *
 * This is the drop-in boundary for deveshjawla/MuZero.jl (reference at /root/reference, pure Julia).
 * The reference has no FFI layer: the seam is a set of Julia functions that read the globals `conf`
 * and `hyper`.  Each entry point below names the reference function (file:line) it replaces; the Julia
 * wrapper that keeps those signatures and forwards to these symbols with `ccall` is
 * muzero.jl_b200/julia/MuZeroB200.jl (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; the caller allocates and owns every host buffer, the library owns all device
 *     memory; no pointer outlives a call except mz_ctx*.
 *   - arrays use the reference's Julia memory order, i.e. a Julia (W,H,C,N) array is a C [N][C][H][W]
 *     array; actions and players are 1-based like the reference.
 *   - every function returns 0 on success, <0 on error (MZ_E_*); mz_last_error() returns the message.
 *     Nothing throws or aborts across the ABI.  There is NO CPU fallback: without a CUDA device
 *     mz_create fails with MZ_E_CUDA.
 *   - a ctx is bound to one CUDA device and must be used by one host thread at a time.
 */
#ifndef MUZERO_B200_H
#define MUZERO_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MZ_MAX_A 16
#define MZ_ABI_VERSION 7

enum { MZ_OK = 0, MZ_E_ARG = -1, MZ_E_CUDA = -2, MZ_E_STATE = -3, MZ_E_NCCL = -4, MZ_E_UNSUPPORTED = -5 };
enum { MZ_GAME_TICTACTOE = 0, MZ_GAME_CONNECT = 1 };
enum { MZ_TIE_PHILOX = 0, MZ_TIE_FIRST = 1 };
enum { MZ_GRAD_REFERENCE_L2 = 0, MZ_GRAD_BPTT = 1 };
/* conf.opponent (src/Constructors.jl:27; select_opponent_action, src/SelfPlay.jl:311-325).  MZ_OPP_NETWORK (mz_arena, mz_play_games):
 * the other side is a second MuZero that searches its plies with the context's opponent networks (mz_set_opponent_weights,
 * mz_snapshot_opponent) */
enum { MZ_OPP_SELF = 0, MZ_OPP_RANDOM = 1, MZ_OPP_EXPERT = 2, MZ_OPP_NETWORK = 3 };
/* network arithmetic of self-play / run_mcts / the network callables:
 *   MZ_NN_FP32_EXACT  fp32 SIMT, sequential-k fmaf: bit-identical to the oracle's arithmetic contract
 *   MZ_NN_BF16_TC     bf16 operands on tcgen05.mma, fp32 accumulation in TMEM
 *   MZ_NN_SPLIT_MMA   tcgen05.mma at near-Float32 accuracy: both operands split into bf16 hi + lo, W_hi X_hi + W_lo X_hi + W_hi X_lo
 *                     accumulated in fp32 in TMEM; network outputs within ~1e-6 of Float32, visit counts identical to the Float32 oracle
 *                     on > 99 % of roots.  In this mode the learner runs on the same path too (mz_learner_path): the unroll forward in split
 *                     precision, MZ_GRAD_BPTT's backward with bf16 operands (gradients within 1e-2 of the largest entry per network). */
enum { MZ_NN_FP32_EXACT = 0, MZ_NN_BF16_TC = 1, MZ_NN_SPLIT_MMA = 2 };
enum { MZ_NET_FEEDFORWARD = 0, MZ_NET_RESNET = 1 };
enum { MZ_NET_REPRESENTATION = 0, MZ_NET_PREDICTION = 1, MZ_NET_DYNAMICS = 2, MZ_NET_ALL = 3 };

/* POD mirror of Config (src/Constructors.jl:18-52, games/tictactoe/params.jl:2-16) and FeedForwardHP
 * (src/Constructors.jl:62-75, params.jl:18-29).  Field names follow the reference. */
typedef struct mz_config {
    int32_t game;                 /* MZ_GAME_* (the reference ships TicTacToe only) */
    int32_t W, H, C;              /* observation_shape */
    int32_t A;                    /* length(action_space) */
    int32_t num_players;          /* length(players) */
    int32_t stacked_observations;
    int32_t max_moves;
    int32_t num_iters;            /* simulations per move */
    int32_t num_unroll_steps;
    int32_t td_steps;
    int32_t batch_size;
    int32_t replay_buffer_size;
    int32_t pb_c_base;
    int32_t intermediate_rewards;
    int32_t tie_mode;             /* UCB tie-break contract (DESIGN.md): MZ_TIE_* */
    float   pb_c_init;
    float   discount;
    float   dirichlet_alpha;      /* dirichlet_α */
    float   exploration_eps;      /* exploration_ϵ; 0 switches the root noise off bit-exactly */
    uint64_t seed;
    int32_t child_order[MZ_MAX_A];/* Julia Dict{Int,Node} iteration order of keys 1..A */
    int32_t width_hidden, depth_representation, depth_prediction, depth_dynamics;
    int32_t depth_policy, depth_value, depth_reward, depth_state_head;
    int32_t hidden_state_size;
    int32_t reward_activation_tanh;
    /* B200 execution parameters (no reference counterpart) */
    int32_t num_slots;            /* concurrent self-play games resident on this GPU (e.g. 4096) */
    int32_t nn_mode;              /* MZ_NN_* */
    /* ResNetHP (src/Constructors.jl:77-90): the residual networks of src/Learning.jl:148-255 in their repaired form
     * (the reference's constructors read undefined names and never ran; DESIGN.md "ResNet").  net_type = MZ_NET_RESNET
     * needs nn_mode = MZ_NN_BF16_TC and hidden_state_size = W*H*rn_num_filters; width_hidden / depth_value are shared. */
    int32_t net_type;               /* MZ_NET_FEEDFORWARD | MZ_NET_RESNET */
    int32_t rn_num_blocks;          /* num_blocks */
    int32_t rn_num_filters;         /* num_filters (64) */
    int32_t rn_kernel;              /* conv_kernel_size = (k,k) of the representation network, 1 or 3 */
    int32_t rn_first_head_filters;  /* num_first_head_filters = 1 */
    int32_t rn_second_head_filters; /* num_second_head_filters = 2 */
    /* prioritised replay (src/Constructors.jl:43-44): repaired specification, DESIGN.md "PER" */
    int32_t per;                    /* conf.PER */
    int32_t per_alpha;              /* conf.PER_alpha, 0..3 */
    /* conf.temperature_threshold (src/Constructors.jl:31): play_game switches to temperature 0 once
     * length(history.action_history) >= threshold (src/SelfPlay.jl:344-346); -1 = nothing (the default) */
    int32_t temperature_threshold;
    /* FeedForwardHP.use_batch_norm (src/Constructors.jl:71): make_dense = Chain(Dense(in, out), BatchNorm(out, relu)) (src/Learning.jl:70-79).
     * BatchNorm runs in test mode everywhere (the reference never differentiates a forward pass and never calls trainmode!).  Runs on the
     * exact-fp32 path and, folded into the weight image (W' = diag(gamma / sqrt(sigma2 + 1f-5)) W), on MZ_NN_SPLIT_MMA; MZ_GRAD_BPTT
     * differentiates the folded layers and maps the result back to W, b, beta, gamma by the chain rule.  MZ_NN_BF16_TC answers MZ_E_UNSUPPORTED.  Blob: such a layer's W, b are followed by
     * beta[out], gamma[out] (Flux.params order) and the running statistics mu[out], sigma2[out] (not parameters: ADAM leaves them alone). */
    int32_t use_batch_norm;
} mz_config;

typedef struct mz_ctx mz_ctx;

/* ---- lifecycle ------------------------------------------------------------------------------ */
int mz_abi_version(void);
int mz_default_config(mz_config *cfg);                       /* games/tictactoe/params.jl:2-29 */
int mz_julia_dict_order(int A, int32_t *order);              /* Dict iteration order used by SelfPlay.jl:158-159,294-295 */
int mz_create(const mz_config *cfg, int device, mz_ctx **out);
int mz_destroy(mz_ctx *ctx);
const char *mz_last_error(mz_ctx *ctx);                      /* ctx may be NULL: last error of this thread */
int mz_set_stream(mz_ctx *ctx, void *cuda_stream);           /* run all work on the caller's cudaStream_t */
int mz_synchronize(mz_ctx *ctx);
int mz_device_info(mz_ctx *ctx, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor, int64_t *free_bytes);

/* ---- networks: init_representation / init_prediction / init_dynamics (src/Learning.jl:87,100,118) ----
 * Weight blob = for each Dense in Flux.params order: W (out,in) column-major (W[o + out*k]) then b[out]. */
int     mz_num_params(const mz_config *cfg, int net);
int     mz_init_weights(mz_ctx *ctx, uint64_t seed);         /* Flux.glorot_uniform, Philox-keyed */
int     mz_set_weights(mz_ctx *ctx, int net, const float *blob, int64_t n);
int     mz_get_weights(mz_ctx *ctx, int net, float *blob, int64_t n);
/* the opponent networks of MZ_OPP_NETWORK: a second weight store, allocated by the first of these calls (a context that never calls them
 * allocates nothing for it).  mz_set_opponent_weights takes the blob, net ids and lengths of mz_set_weights; net < MZ_NET_ALL replaces one
 * network and needs a full opponent set first (MZ_E_STATE otherwise).  mz_snapshot_opponent makes the opponent a copy of the context's
 * current weights, one device-to-device copy in stream order: snapshot, train, then mz_arena(MZ_OPP_NETWORK) measures what training
 * changed.  Neither the learner nor mz_set_weights touches the opponent networks. */
int     mz_set_opponent_weights(mz_ctx *ctx, int net, const float *blob, int64_t n);
int     mz_snapshot_opponent(mz_ctx *ctx);
/* batched callables, host buffers: repr(x (W,H,planes,B)) -> (hidden,B); pred(h) -> (value(1,B), policy(A,B));
 * dyn(sa (W,H,C+1,B)) -> (state(hidden,B), reward(1,B)) */
int mz_representation(mz_ctx *ctx, int B, const float *stacked_obs, float *hidden);
int mz_prediction(mz_ctx *ctx, int B, const float *hidden, float *value, float *policy);
int mz_dynamics(mz_ctx *ctx, int B, const float *state_action, float *next_hidden, float *reward);

/* ---- environment: games/tictactoe/game.jl (reset! :15, env(action) :45-52, legal_action_space :35-43,
 *      is_terminated :85, reward :87-100), batched over n boards in SoA form ---- */
int mz_env_reset(mz_ctx *ctx, int n, uint64_t *p1, uint64_t *p2, int32_t *player);
int mz_env_step(mz_ctx *ctx, int n, uint64_t *p1, uint64_t *p2, int32_t *player, const int32_t *action,
                float *reward /* RLBase.reward(env, mover) */, int32_t *done, uint32_t *legal_mask);
int mz_env_legal(mz_ctx *ctx, int n, const uint64_t *p1, const uint64_t *p2, const int32_t *player, uint32_t *legal_mask);
int mz_env_observation(mz_ctx *ctx, int n, const uint64_t *p1, const uint64_t *p2, float *obs /* [n][C][H][W] */);

/* ---- MCTS: run_mcts (src/SelfPlay.jl:230-285), batched over n independent roots -------------- */
/* Calls with few roots (FeedForwardHP networks without BatchNorm: n <= 148 in MZ_NN_FP32_EXACT contexts, n <= 74 in MZ_NN_SPLIT_MMA
 * contexts) are served by the low-latency kernel mz_k_search_lat -- one tree per two-SM thread-block cluster, networks and tree
 * resident in shared memory, exact fp32, results bit-identical to the batched exact kernel (0.44 ms for one root); the same holds
 * for mz_self_play / mz_arena / mz_play_games calls of <= 16 games.  Environment MUZERO_B200_LAT=n moves both limits (0 = off). */
int mz_run_mcts(mz_ctx *ctx, int n, const float *stacked_obs /* [n][stack] */, const uint32_t *legal_mask,
                const int32_t *to_play, int exploration, const uint64_t *game_id, const int32_t *move_idx,
                int32_t *visit_counts /* [n][A] */, float *root_value /* [n] */, float *root_priors /* [n][A], may be NULL */);
/* select_action (src/SelfPlay.jl:293-306) */
int mz_select_action(mz_ctx *ctx, int n, const int32_t *visit_counts, const uint32_t *legal_mask, float temperature,
                     const uint64_t *game_id, const int32_t *move_idx, int32_t *action);

/* ---- self-play: play_game / self_play! (src/SelfPlay.jl:330-419) + save_game (src/ReplayBuffer.jl:133-161)
 * Plays games first_game .. first_game+n_games-1 on the ctx's num_slots device-resident game slots and
 * appends every finished GameHistory to the device replay ring under the next game number.  With n_games > num_slots the games
 * run as consecutive waves of num_slots games (new games start when every slot is free, which keeps all trees of a launch at the
 * same ply and is 10 - 56 % faster than refilling a slot the moment its game ends; MUZERO_B200_REFILL=immediate in the environment
 * of mz_create selects the latter).  A game's history does not depend on the policy, the number of slots or the sharding. */
int mz_self_play(mz_ctx *ctx, uint64_t first_game, int64_t n_games, float temperature, int64_t *simulations, int64_t *moves);
/* play_game(env, temperature, render, opponent, muzero_player, NNs)::GameHistory (src/SelfPlay.jl:330-382) for n_games games at once:
 * the histories come back to the caller (layout of mz_history_export; order = the order the games finished, game_id[] names them) and are
 * NOT saved -- the reference's self_play! passes them to save_game itself (:414), here mz_history_import.  opponent MZ_OPP_SELF: every
 * ply is searched; otherwise `opponent` moves for the side that is not muzero_player (MZ_OPP_NETWORK: as in mz_arena). */
int mz_play_games(mz_ctx *ctx, uint64_t first_game, int n_games, float temperature, int opponent, int muzero_player, int64_t *game_id,
                  int32_t *T, float *obs, int32_t *actions, float *rewards, int32_t *to_play, float *child_visits, float *root_values,
                  int64_t *simulations /* may be NULL */);
/* competitive_play! (src/SelfPlay.jl:421-435) for n_games games at once: play_game with `opponent` (MZ_OPP_RANDOM: rand over the
 * legal actions, :320; MZ_OPP_EXPERT: the reference's expert_agent() is undefined -- one-ply lookahead: win, else block, else random)
 * moving for the side that is not muzero_player (1 or 2).  The reference passes temperature 0 and, through play_game, still searches
 * with exploration noise (:359).  Finished games go to the replay ring like self-play games (opponent plies repeat the statistics of
 * the previous search, :374; zeros before the first one), so use a context of its own for evaluation.  wins / draws / losses count
 * games for MuZero: the side that completes a line first wins (TicTacToe runs one ply past a win, SURVEY Q14).
 * MZ_OPP_NETWORK: the other side's plies are searched exactly like MuZero's (run_mcts with exploration noise, Philox keys (game id, move
 * index), select_action at `temperature`, that ply's own statistics stored) but with the opponent networks; *simulations counts both
 * sides.  With opponent networks equal to the context's, the games are those of MZ_OPP_SELF bit for bit.  MZ_E_STATE before any opponent
 * weights are set. */
int mz_arena(mz_ctx *ctx, uint64_t first_game, int64_t n_games, int opponent, int muzero_player, float temperature,
             int64_t *wins, int64_t *draws, int64_t *losses, int64_t *simulations);
/* select_opponent_action for n boards (bit masks as in mz_env_step); action[n] 1-based */
int mz_opponent_action(mz_ctx *ctx, int n, const uint64_t *p1, const uint64_t *p2, const int32_t *player, int opponent,
                       const uint64_t *game_id, const int32_t *move_idx, int32_t *action);
/* replay ring state: number of stored games, key (game number) of the oldest one, total stored positions */
int mz_replay_info(mz_ctx *ctx, int64_t *n_games, int64_t *first_key, int64_t *total_samples);
/* GameHistory export (src/Constructors.jl:6-16) for keys key0 .. key0+n-1, padded to Tmax = max_moves+1:
 * game_id[n], T[n], observation_history [n][Tmax][C][H][W], action_history [n][Tmax], reward_history [n][Tmax],
 * to_play_history [n][Tmax], child_visits [n][Tmax][A], root_values [n][Tmax] */
int mz_history_export(mz_ctx *ctx, int64_t key0, int n, int64_t *game_id, int32_t *T, float *obs, int32_t *actions,
                      float *rewards, int32_t *to_play, float *child_visits, float *root_values);
/* load n histories (same layout) into the ring, as save_game would (for learner-only runs and tests) */
int mz_history_import(mz_ctx *ctx, int n, const int64_t *game_id, const int32_t *T, const float *obs, const int32_t *actions,
                      const float *rewards, const int32_t *to_play, const float *child_visits, const float *root_values);
int mz_replay_clear(mz_ctx *ctx);
/* reanalyse: fills GameHistory.reanalysed_predicted_root_values (src/Constructors.jl:13) of games key0 .. key0+n-1 with the value
 * head of the CURRENT networks at every stored position, prediction(representation(get_stacked_observations(history, i))).
 * The reference consumes the field in compute_target_value (src/ReplayBuffer.jl:8) but has no producer (main.jl:18 keeps only a
 * counter); from then on get_batch / mz_learn_step bootstrap those games' value targets from the reanalysed values. */
int mz_reanalyse(mz_ctx *ctx, int64_t key0, int n);
int mz_reanalysed_export(mz_ctx *ctx, int64_t key0, int n, float *values /* [n][Tmax] */, int32_t *is_set /* [n]: 0 = nothing */);
/* MuZero Reanalyze: for every stored position t < T of games key0 .. key0+n-1, run_mcts (src/SelfPlay.jl:230-285) again with the
 * CURRENT networks on the context's network path, from the root self-play searched there: stacked observation
 * get_stacked_observations(history, t+1), the legal actions of the stored board, the stored game id, move index t + 1, and every
 * Philox draw (Dirichlet noise when exploration != 0, tie-breaks) keyed by (game id, t + 1).  child_visits[t] receives the visit
 * distribution (store_search_stats!, src/SelfPlay.jl:115-122) and reanalysed_predicted_root_values[t] node_value(root) (0 for t >= T);
 * the games' values are marked as set, so get_batch bootstraps from them.  Nothing else changes -- in particular root_values and the
 * PER priorities stay as stored.  The results depend neither on num_slots nor on the other games of the call.  Every network path is
 * supported.  *simulations (may be NULL) = simulations run.  MZ_E_ARG for n < 0 or keys outside the buffer, MZ_E_STATE while
 * self-play is in progress. */
int mz_reanalyse_search(mz_ctx *ctx, int64_t key0, int n, int exploration, int64_t *simulations);
/* checkpoint / resume of the replay state (the reference never persists its buffer, main.jl:21 TODO): the three save_game counters
 * (num_played_games, num_played_steps, total_samples; ReplayBuffer.jl:147-152) and, per stored game, what mz_history_import does not carry:
 * history.priorities / game_priority as updated by update_priorities! and reanalysed_predicted_root_values.  Resume = mz_replay_clear,
 * mz_replay_set_counters(first_key - 1, 0, 0), mz_history_import(the stored games), mz_replay_set_counters(saved), then the two setters. */
int mz_replay_counters(mz_ctx *ctx, int64_t out[3]);
int mz_replay_set_counters(mz_ctx *ctx, int64_t num_played_games, int64_t num_played_steps, int64_t total_samples);
int mz_replay_set_priorities(mz_ctx *ctx, int64_t key0, int n, const uint32_t *q_pos /* [n][Tmax] */, const uint32_t *q_game /* [n] */);
int mz_reanalysed_import(mz_ctx *ctx, int64_t key0, int n, const float *values /* [n][Tmax] */, const int32_t *is_set /* [n] */);

/* ---- replay sampling + targets: get_batch (src/ReplayBuffer.jl:188-217) ---------------------- */
int mz_get_batch(mz_ctx *ctx, uint64_t step, int32_t *index_batch /* [B][2] (game key, position) */, float *obs_batch,
                 float *action_batch, float *value_batch, float *reward_batch, float *policy_batch, float *gscale);

/* conf.PER = true: the same batch + the importance-sampling weights (ReplayBuffer.jl:213-215), games / positions drawn by priority */
int mz_get_batch_per(mz_ctx *ctx, uint64_t step, int32_t *index_batch, float *obs_batch, float *action_batch, float *value_batch,
                     float *reward_batch, float *policy_batch, float *gscale, float *weight_batch /* [B] */);
/* fixed-point priorities of games key0 .. key0+n-1: q_pos [n][Tmax], q_game [n] (history.priorities, history.game_priority) */
int mz_replay_priorities(mz_ctx *ctx, int64_t key0, int n, uint32_t *q_pos, uint32_t *q_game);

/* ---- learner: learning! (src/Learning.jl:306-438) --------------------------------------------- */
/* forward unroll + loss on a caller-supplied batch (parity entry point; Learning.jl:347-374, 261-288) */
int mz_learn_forward(mz_ctx *ctx, int B, const float *obs_batch, const float *action_batch, const float *value_batch,
                     const float *reward_batch, const float *policy_batch, const float *gscale, float *pred_values,
                     float *pred_rewards, float *pred_policies, float *losses /* [3] */);
/* one training step t (1-based): get_batch(step=t) on the device ring, unroll, loss, gradients (grad_mode),
 * gradient allreduce when a communicator is attached, ADAM with the Cos schedule (Learning.jl:382-397) */
int mz_learn_step(mz_ctx *ctx, int64_t t, int grad_mode, float *losses /* [3] */);
/* n consecutive iterations t0 .. t0+n-1 queued back to back (no host round trip in between); losses of the last one */
int mz_learn_steps(mz_ctx *ctx, int64_t t0, int n, int grad_mode, float *losses /* [3] */);
/* n learning! iterations t0 .. t0+n-1 with fresh targets (MuZero Reanalyze on the batch): before step t's loss, every distinct game of
 * get_batch(step = t) is reanalysed whole (exactly mz_reanalyse_search on that key, with the weights as they are after step t-1), then
 * the batch is gathered from the refreshed ring and the step proceeds as mz_learn_step(t).  Queued on the device without a host round
 * trip per step (the ResNet path has one: its weight image is packed on the host).  *simulations (may be NULL) = total simulations run.
 * MZ_E_ARG: t0 < 1, n < 1, losses NULL; MZ_E_STATE: empty buffer or self-play in progress; grad_mode errors as mz_learn_step.  Nothing
 * changes on an error. */
int mz_learn_steps_reanalysed(mz_ctx *ctx, int64_t t0, int n, int grad_mode, int exploration, float *losses /* [3] */, int64_t *simulations);
/* gradients of one caller-supplied batch without an update (parity entry point): grad[n_params] in the reference blob
 * order.  MZ_GRAD_REFERENCE_L2: what the reference's three Zygote pullbacks actually return, 2*theta (Learning.jl:385-393
 * differentiate a closure whose predictions were computed outside of it).  MZ_GRAD_BPTT: the gradient of the same loss
 * value (Learning.jl:261-288) through the unroll (Learning.jl:347-370), plus 2*theta.  MZ_GRAD_BPTT is built for the FeedForwardHP
 * networks (with or without BatchNorm) whose hidden layers are at most 64 wide; the observation stack itself may be wider (stacked_observations = 2:
 * 99 inputs); everything else answers MZ_E_UNSUPPORTED. */
int mz_learn_gradients(mz_ctx *ctx, int grad_mode, int B, const float *obs_batch, const float *action_batch, const float *value_batch,
                       const float *reward_batch, const float *policy_batch, const float *gscale, float *grad, float *losses /* [3] */);
/* the same with importance-sampling weights weight_batch [B] (conf.PER; NULL = 1) */
int mz_learn_gradients_w(mz_ctx *ctx, int grad_mode, int B, const float *obs_batch, const float *action_batch, const float *value_batch,
                         const float *reward_batch, const float *policy_batch, const float *gscale, const float *weight_batch, float *grad,
                         float *losses /* [3] */);
/* same update on a caller-supplied batch (parity entry point) */
int mz_learn_step_batch(mz_ctx *ctx, int64_t t, int grad_mode, int B, const float *obs_batch, const float *action_batch,
                        const float *value_batch, const float *reward_batch, const float *policy_batch,
                        const float *gscale, float *losses);
int mz_optimizer_reset(mz_ctx *ctx);
/* checkpoint / resume (Learning.jl:416-435 serialises the networks only; resuming ADAM needs its moments): m, v in the blob order,
 * steps_done = number of updates applied so far (the next step must be called with t = steps_done + 1) */
int mz_get_optimizer_state(mz_ctx *ctx, float *m, float *v, int64_t n, int64_t *steps_done);
int mz_set_optimizer_state(mz_ctx *ctx, const float *m, const float *v, int64_t n, int64_t steps_done);

/* ---- multi-GPU: data-parallel learner, one process per GPU (no reference counterpart; the reference's
 * only transport is Julia Distributed, games/tictactoe/main.jl:1-2,15-21) ------------------------- */
int mz_comm_unique_id(uint8_t id[128]);
int mz_comm_init(mz_ctx *ctx, int rank, int nranks, const uint8_t id[128]);
int mz_comm_destroy(mz_ctx *ctx);
/* How the data-parallel learner exchanges gradients: 0 = no communicator, 1 = ncclAllReduce followed by the ADAM kernel, 2 = one kernel that
 * reads every rank's gradient over peer memory (CUDA IPC mappings, NVLink), sums in rank order and applies ADAM (the default on one node;
 * MUZERO_B200_DP=nccl in the environment of mz_comm_init keeps mode 1). */
int mz_comm_mode(mz_ctx *ctx);
/* Which kernels a learner step of `grad_mode` runs on in this context: 0 = fp32 SIMT (bit-exact forward; nn_mode = MZ_NN_FP32_EXACT / MZ_NN_BF16_TC,
 * or networks the tensor-core learner does not cover), 1 = unroll forward on the tensor cores (MZ_NN_SPLIT_MMA, MZ_GRAD_REFERENCE_L2), 2 = forward and
 * backward on the tensor cores (MZ_NN_SPLIT_MMA, MZ_GRAD_BPTT: split-precision forward, bf16 backward, gradients within 1e-2 of the largest entry per
 * network; MUZERO_B200_BPTT_SIMT=1 in the environment forces path 0), 3 = ResNet networks with MZ_GRAD_REFERENCE_L2 (the unroll runs through the bf16 inference
 * kernel), -1 = not available (ResNet networks with MZ_GRAD_BPTT). */
int mz_learner_path(mz_ctx *ctx, int grad_mode);

/* ---- instrumentation --------------------------------------------------------------------------- */
/* number of kernels this ctx has launched since creation (bench.py's gpu_launches) */
int mz_launch_count(mz_ctx *ctx, int64_t *n);
/* device time (ms) and launch count accumulated per kernel family since the last reset;
 * family: 0 self-play move kernel, 1 save/refill, 2 replay gather, 3 learner fwd/loss, 4 adam, 5 nn batch, 6 env */
int mz_kernel_time(mz_ctx *ctx, int family, double *ms, int64_t *launches);
int mz_kernel_time_reset(mz_ctx *ctx, int enable);
/* phase timers of the last mz_self_play call (profiling builds with -DMZ_PHASE_TIMERS, zeros otherwise):
 * out[6*g + p] = clock cycles summed over CTAs, g = 0 prediction group / tree lane 0, g = 1 dynamics group,
 * p = 0 select+stage, 1 wait, 2 network, 3 wait, 4 expand+backup, 5 = number of CTAs that reported */
int mz_phase_cycles(mz_ctx *ctx, uint64_t out[60]);   /* raw profiling counters, see profiles/phase_timers.py */
/* tree statistics of the last mz_self_play call: mean legal actions L and mean selection depth d */
int mz_search_stats(mz_ctx *ctx, double *mean_legal, double *mean_depth);

#ifdef __cplusplus
}
#endif
#endif
