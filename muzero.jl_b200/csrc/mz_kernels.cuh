// mz_kernels.cuh -- the self-play kernels.
//
//   mz_k_search<MODE>   one CTA = 32 trees.  Root inference (representation + prediction), root expansion,
//                       then S simulations of {PUCT select -> prediction(parent) + dynamics -> expand -> backup}
//                       without leaving the SM: weights stream through shared memory (TMA bulk copies),
//                       activations stay in shared memory, node pools live in HBM/L2.
//                       MODE_API  : roots come from caller arrays (run_mcts, src/SelfPlay.jl:230-285)
//                       MODE_SLOTS: roots come from the device-resident game slots; after the search the same
//                                   kernel samples the action, steps the environment and appends to the game
//                                   history (play_game's loop body, src/SelfPlay.jl:343-380).
//                       MODE_REPLAY: roots are stored positions of the replay ring (MuZero Reanalyze); the results
//                                   replace the position's policy target and reanalysed root value.
//   mz_k_save_refill    save_game (src/ReplayBuffer.jl:133-161) for finished slots, in slot order, into the
//                       device replay ring + assignment of the next game ids to free slots.
#pragma once
#include "mz_device.cuh"

enum { MZ_MODE_API = 0, MZ_MODE_SLOTS = 1, MZ_MODE_REPLAY = 2 };

// Optional phase timers (make EXTRA=-DMZ_PHASE_TIMERS): threads 0 (tree lane 0 / prediction group) and 128 (dynamics
// group) of every CTA accumulate clock64() deltas of the simulation loop into stats[4 + 6*g + phase]:
// 0->1 select+stage, 1->2 wait, 2->3 network, 3->4 wait, 4->5 expand+backup.  Compiled out of the product build.
#ifdef MZ_PHASE_TIMERS
#define MZ_TIMER_DECL long long mz_tk[1] = {0}; long long mz_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define MZ_TIMER(i) do { long long c_ = clock64(); if ((i) > 0) mz_acc[(i) - 1] += c_ - mz_tk[0]; mz_tk[0] = c_; } while (0)
#define MZ_TIMER_FLUSH(stats) do { if ((stats) && (threadIdx.x == 0 || threadIdx.x == MZ_GROUP)) { int g_ = threadIdx.x ? 1 : 0; \
    for (int i_ = 0; i_ < 8; i_++) atomicAdd(&(stats)[32 + 9 * g_ + i_], (unsigned long long)mz_acc[i_]); atomicAdd(&(stats)[32 + 9 * g_ + 8], 1ull); } } while (0)
#else
#define MZ_TIMER_DECL
#define MZ_TIMER(i)
#define MZ_TIMER_FLUSH(stats)
#endif
enum { MZ_SLOT_IDLE = 0, MZ_SLOT_ACTIVE = 1, MZ_SLOT_FINISHED = 2 /* + P.fin_tag: 2 or 3 */ };

struct mz_slots {          // device-resident concurrent games, SoA
    uint64_t *p1, *p2; int32_t *player, *T, *status; int64_t *game_id;
    int32_t *fin_list;       // [G + 6] scratch of mz_k_save_refill: the finished slots in slot order, their number, the first key - 1
    // per-slot GameHistory under construction (src/Constructors.jl:6-16); boards are kept as bit masks
    uint64_t *h_p1, *h_p2;   // [G][Tmax] board before move i
    int32_t *h_action;       // [G][Tmax]
    float *h_reward;         // [G][Tmax]
    uint8_t *h_to_play;      // [G][Tmax]
    float *h_cv;             // [G][Tmax][A]
    float *h_rv;             // [G][Tmax]
};
struct mz_ring {           // device replay buffer: key k lives at (k-1) % capacity
    int64_t capacity;
    int64_t *game_id; int32_t *T;
    uint64_t *h_p1, *h_p2; int32_t *h_action; float *h_reward; uint8_t *h_to_play; float *h_cv; float *h_rv;
    uint32_t *q_pos, *q_game;             // conf.PER: history.priorities [R][Tmax], history.game_priority [R] (fixed point)
    unsigned long long *prefix, *upd;     // inclusive prefix sums of q_game in key order [R]; update_priorities! scratch [R][Tmax]
    float *h_rrv; uint8_t *reanalysed;   // GameHistory.reanalysed_predicted_root_values (Constructors.jl:13): [R][Tmax] + "is not nothing" flag per game
    // counters (device): [0] num_played_games, [1] num_played_steps, [2] total_samples, [3] next game id to hand out,
    // [4] end game id (exclusive), [5] active slots after the last refill
    int64_t *counters;
};
struct mz_search_args {
    const float *wglob; const double *pbc0; const double *sqrtN; void *tree_pool;
    int32_t n, max_dim, max_layer_floats, exploration;
    int32_t persist;             // MODE_SLOTS, mz_k_search_sp: 1 = the kernel plays every game of its CTA to the end (one launch per wave: a CTA starts its next
                                 // move when ITS trees are done instead of waiting for the slowest CTA of the grid)
    // MODE_API inputs / outputs
    const float *stacked; const uint32_t *legal; const uint64_t *game_id; const int32_t *move_idx;
    int32_t *visit_counts; float *root_value; float *root_priors;
    // MODE_SLOTS
    mz_slots slots; float temperature;
    unsigned long long *stats;   // [0] sum depth, [1] simulations, [2] sum legal, [3] roots
    // MODE_REPLAY: root i is position t of the game at ring position pos, replay[i] = pos * Tmax + t (the index of its [R][Tmax] entries).
    // Last, so that the fields the other modes read keep their offsets.
    mz_ring ring; const int64_t *replay;
};

// ---- lane-parallel tree operations: MZ_LANES (8) lanes of a warp cooperate on one tree.  They are the GPU-only
// counterparts of the scalar mz_tree_select / mz_tree_expand / mz_tree_backup in mz_common.h (which the CPU harness
// checks against the oracle) and must produce the same bits; tests/test_gpu_parity.py holds them to that. ----
__device__ __forceinline__ float mz_seg_max(float v, uint32_t segmask) {
#pragma unroll
    for (int m = 1; m < MZ_LANES; m <<= 1) { float o = __shfl_xor_sync(segmask, v, m, MZ_LANES); v = o > v ? o : v; }
    return v;
}
__device__ __forceinline__ uint32_t mz_seg_or(uint32_t v, uint32_t segmask) {
#pragma unroll
    for (int m = 1; m < MZ_LANES; m <<= 1) v |= __shfl_xor_sync(segmask, v, m, MZ_LANES);
    return v;
}
__device__ __forceinline__ int mz_seg_add(int v, uint32_t segmask) {
#pragma unroll
    for (int m = 1; m < MZ_LANES; m <<= 1) v += __shfl_xor_sync(segmask, v, m, MZ_LANES);
    return v;
}

// select_child loop (src/SelfPlay.jl:157-166, 261-268): lane ln scores the children at Dict positions ln and ln+8.
// One dependent memory round trip per level: the chosen child's packed word (expanded? where are its children?) and
// prior come by shuffle from the lane that loaded its record to score it.
__device__ __forceinline__ mz_leaf mz_tree_select_lanes(const mz_params &P, const mz_tree &t, const double *pbc0, const double *sqrtN, uint32_t legal,
                                                        uint32_t posmask, mz_minmax mm, uint32_t game, uint32_t move, uint32_t sim, int ln,
                                                        uint32_t segmask, uint16_t *path, bool tri = false) {
    mz_leaf L; L.node = 0; L.parent = 0; L.action = 0; L.depth = 0; L.prior = 0.0f; L.parent_x = 0;
    const int a0 = ln < P.A ? P.order[ln] : 1, a1 = ln + 8 < P.A ? P.order[ln + 8] : 1;
    const bool ok0 = (posmask >> ln) & 1u, ok1 = (posmask >> (ln + 8)) & 1u;
    uint32_t x = mz_f2bits(t.A[0].x);
    if (ln == 0) path[0] = 0;
    while (mz_nx_exp(x) >= 0) {
        L.depth++;
        const int base = 1 + mz_nx_exp(x) * P.A;
        const int N = mz_nx_visit(x);
        mz_f4 c0, c1; c0.x = c0.y = c0.z = c0.w = 0.0f; c1 = c0;
        if (ok0) c0 = t.A[base + a0 - 1];
        if (ok1) c1 = t.A[base + a1 - 1];
        float s0 = 0.0f, s1 = 0.0f;
        // tri: pbc0 is a compact (triangular) copy of the table: a child has at most as many visits as its parent, so row N holds n = 0..N
        const double *row = pbc0 + (tri ? (N * (N + 1)) / 2 : N * (P.S + 2));
        if (ok0) s0 = mz_ucb_row(P, row, c0, mm);
        if (ok1) s1 = mz_ucb_row(P, row, c1, mm);
        float b = ok0 ? s0 : -INFINITY;
        if (ok1) b = s1 > b ? s1 : b;
        const float best = mz_seg_max(b, segmask);
        uint32_t tied = ((ok0 && s0 == best) ? (1u << ln) : 0u) | ((ok1 && s1 == best) ? (1u << (ln + 8)) : 0u);
        tied = mz_seg_or(tied, segmask);
        if (tied == 0) tied = posmask & (0u - posmask);
        const int nt = __popc(tied);
        int pick = 0;
        if (nt > 1 && P.tie_mode == MZ_TIE_PHILOX) pick = (int)mz_u32_below(mz_philox(P.seed, MZ_STREAM_TIE, game, move, sim, (uint32_t)L.depth).x, (uint32_t)nt);
        uint32_t m = tied;
        for (int i = 0; i < pick; i++) m &= m - 1;
        const int j = __ffs((int)m) - 1;
        L.action = P.order[j];
        L.parent = L.node; L.parent_x = x;
        L.node = base + L.action - 1;
        x = __shfl_sync(segmask, j < 8 ? mz_f2bits(c0.x) : mz_f2bits(c1.x), j & 7, MZ_LANES);
        L.prior = __shfl_sync(segmask, j < 8 ? c0.z : c1.z, j & 7, MZ_LANES);
        if (ln == 0) path[L.depth] = (uint16_t)L.node;
    }
    return L;
}

// softmax(logits) (Learning.jl:114) then expand_node!'s second softmax over the legal subset (SelfPlay.jl:88-96, Q1);
// exp() calls are spread over the lanes, both sums run in ascending action order like the scalar code.  The expanded
// node's record is rebuilt from what is known (unvisited, prior, reward): no load.
__device__ __forceinline__ void mz_tree_expand_lanes(const mz_params &P, const mz_tree &t, int node, int e, uint32_t legal, const float *logits /* [a*ls] */,
                                                     float reward, float prior, int ln, uint32_t segmask, int ls = MZ_ROWS /* stride between logits */) {
    const bool v0 = ln < P.A, v1 = ln + 8 < P.A;
    const float l0 = v0 ? logits[ln * ls] : -INFINITY, l1 = v1 ? logits[(ln + 8) * ls] : -INFINITY;
    float m = mz_seg_max(l1 > l0 ? l1 : l0, segmask);
    float e0 = v0 ? mz_expf(l0 - m) : 0.0f, e1 = v1 ? mz_expf(l1 - m) : 0.0f;
    // ordered sums (ascending action, like the scalar code): all shuffles are issued first, then the dependent adds
    float ev[MZ_MAX_A];
#pragma unroll
    for (int a = 0; a < MZ_MAX_A; a++) ev[a] = __shfl_sync(segmask, a < 8 ? e0 : e1, a & 7, MZ_LANES);
    float s = 0.0f;
#pragma unroll
    for (int a = 0; a < MZ_MAX_A; a++) if (a < P.A) s = s + ev[a];
    const float p0 = e0 / s, p1 = e1 / s;                       // policy[ln], policy[ln+8]
    const bool g0 = v0 && ((legal >> ln) & 1u), g1 = v1 && ((legal >> (ln + 8)) & 1u);
    float q = g0 ? p0 : -INFINITY; if (g1) q = p1 > q ? p1 : q;
    const float m2 = mz_seg_max(q, segmask);
    const float f0 = g0 ? mz_expf(p0 - m2) : 0.0f, f1 = g1 ? mz_expf(p1 - m2) : 0.0f;
#pragma unroll
    for (int a = 0; a < MZ_MAX_A; a++) ev[a] = __shfl_sync(segmask, a < 8 ? f0 : f1, a & 7, MZ_LANES);
    float s2 = 0.0f;
#pragma unroll
    for (int a = 0; a < MZ_MAX_A; a++) if (a < P.A && ((legal >> a) & 1u)) s2 = s2 + ev[a];
    const int base = 1 + e * P.A;
    mz_f4 c; c.x = mz_bits2f(mz_nx_pack(0, -1, 0)); c.y = 0.0f; c.w = 0.0f;
    if (v0) { c.z = g0 ? f0 / s2 : 0.0f; t.A[base + ln] = c; }
    if (v1) { c.z = g1 ? f1 / s2 : 0.0f; t.A[base + ln + 8] = c; }
    if (ln == 0) { mz_f4 me; me.x = mz_bits2f(mz_nx_pack(0, e, 0)); me.y = 0.0f; me.z = prior; me.w = reward; t.A[node] = me; }
    __syncwarp(segmask);
}

// backpropagate! (SelfPlay.jl:190-217, Q8) over the recorded path: the node records of 8 path entries are loaded in
// parallel, the (cheap, sequential) value recurrence is replayed by every lane, the owning lane writes back.
__device__ __forceinline__ void mz_tree_backup_lanes(const mz_params &P, const mz_tree &t, const uint16_t *path, int depth, float value, mz_minmax &mm,
                                                     int ln, uint32_t segmask) {
    for (int top = depth; top >= 0; top -= MZ_LANES) {
        const int idx = top - ln;
        const int nd = idx >= 0 ? (int)path[idx] : 0;
        mz_f4 rec = t.A[nd];
        const int cnt = top + 1 < MZ_LANES ? top + 1 : MZ_LANES;
        for (int u = 0; u < cnt; u++) {
            const uint32_t x = __shfl_sync(segmask, mz_f2bits(rec.x), u, MZ_LANES) + 1u;     // visit_count += 1
            const float y = __shfl_sync(segmask, rec.y, u, MZ_LANES), w = __shfl_sync(segmask, rec.w, u, MZ_LANES);
            const int j = depth - (top - u);
            const bool same = (P.P == 1) || ((j & 1) == 0);       // j % P, P <= 2
            const float ny = same ? y + value : y - value;
            const int vc = mz_nx_visit(x);
            const float upd = w + P.discount * (ny / (float)vc);
            mm.mn = mm.mn < upd ? mm.mn : upd;
            mm.mx = mm.mx > upd ? mm.mx : upd;
            if (P.P == 1) value = w + P.discount * value;
            else value = same ? -w : w + P.discount * value;
            if (ln == u) { rec.x = mz_bits2f(x); rec.y = ny; t.A[nd] = rec; }
        }
    }
    __syncwarp(segmask);
}

// store_search_stats! (src/SelfPlay.jl:115-122, Q12): the root's visit distribution over the legal actions, the policy target of the
// position.  Self-play (mz_slot_epilogue) and reanalysis (mz_root_finish<MODE_REPLAY>) both write it through here.
__device__ __forceinline__ void mz_store_search_stats(const mz_params &P, float *cv, const int32_t *vc, uint32_t legal, int sum_visits) {
    for (int i = 0; i < P.A; i++) cv[i] = ((legal >> i) & 1u) ? (float)((double)vc[i] / (double)sum_visits) : 0.0f;
}

// play_game's loop body after run_mcts (src/SelfPlay.jl:344-346, 360-379) for one game slot: temperature rule, select_action, environment
// step, store_search_stats! (Q12), history append, termination.  Lane 0 of the tree, from mz_root_finish.
__device__ __forceinline__ void mz_slot_epilogue(const mz_params &P, const mz_slots &s, int64_t g, const int32_t *vc, int sum_visits, uint32_t legal, float rv,
                                                 float temperature, uint32_t game, uint32_t move) {
    int T = s.T[g];
    const int action = mz_select_action_counts(P, vc, legal, mz_play_temperature(P, T, temperature), game, move);  // :344-346, :360
    mz_board b; b.p1 = s.p1[g]; b.p2 = s.p2[g]; b.player = s.player[g];
    const int p = b.player;
    mz_env_step_b(P, b, action);                                                    // :366
    const float reward = (float)mz_env_reward_b(P, b, p);                           // :367
    const bool done = mz_env_terminated_b(P, b);                                    // :368
    mz_store_search_stats(P, s.h_cv + ((size_t)g * P.Tmax + T) * P.A, vc, legal, sum_visits);
    s.h_rv[(size_t)g * P.Tmax + T] = rv;
    s.h_action[(size_t)g * P.Tmax + T] = action;                                    // :377-379
    s.h_reward[(size_t)g * P.Tmax + T] = reward;
    s.h_to_play[(size_t)g * P.Tmax + T] = (uint8_t)p;
    T += 1;
    s.p1[g] = b.p1; s.p2[g] = b.p2; s.player[g] = b.player; s.T[g] = T;
    if (T < P.Tmax) { s.h_p1[(size_t)g * P.Tmax + T] = b.p1; s.h_p2[(size_t)g * P.Tmax + T] = b.p2; }
    if (done || T > P.max_moves) s.status[g] = MZ_SLOT_FINISHED + P.fin_tag;                    // loop condition :343
}

// ---- run_mcts for one root (SelfPlay.jl:230-285), the part every search kernel shares: the root's state, its stacked observation, the
// root node and its expansion, the results.  The kernels differ in how they run the networks and in which threads own a tree. ----
struct mz_root { bool active; uint32_t legal, game, move, posmask; };
// root g: MODE_API from the caller's arrays, MODE_SLOTS from the slot's board (SelfPlay.jl:351,359); in competitive play a slot is searched
// only on MuZero's plies.  MODE_REPLAY: stored position t of a ring game, with the root self-play searched there (board before move t,
// its side to move, game id, move index t + 1).  valid = false (no root g for this thread: g >= a.n, or not a tree lane) gives an inactive
// root with no legal action.
template <int MODE>
__device__ __forceinline__ mz_root mz_root_begin(const mz_params &P, const mz_search_args &a, int64_t g, bool valid) {
    mz_root R; R.active = false; R.legal = 0; R.game = 0; R.move = 0; R.posmask = 0;
    if (MODE == MZ_MODE_API) {
        if (valid) { R.legal = a.legal[g]; R.game = (uint32_t)a.game_id[g]; R.move = (uint32_t)a.move_idx[g]; }
        R.active = R.legal != 0;   // run_mcts asserts !isempty(legal_actions) (SelfPlay.jl:243)
    } else if (MODE == MZ_MODE_REPLAY) {
        if (valid) {
            const int64_t e = a.replay[g], pos = e / P.Tmax;
            mz_board b; b.p1 = a.ring.h_p1[e]; b.p2 = a.ring.h_p2[e]; b.player = a.ring.h_to_play[e];
            R.legal = mz_env_legal_b(P, b); R.game = (uint32_t)a.ring.game_id[pos]; R.move = (uint32_t)(e - pos * P.Tmax) + 1u;
        }
        R.active = R.legal != 0;   // a stored position precedes a move: it has a legal action
    } else if (valid) {            // MODE_SLOTS
        R.active = a.slots.status[g] == MZ_SLOT_ACTIVE && (P.arena_player == 0 || a.slots.player[g] == P.arena_player);
        if (R.active) {
            mz_board b; b.p1 = a.slots.p1[g]; b.p2 = a.slots.p2[g]; b.player = a.slots.player[g];
            R.legal = mz_env_legal_b(P, b); R.game = (uint32_t)a.slots.game_id[g]; R.move = (uint32_t)a.slots.T[g] + 1u;
        }
        if (R.legal == 0) R.active = false;   // never reached in play
    }
    for (int j = 0; j < P.A; j++) if ((R.legal >> (P.order[j] - 1)) & 1u) R.posmask |= 1u << j;   // legal actions as a mask over Dict positions
    return R;
}
// entry k of root gg's stacked observations (get_stacked_observations, SelfPlay.jl:128-149); 0 past the launch's roots and for a slot
// that has no ply to search.  MODE_REPLAY reads the stored history as mz_k_reanalyse and get_batch do: index t + 1 of the game.
template <int MODE>
__device__ __forceinline__ float mz_root_obs(const mz_params &P, const mz_search_args &a, int64_t gg, int k) {
    if (gg >= a.n) return 0.0f;
    if (MODE == MZ_MODE_API) return a.stacked[gg * P.stack_size + k];
    if (MODE == MZ_MODE_REPLAY) {
        const int64_t e = a.replay[gg], pos = e / P.Tmax, row = pos * P.Tmax;
        return mz_stacked_value(P, a.ring.h_p1 + row, a.ring.h_p2 + row, a.ring.h_action + row, (int)(e - row) + 1, k);
    }
    if (a.slots.status[gg] != MZ_SLOT_ACTIVE) return 0.0f;
    return mz_stacked_value(P, a.slots.h_p1 + gg * P.Tmax, a.slots.h_p2 + gg * P.Tmax, a.slots.h_action + gg * P.Tmax, a.slots.T[gg] + 1, k);
}
// the 8 lanes of an active tree, after the root prediction: Node(prior=0) (:232), its expansion (:245; logits[a * ls] = logit of action
// a + 1), then the exploration noise (:247-249; eps = 0 is the identity)
__device__ __forceinline__ void mz_root_init(const mz_params &P, const mz_tree &t, const mz_root &R, int exploration, const float *logits, int ls, int ln,
                                             uint32_t segmask) {
    if (ln == 0) { mz_f4 root; root.x = mz_bits2f(mz_nx_pack(0, -1, 0)); root.y = 0.0f; root.z = 0.0f; root.w = 0.0f; t.A[0] = root; }
    __syncwarp(segmask);
    mz_tree_expand_lanes(P, t, 0, 0, R.legal, logits, 0.0f, 0.0f, ln, segmask, ls);
    if (ln == 0 && exploration && P.exploration_eps != 0.0f) mz_tree_add_noise(P, t, R.legal, R.game, R.move);
    __syncwarp(segmask);
}
// results of root g, lane 0 of an active tree: the launch's statistics (stats[0] sum of leaf depths, [1] simulations, [2] sum of legal
// actions, [3] roots), then visit counts, root value and priors to the caller (MODE_API), the move of the game (MODE_SLOTS), or the
// stored position's policy target and reanalysed root value (MODE_REPLAY)
template <int MODE>
__device__ __forceinline__ void mz_root_finish(const mz_params &P, const mz_search_args &a, int64_t g, const mz_tree &t, const mz_root &R,
                                               unsigned long long depth_sum) {
    int32_t vc[MZ_MAX_A]; int sum_visits = 0, nlegal = 0;
    for (int i = 0; i < P.A; i++) {
        vc[i] = ((R.legal >> i) & 1u) ? (int32_t)mz_nx_visit(mz_f2bits(t.A[1 + i].x)) : 0;
        sum_visits += vc[i]; nlegal += (int)((R.legal >> i) & 1u);
    }
    const mz_f4 root = t.A[0];
    const int rvc = mz_nx_visit(mz_f2bits(root.x));
    const float rv = rvc == 0 ? 0.0f : root.y / (float)rvc;                                 // node_value(root)
    if (a.stats) {
        atomicAdd(&a.stats[0], depth_sum); atomicAdd(&a.stats[1], (unsigned long long)P.S);
        atomicAdd(&a.stats[2], (unsigned long long)nlegal); atomicAdd(&a.stats[3], 1ull);
    }
    if (MODE == MZ_MODE_API) {
        for (int i = 0; i < P.A; i++) {
            a.visit_counts[g * P.A + i] = vc[i];
            if (a.root_priors) a.root_priors[g * P.A + i] = ((R.legal >> i) & 1u) ? t.A[1 + i].z : 0.0f;
        }
        a.root_value[g] = rv;
    } else if (MODE == MZ_MODE_REPLAY) {
        const int64_t e = a.replay[g];
        mz_store_search_stats(P, a.ring.h_cv + e * P.A, vc, R.legal, sum_visits);
        a.ring.h_rrv[e] = rv;
    } else mz_slot_epilogue(P, a.slots, g, vc, sum_visits, R.legal, rv, a.temperature, R.game, R.move);
}

// Self-play launches run one iteration ahead of the host (run_wave, mz_api.cu): a CTA none of whose slots has a ply to search -- every
// CTA of the iteration queued past the end of a wave -- returns at its first instruction, before any barrier, TMA or TMEM state exists.
// MODE_API and MODE_REPLAY launches cover exactly their roots (the replay root list is dense): no CTA is idle.
template <int MODE>
__device__ __forceinline__ bool mz_cta_idle(const mz_params &P, const mz_search_args &a, int rows_per_cta) {
    if (MODE != MZ_MODE_SLOTS) return false;
    int any = 0;
    const int64_t g = (int64_t)blockIdx.x * rows_per_cta + threadIdx.x;
    if ((int)threadIdx.x < rows_per_cta && g < a.n) any = a.slots.status[g] == MZ_SLOT_ACTIVE && (P.arena_player == 0 || a.slots.player[g] == P.arena_player);
    return __syncthreads_or(any) == 0;
}

template <int MODE, bool BN = false>
__global__ void __launch_bounds__(MZ_THREADS) mz_k_search(const __grid_constant__ mz_params P, const mz_search_args a) {
    extern __shared__ __align__(128) unsigned char mz_smem[];
    if (mz_cta_idle<MODE>(P, a, MZ_ROWS)) return;
    const mz_smem_plan sp = mz_smem_carve(mz_smem, a.max_dim, a.max_layer_floats, P.hidden_pad, P.S);
    const int tid = threadIdx.x;
    const int r = tid >> 3, ln = tid & (MZ_LANES - 1);              // tree (row) of this thread and its lane within the tree
    const uint32_t segmask = 0xffu << ((tid & 31) & ~7);
    const int64_t g = (int64_t)blockIdx.x * MZ_ROWS + r;
    mz_nn_pipe pipe;
    mz_pipe_init(pipe, sp, a.wglob);
    mz_zero_activations(sp, a.max_dim);
    uint16_t *path = sp.path + (size_t)r * (P.S + 2);

    // ---- per-tree state, replicated in the 8 lanes of the tree ----
    mz_tree tree; tree.A = nullptr; tree.hidden = nullptr;
    if (g < a.n) tree = mz_tree_at(P, a.tree_pool, g);
    const mz_root root = mz_root_begin<MODE>(P, a, g, g < a.n);
    const bool active = root.active;
    __syncthreads();   // mbarrier init + zeroed buffers visible
    const int pred_first = P.nets[1].first, dyn_first = P.nets[2].first;
    if (tid == 0) mz_nn_issue(pipe, P, P.nets[0].first, 0);            // group 0: representation, then prediction
    if (tid == MZ_GROUP) mz_nn_issue(pipe, P, dyn_first, 0);     // group 1: dynamics (first used in simulation 1)

    // ---- stage the stacked observations, k-major (get_stacked_observations, SelfPlay.jl:128-149) ----
    for (int i = tid; i < MZ_ROWS * P.stack_size; i += MZ_THREADS) {
        int rr, k;
        if (MODE == MZ_MODE_API) { rr = i / P.stack_size; k = i % P.stack_size; }   // the caller's rows are contiguous
        else { k = i / MZ_ROWS; rr = i % MZ_ROWS; }                                  // slots, replay positions: every entry is computed
        sp.in0[k * MZ_ROWS + rr] = mz_root_obs<MODE>(P, a, (int64_t)blockIdx.x * MZ_ROWS + rr, k);
    }
    __syncthreads();

    // ---- root: representation -> h0; prediction(h0) -> (v0, p0)  (SelfPlay.jl:233-245), group 0 only ----
    if (pipe.grp == 0) {
        mz_nn_net<BN>(pipe, P, 0, pred_first, sp.in0, sp.bufT[0], sp.outH, nullptr, sp.t0[0], sp.t1[0]);
        mz_nn_net<BN>(pipe, P, 1, pred_first, sp.outH, sp.bufT[0], sp.outV, sp.outL, sp.t0[0], sp.t1[0]);   // prefetches simulation 1's first layer
    }
    __syncthreads();

    mz_minmax mm; mm.mn = INFINITY; mm.mx = -INFINITY;                                    // SelfPlay.jl:251
    unsigned long long depth_sum = 0;
    MZ_TIMER_DECL;
    if (active) {
        for (int k = ln; k < P.hidden; k += MZ_LANES) tree.hidden[k] = sp.outH[k * MZ_ROWS + r];
        mz_root_init(P, tree, root, a.exploration, sp.outL + r, MZ_ROWS, ln, segmask);
    }

    // ---- simulations (SelfPlay.jl:254-283) ----
    for (int sim = 1; sim <= P.S; sim++) {
        mz_leaf leaf; leaf.node = 0; leaf.parent = 0; leaf.action = 1; leaf.depth = 0; leaf.prior = 0.0f; leaf.parent_x = 0;
        MZ_TIMER(0);
        if (active) {
            leaf = mz_tree_select_lanes(P, tree, a.pbc0, a.sqrtN, root.legal, root.posmask, mm, root.game, root.move, (uint32_t)sim, ln, segmask, path);
            depth_sum += (unsigned long long)leaf.depth;
            MZ_TIMER(1);
            const int pe = mz_nx_exp(leaf.parent_x), dbl = mz_nx_dbl(leaf.parent_x);
            const float *h = tree.hidden + (size_t)pe * P.hidden_pad;
            const float sc = mz_bits2f((uint32_t)(127 + dbl) << 23);                       // 2^dbl: state after dbl in-place doublings (Q6)
            for (int k = ln; k < P.hidden; k += MZ_LANES) {
                float v = h[k] * sc;
                sp.in1[k * MZ_ROWS + r] = v;                                                // prediction(parent.hidden_state), :271 (Q5)
                sp.in0[k * MZ_ROWS + r] = v * 2.0f;                                         // make_state_action: state .*= 2, :11
            }
            const float plane = P.act_plane_play[leaf.action];                              // :8-9
            for (int k = P.obs_size + ln; k < P.sa_size; k += MZ_LANES) sp.in0[k * MZ_ROWS + r] = plane;
            __syncwarp(segmask);
            if (ln == 0) reinterpret_cast<uint32_t *>(&tree.A[leaf.parent])[0] = leaf.parent_x + (1u << 24);   // one more doubling (Q6)
        }
        MZ_TIMER(2);
        __syncthreads();
        MZ_TIMER(3);
        if (pipe.grp == 0) mz_nn_net<BN>(pipe, P, 1, sim < P.S ? pred_first : -1, sp.in1, sp.bufT[0], sp.outV, sp.outL, sp.t0[0], sp.t1[0]);
        else               mz_nn_net<BN>(pipe, P, 2, sim < P.S ? dyn_first : -1, sp.in0, sp.bufT[1], sp.outH, sp.outR, sp.t0[1], sp.t1[1]);
        MZ_TIMER(4);
        __syncthreads();
        MZ_TIMER(5);
        if (active) {
            float *nh = tree.hidden + (size_t)sim * P.hidden_pad;
            for (int k = ln; k < P.hidden; k += MZ_LANES) nh[k] = sp.outH[k * MZ_ROWS + r];
            MZ_TIMER(6);
            mz_tree_expand_lanes(P, tree, leaf.node, sim, root.legal, sp.outL + r, sp.outR[r], leaf.prior, ln, segmask);   // :280 (root's legal set, Q7)
            MZ_TIMER(7);
            mz_tree_backup_lanes(P, tree, path, leaf.depth, sp.outV[r], mm, ln, segmask);                  // :281
        }
        MZ_TIMER(8);
        // no CTA barrier needed here: the lanes that stage the next inputs are the ones that just read the outputs, and
        // every network read of in0/in1 finished before the barrier above
    }

    MZ_TIMER_FLUSH(a.stats);
    if (active && ln == 0) mz_root_finish<MODE>(P, a, g, tree, root, depth_sum);
}

// Initial priorities of one stored game (save_game, ReplayBuffer.jl:136-145): |root_value - compute_target_value|^alpha per
// position, game priority = their maximum.
__device__ __forceinline__ void mz_per_init_game(const mz_params &P, const mz_ring &r, int64_t pos) {
    const int T = r.T[pos];
    const float *rew = r.h_reward + (size_t)pos * P.Tmax, *rv = r.h_rv + (size_t)pos * P.Tmax; const uint8_t *tp = r.h_to_play + (size_t)pos * P.Tmax;
    uint32_t mx = 0;
    for (int i = 1; i <= P.Tmax; i++) {
        uint32_t q = 0;
        if (i <= T) { q = mz_per_quantise(mz_pow_int(fabsf(rv[i - 1] - mz_target_value(P, T, rew, tp, rv, i)), P.per_alpha)); mx = q > mx ? q : mx; }
        r.q_pos[(size_t)pos * P.Tmax + i - 1] = q;
    }
    r.q_game[pos] = mx;
}
__global__ void mz_k_per_init(const __grid_constant__ mz_params P, mz_ring r, int64_t key0, int n) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) mz_per_init_game(P, r, (key0 + j - 1) % r.capacity);
}
// Inclusive prefix sums of the game priorities in ascending key order (single CTA; integer sums: exact and order independent).
// counters[6] = their total.
__global__ void __launch_bounds__(1024) mz_k_per_scan(const __grid_constant__ mz_params P, mz_ring r) {
    __shared__ unsigned long long part[1024];
    const int tid = threadIdx.x;
    const int64_t played = r.counters[0], n = played < r.capacity ? played : r.capacity, first_key = played - n + 1;
    const int64_t per = (n + 1023) / 1024, lo = (int64_t)tid * per, hi = lo + per < n ? lo + per : n;
    unsigned long long s = 0;
    for (int64_t i = lo; i < hi; i++) s += r.q_game[(first_key + i - 1) % r.capacity];
    part[tid] = s; __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) { unsigned long long t = tid >= off ? part[tid - off] : 0ull; __syncthreads(); part[tid] += t; __syncthreads(); }
    unsigned long long run = tid ? part[tid - 1] : 0ull;
    for (int64_t i = lo; i < hi; i++) { run += r.q_game[(first_key + i - 1) % r.capacity]; r.prefix[i] = run; }
    if (tid == 1023) r.counters[6] = (int64_t)part[1023];
}
// update_priorities! (ReplayBuffer.jl:168-183, repaired bounds; Learning.jl:400-404): rows k = 0 .. min(K, T - pos) of
// |predicted_values - target_values|^alpha go to positions pos + k.  Batch elements apply in order (the last one wins where they
// overlap): phase 1 marks every slot with the largest (b + 1, q) by a 64-bit atomicMax, phase 2 lets the winner write, phase 3
// recomputes the game priorities.
__global__ void mz_k_per_update(const __grid_constant__ mz_params P, mz_ring r, int B, const int32_t *index, const float *pv, const float *tv, int phase) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, K1 = P.K + 1;
    if (i >= B * K1) return;
    const int b = i / K1, k = i % K1;
    const int64_t key = index[2 * b], played = r.counters[0], n = played < r.capacity ? played : r.capacity;
    if (key < played - n + 1 || key > played) return;                       // the game has left the buffer (:172)
    const int64_t pos = (key - 1) % r.capacity;
    const int T = r.T[pos], p = index[2 * b + 1];
    if (phase == 2) {
        if (k == 0) { uint32_t mx = 0; for (int t = 0; t < T; t++) { uint32_t q = r.q_pos[(size_t)pos * P.Tmax + t]; mx = q > mx ? q : mx; } r.q_game[pos] = mx; }
        return;
    }
    if (p + k > T) return;
    const size_t slot = (size_t)pos * P.Tmax + p + k - 1;
    const uint32_t q = mz_per_quantise(mz_pow_int(fabsf(pv[(size_t)b * K1 + k] - tv[(size_t)b * K1 + k]), P.per_alpha));
    const unsigned long long mine = ((unsigned long long)(b + 1) << 32) | q;
    if (phase == 0) atomicMax(&r.upd[slot], mine);
    else if (r.upd[slot] == mine) { r.q_pos[slot] = q; r.upd[slot] = 0ull; }
}

// competitive play (play_game with an opponent, src/SelfPlay.jl:358-363): the opponent's ply for every active slot whose side to move
// is not MuZero's.  The history entry repeats the statistics of the previous search (store_search_stats! is called with the stale
// root, :374); before the first search the reference's `root` is the Int 0 and it would throw: zeros.
__global__ void mz_k_opponent_move(const __grid_constant__ mz_params P, mz_slots s, int n_slots) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_slots || s.status[g] != MZ_SLOT_ACTIVE || s.player[g] == P.arena_player) return;
    mz_board b; b.p1 = s.p1[g]; b.p2 = s.p2[g]; b.player = s.player[g];
    int T = s.T[g];
    const int p = b.player;
    const int action = mz_opponent_action(P, b, P.arena_opponent, (uint32_t)s.game_id[g], (uint32_t)T + 1u);
    mz_env_step_b(P, b, action);
    const float reward = (float)mz_env_reward_b(P, b, p);
    const bool done = mz_env_terminated_b(P, b);
    const size_t o = (size_t)g * P.Tmax + T;
    for (int i = 0; i < P.A; i++) s.h_cv[o * P.A + i] = T > 0 ? s.h_cv[(o - 1) * P.A + i] : 0.0f;
    s.h_rv[o] = T > 0 ? s.h_rv[o - 1] : 0.0f;
    s.h_action[o] = action; s.h_reward[o] = reward; s.h_to_play[o] = (uint8_t)p;
    T += 1;
    s.p1[g] = b.p1; s.p2[g] = b.p2; s.player[g] = b.player; s.T[g] = T;
    if (T < P.Tmax) { s.h_p1[(size_t)g * P.Tmax + T] = b.p1; s.h_p2[(size_t)g * P.Tmax + T] = b.p2; }
    if (done || T > P.max_moves) s.status[g] = MZ_SLOT_FINISHED + P.fin_tag;
}
__global__ void mz_k_opponent_action(const __grid_constant__ mz_params P, int n, const uint64_t *p1, const uint64_t *p2, const int32_t *player, int opponent,
                                     const uint64_t *game_id, const int32_t *move_idx, int32_t *action) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    mz_board b; b.p1 = p1[g]; b.p2 = p2[g]; b.player = player[g];
    action[g] = mz_opponent_action(P, b, opponent, (uint32_t)game_id[g], (uint32_t)move_idx[g]);
}

// save_game (src/ReplayBuffer.jl:133-161) for every finished slot in slot order, then hand the next game ids to
// free slots.  Single CTA: the order in which games receive their game number must be deterministic.
#define MZ_SAVE_MAX_K 64   // slots per thread of mz_k_save_refill: num_slots <= 65536
#define MZ_FIN_KEY(n) (((n) + 3) & ~1)   // fin_list[n] = number of games; the 64-bit first key - 1 sits at the next 8-byte aligned pair (fin_list has n + 6 entries)
__global__ void __launch_bounds__(1024) mz_k_save_refill(const __grid_constant__ mz_params P, mz_slots s, mz_ring r, int n_slots, unsigned long long *arena_tally = nullptr, int wave_sync = 0,
                                                          int64_t *snap = nullptr /* mapped host memory: the counters after this kernel, read by the self-play loop */) {
    __shared__ unsigned long long warp_tot[32];
    __shared__ int active_count;
    __shared__ long long add_steps, add_samples;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t base_key = r.counters[0], next_game = r.counters[3], end_game = r.counters[4];
    if (tid == 0) { active_count = 0; add_steps = 0; add_samples = 0; }
    // (1) thread t owns the contiguous slots [t*K, (t+1)*K): one exclusive scan over the CTA gives every finished slot its rank in slot
    //     order (= the order game numbers are handed out in) and every free slot its rank among the free ones
    const int K = (n_slots + 1023) / 1024, lo = tid * K, hi = lo + K < n_slots ? lo + K : n_slots;
    unsigned long long fin_bits = 0, free_bits = 0;                        // per owned slot (K <= 64)
    for (int i = 0; lo + i < hi; i++) {
        const int st = s.status[lo + i];
        // finished in THIS iteration (tag = its parity); a slot the search of the next iteration -- which may run beside this kernel -- is
        // finishing right now carries the other tag and counts as active: the next save / refill takes it
        if (st == MZ_SLOT_FINISHED + P.fin_tag) fin_bits |= 1ull << i;
        if (st == MZ_SLOT_FINISHED + P.fin_tag || st == MZ_SLOT_IDLE) free_bits |= 1ull << i;
    }
    const unsigned long long mine = ((unsigned long long)__popcll(fin_bits) << 32) | (unsigned long long)__popcll(free_bits);
    unsigned long long inc = mine;
    for (int off = 1; off < 32; off <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, off); if (lane >= off) inc += t; }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    unsigned long long before = 0, total = 0;
    for (int w = 0; w < 32; w++) { const unsigned long long t = warp_tot[w]; if (w < warp) before += t; total += t; }
    const unsigned long long excl = before + inc - mine;
    const int fin_rank0 = (int)(excl >> 32), free_rank0 = (int)(excl & 0xffffffffu);
    const int total_fin = (int)(total >> 32), total_free = (int)(total & 0xffffffffu);
    for (unsigned long long m = fin_bits; m; m &= m - 1) s.fin_list[fin_rank0 + __popcll(fin_bits & ((m & (0ull - m)) - 1ull))] = lo + __ffsll((long long)m) - 1;
    __syncthreads();
    // (2) save_game for finished game j (slot fin_list[j]) under key = num_played_games + j + 1 (:149-154); all games in parallel
    long long steps = 0, samples = 0;
    for (int j = tid; j < total_fin; j += 1024) {
        const int g = s.fin_list[j];
        const int64_t key = base_key + j + 1, pos = (key - 1) % r.capacity;
        const int T = s.T[g];
        if (key > r.capacity) samples -= (long long)r.T[pos];              // evicted history (:156-160)
        r.game_id[pos] = s.game_id[g]; r.T[pos] = T; r.reanalysed[pos] = 0;
        steps += T; samples += T;
        if (arena_tally && P.arena_tally != 0)                               // competitive play: wins / draws / losses for MuZero
            atomicAdd(&arena_tally[1 - mz_arena_outcome(P, T, s.h_action + (size_t)g * P.Tmax, P.arena_tally)], 1ull);
    }
    if (steps) atomicAdd((unsigned long long *)&add_steps, (unsigned long long)steps);
    if (samples) atomicAdd((unsigned long long *)&add_samples, (unsigned long long)samples);
    //     the histories themselves are copied by mz_k_save_copy (many CTAs: one CTA moves ~1 MB far too slowly), which reads
    //     {first key - 1, number of games} from the two words after the list
    if (tid == 0) { s.fin_list[n_slots] = total_fin; reinterpret_cast<int64_t *>(s.fin_list + MZ_FIN_KEY(n_slots))[0] = base_key; }
    __syncthreads();
    // (3) hand the next game ids to the free slots, in slot order; reset! (game.jl:15-20).  The board before move 0 is empty in every
    //     history, so h_p1 / h_p2 [g][0] stay zero.
    //     wave_sync: new games start only when EVERY slot is free, so that all trees of a launch are at the same ply (a launch lasts as
    //     long as its deepest tree, and late plies search deeper: mixing plies makes every launch as slow as the last plies')
    const bool hand_out = !wave_sync || total_free == n_slots;
    int nact = 0, free_rank = free_rank0;
    for (int i = 0; lo + i < hi; i++) {
        const int g = lo + i;
        if ((free_bits >> i) & 1ull) {
            const int64_t id = next_game + free_rank++;
            if (hand_out && id < end_game) { s.game_id[g] = id; s.status[g] = MZ_SLOT_ACTIVE; s.T[g] = 0; s.p1[g] = 0; s.p2[g] = 0; s.player[g] = 1; nact++; }
            else s.status[g] = MZ_SLOT_IDLE;
        } else nact++;                                                     // neither finished nor idle: active
    }
    if (nact) atomicAdd(&active_count, nact);
    __syncthreads();
    if (tid == 0) {
        const int64_t handed = !hand_out ? 0 : next_game + total_free < end_game ? total_free : (end_game - next_game > 0 ? end_game - next_game : 0);
        r.counters[0] = base_key + total_fin;
        r.counters[1] += add_steps;
        r.counters[2] += add_samples;
        r.counters[3] = next_game + handed;
        r.counters[5] = active_count;
        if (snap) {   // instead of a device-to-host copy between the kernels of every move (a copy-engine operation in the stream costs more than the kernel)
            snap[0] = base_key + total_fin; snap[1] = r.counters[1]; snap[2] = r.counters[2]; snap[3] = next_game + handed; snap[4] = end_game; snap[5] = active_count;
            snap[6] = r.counters[6]; snap[7] = r.counters[7];
            __threadfence_system();
        }
    }
}

// The GameHistory arrays of the games mz_k_save_refill has just numbered: slot fin_list[j] -> ring position of key base_key + j + 1.
// Reads nothing that the refill resets (the per-slot history arrays are overwritten only by the next game's plies, after this kernel).
__global__ void __launch_bounds__(256) mz_k_save_copy(const __grid_constant__ mz_params P, mz_slots s, mz_ring r, int n_slots) {
    const int total_fin = s.fin_list[n_slots];
    if (total_fin == 0) return;
    const int64_t base_key = reinterpret_cast<const int64_t *>(s.fin_list + MZ_FIN_KEY(n_slots))[0];
    const int nthreads = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
    const int rows = total_fin * P.Tmax;
    for (int idx = t0; idx < rows; idx += nthreads) {
        const int j = idx / P.Tmax, i = idx - j * P.Tmax;
        const size_t so = (size_t)s.fin_list[j] * P.Tmax + i, ro = (size_t)((base_key + j) % r.capacity) * P.Tmax + i;
        r.h_p1[ro] = s.h_p1[so]; r.h_p2[ro] = s.h_p2[so]; r.h_action[ro] = s.h_action[so]; r.h_reward[ro] = s.h_reward[so];
        r.h_to_play[ro] = s.h_to_play[so]; r.h_rv[ro] = s.h_rv[so];
    }
    const int row_cv = P.Tmax * P.A;
    for (int idx = t0; idx < total_fin * row_cv; idx += nthreads) {
        const int j = idx / row_cv, e = idx - j * row_cv;
        r.h_cv[(size_t)((base_key + j) % r.capacity) * row_cv + e] = s.h_cv[(size_t)s.fin_list[j] * row_cv + e];
    }
}
// initial priorities of the games just saved (save_game, ReplayBuffer.jl:136-145), from the stored histories
__global__ void mz_k_save_per(const __grid_constant__ mz_params P, mz_slots s, mz_ring r, int n_slots) {
    const int total_fin = s.fin_list[n_slots];
    const int64_t base_key = reinterpret_cast<const int64_t *>(s.fin_list + MZ_FIN_KEY(n_slots))[0];
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < total_fin; j += gridDim.x * blockDim.x) mz_per_init_game(P, r, (base_key + j) % r.capacity);
}

// ---- batched network callables (init_*(hyper) callables, src/Learning.jl:87-142) -------------------
struct mz_nn_args { const float *wglob; int32_t B, max_dim, max_layer_floats, net; const float *in; float *out1; float *out2; };
template <bool BN = false>
__global__ void __launch_bounds__(MZ_THREADS) mz_k_nn_forward(const __grid_constant__ mz_params P, const mz_nn_args a) {
    extern __shared__ __align__(128) unsigned char mz_smem[];
    const mz_smem_plan sp = mz_smem_carve(mz_smem, a.max_dim, a.max_layer_floats, P.hidden_pad, P.S);
    const int tid = threadIdx.x;
    mz_nn_pipe pipe;
    mz_pipe_init(pipe, sp, a.wglob);
    mz_zero_activations(sp, a.max_dim);
    __syncthreads();
    const mz_net &N = P.nets[a.net];
    if (tid == 0) mz_nn_issue(pipe, P, N.first, 0);
    const int in = P.layers[N.first].in;
    for (int i = tid; i < MZ_ROWS * in; i += MZ_THREADS) {
        int r = i / in, k = i % in;
        int64_t gg = (int64_t)blockIdx.x * MZ_ROWS + r;
        sp.in0[k * MZ_ROWS + r] = gg < a.B ? a.in[gg * in + k] : 0.0f;
    }
    __syncthreads();
    float *h1 = a.net == 1 ? sp.outV : sp.outH, *h2 = a.net == 1 ? sp.outL : sp.outR;
    if (pipe.grp == 0) mz_nn_net<BN>(pipe, P, a.net, -1, sp.in0, sp.bufT[0], h1, h2, sp.t0[0], sp.t1[0]);
    __syncthreads();
    const int64_t g = (int64_t)blockIdx.x * MZ_ROWS + tid;
    if (tid < MZ_ROWS && g < a.B) {
        if (a.net == 1) {
            float logits[MZ_MAX_A], policy[MZ_MAX_A];
            for (int i = 0; i < P.A; i++) logits[i] = sp.outL[i * MZ_ROWS + tid];
            mz_softmax(logits, P.A, policy);
            a.out1[g] = sp.outV[tid];
            for (int i = 0; i < P.A; i++) a.out2[g * P.A + i] = policy[i];
        } else {
            for (int k = 0; k < P.hidden; k++) a.out1[g * P.hidden + k] = sp.outH[k * MZ_ROWS + tid];
            if (a.net == 2) a.out2[g] = sp.outR[tid];
        }
    }
}

// ---- reanalyse: fills GameHistory.reanalysed_predicted_root_values (Constructors.jl:13) -------------------------------
// The reference consumes the field (compute_target_value, ReplayBuffer.jl:8) but nothing produces it (main.jl:18 only keeps a
// counter).  Producer, as in MuZero Reanalyze: for every stored position of games key0 .. key0+n-1 the value head of the CURRENT
// networks on the stacked observation, prediction(representation(get_stacked_observations(history, i))).  32 positions per CTA.
struct mz_reanalyse_args { const float *wglob; int32_t max_dim, max_layer_floats, n; int64_t key0; mz_ring ring; };
template <bool BN = false>
__global__ void __launch_bounds__(MZ_THREADS) mz_k_reanalyse(const __grid_constant__ mz_params P, const mz_reanalyse_args a) {
    extern __shared__ __align__(128) unsigned char mz_smem[];
    const mz_smem_plan sp = mz_smem_carve(mz_smem, a.max_dim, a.max_layer_floats, P.hidden_pad, P.S);
    const int tid = threadIdx.x;
    mz_nn_pipe pipe;
    mz_pipe_init(pipe, sp, a.wglob);
    mz_zero_activations(sp, a.max_dim);
    __syncthreads();
    if (tid == 0) mz_nn_issue(pipe, P, P.nets[0].first, 0);
    const int64_t total = (int64_t)a.n * P.Tmax;
    for (int i = tid; i < MZ_ROWS * P.stack_size; i += MZ_THREADS) {
        const int k = i / MZ_ROWS, rr = i % MZ_ROWS;
        const int64_t item = (int64_t)blockIdx.x * MZ_ROWS + rr;
        float v = 0.0f;
        if (item < total) {
            const int64_t pos = (a.key0 + item / P.Tmax - 1) % a.ring.capacity; const int t = (int)(item % P.Tmax);
            if (t < a.ring.T[pos]) v = mz_stacked_value(P, a.ring.h_p1 + pos * P.Tmax, a.ring.h_p2 + pos * P.Tmax, a.ring.h_action + pos * P.Tmax, t + 1, k);
        }
        sp.in0[k * MZ_ROWS + rr] = v;
    }
    __syncthreads();
    if (pipe.grp == 0) {
        mz_nn_net<BN>(pipe, P, 0, P.nets[1].first, sp.in0, sp.bufT[0], sp.outH, nullptr, sp.t0[0], sp.t1[0]);
        mz_nn_net<BN>(pipe, P, 1, -1, sp.outH, sp.bufT[0], sp.outV, sp.outL, sp.t0[0], sp.t1[0]);
    }
    __syncthreads();
    const int64_t item = (int64_t)blockIdx.x * MZ_ROWS + tid;
    if (tid < MZ_ROWS && item < total) {
        const int64_t pos = (a.key0 + item / P.Tmax - 1) % a.ring.capacity; const int t = (int)(item % P.Tmax);
        a.ring.h_rrv[pos * P.Tmax + t] = t < a.ring.T[pos] ? sp.outV[tid] : 0.0f;
        if (t == 0) a.ring.reanalysed[pos] = 1;
    }
}

// mz_reanalyse_search: the entries the search does not write -- reanalysed values of positions t >= T are 0, as mz_k_reanalyse leaves
// them -- and the "is set" flag of every game of the range.  One thread per (game, position).
__global__ void mz_k_reanalyse_mark(const __grid_constant__ mz_params P, mz_ring r, int64_t key0, int n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)n * P.Tmax) return;
    const int64_t pos = (key0 + i / P.Tmax - 1) % r.capacity; const int t = (int)(i % P.Tmax);
    if (t >= r.T[pos]) r.h_rrv[pos * P.Tmax + t] = 0.0f;
    if (t == 0) r.reanalysed[pos] = 1;
}

// ---- batched environment verbs (games/tictactoe/game.jl) --------------------------------------------
__global__ void mz_k_env_step(const __grid_constant__ mz_params P, int n, uint64_t *p1, uint64_t *p2, int32_t *player,
                              const int32_t *action, float *reward, int32_t *done, uint32_t *legal) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    mz_board b; b.p1 = p1[i]; b.p2 = p2[i]; b.player = player[i];
    if (action) {
        int p = b.player;
        mz_env_step_b(P, b, action[i]);
        p1[i] = b.p1; p2[i] = b.p2; player[i] = b.player;
        if (reward) reward[i] = (float)mz_env_reward_b(P, b, p);
    }
    if (done) done[i] = mz_env_terminated_b(P, b) ? 1 : 0;
    if (legal) legal[i] = mz_env_legal_b(P, b);
}
__global__ void mz_k_env_obs(const __grid_constant__ mz_params P, int n, const uint64_t *p1, const uint64_t *p2, float *obs) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)n * P.obs_size) return;
    int g = (int)(i / P.obs_size), k = (int)(i % P.obs_size);
    mz_board b; b.p1 = p1[g]; b.p2 = p2[g]; b.player = 1;
    obs[i] = mz_env_obs_value(P, b, k / P.cells, k % P.cells);
}
__global__ void mz_k_select_action(const __grid_constant__ mz_params P, int n, const int32_t *vc, const uint32_t *legal, float temperature,
                                   const uint64_t *game_id, const int32_t *move_idx, int32_t *action) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t c[MZ_MAX_A];
    for (int k = 0; k < P.A; k++) c[k] = vc[(size_t)i * P.A + k];
    action[i] = mz_select_action_counts(P, c, legal[i], temperature, (uint32_t)game_id[i], (uint32_t)move_idx[i]);
}

// ---- GameHistory export / import (src/Constructors.jl:6-16) --------------------------------------------
__global__ void mz_k_history_export(const __grid_constant__ mz_params P, mz_ring r, int64_t key0, int n, int64_t *game_id, int32_t *T,
                                    float *obs, int32_t *actions, float *rewards, int32_t *to_play, float *cv, float *rv) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t per = (int64_t)P.Tmax * P.obs_size;
    if (i >= (int64_t)n * per) return;
    int j = (int)(i / per); int rem = (int)(i % per); int t = rem / P.obs_size, k = rem % P.obs_size;
    int64_t pos = (key0 + j - 1) % r.capacity;
    int Tg = r.T[pos];
    size_t ro = (size_t)pos * P.Tmax + t;
    mz_board b; b.p1 = r.h_p1[ro]; b.p2 = r.h_p2[ro]; b.player = 1;
    obs[i] = t < Tg ? mz_env_obs_value(P, b, k / P.cells, k % P.cells) : 0.0f;
    if (k == 0) {
        size_t oo = (size_t)j * P.Tmax + t;
        bool v = t < Tg;
        actions[oo] = v ? r.h_action[ro] : 0; rewards[oo] = v ? r.h_reward[ro] : 0.0f; to_play[oo] = v ? (int32_t)r.h_to_play[ro] : 0;
        rv[oo] = v ? r.h_rv[ro] : 0.0f;
        for (int a = 0; a < P.A; a++) cv[oo * P.A + a] = v ? r.h_cv[ro * P.A + a] : 0.0f;
        if (t == 0) { game_id[j] = r.game_id[pos]; T[j] = Tg; }
    }
}
// import: observations come as float planes; boards are recovered from planes 0 and 1.  One thread per (game, move).
__global__ void mz_k_history_import(const __grid_constant__ mz_params P, mz_ring r, int64_t key0, int n, const int64_t *game_id, const int32_t *T,
                                    const float *obs, const int32_t *actions, const float *rewards, const int32_t *to_play,
                                    const float *cv, const float *rv) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * P.Tmax) return;
    int j = i / P.Tmax, t = i % P.Tmax;
    int64_t pos = (key0 + j - 1) % r.capacity;
    size_t ro = (size_t)pos * P.Tmax + t, oo = (size_t)j * P.Tmax + t;
    uint64_t b1 = 0, b2 = 0;
    const float *o = obs + oo * P.obs_size;
    for (int c = 0; c < P.cells; c++) {
        int bit = c;
        if (P.game == MZ_GAME_CONNECT) bit = (c % P.W) + (P.W + 1) * (c / P.W);
        if (o[c] != 0.0f) b1 |= 1ull << bit;
        if (o[P.cells + c] != 0.0f) b2 |= 1ull << bit;
    }
    r.h_p1[ro] = b1; r.h_p2[ro] = b2; r.h_action[ro] = actions[oo]; r.h_reward[ro] = rewards[oo]; r.h_to_play[ro] = (uint8_t)to_play[oo];
    r.h_rv[ro] = rv[oo];
    for (int a = 0; a < P.A; a++) r.h_cv[ro * P.A + a] = cv[oo * P.A + a];
    if (t == 0) { r.game_id[pos] = game_id[j]; r.T[pos] = T[j]; r.reanalysed[pos] = 0; }
}
