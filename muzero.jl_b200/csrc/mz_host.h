// mz_host.h -- host-side construction of the device parameter block, the padded weight layout and the
// integer-only UCB tables from an mz_config.  Plain C++ (no CUDA) so the CPU harness can share it.
#pragma once
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "mz_common.h"

namespace mzh {

// Julia (<= 1.10) Dict{Int,V} iteration order for keys 1..A inserted in ascending order: 16 slots (x4 growth
// once count*3 > 2*slots), slot = hash_64_64(3|x| + bits(Float64(x))) & (sz-1), linear probing.  This is the
// order SelfPlay.jl:158-159 (select_child), :103 (noise) and :294-295 (select_action) iterate children in.
inline uint64_t hash_64_64(uint64_t a) {
    a = ~a + (a << 21); a = a ^ (a >> 24); a = a + (a << 3) + (a << 8); a = a ^ (a >> 14);
    a = a + (a << 2) + (a << 4); a = a ^ (a >> 28); a = a + (a << 31);
    return a;
}
inline void julia_dict_order(int A, int32_t *order) {
    int sz = 16;
    while (A * 3 > sz * 2) sz *= 4;
    std::vector<int> slots((size_t)sz, 0);
    for (int k = 1; k <= A; k++) {
        double d = (double)k; uint64_t b; memcpy(&b, &d, 8);
        int i = (int)(hash_64_64(3ull * (uint64_t)k + b) & (uint64_t)(sz - 1));
        while (slots[(size_t)i]) i = (i + 1) & (sz - 1);
        slots[(size_t)i] = k;
    }
    int n = 0;
    for (int i = 0; i < sz; i++) if (slots[(size_t)i]) order[n++] = slots[(size_t)i];
}

inline void default_config(mz_config *c) {   // games/tictactoe/params.jl:2-29, src/Constructors.jl:18-52
    memset(c, 0, sizeof(*c));
    c->game = MZ_GAME_TICTACTOE; c->W = 3; c->H = 3; c->C = 3; c->A = 9; c->num_players = 2;
    c->stacked_observations = 1; c->max_moves = 9; c->num_iters = 10; c->num_unroll_steps = 5; c->td_steps = 5;
    c->batch_size = 32; c->replay_buffer_size = 10000; c->pb_c_base = 19652; c->intermediate_rewards = 0;
    c->tie_mode = MZ_TIE_PHILOX; c->pb_c_init = 1.25f; c->discount = 0.997f; c->dirichlet_alpha = 0.25f;
    c->exploration_eps = 0.25f; c->seed = 1337;
    julia_dict_order(c->A, c->child_order);
    c->width_hidden = 64; c->depth_representation = 3; c->depth_prediction = 3; c->depth_dynamics = 3;
    c->depth_policy = 1; c->depth_value = 1; c->depth_reward = 1; c->depth_state_head = 3;
    c->hidden_state_size = 27; c->reward_activation_tanh = 1;
    c->num_slots = 4096; c->nn_mode = MZ_NN_FP32_EXACT;
    c->per = 0; c->per_alpha = 1;
    c->temperature_threshold = -1;
    c->use_batch_norm = 0;
    c->net_type = MZ_NET_FEEDFORWARD; c->rn_num_blocks = 2; c->rn_num_filters = 64; c->rn_kernel = 3; c->rn_first_head_filters = 1; c->rn_second_head_filters = 2;
}

inline const char *validate(const mz_config &c) {
    if (c.game != MZ_GAME_TICTACTOE && c.game != MZ_GAME_CONNECT) return "unknown game";
    if (c.A < 1 || c.A > MZ_MAX_A) return "action space size must be in 1..16";
    if (c.W < 1 || c.H < 1 || c.C != 3) return "observation_shape must be (W,H,3)";
    if (c.game == MZ_GAME_TICTACTOE && (c.W != 3 || c.H != 3 || c.A != 9)) return "TicTacToe needs observation_shape (3,3,3) and 9 actions";
    if (c.game == MZ_GAME_CONNECT && (c.A != c.H || (c.W + 1) * c.H > 64)) return "Connect needs A == H columns and (W+1)*H <= 64";
    if (c.net_type != MZ_NET_FEEDFORWARD && c.net_type != MZ_NET_RESNET) return "unknown net_type";
    if (c.temperature_threshold < -1) return "temperature_threshold must be >= 0, or -1 for nothing";
    if (c.per && (c.per_alpha < 0 || c.per_alpha > 3)) return "PER_alpha must be in 0..3";
    if (c.per && c.net_type != MZ_NET_FEEDFORWARD) return "PER belongs to the learner, which is implemented for the FeedForwardHP networks";
    if (c.net_type == MZ_NET_FEEDFORWARD && c.hidden_state_size != c.W * c.H * c.C) return "hidden_state_size must equal prod(observation_shape) (Constructors.jl:73)";
    if (c.num_players < 1 || c.num_players > 2) return "1 or 2 players";
    if (c.num_iters < 1 || c.num_iters > 1000) return "num_iters must be in 1..1000";
    if (1 + (c.num_iters + 1) * c.A > 65535) return "tree too large for 16-bit path entries";
    if (c.max_moves < 1 || c.max_moves > 63) return "max_moves must be in 1..63";
    if (c.stacked_observations < 0 || c.stacked_observations > 8) return "stacked_observations out of range";
    if (c.num_unroll_steps < 0 || c.num_unroll_steps > 32 || c.td_steps < 0 || c.td_steps > 64) return "unroll/td steps out of range";
    if (c.width_hidden < 4 || c.width_hidden % 4) return "width_hidden must be a positive multiple of 4";
    if (c.batch_size < 1 || c.replay_buffer_size < 1 || c.num_slots < 1) return "batch_size, replay_buffer_size, num_slots must be positive";
    if (c.num_slots > 65536) return "num_slots must be <= 65536 (mz_k_save_refill keeps a 64-bit mask of the slots each of its 1024 threads owns)";
    int order_seen = 0;
    for (int i = 0; i < c.A; i++) { if (c.child_order[i] < 1 || c.child_order[i] > c.A) return "child_order must be a permutation of 1..A"; order_seen |= 1 << (c.child_order[i] - 1); }
    if (order_seen != (1 << c.A) - 1) return "child_order must be a permutation of 1..A";
    return nullptr;
}

struct model {
    mz_params P;
    std::vector<double> pbc0, sqrtN;   // ucb_score's Float64 terms, functions of integers only (Q3)
    int max_dim;                       // largest layer in/out_pad: activation buffer rows
    int max_layer_floats;              // largest bulk-copied layer
};

// bn: the layer comes from make_dense with use_batch_norm (Learning.jl:70-79): exactly the relu layers
inline void add_layer(mz_params &P, int in, int out, int act, int &src_off, int &dev_off, bool bn = false) {
    mz_layer &l = P.layers[P.n_layers++];
    l.in = in; l.out = out; l.out_pad = (out + 3) & ~3; l.act = act; l.bn = bn && act == MZ_ACT_RELU ? 1 : 0;
    l.src_w_off = src_off; src_off += in * out; l.src_b_off = src_off; src_off += out + (l.bn ? 4 * out : 0);
    l.w_off = dev_off; dev_off += in * l.out_pad; l.b_off = dev_off; dev_off += l.out_pad * (l.bn ? 5 : 1);
    l.floats = in * l.out_pad + l.out_pad * (l.bn ? 5 : 1);
}

inline int count_layers(const mz_config &c) {
    return (c.depth_representation + 2) + (c.depth_prediction + 1 + c.depth_value + 1 + c.depth_policy + 1) +
           (c.depth_dynamics + 1 + c.depth_state_head + 1 + c.depth_reward + 1);
}

// Conf.discount^i exactly as Julia evaluates Float32^Int64 (Base: products for i<=3, llvm.pow.f32 beyond).
inline float discount_pow(float g, int i) {
    if (i == 0) return 1.0f;
    if (i == 1) return g;
    if (i == 2) return g * g;
    if (i == 3) return g * g * g;
    return powf(g, (float)i);
}

inline const char *build_model(const mz_config &c, model &M) {
    if (const char *e = validate(c)) return e;
    if (c.net_type == MZ_NET_FEEDFORWARD && count_layers(c) > MZ_MAX_LAYERS) return "too many layers";
    mz_params &P = M.P;
    memset(&P, 0, sizeof(P));
    P.game = c.game; P.W = c.W; P.H = c.H; P.C = c.C; P.A = c.A; P.P = c.num_players;
    P.stacked = c.stacked_observations; P.max_moves = c.max_moves; P.Tmax = c.max_moves + 1;
    P.S = c.num_iters; P.K = c.num_unroll_steps; P.td = c.td_steps;
    P.cells = c.W * c.H; P.obs_size = P.cells * c.C;
    P.planes = c.C * (c.stacked_observations + 1) + c.stacked_observations;      // Learning.jl:88
    P.stack_size = P.cells * P.planes; P.sa_size = P.cells * (c.C + 1);            // Learning.jl:120
    P.hidden = c.hidden_state_size; P.hidden_pad = (P.hidden + 3) & ~3;
    P.tie_mode = c.tie_mode; P.pb_c_base = c.pb_c_base; P.intermediate_rewards = c.intermediate_rewards;
    P.batch_size = c.batch_size;
    P.pb_c_init = c.pb_c_init; P.discount = c.discount; P.dirichlet_alpha = c.dirichlet_alpha; P.exploration_eps = c.exploration_eps;
    P.seed = c.seed; P.per = c.per ? 1 : 0; P.per_alpha = c.per_alpha; P.temp_threshold = c.temperature_threshold;
    P.arena_player = 0; P.arena_opponent = MZ_OPP_SELF; P.arena_tally = 0;
    for (int i = 0; i < MZ_MAX_A; i++) P.order[i] = c.child_order[i];
    for (int a = 0; a <= c.A; a++) {
        P.act_plane_play[a] = (float)((double)a / (double)c.A);   // SelfPlay.jl:8-9: Int/Int -> Float64, stored Float32
        P.act_plane_learn[a] = (float)a / (float)c.A;             // Learning.jl:294: Float32 ./ Int
    }
    for (int i = 0; i < 72; i++) P.disc_pow[i] = discount_pow(c.discount, i);
    // tree pool geometry
    P.nodes_per_tree = 1 + (c.num_iters + 1) * c.A;
    int a_bytes = P.nodes_per_tree * 16;
    int h_bytes = (c.num_iters + 1) * P.hidden_pad * 4;
    P.nodeB_off_bytes = 0; P.hidden_off_bytes = a_bytes;
    P.tree_stride_bytes = (a_bytes + h_bytes + 127) & ~127;
    // ucb_score (SelfPlay.jl:172-174): pb_c = log2((N + base + 1) / base) + init, then * sqrt(N)/(n+1); all Float64
    // evaluated for every (parent visits N, child visits n) pair on the host: pbc0[N * (S + 2) + n] = pbc0(N) * (sqrt(N) / (n + 1))
    {
        const size_t W = (size_t)c.num_iters + 2;
        M.pbc0.resize(W * W); M.sqrtN.resize(W);
        for (size_t N = 0; N < W; N++) {
            const double p0 = log2((double)((int)N + c.pb_c_base + 1) / (double)c.pb_c_base) + (double)c.pb_c_init;
            M.sqrtN[N] = sqrt((double)N);
            for (size_t n = 0; n < W; n++) M.pbc0[N * W + n] = p0 * (M.sqrtN[N] / (double)(n + 1));
        }
    }
    if (c.net_type == MZ_NET_RESNET) {   // the residual networks have their own description (mz_rn_host.h); the state is (W,H,nf)
        P.sa_size = P.hidden + P.cells; P.tc_ok = 0; M.max_dim = 4; M.max_layer_floats = 0;
        return nullptr;
    }
    // networks (src/Learning.jl:87-142), Flux.params order
    int src = 0, dev = 0, w = c.width_hidden;
    const bool bn = c.use_batch_norm != 0;
    P.nets[0].first = P.n_layers;
    add_layer(P, P.stack_size, w, MZ_ACT_RELU, src, dev, bn);
    for (int i = 0; i < c.depth_representation; i++) add_layer(P, w, w, MZ_ACT_RELU, src, dev, bn);
    add_layer(P, w, P.hidden, MZ_ACT_ID, src, dev);
    P.nets[0].n_trunk = c.depth_representation + 2; P.nets[0].n_h1 = 0; P.nets[0].n_h2 = 0;
    P.nets[1].first = P.n_layers;
    add_layer(P, P.hidden, w, MZ_ACT_RELU, src, dev, bn);
    for (int i = 0; i < c.depth_prediction; i++) add_layer(P, w, w, MZ_ACT_RELU, src, dev, bn);
    for (int i = 0; i < c.depth_value; i++) add_layer(P, w, w, MZ_ACT_RELU, src, dev, bn);
    add_layer(P, w, 1, MZ_ACT_TANH, src, dev);
    for (int i = 0; i < c.depth_policy; i++) add_layer(P, w, w, MZ_ACT_RELU, src, dev, bn);
    add_layer(P, w, c.A, MZ_ACT_ID, src, dev);
    P.nets[1].n_trunk = c.depth_prediction + 1; P.nets[1].n_h1 = c.depth_value + 1; P.nets[1].n_h2 = c.depth_policy + 1;
    P.nets[2].first = P.n_layers;
    add_layer(P, P.sa_size, w, MZ_ACT_RELU, src, dev, bn);
    for (int i = 0; i < c.depth_dynamics; i++) add_layer(P, w, w, MZ_ACT_RELU, src, dev, bn);
    for (int i = 0; i < c.depth_state_head; i++) add_layer(P, w, w, MZ_ACT_RELU, src, dev, bn);
    add_layer(P, w, P.hidden, MZ_ACT_ID, src, dev);
    for (int i = 0; i < c.depth_reward; i++) add_layer(P, w, w, MZ_ACT_RELU, src, dev, bn);
    add_layer(P, w, 1, c.reward_activation_tanh ? MZ_ACT_TANH : MZ_ACT_ID, src, dev);
    P.nets[2].n_trunk = c.depth_dynamics + 1; P.nets[2].n_h1 = c.depth_state_head + 1; P.nets[2].n_h2 = c.depth_reward + 1;
    P.n_params = src; P.total_floats = dev;
    // tensor-core image geometry: usable when every layer has in <= 64 and out <= 64 (one K block, one M=64 tile)
    P.tc_ok = 1;
    {
        int off = 0, boff = 0;
        for (int n = 0; n < 3; n++) {
            P.tc_net_off[n] = off;
            int first = P.nets[n].first, cnt = P.nets[n].n_trunk + P.nets[n].n_h1 + P.nets[n].n_h2;
            for (int i = first; i < first + cnt; i++) {
                const mz_layer &l = P.layers[i];
                if (l.in > 64 || l.out > 64) P.tc_ok = 0;   // (BatchNorm layers: folded into the image by mz_k_pack_images)
                P.tc_a_off[i] = off; P.tc_ksteps[i] = (l.in + 15) / 16; P.tc_bias_off[i] = boff;
                off += ((l.out + 7) / 8) * 1024; boff += 64;
            }
        }
        P.tc_net_off[3] = off; P.tc_bias_floats = boff;
    }
    M.max_dim = 4; M.max_layer_floats = 0;
    for (int i = 0; i < P.n_layers; i++) {
        if (P.layers[i].in > M.max_dim) M.max_dim = P.layers[i].in;
        if (P.layers[i].out_pad > M.max_dim) M.max_dim = P.layers[i].out_pad;
        if (P.layers[i].floats > M.max_layer_floats) M.max_layer_floats = P.layers[i].floats;
    }
    M.max_dim = (M.max_dim + 3) & ~3;
    return nullptr;
}

inline int net_params(const mz_params &P, int net) {
    if (net == MZ_NET_ALL) return P.n_params;
    int first = P.nets[net].first, n = P.nets[net].n_trunk + P.nets[net].n_h1 + P.nets[net].n_h2, s = 0;
    for (int i = first; i < first + n; i++) s += P.layers[i].in * P.layers[i].out + P.layers[i].out * (P.layers[i].bn ? 5 : 1);
    return s;
}
inline int net_src_offset(const mz_params &P, int net) { return net == MZ_NET_ALL ? 0 : P.layers[P.nets[net].first].src_w_off; }

// reference-order blob (W (out,in) column-major: W[o + out*k], then b) <-> padded device layout (W[k][out_pad], b[out_pad])
inline void pack_weights(const mz_params &P, const float *src, float *dev) {
    memset(dev, 0, sizeof(float) * (size_t)P.total_floats);
    for (int i = 0; i < P.n_layers; i++) {
        const mz_layer &l = P.layers[i];
        for (int k = 0; k < l.in; k++) for (int o = 0; o < l.out; o++) dev[l.w_off + k * l.out_pad + o] = src[l.src_w_off + k * l.out + o];
        for (int o = 0; o < l.out; o++) dev[l.b_off + o] = src[l.src_b_off + o];
        if (l.bn) for (int j = 0; j < 4; j++) for (int o = 0; o < l.out; o++) dev[l.b_off + (j + 1) * l.out_pad + o] = src[l.src_b_off + (j + 1) * l.out + o];
    }
}
inline void unpack_weights(const mz_params &P, const float *dev, float *src) {
    for (int i = 0; i < P.n_layers; i++) {
        const mz_layer &l = P.layers[i];
        for (int k = 0; k < l.in; k++) for (int o = 0; o < l.out; o++) src[l.src_w_off + k * l.out + o] = dev[l.w_off + k * l.out_pad + o];
        for (int o = 0; o < l.out; o++) src[l.src_b_off + o] = dev[l.b_off + o];
        if (l.bn) for (int j = 0; j < 4; j++) for (int o = 0; o < l.out; o++) src[l.src_b_off + (j + 1) * l.out + o] = dev[l.b_off + (j + 1) * l.out_pad + o];
    }
}

// float -> bfloat16, round to nearest even (the same rounding as __float2bfloat16_rn on the device)
inline uint16_t f2bf16(float f) {
    uint32_t u; memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
// Byte offset of element (row r, k) inside a K-major SWIZZLE_128B tile with 64 bf16 (128 B) per row: 8-row groups of
// 1024 B, 16-byte chunk index XOR-ed with the row index inside the group (Swizzle<3,4,3>).
inline int tc_tile_offset(int r, int k) { return (r >> 3) * 1024 + (r & 7) * 128 + ((((k >> 3) ^ (r & 7)) & 7) << 4) + (k & 7) * 2; }
// reference-order blob -> bf16 A-operand image (rows = output features, K = input features) + fp32 bias block
inline void pack_weights_tc(const mz_params &P, const float *src, std::vector<uint16_t> &image, std::vector<float> &bias) {
    image.assign((size_t)P.tc_net_off[3] / 2 + 4096, 0); bias.assign((size_t)P.tc_bias_floats, 0.0f);
    for (int i = 0; i < P.n_layers; i++) {
        const mz_layer &l = P.layers[i];
        for (int o = 0; o < l.out; o++) {
            for (int k = 0; k < l.in; k++) image[(size_t)(P.tc_a_off[i] + tc_tile_offset(o, k)) / 2] = f2bf16(src[l.src_w_off + k * l.out + o]);
            bias[(size_t)P.tc_bias_off[i] + o] = src[l.src_b_off + o];
        }
    }
}

// ---- split-precision tensor-core path (mz_sp.cuh, mz_kernels_sp.cuh): rounds, weight sets, hi / lo weight image ----------------
inline float bf16_to_f(uint16_t h) { uint32_t u = (uint32_t)h << 16; float f; memcpy(&f, &u, 4); return f; }

struct sp_builder { const mz_params *P; mz_sp_plan *S; };
inline mz_sp_job sp_job(const mz_params &P, const mz_sp_plan &S, int layer, int src, int dst, int f32_off, int perm) {
    const mz_layer &l = P.layers[layer];
    mz_sp_job j; memset(&j, 0, sizeof(j));
    j.a_off = 0; j.a_bytes = S.w_bytes[layer]; j.bias_off = layer * 64; j.f32_off = f32_off;
    j.src_tile = (int16_t)src; j.dst_tile = (int16_t)dst; j.ks = (int16_t)((l.in + 15) / 16); j.out = (int16_t)l.out; j.act = (int16_t)l.act;
    j.perm = (int16_t)perm; j.layer = (int16_t)layer;
    return j;
}
inline void sp_emit(mz_sp_plan &S, const mz_sp_job *j0, const mz_sp_job *j1) {
    if (S.total_rounds >= MZ_SP_MAX_ROUNDS) { S.ok = 0; return; }
    mz_sp_round &R = S.round[S.total_rounds++];
    memset(&R, 0, sizeof(R));
    R.job[0] = *j0; R.njobs = 1;
    if (j1) { R.job[1] = *j1; R.njobs = 2; }
    R.set = -1; R.next = -1;
}
// Rounds of one network.  Three operand tiles per group: 0 = the network input (free again once the first layer has run), 1, 2.
// Trunk layers ping-pong; the two heads advance in lock-step when the second head is at most two layers deep (so three tiles suffice),
// otherwise one after the other.  Every hidden layer flips the column order of the activations (mz_sp.cuh: the epilogue writes the
// eight columns a thread holds as one 16-byte chunk), `perm` tracks it so the final layer can undo it.
inline void sp_build_net(const mz_params &P, mz_sp_plan &S, int net, int h1_off, int h2_off) {
    const mz_net &N = P.nets[net];
    const int f = N.first;
    S.first[net] = S.total_rounds;
    int cur = 0, perm = 0;
    for (int i = 0; i < N.n_trunk; i++) {
        const bool last = i == N.n_trunk - 1;
        if (last && N.n_h1 == 0) { mz_sp_job j = sp_job(P, S, f + i, cur, -1, h1_off, perm); sp_emit(S, &j, nullptr); }
        else { const int d = cur == 1 ? 2 : 1; mz_sp_job j = sp_job(P, S, f + i, cur, d, -1, perm); sp_emit(S, &j, nullptr); cur = d; perm ^= 1; }
    }
    if (N.n_h1 > 0) {
        const int f1 = f + N.n_trunk, f2 = f1 + N.n_h1, T = cur;
        int other[2], k = 0;
        for (int t = 0; t < 3; t++) if (t != T) other[k++] = t;
        if (N.n_h2 <= 2 && N.n_h2 <= N.n_h1) {
            int c1 = T, c2 = T, p1 = perm, p2 = perm;
            for (int i = 0; i < N.n_h1; i++) {
                const bool last1 = i == N.n_h1 - 1, has2 = i < N.n_h2, last2 = i == N.n_h2 - 1;
                int d1 = -1, d2 = -1;
                if (!last1) { for (int t = 0; t < 3; t++) if (t != c1 && !(has2 && t == c2)) { d1 = t; break; } }
                if (has2 && !last2) { for (int t = 0; t < 3; t++) if (t != c1 && t != c2 && t != d1) { d2 = t; break; } }
                mz_sp_job j1 = sp_job(P, S, f1 + i, c1, d1, last1 ? h1_off : -1, p1);
                if (has2) { mz_sp_job j2 = sp_job(P, S, f2 + i, c2, d2, last2 ? h2_off : -1, p2); sp_emit(S, &j1, &j2); }
                else sp_emit(S, &j1, nullptr);
                if (!last1) { c1 = d1; p1 ^= 1; }
                if (has2 && !last2) { c2 = d2; p2 ^= 1; }
            }
        } else {
            for (int h = 0; h < 2; h++) {
                const int fh = h == 0 ? f1 : f2, nh = h == 0 ? N.n_h1 : N.n_h2, off = h == 0 ? h1_off : h2_off;
                int c = T, p = perm;
                for (int i = 0; i < nh; i++) {
                    const bool last = i == nh - 1;
                    const int d = last ? -1 : (c == other[0] ? other[1] : other[0]);
                    mz_sp_job j = sp_job(P, S, fh + i, c, d, last ? off : -1, p); sp_emit(S, &j, nullptr);
                    if (!last) { c = d; p ^= 1; }
                }
            }
        }
    }
    S.n_rounds[net] = S.total_rounds - S.first[net];
}
inline int sp_round_bytes(const mz_sp_round &R) { int b = 0; for (int j = 0; j < R.njobs; j++) b += 2 * R.job[j].a_bytes; return b; }
// places the weights of network `net` at `base` with its rounds spread over n weight sets (round i of the network uses set i % n);
// returns the bytes used
inline int sp_place(mz_sp_plan &S, int net, int n, int base, int set_first) {
    const int f = S.first[net], R = S.n_rounds[net];
    int off = base;
    for (int s = 0; s < n; s++) {
        int size = 0;
        for (int i = s; i < R; i += n) { const int b = sp_round_bytes(S.round[f + i]); if (b > size) size = b; }
        for (int i = s; i < R; i += n) {
            mz_sp_round &Rd = S.round[f + i];
            Rd.set = (int16_t)(set_first + s);
            const int nx = i + n < R ? i + n : s;
            Rd.next = (int16_t)(nx == i ? -1 : f + nx);
            const int members = (R - s + n - 1) / n;
            Rd.per_pass = (int16_t)(members > 1 ? members : 0); Rd.ord = (int16_t)(members > 1 ? i / n : 0);
            int o = off; Rd.ncopy = Rd.njobs;
            for (int j = 0; j < Rd.njobs; j++) {
                Rd.job[j].a_off = o;
                Rd.copy[j].src_off = S.w_off[Rd.job[j].layer]; Rd.copy[j].bytes = 2 * Rd.job[j].a_bytes; Rd.copy[j].dst_off = o; Rd.copy[j].pad_ = 0;
                o += 2 * Rd.job[j].a_bytes;
            }
        }
        off += size;
    }
    S.set_first[net] = set_first; S.n_sets[net] = n;
    return off - base;
}
// the representation: every round's weights side by side, one set (mbarrier), loaded once per kernel
inline int sp_place_linear(mz_sp_plan &S, int net, int base, int set) {
    const int f = S.first[net], R = S.n_rounds[net];
    int off = base;
    for (int i = 0; i < R; i++) {
        mz_sp_round &Rd = S.round[f + i];
        Rd.set = (int16_t)set; Rd.next = -1; Rd.per_pass = 0; Rd.ord = 0; Rd.ncopy = Rd.njobs;
        for (int j = 0; j < Rd.njobs; j++) {
            Rd.job[j].a_off = off;
            Rd.copy[j].src_off = S.w_off[Rd.job[j].layer]; Rd.copy[j].bytes = 2 * Rd.job[j].a_bytes; Rd.copy[j].dst_off = off; Rd.copy[j].pad_ = 0;
            off += 2 * Rd.job[j].a_bytes;
        }
    }
    S.set_first[net] = set; S.n_sets[net] = 1;
    return off - base;
}
inline void build_sp_plan(const mz_params &P, size_t smem_limit, mz_sp_plan &S) {
    memset(&S, 0, sizeof(S));
    S.ok = 1;
    int off = 0;
    for (int i = 0; i < P.n_layers; i++) {
        const mz_layer &l = P.layers[i];
        if (l.in > 64 || l.out > 64) S.ok = 0;
        S.w_off[i] = off; S.w_bytes[i] = ((l.out + 7) / 8) * 1024;
        off += 2 * S.w_bytes[i];
    }
    S.image_bytes = off; S.bias_floats = P.n_layers * 64;
    if (!S.ok) return;
    S.out_off[0] = 0; S.out_off[1] = 4 * MZ_SP_OS; S.out_off[2] = 20 * MZ_SP_OS; S.out_off[3] = 24 * MZ_SP_OS;
    sp_build_net(P, S, 0, S.out_off[3], -1);
    sp_build_net(P, S, 1, S.out_off[0], S.out_off[1]);
    sp_build_net(P, S, 2, S.out_off[3], S.out_off[2]);
    if (!S.ok) return;
    // the dynamics rounds after the reward is final: with the heads side by side, the state head's last n_h1 - n_h2 layers.  Nothing
    // but the next simulation's staging reads their output, so mz_k_search_sp runs them beside the tree phases.  Heads one after the
    // other end with the reward head: no tail.
    const mz_net &D = P.nets[2];
    S.tail = D.n_h1 > 0 && D.n_h2 > 0 && D.n_h2 <= 2 && D.n_h2 <= D.n_h1 ? D.n_h1 - D.n_h2 : 0;
    // smallest divisor d (sets per network = ceil(rounds / d)) whose weight area fits; d = 1 keeps every weight resident
    for (int d = 1; d <= MZ_SP_MAX_ROUNDS; d++) {
        const int np = (S.n_rounds[1] + d - 1) / d, nd = (S.n_rounds[2] + d - 1) / d;
        if (np + nd + 1 > MZ_SP_MAX_SETS) continue;
        const int pb = sp_place(S, 1, np, 0, 0);
        const int db = sp_place(S, 2, nd, pb, np);
        const int rb = sp_place_linear(S, 0, pb, np + nd);      // over the dynamics area: the representation runs before the first dynamics pass
        S.total_sets = np + nd + 1; S.divisor = d;
        S.warea_bytes = pb + (db > rb ? db : rb);
        for (S.pbc_smem = 1; S.pbc_smem >= 0; S.pbc_smem--)
            if (mz_sp_smem_bytes(S.warea_bytes, S.bias_floats, S.total_rounds, P.hidden_pad, P.S, S.pbc_smem) <= smem_limit) return;
    }
    S.ok = 0;
}
// reference-order blob -> per layer a bf16 hi block (round to nearest) followed by a bf16 lo block (w - hi, round to nearest), each a
// [rows8(out) x 64] K-major SWIZZLE_128B A-operand tile (tc_tile_offset); biases fp32, 64 per layer
inline void pack_weights_sp(const mz_params &P, const mz_sp_plan &S, const float *src, std::vector<uint16_t> &image, std::vector<float> &bias) {
    image.assign((size_t)S.image_bytes / 2 + 8, 0); bias.assign((size_t)S.bias_floats, 0.0f);
    for (int i = 0; i < P.n_layers; i++) {
        const mz_layer &l = P.layers[i];
        for (int o = 0; o < l.out; o++) {
            for (int k = 0; k < l.in; k++) {
                const float w = src[l.src_w_off + k * l.out + o];
                const uint16_t hi = f2bf16(w), lo = f2bf16(w - bf16_to_f(hi));
                image[(size_t)(S.w_off[i] + tc_tile_offset(o, k)) / 2] = hi;
                image[(size_t)(S.w_off[i] + S.w_bytes[i] + tc_tile_offset(o, k)) / 2] = lo;
            }
            bias[(size_t)i * 64 + o] = src[l.src_b_off + o];
        }
    }
}

// ---- learner on the tensor cores: backward rounds (mz_learner_tc.cuh) ------------------------------------------------------------
inline mz_lr_bjob lr_bjob(const mz_params &P, const mz_lr_plan &L, int l0, int src0, int l1, int src1, int dst, int f32_off, int rows, int mask, int discard) {
    mz_lr_bjob j; memset(&j, 0, sizeof(j));
    j.a_off[0] = 0; j.a_off[1] = -1; j.f32_off = f32_off;
    j.layer[0] = (int16_t)l0; j.layer[1] = (int16_t)l1; j.src_tile[0] = (int16_t)src0; j.src_tile[1] = (int16_t)src1; j.dst_tile = (int16_t)dst;
    j.ks[0] = (int16_t)((P.layers[l0].out + 15) / 16); j.ks[1] = (int16_t)(l1 >= 0 ? (P.layers[l1].out + 15) / 16 : 0);
    j.rows = (int16_t)rows; j.mask = (int16_t)mask; j.perm = (int16_t)L.fwd_perm[l0]; j.discard = (int16_t)discard;
    return j;
}
inline void lr_emit(mz_lr_plan &L, const mz_lr_bjob *j0, const mz_lr_bjob *j1) {
    if (L.btotal_rounds >= MZ_LR_MAX_ROUNDS) { L.ok = 0; return; }
    mz_lr_bround &R = L.bround[L.btotal_rounds++];
    memset(&R, 0, sizeof(R));
    R.job[0] = *j0; R.njobs = 1;
    if (j1) { R.job[1] = *j1; R.njobs = 2; }
}
// Backward rounds of one network, last layer first.  Six 4 KB tiles per group: head 1 walks tiles 0 <-> 1, head 2 tiles 2 <-> 3 (in
// lock-step, aligned so that both reach their first layer together), the merged gradient of the trunk output lands in tile 4 and the
// trunk walks 4 <-> 5.  f32_off: where the gradient w.r.t. the network input goes (-1: not needed -- the representation).
inline void lr_build_net(const mz_params &P, mz_lr_plan &L, int net, int f32_off, int in_rows) {
    const mz_net &N = P.nets[net];
    const int f = N.first, nt = N.n_trunk, n1 = N.n_h1, n2 = N.n_h2;
    L.bfirst[net] = L.btotal_rounds;
    auto relu_below = [&](int l) { return l > f && P.layers[(l == f + nt || l == f + nt + n1) ? f + nt - 1 : l - 1].act == MZ_ACT_RELU ? 1 : 0; };
    int cur;
    if (n1 == 0) {
        L.start_tile[net][0] = 0; L.start_layer[net][0] = f + nt - 1; L.start_tile[net][1] = -1; L.start_layer[net][1] = -1;
        cur = 0;
    } else {
        const int fa = f + nt, fb = fa + n1;
        L.start_tile[net][0] = 0; L.start_layer[net][0] = fa + n1 - 1; L.start_tile[net][1] = 2; L.start_layer[net][1] = fb + n2 - 1;
        if (L.fwd_perm[fa] != L.fwd_perm[fb]) L.ok = 0;
        int ca = 0, cb = 2;
        const int la = n1 - 1, lb = n2 - 1, maxl = la > lb ? la : lb;
        for (int i = 0; i < maxl; i++) {
            const bool ha = i >= maxl - la, hb = i >= maxl - lb;
            mz_lr_bjob ja, jb;
            if (ha) { const int l = fa + n1 - 1 - (i - (maxl - la)); ja = lr_bjob(P, L, l, ca, -1, -1, ca ^ 1, -1, P.layers[l].in, relu_below(l), 0); ca ^= 1; }
            if (hb) { const int l = fb + n2 - 1 - (i - (maxl - lb)); jb = lr_bjob(P, L, l, cb, -1, -1, cb == 2 ? 3 : 2, -1, P.layers[l].in, relu_below(l), 0); cb = cb == 2 ? 3 : 2; }
            if (ha && hb) lr_emit(L, &ja, &jb); else lr_emit(L, ha ? &ja : &jb, nullptr);
        }
        mz_lr_bjob jm = lr_bjob(P, L, fa, ca, fb, cb, 4, -1, P.layers[fa].in, relu_below(fa), 0);
        lr_emit(L, &jm, nullptr);
        cur = 4;
    }
    for (int i = nt - 1; i >= 1; i--) {
        const int d = n1 == 0 ? (cur ^ 1) : (cur == 4 ? 5 : 4);
        mz_lr_bjob j = lr_bjob(P, L, f + i, cur, -1, -1, d, -1, P.layers[f + i].in, relu_below(f + i), 0);
        lr_emit(L, &j, nullptr);
        cur = d;
    }
    { mz_lr_bjob j = lr_bjob(P, L, f, cur, -1, -1, -1, f32_off, in_rows, 0, f32_off < 0 ? 1 : 0); lr_emit(L, &j, nullptr); }
    L.bn_rounds[net] = L.btotal_rounds - L.bfirst[net];
    for (int h = 0; h < 2; h++) L.start_perm[net][h] = L.start_layer[net][h] >= 0 ? L.fwd_perm[L.start_layer[net][h]] : 0;
}
inline int lr_place(mz_lr_plan &L, const mz_sp_plan &S, int net, int base, int set) {
    int off = base;
    for (int r = L.bfirst[net]; r < L.bfirst[net] + L.bn_rounds[net]; r++) {
        mz_lr_bround &R = L.bround[r];
        R.set = (int16_t)set; R.next = -1; R.per_pass = 0; R.ord = 0; R.ncopy = 0;
        for (int j = 0; j < R.njobs; j++) for (int t = 0; t < 2; t++) {
            const int l = R.job[j].layer[t];
            if (l < 0 || R.job[j].discard) continue;
            R.job[j].a_off[t] = off;
            mz_sp_copy &c = R.copy[R.ncopy++]; c.src_off = S.w_off[l]; c.bytes = S.w_bytes[l]; c.dst_off = off; c.pad_ = 0;
            off += S.w_bytes[l];
        }
    }
    L.bset_first[net] = set; L.bn_sets[net] = 1;
    return off - base;
}
// dh buffers of the backward pass: float offsets in the learner kernel's gradient area ([feature][MZ_SP_OS], hidden_pad rows each)
inline void build_lr_plan(const mz_params &P, const mz_sp_plan &S, mz_lr_plan &L) {
    memset(&L, 0, sizeof(L));
    L.ok = S.ok;
    if (!L.ok) return;
    L.n_eval = P.K > 0 ? P.K : 1;
    for (int n = 0; n < 3; n++) L.layers_in_net[n] = P.nets[n].n_trunk + P.nets[n].n_h1 + P.nets[n].n_h2;
    L.slot_base[0] = 0; L.slot_base[1] = L.layers_in_net[0]; L.slot_base[2] = L.slot_base[1] + L.n_eval * L.layers_in_net[1];
    L.slots_per_cta = L.slot_base[2] + L.n_eval * L.layers_in_net[2];
    for (int r = 0; r < S.total_rounds; r++) for (int j = 0; j < S.round[r].njobs; j++) L.fwd_perm[S.round[r].job[j].layer] = S.round[r].job[j].perm;
    lr_build_net(P, L, 0, -1, P.stack_size);
    lr_build_net(P, L, 1, 0, P.hidden);                                  // d loss / d h_e through prediction: rows [0, hidden_pad)
    lr_build_net(P, L, 2, P.hidden_pad * MZ_SP_OS, P.hidden);            // ... through dynamics (the state rows of its input; the action plane's gradient is not needed)
    if (!L.ok) return;
    const int pb = lr_place(L, S, 1, 0, 0), db = lr_place(L, S, 2, pb, 1), rb = lr_place(L, S, 0, pb, 2);
    L.btotal_sets = 3;
    L.bwarea_bytes = pb + (db > rb ? db : rb);
    if (L.bwarea_bytes > S.warea_bytes) L.ok = 0;                        // the backward weights (hi blocks only) must fit the forward's weight area
}

// Flux.glorot_uniform (un-vendored): (rand(Float32,out,in) .- 0.5f0) .* sqrt(24f0/(in+out)); bias zeros.  The reference
// never seeds it (Constructors.jl:19); contract: element i of layer l of net n = Philox(seed, INIT, n, l, i/4)[i%4].
inline void init_weights(const mz_params &P, uint64_t seed, float *src) {
    for (int n = 0; n < 3; n++) {
        int first = P.nets[n].first, cnt = P.nets[n].n_trunk + P.nets[n].n_h1 + P.nets[n].n_h2;
        for (int li = 0; li < cnt; li++) {
            const mz_layer &l = P.layers[first + li];
            float scale = sqrtf(24.0f / (float)(l.in + l.out));
            int nw = l.in * l.out;
            for (int i = 0; i < nw; i += 4) {
                mz_u4 r = mz_philox(seed, MZ_STREAM_INIT, (uint32_t)n, (uint32_t)li, (uint32_t)(i / 4), 0);
                uint32_t rr[4] = {r.x, r.y, r.z, r.w};
                for (int j = 0; j < 4 && i + j < nw; j++) src[l.src_w_off + i + j] = (mz_u32_to_unit(rr[j]) - 0.5f) * scale;
            }
            for (int o = 0; o < l.out; o++) src[l.src_b_off + o] = 0.0f;
            if (l.bn) for (int o = 0; o < l.out; o++) { src[l.src_b_off + l.out + o] = 0.0f; src[l.src_b_off + 2 * l.out + o] = 1.0f; src[l.src_b_off + 3 * l.out + o] = 0.0f; src[l.src_b_off + 4 * l.out + o] = 1.0f; }   // Flux.BatchNorm(out): beta, gamma, mu, sigma2
        }
    }
}

// Backward program of one 32-sample tile for grad_mode = MZ_GRAD_BPTT (kernel: mz_k_learn_bptt).  Follows the unroll
// of Learning.jl:347-370 backwards: rows K..1 of the prediction net on group 0, dynamics steps K..1 on group 1, one
// lock-step per unroll step (the gradient w.r.t. h_{i-1} needs both), then the representation net.  Rows 0 and 1 of the
// predictions are the same forward evaluation prediction(h_0) (Q19), so their loss gradients are summed before one
// backward walk (the backward pass is linear in the upstream gradient).
struct bptt_program { mz_bptt_plan plan; std::vector<mz_bstage> stages[2]; };

inline void bptt_chain(const mz_params &P, const mz_bptt_plan &pl, std::vector<mz_bstage> &out, int eval_base, int first_layer, int n,
                       int in_prev_act, int dz_first, int pre, int row, int merge0, int dx_last_buf, int dx_last_mode, float dx_last_scale,
                       uint64_t &used) {
    int cur = dz_first;
    for (int j = n - 1; j >= 0; j--) {
        mz_bstage s; memset(&s, 0, sizeof(s));
        s.layer = (int16_t)(first_layer + j); s.row = (int16_t)row;
        s.x_off = eval_base + pl.x_off[first_layer + j];
        s.dz_buf = (uint8_t)cur;
        s.pre = (uint8_t)(j == n - 1 ? pre : MZ_PRE_NONE); s.merge0 = (uint8_t)(j == n - 1 ? merge0 : 0);
        if (j > 0) { s.dx_buf = (uint8_t)(cur == MZ_BUF_Z0 ? MZ_BUF_Z1 : MZ_BUF_Z0); s.dx_mode = MZ_DX_STORE; s.prev_act = (uint8_t)P.layers[first_layer + j - 1].act; s.dx_scale = 1.0f; }
        else { s.dx_buf = (uint8_t)dx_last_buf; s.dx_mode = (uint8_t)dx_last_mode; s.prev_act = (uint8_t)in_prev_act; s.dx_scale = dx_last_scale; }
        s.first = (uint8_t)(((used >> (first_layer + j)) & 1ull) ? 0 : 1);
        used |= 1ull << (first_layer + j);
        out.push_back(s);
        cur = s.dx_buf;
    }
}

inline const char *build_bptt(const mz_params &P, bptt_program &bp) {
    mz_bptt_plan &pl = bp.plan; memset(&pl, 0, sizeof(pl));
    bp.stages[0].clear(); bp.stages[1].clear();
    if (P.K + 2 > MZ_MAX_BSTEPS) return "too many unroll steps for the backward program";
    for (int n = 0; n < 3; n++) {
        const mz_net &N = P.nets[n];
        int off = ((P.layers[N.first].in + 3) & ~3) * 32;
        int cnt = N.n_trunk + N.n_h1 + N.n_h2;
        for (int i = 0; i < cnt; i++) {
            int l = N.first + i;
            pl.y_off[l] = off; off += P.layers[l].out_pad * 32;
            if (i == 0) pl.x_off[l] = 0;
            else if (i == N.n_trunk || i == N.n_trunk + N.n_h1) pl.x_off[l] = pl.y_off[N.first + N.n_trunk - 1];
            else pl.x_off[l] = pl.y_off[l - 1];
        }
        pl.net_block[n] = off;
    }
    pl.n_pred_evals = P.K > 0 ? P.K : 1;
    pl.net_base[0] = 0; pl.net_base[1] = pl.net_block[0]; pl.net_base[2] = pl.net_base[1] + pl.n_pred_evals * pl.net_block[1];
    pl.tile_floats = pl.net_base[2] + P.K * pl.net_block[2];
    pl.rewards = P.intermediate_rewards ? 1 : 0;
    const mz_net &NR = P.nets[0], &NP = P.nets[1], &ND = P.nets[2];
    const int trunk_act_p = P.layers[NP.first + NP.n_trunk - 1].act, trunk_act_d = P.layers[ND.first + ND.n_trunk - 1].act;
    uint64_t used = 0;
    int step = 0;
    const int nrows = P.K > 0 ? P.K : 1;
    for (int s = 0; s < nrows; s++, step++) {
        // group 0: prediction row i (evaluation e = prediction(h_e), e = i - 1; row 0 shares evaluation 0)
        const int i = P.K > 0 ? P.K - s : 0, e = i > 0 ? i - 1 : 0, merge0 = (P.K > 0 && i == 1) ? 1 : 0;
        const int pbase = pl.net_base[1] + e * pl.net_block[1];
        bptt_chain(P, pl, bp.stages[0], pbase, NP.first + NP.n_trunk, NP.n_h1, trunk_act_p, MZ_BUF_Z0, MZ_PRE_VALUE, i, merge0, MZ_BUF_TA, MZ_DX_STORE, 1.0f, used);
        bptt_chain(P, pl, bp.stages[0], pbase, NP.first + NP.n_trunk + NP.n_h1, NP.n_h2, trunk_act_p, MZ_BUF_Z0, MZ_PRE_POLICY, i, merge0, MZ_BUF_TA, MZ_DX_ACCUM, 1.0f, used);
        bptt_chain(P, pl, bp.stages[0], pbase, NP.first, NP.n_trunk, MZ_ACT_ID, MZ_BUF_TA, MZ_PRE_NONE, i, 0, MZ_BUF_DHP, MZ_DX_STORE, 1.0f, used);
        pl.step_end[0][step] = (int32_t)bp.stages[0].size();
        // group 1: dynamics step i (produced h_i and r_i from h_{i-1}); h_K feeds nothing, so step K has no state-head gradient
        if (P.K > 0) {
            const int dbase = pl.net_base[2] + (i - 1) * pl.net_block[2];
            const bool state = i < P.K, reward = P.intermediate_rewards != 0;
            if (state) bptt_chain(P, pl, bp.stages[1], dbase, ND.first + ND.n_trunk, ND.n_h1, trunk_act_d, MZ_BUF_DH, MZ_PRE_NONE, i, 0, MZ_BUF_TA, MZ_DX_STORE, 1.0f, used);
            if (reward) bptt_chain(P, pl, bp.stages[1], dbase, ND.first + ND.n_trunk + ND.n_h1, ND.n_h2, trunk_act_d, MZ_BUF_Z0, MZ_PRE_REWARD, i, 0, MZ_BUF_TA, state ? MZ_DX_ACCUM : MZ_DX_STORE, 1.0f, used);
            if (state || reward) {   // make_dynamics_input: state * 2.0f0 (Learning.jl:299)
                bptt_chain(P, pl, bp.stages[1], dbase, ND.first, ND.n_trunk, MZ_ACT_ID, MZ_BUF_TA, MZ_PRE_NONE, i, 0, MZ_BUF_DHD, MZ_DX_STORE, 2.0f, used);
                pl.dhd_valid[step] = 1;
            }
        }
        pl.step_end[1][step] = (int32_t)bp.stages[1].size();
    }
    // representation (group 0): upstream = d loss / d h_0 in DH
    {
        int cur = MZ_BUF_DH;
        for (int j = NR.n_trunk - 1; j >= 0; j--) {
            mz_bstage s; memset(&s, 0, sizeof(s));
            s.layer = (int16_t)(NR.first + j); s.x_off = pl.net_base[0] + pl.x_off[NR.first + j]; s.dz_buf = (uint8_t)cur;
            if (j > 0) { s.dx_buf = (uint8_t)(cur == MZ_BUF_Z0 ? MZ_BUF_Z1 : MZ_BUF_Z0); s.dx_mode = MZ_DX_STORE; s.prev_act = (uint8_t)P.layers[NR.first + j - 1].act; s.dx_scale = 1.0f; }
            s.first = 1; used |= 1ull << (NR.first + j);
            bp.stages[0].push_back(s);
            cur = s.dx_buf;
        }
        pl.step_end[0][step] = (int32_t)bp.stages[0].size(); pl.step_end[1][step] = (int32_t)bp.stages[1].size();
        step++;
    }
    pl.n_steps = step;
    pl.n_stages[0] = (int32_t)bp.stages[0].size(); pl.n_stages[1] = (int32_t)bp.stages[1].size();
    pl.dead_layers = ~used & ((P.n_layers >= 64 ? 0ull : (1ull << P.n_layers)) - 1ull);
    return nullptr;
}

// ParameterSchedulers.Cos(l0=1e-4, l1=1e-1, period=10) (Learning.jl:319), 1-based step.
inline double cos_schedule(int64_t t) {
    double l0 = 1e-4, l1 = 1e-1, period = 10.0;
    double g = (1.0 + cos(2.0 * 3.14159265358979323846 * (double)(t - 1) / period)) / 2.0;
    return fabs(l0 - l1) * g + (l0 < l1 ? l0 : l1);
}

}  // namespace mzh
