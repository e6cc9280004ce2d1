// mz_common.h -- scalar building blocks shared by every kernel of libmuzero_b200: counter-based RNG,
// the fp32 math contract, game rules, observation stacking, and the per-tree MCTS operations
// (PUCT select with min-max normalised Q, expansion, discounted backup) over a flat node pool.
//
// Everything here is MZ_HD (__host__ __device__) and free of CUDA-only intrinsics so that the same code
// can be compiled by g++ into tests/host_harness and checked against the oracle on the CPU before it
// ever runs on a GPU.  The product itself only ever runs it on the device.
//
// Reference behaviour is cited as file:line under /root/reference (deveshjawla/MuZero.jl).
#pragma once
#include <stdint.h>
#include <math.h>
#include <string.h>
#include "../../include/muzero_b200.h"

#if defined(__CUDACC__)
#define MZ_HD __host__ __device__ __forceinline__
#else
#define MZ_HD static inline
#endif

#define MZ_MAX_LAYERS 40
#define MZ_MAX_WIDTH 64   /* width_hidden of the fp32 SIMT path (reference: 64) */

enum { MZ_STREAM_TIE = 1, MZ_STREAM_ACTION = 2, MZ_STREAM_DIRICHLET = 3, MZ_STREAM_REPLAY = 4, MZ_STREAM_ABSORB = 5, MZ_STREAM_INIT = 7, MZ_STREAM_OPPONENT = 8 };
enum { MZ_ACT_ID = 0, MZ_ACT_RELU = 1, MZ_ACT_TANH = 2 };

// ------------------------------------------------------------------------------------------------
// Philox4x32-10.  All randomness of the path is keyed (seed, stream) x counter so results do not depend
// on how games are batched or sharded (the reference uses an unseeded global RNG / MersenneTwister(1234),
// src/SelfPlay.jl:152,164).
// ------------------------------------------------------------------------------------------------
struct mz_u4 { uint32_t x, y, z, w; };
MZ_HD mz_u4 mz_philox(uint64_t seed, uint32_t stream, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ stream;
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    mz_u4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
    return o;
}
MZ_HD float mz_u32_to_unit(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }
MZ_HD uint32_t mz_u32_below(uint32_t x, uint32_t n) { return (uint32_t)(((uint64_t)x * n) >> 32); }

// ------------------------------------------------------------------------------------------------
// fp32 math contract: every multiply-add that is fused is an explicit fmaf(); everything else is a
// separately rounded IEEE op (device code is compiled with -fmad=false, host with -ffp-contract=off).
// ------------------------------------------------------------------------------------------------
MZ_HD float mz_bits2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
MZ_HD uint32_t mz_f2bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

MZ_HD float mz_expf(float x) {
    x = x > 88.0f ? 88.0f : x;
    x = x < -87.0f ? -87.0f : x;
    float fn = rintf(x * 1.44269504088896341f);
    float r = fmaf(fn, -0.693359375f, x);
    r = fmaf(fn, 2.12194440e-4f, r);
    float p = 1.9875691500e-4f;
    p = fmaf(p, r, 1.3981999507e-3f);
    p = fmaf(p, r, 8.3334519073e-3f);
    p = fmaf(p, r, 4.1665795894e-2f);
    p = fmaf(p, r, 1.6666665459e-1f);
    p = fmaf(p, r, 5.0000001201e-1f);
    float r2 = r * r;
    float y = fmaf(p, r2, r) + 1.0f;
    int n = (int)fn;
    return y * mz_bits2f((uint32_t)(n + 127) << 23);
}
MZ_HD float mz_logf(float x) {
    uint32_t u = mz_f2bits(x);
    int e = (int)((u >> 23) & 0xff) - 126;
    float m = mz_bits2f((u & 0x007fffffu) | 0x3f000000u);
    if (m < 0.707106781186547524f) { e -= 1; m = (m + m) - 1.0f; } else { m = m - 1.0f; }
    float z = m * m;
    float y = 7.0376836292e-2f;
    y = fmaf(y, m, -1.1514610310e-1f);
    y = fmaf(y, m, 1.1676998740e-1f);
    y = fmaf(y, m, -1.2420140846e-1f);
    y = fmaf(y, m, 1.4249322787e-1f);
    y = fmaf(y, m, -1.6668057665e-1f);
    y = fmaf(y, m, 2.0000714765e-1f);
    y = fmaf(y, m, -2.4999993993e-1f);
    y = fmaf(y, m, 3.3333331174e-1f);
    y = (y * m) * z;
    float fe = (float)e;
    y = fmaf(fe, -2.12194440e-4f, y);
    y = fmaf(z, -0.5f, y);
    float r = m + y;
    r = fmaf(fe, 0.693359375f, r);
    return r;
}
MZ_HD float mz_tanhf(float x) {
    float z = fabsf(x);
    if (z > 44.0f) return x > 0.0f ? 1.0f : -1.0f;
    if (z >= 0.625f) {
        float s = mz_expf(z + z);
        z = 1.0f - 2.0f / (s + 1.0f);
        return x < 0.0f ? -z : z;
    }
    float w = x * x;
    float p = -5.70498872745e-3f;
    p = fmaf(p, w, 2.06390887954e-2f);
    p = fmaf(p, w, -5.37397155531e-2f);
    p = fmaf(p, w, 1.33314422036e-1f);
    p = fmaf(p, w, -3.33332819422e-1f);
    return fmaf(p * w, x, x);
}
MZ_HD float mz_pow_contract(float x, float e) {   // visit_counts .^ (1/T), src/SelfPlay.jl:301
    if (x == 0.0f) return 0.0f;
    if (e == rintf(e) && e >= 1.0f && e <= 16.0f) {
        float r = x;
        for (int i = 1; i < (int)e; i++) r = r * x;
        return r;
    }
    return mz_expf(e * mz_logf(x));
}
MZ_HD float mz_activate(float v, int act) {
    if (act == MZ_ACT_RELU) return v > 0.0f ? v : 0.0f;     // NNlib relu(x) = max(0, x)
    if (act == MZ_ACT_TANH) return mz_tanhf(v);
    return v;
}

// ------------------------------------------------------------------------------------------------
// Device-side parameter block (built on the host from mz_config; lives in __constant__ memory).
// ------------------------------------------------------------------------------------------------
struct mz_layer {            // one Dense layer in the padded device layout
    int32_t in, out, out_pad, act;
    int32_t w_off, b_off;    // float offsets into the padded device blob (16-byte aligned)
    int32_t src_w_off, src_b_off; // float offsets into the reference-order blob
    int32_t floats;          // in*out_pad + out_pad (+ 4 * out_pad: BatchNorm): one contiguous bulk copy
    int32_t bn;              // 1: followed by BatchNorm (FeedForwardHP.use_batch_norm): device block = W | b | beta | gamma | mu | sigma2 (out_pad floats each);
                             // reference-order blob: W, b, beta[out], gamma[out], mu[out], sigma2[out]
};
// BatchNorm in test mode (Flux 0.12.4): gamma .* (x .- mu) ./ sqrt.(sigma2 .+ 1f-5) .+ beta, every operation rounded on its own
MZ_HD float mz_batchnorm(float v, float beta, float gamma, float mu, float var) { return ((gamma * (v - mu)) / sqrtf(var + 1e-5f)) + beta; }
struct mz_net {              // trunk + two heads (representation has no heads)
    int32_t n_trunk, n_h1, n_h2, first;  // layers [first, first+n_trunk) trunk, then h1, then h2
};
struct mz_params {
    int32_t game, W, H, C, A, P;               // P = num_players
    int32_t stacked, max_moves, Tmax, S, K, td;
    int32_t cells, obs_size, planes, stack_size, sa_size, hidden, hidden_pad;
    int32_t tie_mode, pb_c_base, intermediate_rewards, batch_size;
    int32_t nodes_per_tree, tree_stride_bytes, nodeB_off_bytes, hidden_off_bytes;
    float pb_c_init, discount, dirichlet_alpha, exploration_eps;
    uint64_t seed;
    int32_t order[MZ_MAX_A];                   // Dict iteration order (1-based actions)
    float act_plane_play[MZ_MAX_A + 1];        // Float32(Float64(a)/A)      (src/SelfPlay.jl:8-9)
    float act_plane_learn[MZ_MAX_A + 1];       // Float32(a) / Float32(A)    (src/Learning.jl:294)
    float disc_pow[72];                        // conf.discount^i as Julia computes Float32^Int
    int32_t n_layers, total_floats, n_params, per;   // per: conf.PER
    int32_t per_alpha;
    int32_t temp_threshold;                    // conf.temperature_threshold (SelfPlay.jl:344-346), -1 = nothing
    int32_t arena_player, arena_opponent;      // competitive play (SelfPlay.jl:421-435): the side MuZero plays (0 = self-play) and who moves for the other
    int32_t arena_tally;                       // the side whose wins / draws / losses mz_k_save_refill counts (0 = none)
    mz_net nets[3];
    mz_layer layers[MZ_MAX_LAYERS];
    // tensor-core (MZ_NN_BF16_TC) weight image: per layer a [rows8(out) x 64] bf16 tile in the UMMA K-major
    // SWIZZLE_128B shared-memory layout, pre-swizzled on the host so one bulk copy per network stages it
    int32_t tc_a_off[MZ_MAX_LAYERS];   // byte offset of the layer's A tile inside the image (1024-aligned)
    int32_t tc_ksteps[MZ_MAX_LAYERS];  // ceil(in / 16) tcgen05.mma instructions per layer
    int32_t tc_net_off[4];             // byte offset of each network's block; [3] = total image bytes
    int32_t tc_bias_off[MZ_MAX_LAYERS];// float offset of the layer's bias inside the bias block
    int32_t tc_bias_floats, tc_ok;
    int32_t fin_tag, tc_pad_;          // fin_tag: parity of the self-play iteration (set per launch): a slot finished in iteration k carries status MZ_SLOT_FINISHED + (k & 1),
                                       // so that the save / refill kernels of iteration k can run beside the search of iteration k + 1 without taking its finishes
};

// ------------------------------------------------------------------------------------------------
// Split-precision network path (nn_mode = MZ_NN_SPLIT_MMA; mz_sp.cuh, mz_kernels_sp.cuh): every Dense layer on the tcgen05 tensor
// cores with BOTH operands split into bf16 hi + lo parts, x = hi + lo, and the three products W_hi X_hi + W_lo X_hi + W_hi X_lo
// accumulated in fp32 in TMEM: 16 mantissa bits per operand.  The host compiles the three networks into ROUNDS (up to two independent
// layers that are issued together: e.g. the first layers of the two heads of a network) and decides where each round's weights live:
// hi + lo images of prediction + dynamics (240 KB) do not fit an SM next to the activation tiles, so the rounds of a network share
// WEIGHT SETS -- shared-memory regions that alternate between the rounds assigned to them (round r and round r + n_sets): when a round's
// MMAs have completed, its set is refilled by TMA with the weights of the round that uses the set next.  The sequence is the same in
// every simulation, so addresses (and UMMA descriptors) are static and the refill runs half a network pass ahead of its use.
// ------------------------------------------------------------------------------------------------
#define MZ_SP_MAX_ROUNDS 40
#define MZ_SP_MAX_SETS 48
#define MZ_SP_TILE_BYTES 4096                      // one operand tile: [64 k][32 trees] bf16, N-major, SWIZZLE_64B
#define MZ_SP_OS 36                               // floats per feature row of the fp32 network outputs [feature][tree]: 36 = 4 mod 32 keeps the
                                                   // trees' reads (8 lanes per tree, lane = feature) free of bank conflicts; 16-byte aligned rows
#define MZ_SP_TILES_PER_GROUP 3                    // input / ping / pong, each as a hi tile followed by a lo tile
struct mz_sp_job {
    int32_t a_off;                                  // byte offset of the layer's hi weight block in the CTA's weight area (lo block = + a_bytes)
    int32_t a_bytes;                                // bytes of one block: rows8(out) x 128
    int32_t bias_off;                               // float offset of the layer's bias in the bias block
    int32_t f32_off;                                // final layer: float offset of its fp32 output in the output area, else -1
    int16_t src_tile, dst_tile;                     // operand tiles of the group (0 = input, 1, 2); dst_tile = -1 for a final layer
    int16_t ks, out, act, perm;                     // k-steps, real outputs, activation, column order of the input tile (0 natural, 1 permuted)
    int16_t layer, pad_[3];
};
struct mz_sp_copy { int32_t src_off, bytes, dst_off, pad_; };   // global image offset -> weight-area offset
struct mz_sp_round {
    mz_sp_job job[2];
    mz_sp_copy copy[2];
    int16_t njobs, ncopy;
    int16_t set;                                    // weight set = mbarrier index
    int16_t next;                                   // global index of the round whose weights replace this round's when it has completed (-1: none)
    int16_t per_pass, ord;                          // fills of the set per pass over the network (0: loaded once) and which of them this round consumes
};
struct mz_sp_plan {
    int32_t first[3], n_rounds[3];                  // per network (representation, prediction, dynamics): rounds [first, first + n)
    int32_t set_first[3], n_sets[3];                // per network: its weight sets (the representation has one, loaded once, over the dynamics area)
    int32_t total_rounds, total_sets;
    int32_t image_bytes, warea_bytes, bias_floats, divisor, ok, pbc_smem;
    int32_t tail;                                   // trailing rounds of the dynamics network without a reward job (the state head alone)
    int32_t out_off[4];                            // float offsets of value / logits / reward / hidden outputs in the output area
    int32_t w_off[MZ_MAX_LAYERS], w_bytes[MZ_MAX_LAYERS];   // image: hi block at w_off, lo block at w_off + w_bytes
    mz_sp_round round[MZ_SP_MAX_ROUNDS];
};

#define MZ_SP_RDESC_BYTES 128                       // sizeof(mz_sp_rdesc), the device form of a round (mz_sp.cuh)
#define MZ_SP_CTRL_BYTES 1024                       // mbarriers, TMEM slot, active-tree flags
// dynamic shared memory of a kernel on this path (the carve-up is mz_sp_carve in mz_sp.cuh)
// pbc_smem: the kernel keeps a compact copy of ucb_score's Float64 table (rows N = 0..S+1, entries n = 0..N) in shared memory
MZ_HD size_t mz_sp_smem_bytes(int warea_bytes, int bias_floats, int total_rounds, int hidden_pad, int S, int pbc_smem) {
    size_t tiles = (size_t)2 * MZ_SP_TILES_PER_GROUP * 2 * MZ_SP_TILE_BYTES;
    size_t bias = ((size_t)bias_floats * 4 + 127) & ~(size_t)127;
    size_t out = (size_t)(24 + hidden_pad) * MZ_SP_OS * 4;
    size_t tab = pbc_smem ? ((((size_t)S + 2) * ((size_t)S + 3) / 2) * 8 + 127) & ~(size_t)127 : 0;
    size_t path = (((size_t)S + 2) * 2 * 32 + 127) & ~(size_t)127;
    size_t prog = ((size_t)total_rounds * MZ_SP_RDESC_BYTES + 127) & ~(size_t)127;
    return 1024 + (size_t)warea_bytes + tiles + MZ_SP_CTRL_BYTES + bias + out + tab + path + prog;
}

// ------------------------------------------------------------------------------------------------
// Learner on the tensor cores (grad_mode = MZ_GRAD_BPTT with nn_mode = MZ_NN_SPLIT_MMA; mz_learner_tc.cuh).  32 samples per CTA.
//   forward   the rounds of mz_sp_plan (split precision); every round also stores the hi tile of each job's INPUT to global memory
//             (TMA bulk store): X[slot], slot = slot_base[net] + evaluation * layers(net) + (layer - first layer of net)
//   backward  per evaluation, last to first: dX = W^T dZ through BACKWARD ROUNDS (the hi weight block read as an M-major A operand,
//             bf16 operands), relu mask from X[slot], the result is the previous layer's dZ tile; every round stores its dZ input
//             tiles: dZ[slot].  The first layers of the two heads accumulate into one accumulator (the trunk output's gradient).
//   weights   a second kernel computes dW[layer] = sum over (CTA, evaluation) dZ[slot] X[slot]^T with the samples as the K dimension.
// ------------------------------------------------------------------------------------------------
#define MZ_LR_MAX_ROUNDS 40
struct mz_lr_bjob {
    int32_t a_off[2];                               // weight-area offsets of the hi blocks (two for the merge of the heads' first layers, else [1] = -1)
    int32_t f32_off;                                // first layer of a network: float offset of the fp32 input gradient in the output area, else -1
    int16_t layer[2];                               // the layer(s) whose input gradient this job computes
    int16_t src_tile[2], dst_tile;                  // 4 KB tiles of the group (0..5): dZ of layer[i]; dst = dZ of the layer below (-1: none)
    int16_t ks[2];                                  // k-steps = ceil(out / 16) of layer[i]
    int16_t rows;                                   // real rows of the result = inputs of layer[0]
    int16_t mask;                                   // 1: multiply by (X[slot of layer[0]] > 0) (the layer below ends in relu)
    int16_t perm;                                   // column order of the src tiles (= the forward tile order of layer[0]'s input)
    int16_t discard;                                // 1: the result is not needed (first layer of the representation): no MMA, only the dZ store
    int16_t pad_;
};
struct mz_lr_bround {
    mz_lr_bjob job[2];
    mz_sp_copy copy[4];                             // this round's hi weight blocks
    int16_t njobs, ncopy, set, next, per_pass, ord, pad_[2];
};
struct mz_lr_plan {
    int32_t ok, n_eval, slots_per_cta;
    int32_t slot_base[3], layers_in_net[3];
    int32_t bfirst[3], bn_rounds[3];                // backward rounds per network
    int32_t bset_first[3], bn_sets[3], btotal_rounds, btotal_sets, bwarea_bytes;
    int32_t start_tile[3][2], start_layer[3][2], start_perm[3][2];   // where the loss / hidden-state gradients are staged: tile, layer (-1: none), column order
    int32_t fwd_perm[MZ_MAX_LAYERS];                // column order of every layer's forward input tile
    mz_lr_bround bround[MZ_LR_MAX_ROUNDS];
};

// ------------------------------------------------------------------------------------------------
// Learner backward pass (grad_mode = MZ_GRAD_BPTT): host-built program of backward layer applications.
// One CTA = 32 samples; group 0 walks the prediction rows (and finally the representation), group 1 the
// dynamics steps, in lock-step "steps" separated by CTA barriers (see mz_learner_bptt.cuh).
// ------------------------------------------------------------------------------------------------
enum { MZ_BUF_Z0 = 0, MZ_BUF_Z1 = 1, MZ_BUF_TA = 2, MZ_BUF_DH = 3, MZ_BUF_DHP = 4, MZ_BUF_DHD = 5 };
enum { MZ_PRE_NONE = 0, MZ_PRE_VALUE = 1, MZ_PRE_POLICY = 2, MZ_PRE_REWARD = 3 };
enum { MZ_DX_NONE = 0, MZ_DX_STORE = 1, MZ_DX_ACCUM = 2 };
#define MZ_MAX_BSTEPS 40
struct mz_bstage {
    int16_t layer;        // index into mz_params::layers
    int16_t row;          // prediction row / dynamics step (1-based) the loss terms of `pre` belong to
    int32_t x_off;        // float offset of the layer's input activations inside the tile's activation block
    uint8_t dz_buf, dx_buf, dx_mode, prev_act;   // prev_act: activation of the layer that produced the input (applied to dX)
    uint8_t first, pre, merge0, pad_;            // first: this is the tile's first gradient contribution to the layer (store, not add)
    float dx_scale;
};
struct mz_bptt_plan {
    int32_t y_off[MZ_MAX_LAYERS];     // float offset of each layer's output inside its network's evaluation block
    int32_t x_off[MZ_MAX_LAYERS];     // float offset of each layer's input inside the block
    int32_t net_base[3], net_block[3];// activation block = [repr | pred evals | dyn evals]
    int32_t tile_floats, n_pred_evals, n_steps, rewards;
    int32_t n_stages[2];
    int32_t step_end[2][MZ_MAX_BSTEPS];   // exclusive end of each step's stages in the group's program
    uint8_t dhd_valid[MZ_MAX_BSTEPS];     // group 1 produced a dynamics-input gradient in this step
    uint64_t dead_layers;                 // layers that receive no data gradient at all (their partial sums are zero-filled)
};

// ------------------------------------------------------------------------------------------------
// ResNet networks on the tensor cores (net_type = MZ_NET_RESNET): host-built step program (mz_rn_host.h) executed by
// mz_kernels_rn.cuh.  Activations are bf16 tiles of 128 rows x 64 channels (rows = (tree, cell) pairs for the
// convolution towers, rows = trees for the dense heads), UMMA K-major SWIZZLE_128B; a step = up to 4 jobs (one MMA
// chain + epilogue each) sharing one staged weight block.
// ------------------------------------------------------------------------------------------------
#define MZ_RN_TILES 4
enum { MZ_RN_BUF_X0 = 0, MZ_RN_BUF_T0 = 4, MZ_RN_BUF_HV = 8, MZ_RN_BUF_HP = 9, MZ_RN_BUF_S0 = 10, MZ_RN_BUF_S1 = 11 };
enum { MZ_RN_EPI_TILE = 0, MZ_RN_EPI_HEAD = 1, MZ_RN_EPI_F32 = 2 };
enum { MZ_RN_F_PLANE = 1, MZ_RN_F_POOL = 2, MZ_RN_F_TREES = 4 };
enum { MZ_RN_OUT_V = 0, MZ_RN_OUT_L = 1, MZ_RN_OUT_R = 2 };
struct mz_rn_job {
    uint8_t a_buf, dst_buf, dst2_buf, skip_buf;   // buffer ids (0xff = none)
    uint8_t epi, n16, kblocks, act;
    uint8_t wg, acc, flags, nfa;                  // wg: warpgroup running the epilogue; acc: TMEM accumulator slot (64 columns each)
    uint8_t nfb, out, out_id, pad_;
    int32_t w_sub, p_sub;                         // byte offsets inside the step's staged block: B image; {S[64], T[64], E[64]} floats
    int32_t wref;                                 // host-side bookkeeping
};
struct mz_rn_step {
    int32_t w_off, w_bytes;                       // the step's block inside the global weight image
    uint8_t njobs, ntaps, tap, last;              // k x k convolutions: one step per tap, epilogue after the last
    int8_t dx, dy; uint8_t accumulate;            // tap: A = copy of a_buf shifted by (dx, dy) cells
    uint8_t rowlocal;                             // 1/2: every job is a (tree,cell)-tile job of warpgroup j on its own tile, so the warpgroups need not
                                                  // meet after the step (1), except before a step that is not row-local / the end of a range (2)
    mz_rn_job jobs[MZ_RN_TILES];
    int8_t wgjob[4];                              // the job warpgroup w runs the epilogue of (at most one per step), or -1
};
struct mz_rn_params {
    int32_t cells, nf, tpt, ntrees, rows_valid, node_bytes;
    int32_t planes, ksize, nvf, npf;
    int32_t prog_repr[2], prog_pred[2], prog_dyn[2], n_steps, smem_first;   // steps >= smem_first are copied to shared memory
    int32_t image_bytes, slot_bytes, hidden_off_bytes, tree_stride_bytes;
};

// ------------------------------------------------------------------------------------------------
// Games.  TicTacToe follows games/tictactoe/game.jl including its quirks (SURVEY Q14-Q16); boards are
// two bit masks (bit a-1 = cell of action a, column-major like CartesianIndices((3,3))[a]).
// MZ_GAME_CONNECT is the synthetic larger-board game of BASELINE.json config 4 (no reference code):
// H x W... see mz_connect_* below.
// ------------------------------------------------------------------------------------------------
struct mz_board { uint64_t p1, p2; int32_t player; };

MZ_HD bool mz_ttt_line(uint32_t b) {  // game.jl:106-113
    return ((b & 0x049u) == 0x049u) || ((b & 0x092u) == 0x092u) || ((b & 0x124u) == 0x124u) ||
           ((b & 0x007u) == 0x007u) || ((b & 0x038u) == 0x038u) || ((b & 0x1c0u) == 0x1c0u) ||
           ((b & 0x111u) == 0x111u) || ((b & 0x054u) == 0x054u);
}
// Connect game (synthetic, config 4): board of `W` rows x `H` columns in the (W,H,C) observation, a move
// drops a mark into column a (lowest free row); 4 in a row wins for the mover, clean termination.
MZ_HD bool mz_connect_has4(uint64_t b, int rows) {
    int s = rows + 1;  // padded column stride so vertical runs cannot wrap
    uint64_t m;
    m = b & (b >> 1);       if (m & (m >> 2)) return true;            // vertical
    m = b & (b >> s);       if (m & (m >> (2 * s))) return true;      // horizontal
    m = b & (b >> (s + 1)); if (m & (m >> (2 * (s + 1)))) return true; // diagonal /
    m = b & (b >> (s - 1)); if (m & (m >> (2 * (s - 1)))) return true; // diagonal \.
    return false;
}
// Connect boards are stored in the padded layout: bit (r + (rows+1)*c).
MZ_HD int mz_connect_height(uint64_t occ, int rows, int c) {
    uint64_t col = (occ >> ((rows + 1) * c)) & ((1ull << rows) - 1ull);
    int h = 0;
    while (col & 1ull) { h++; col >>= 1; }
    return h;
}

MZ_HD void mz_env_reset_b(const mz_params &P, mz_board &b) { b.p1 = 0; b.p2 = 0; b.player = 1; }  // game.jl:15-20

MZ_HD bool mz_env_win_side_to_move(const mz_params &P, const mz_board &b) {  // is_win ignores `player` (game.jl:102-104)
    return mz_ttt_line((uint32_t)(b.player == 1 ? b.p1 : b.p2));
}
MZ_HD bool mz_connect_last_mover_won(const mz_params &P, const mz_board &b) {
    return mz_connect_has4(b.player == 1 ? b.p2 : b.p1, P.W);
}
MZ_HD uint32_t mz_env_legal_b(const mz_params &P, const mz_board &b) {       // game.jl:35-43
    if (P.game == MZ_GAME_TICTACTOE) {
        if (mz_env_win_side_to_move(P, b)) return 0u;
        return (uint32_t)(~(b.p1 | b.p2)) & ((1u << P.cells) - 1u);
    }
    uint32_t m = 0;
    if (mz_connect_last_mover_won(P, b)) return 0u;
    for (int c = 0; c < P.A; c++) if (mz_connect_height(b.p1 | b.p2, P.W, c) < P.W) m |= 1u << c;
    return m;
}
MZ_HD void mz_env_step_b(const mz_params &P, mz_board &b, int action) {       // game.jl:45-52
    uint64_t bit;
    if (P.game == MZ_GAME_TICTACTOE) bit = 1ull << (action - 1);
    else { int c = action - 1; bit = 1ull << ((P.W + 1) * c + mz_connect_height(b.p1 | b.p2, P.W, c)); }
    if (b.player == 1) b.p1 |= bit; else b.p2 |= bit;
    b.player = b.player % P.P + 1;                                            // mod1(player+1, 2)
}
MZ_HD bool mz_env_full(const mz_params &P, const mz_board &b) {
    if (P.game == MZ_GAME_TICTACTOE) return ((uint32_t)(b.p1 | b.p2) & ((1u << P.cells) - 1u)) == ((1u << P.cells) - 1u);
    for (int c = 0; c < P.A; c++) if (mz_connect_height(b.p1 | b.p2, P.W, c) < P.W) return false;
    return true;
}
MZ_HD bool mz_env_terminated_b(const mz_params &P, const mz_board &b) {       // game.jl:85,128-139
    if (P.game == MZ_GAME_TICTACTOE) return mz_env_full(P, b) || mz_env_win_side_to_move(P, b);
    return mz_env_full(P, b) || mz_connect_last_mover_won(P, b);
}
MZ_HD int mz_env_reward_b(const mz_params &P, const mz_board &b, int player) { // game.jl:87-100 (winner is always 1, Q15)
    if (P.game == MZ_GAME_TICTACTOE) {
        if (!mz_env_terminated_b(P, b)) return 0;
        if (!mz_env_win_side_to_move(P, b)) return 0;
        return player == 1 ? 1 : -1;
    }
    if (!mz_connect_last_mover_won(P, b)) return 0;
    int last = b.player == 1 ? 2 : 1;
    return player == last ? 1 : -1;
}
// observation planes (player-1 marks, player-2 marks, empty), Julia (W,H,C) order: cell index fastest
MZ_HD float mz_env_obs_value(const mz_params &P, const mz_board &b, int plane, int cell) {
    int bit = cell;
    if (P.game == MZ_GAME_CONNECT) { int r = cell % P.W, c = cell / P.W; bit = r + (P.W + 1) * c; }
    int a = (int)((b.p1 >> bit) & 1ull), o = (int)((b.p2 >> bit) & 1ull);
    return plane == 0 ? (float)a : plane == 1 ? (float)o : (float)(!(a | o));
}
// get_stacked_observations (src/SelfPlay.jl:128-149): element k of the stacked observation at 1-based
// `index`; boards h1/h2 hold the boards BEFORE move i at [i-1]; the action plane is the RAW index (Q13).
MZ_HD float mz_stacked_value(const mz_params &P, const uint64_t *h1, const uint64_t *h2, const int32_t *acts, int index, int k) {
    int per = P.cells + P.obs_size;  // one (action plane + observation) group
    mz_board b; b.player = 1;
    if (k < P.obs_size) { b.p1 = h1[index - 1]; b.p2 = h2[index - 1]; return mz_env_obs_value(P, b, k / P.cells, k % P.cells); }
    int g = (k - P.obs_size) / per, r = (k - P.obs_size) % per;
    int past = index - 1 - g;   // 1-based past index
    if (past < 1) return 0.0f;
    if (r < P.cells) return (float)acts[past - 1];
    r -= P.cells;
    b.p1 = h1[past - 1]; b.p2 = h2[past - 1];
    return mz_env_obs_value(P, b, r / P.cells, r % P.cells);
}

// ------------------------------------------------------------------------------------------------
// Flat per-tree node pool.  Q7 (every expanded node gets children for the ROOT's legal set) makes the
// pool regular: expansion e (0 = root, 1..S = simulations) owns the child block [1+e*A, 1+(e+1)*A) and
// the hidden state slot e.  One 16-byte record per node:
//   node[n] = { x = visit_count (bits 0-11) | expansion id + 1 (bits 12-23) | doublings (bits 24-29),
//               y = value_sum, z = prior, w = reward }
// Everything the next selection level needs about a child (is it expanded, where are ITS children) travels with
// the record that was loaded to score it, so a selection level costs one dependent memory round trip.
// `doublings` implements make_state_action's in-place `state .*= 2` (Q6) as an exact power-of-two scale on read.
// ------------------------------------------------------------------------------------------------
struct alignas(16) mz_f4 { float x, y, z, w; };
struct mz_tree {
    mz_f4 *A;
    float *hidden;
};
MZ_HD mz_tree mz_tree_at(const mz_params &P, void *pool, int64_t tree) {
    char *base = (char *)pool + tree * (int64_t)P.tree_stride_bytes;
    mz_tree t; t.A = (mz_f4 *)base; t.hidden = (float *)(base + P.hidden_off_bytes);
    return t;
}
MZ_HD uint32_t mz_nx_pack(int visit, int exp_id, int dbl) { return (uint32_t)visit | ((uint32_t)(exp_id + 1) << 12) | ((uint32_t)dbl << 24); }
MZ_HD int mz_nx_visit(uint32_t x) { return (int)(x & 0xfffu); }
MZ_HD int mz_nx_exp(uint32_t x) { return (int)((x >> 12) & 0xfffu) - 1; }
MZ_HD int mz_nx_dbl(uint32_t x) { return (int)(x >> 24); }
MZ_HD uint32_t mz_node_x(const mz_f4 &r) { return mz_f2bits(r.x); }

struct mz_minmax { float mn, mx; };

// ucb_score (src/SelfPlay.jl:171-184): Float64 exploration term from integer-only tables
// (pbc0[N] = log2((N+base+1)/base) + init, sqrtN[N] = sqrt(N)), Float32 value term, Float32 result.
// `pbc` is the host-built table pbc[N * (S + 2) + n] = pbc0[N] * (sqrtN[N] / (double)(n + 1)): the same IEEE double operations in
// the same order, evaluated once on the host -- the device does no Float64 division (slow on this part) in the selection loop.
// `row` = the table row of the parent's visit count N (pbc + N * (S + 2), or the kernel's own compact copy of it)
MZ_HD float mz_ucb_row(const mz_params &P, const double *row, mz_f4 child, mz_minmax mm) {
    int n = mz_nx_visit(mz_f2bits(child.x));
    double pb_c = row[n];
    double prior_score = pb_c * (double)child.z;
    if (n > 0) {
        float nv = child.y / (float)n;                                    // node_value :76-82
        float q = child.w + P.discount * (P.P == 1 ? nv : -nv);
        float vs = (mm.mx > mm.mn) ? (q - mm.mn) / (mm.mx - mm.mn) : q;   // normalize_tree_value :33-39
        return (float)(prior_score + (double)vs);
    }
    return (float)(prior_score + 0.0);
}
MZ_HD float mz_ucb(const mz_params &P, const double *pbc, const double *unused_, int N, mz_f4 child, mz_minmax mm) {
    (void)unused_;
    return mz_ucb_row(P, pbc + N * (P.S + 2), child, mm);
}

// leaf of a selection: node indices, the leaf's prior (its record is rebuilt by expand), the parent's packed x word
struct mz_leaf { int node, parent, action, depth; float prior; uint32_t parent_x; };

// select_child loop of run_mcts (src/SelfPlay.jl:157-166, 261-268); records the path (root .. leaf) for the backup.
MZ_HD mz_leaf mz_tree_select(const mz_params &P, const mz_tree &t, const double *pbc0, const double *sqrtN, uint32_t legal,
                             mz_minmax mm, uint32_t game, uint32_t move, uint32_t sim, uint16_t *path) {
    mz_leaf L; L.node = 0; L.parent = 0; L.action = 0; L.depth = 0; L.prior = 0.0f; L.parent_x = 0;
    uint32_t x = mz_f2bits(t.A[0].x);
    path[0] = 0;
    while (mz_nx_exp(x) >= 0) {
        L.depth++;
        int base = 1 + mz_nx_exp(x) * P.A;
        int N = mz_nx_visit(x);
        float best = 0.0f; uint32_t tied = 0;
        for (int j = 0; j < P.A; j++) {
            int a = P.order[j];
            if (!((legal >> (a - 1)) & 1u)) continue;
            float s = mz_ucb(P, pbc0, sqrtN, N, t.A[base + a - 1], mm);
            if (tied == 0 || s > best) { best = s; tied = 1u << j; }
            else if (s == best) tied |= 1u << j;
        }
        int nt = 0; for (uint32_t m = tied; m; m &= m - 1) nt++;
        int pick = 0;
        if (nt > 1 && P.tie_mode == MZ_TIE_PHILOX) pick = (int)mz_u32_below(mz_philox(P.seed, MZ_STREAM_TIE, game, move, sim, (uint32_t)L.depth).x, (uint32_t)nt);
        uint32_t m = tied;
        for (int i = 0; i < pick; i++) m &= m - 1;
        int j = 0; while (!((m >> j) & 1u)) j++;
        L.action = P.order[j];
        L.parent = L.node; L.parent_x = x;
        L.node = base + L.action - 1;
        path[L.depth] = (uint16_t)L.node;
        mz_f4 c = t.A[L.node];
        x = mz_f2bits(c.x); L.prior = c.z;
    }
    return L;
}

// NNlib.softmax over n values in index order.
MZ_HD void mz_softmax(const float *x, int n, float *y) {
    float m = x[0];
    for (int i = 1; i < n; i++) m = x[i] > m ? x[i] : m;
    float s = 0.0f;
    for (int i = 0; i < n; i++) { y[i] = mz_expf(x[i] - m); s = s + y[i]; }
    for (int i = 0; i < n; i++) y[i] = y[i] / s;
}

// expand_node! (src/SelfPlay.jl:88-96): second softmax over the legal subset (ascending actions, Q1) of the
// already-softmaxed policy; children block e; the node (unvisited until the backup, prior `prior`) becomes expanded
// with reward r.
MZ_HD void mz_tree_expand(const mz_params &P, const mz_tree &t, int node, int e, uint32_t legal, const float *policy, float reward, float prior) {
    float sub[MZ_MAX_A], pv[MZ_MAX_A]; int n = 0;
    for (int a = 1; a <= P.A; a++) if ((legal >> (a - 1)) & 1u) sub[n++] = policy[a - 1];
    mz_softmax(sub, n, pv);
    int base = 1 + e * P.A; n = 0;
    for (int a = 1; a <= P.A; a++) {
        mz_f4 c; c.x = mz_bits2f(mz_nx_pack(0, -1, 0)); c.y = 0.0f; c.w = 0.0f;
        c.z = ((legal >> (a - 1)) & 1u) ? pv[n++] : 0.0f;
        t.A[base + a - 1] = c;
    }
    mz_f4 me; me.x = mz_bits2f(mz_nx_pack(0, e, 0)); me.y = 0.0f; me.z = prior; me.w = reward;
    t.A[node] = me;
}

// backpropagate! (src/SelfPlay.jl:190-217) over the recorded path, leaf -> root.  Two players: a node j steps
// above the leaf has node.to_play == to_play iff j is even; includes the dropped-bootstrap bug (Q8).
MZ_HD void mz_tree_backup(const mz_params &P, const mz_tree &t, const uint16_t *path, int depth, float value, mz_minmax &mm) {
    for (int j = 0; j <= depth; j++) {
        int node = path[depth - j];
        mz_f4 a = t.A[node];
        uint32_t x = mz_f2bits(a.x) + 1u;                                 // visit_count += 1 (low bits of the packed word)
        int vc = mz_nx_visit(x);
        bool same = (P.P == 1) || ((j % P.P) == 0);
        a.y = same ? a.y + value : a.y - value;
        a.x = mz_bits2f(x);
        t.A[node] = a;
        float u = a.w + P.discount * (a.y / (float)vc);
        mm.mn = mm.mn < u ? mm.mn : u;                                   // update_tree! :27-31
        mm.mx = mm.mx > u ? mm.mx : u;
        if (P.P == 1) value = a.w + P.discount * value;
        else value = same ? -a.w : a.w + P.discount * value;
    }
}

// Gamma(alpha) draws for the root Dirichlet noise (add_exploration_noise!, src/SelfPlay.jl:102-109).
// Contract (Distributions.jl is un-vendored): Marsaglia-Tsang on alpha+1 with polar normals, times
// u^(1/alpha), in Float32, from Philox(seed, DIRICHLET, game, move, child j, counter).
struct mz_rstream { uint64_t seed; uint32_t c0, c1, c2, ctr; uint32_t buf[4]; int have; };
MZ_HD uint32_t mz_rs_next(mz_rstream &s) {
    if (s.have == 0) { mz_u4 r = mz_philox(s.seed, MZ_STREAM_DIRICHLET, s.c0, s.c1, s.c2, s.ctr++); s.buf[0] = r.x; s.buf[1] = r.y; s.buf[2] = r.z; s.buf[3] = r.w; s.have = 4; }
    uint32_t v = s.buf[4 - s.have]; s.have--;
    return v;
}
MZ_HD float mz_rs_unit_open(mz_rstream &s) { return ((float)(mz_rs_next(s) >> 8) + 0.5f) * 5.9604644775390625e-8f; }
MZ_HD float mz_rs_normal(mz_rstream &s) {
    for (;;) {
        float a = 2.0f * mz_rs_unit_open(s) - 1.0f, b = 2.0f * mz_rs_unit_open(s) - 1.0f;
        float q = a * a + b * b;
        if (q >= 1.0f || q == 0.0f) continue;
        return a * sqrtf(-2.0f * mz_logf(q) / q);
    }
}
MZ_HD float mz_rs_gamma(mz_rstream &s, float alpha) {
    float a1 = alpha < 1.0f ? alpha + 1.0f : alpha;
    float d = a1 - 0.333333343f, cc = 1.0f / sqrtf(9.0f * d), g;
    for (;;) {
        float x = mz_rs_normal(s), v = 1.0f + cc * x;
        if (v <= 0.0f) continue;
        v = v * v * v;
        float u = mz_rs_unit_open(s);
        if (mz_logf(u) < 0.5f * x * x + d - d * v + d * mz_logf(v)) { g = d * v; break; }
    }
    if (alpha < 1.0f) { float u = mz_rs_unit_open(s); g = g * mz_expf(mz_logf(u) / alpha); }
    return g;
}
MZ_HD void mz_tree_add_noise(const mz_params &P, const mz_tree &t, uint32_t legal, uint32_t game, uint32_t move) {
    float noise[MZ_MAX_A], sum = 0.0f; int n = 0;
    for (int j = 0; j < P.A; j++) {
        int a = P.order[j];
        if (!((legal >> (a - 1)) & 1u)) continue;
        mz_rstream s; s.seed = P.seed; s.c0 = game; s.c1 = move; s.c2 = (uint32_t)n; s.ctr = 0; s.have = 0;
        noise[n] = mz_rs_gamma(s, P.dirichlet_alpha); sum = sum + noise[n]; n++;
    }
    n = 0;
    for (int j = 0; j < P.A; j++) {
        int a = P.order[j];
        if (!((legal >> (a - 1)) & 1u)) continue;
        float nz = noise[n++] / sum;
        mz_f4 c = t.A[1 + a - 1];
        c.z = c.z * (1.0f - P.exploration_eps) + nz * P.exploration_eps;
        t.A[1 + a - 1] = c;
    }
}

// ---- competitive play: select_opponent_action (src/SelfPlay.jl:311-325) ------------------------------------------
// a completed line of one side's marks (the real rule, not is_win's side-to-move test)
MZ_HD bool mz_env_has_line(const mz_params &P, uint64_t b) { return P.game == MZ_GAME_TICTACTOE ? mz_ttt_line((uint32_t)b) : mz_connect_has4(b, P.W); }
// "random": rand(rng, las), uniform over the ascending legal actions from the Philox stream (seed, OPPONENT, game, move) -- as written
// the branch reads `las` before defining it.  "expert": expert_agent() is not defined in the reference; repaired as one-ply
// lookahead: the first legal action that completes a line for the mover, else the first that would complete one for the other
// side, else the random action.
MZ_HD int mz_opponent_action(const mz_params &P, const mz_board &b, int opponent, uint32_t game, uint32_t move) {
    const uint32_t legal = mz_env_legal_b(P, b);
    int las[MZ_MAX_A], n = 0;
    for (int a = 1; a <= P.A; a++) if ((legal >> (a - 1)) & 1u) las[n++] = a;
    if (n == 0) return 1;
    if (opponent == MZ_OPP_EXPERT) {
        for (int pass = 0; pass < 2; pass++) for (int i = 0; i < n; i++) {
            mz_board t = b;
            if (pass == 1) t.player = t.player % P.P + 1;
            const int who = t.player;
            mz_env_step_b(P, t, las[i]);
            if (mz_env_has_line(P, who == 1 ? t.p1 : t.p2)) return las[i];
        }
    }
    return las[mz_u32_below(mz_philox(P.seed, MZ_STREAM_OPPONENT, game, move, 0, 0).x, (uint32_t)n)];
}
// +1 / 0 / -1 for MuZero: the side that completes a line first wins (TicTacToe runs one ply past a win, Q14)
MZ_HD int mz_arena_outcome(const mz_params &P, int T, const int32_t *actions, int muzero_player) {
    mz_board b; mz_env_reset_b(P, b);
    for (int i = 0; i < T; i++) {
        const int who = b.player;
        mz_env_step_b(P, b, actions[i]);
        if (mz_env_has_line(P, who == 1 ? b.p1 : b.p2)) return who == muzero_player ? 1 : -1;
    }
    return 0;
}

// play_game's temperature for the ply searched after T plies (src/SelfPlay.jl:344-346): 0 from conf.temperature_threshold plies on
MZ_HD float mz_play_temperature(const mz_params &P, int T, float temperature) {
    return (P.temp_threshold >= 0 && T >= P.temp_threshold) ? 0.0f : temperature;
}

// select_action (src/SelfPlay.jl:293-306) over the root's children in Dict order (Q9-Q10).
MZ_HD int mz_select_action_counts(const mz_params &P, const int32_t *visit_counts /* [A] by action-1 */, uint32_t legal,
                                  float temperature, uint32_t game, uint32_t move) {
    int counts[MZ_MAX_A], acts[MZ_MAX_A], n = 0;
    for (int j = 0; j < P.A; j++) { int a = P.order[j]; if ((legal >> (a - 1)) & 1u) { counts[n] = visit_counts[a - 1]; acts[n] = a; n++; } }
    if (temperature == 0.0f) {
        int best = 0;
        for (int i = 1; i < n; i++) if (counts[i] > counts[best]) best = i;
        return acts[best];
    }
    mz_u4 r = mz_philox(P.seed, MZ_STREAM_ACTION, game, move, 0, 0);
    if (isinf(temperature)) return acts[mz_u32_below(r.x, (uint32_t)n)];
    float d[MZ_MAX_A], s = 0.0f, e = 1.0f / temperature;
    for (int i = 0; i < n; i++) { d[i] = mz_pow_contract((float)counts[i], e); s = s + d[i]; }
    for (int i = 0; i < n; i++) d[i] = d[i] / s;
    float draw = mz_u32_to_unit(r.x), cp = d[0]; int i = 0;
    while (cp <= draw && i < n - 1) { i++; cp = cp + d[i]; }
    return acts[i];
}

// Prioritised replay (conf.PER, repaired specification: DESIGN.md / oracle/mz_oracle.c): priority |root value - target value|^alpha
// (Float32 ^ Int as Julia evaluates it for alpha <= 3) in fixed point, q = max(1, round(p * 2^16)): integer sums are exact, so the
// device prefix scan and the oracle's sequential sums agree bit for bit.
MZ_HD float mz_pow_int(float x, int i) { return i == 0 ? 1.0f : i == 1 ? x : i == 2 ? x * x : x * x * x; }
MZ_HD uint32_t mz_per_quantise(float p) {
    float s = p * 65536.0f;
    if (!(s >= 1.0f)) return 1u;
    if (s > 4.0e9f) return 4000000000u;
    return (uint32_t)llrintf(s);
}

// compute_target_value (src/ReplayBuffer.jl:5-20), Q17; 1-based index.
MZ_HD float mz_target_value(const mz_params &P, int T, const float *rewards, const uint8_t *to_play, const float *root_values, int index) {
    int bootstrap = index + P.td;
    if (bootstrap < T) {
        float last = to_play[bootstrap - 1] == to_play[index - 1] ? root_values[bootstrap - 1] : -root_values[bootstrap - 1];
        float value = last * P.disc_pow[P.td];
        int i = 1;
        for (int ri = index; ri <= bootstrap; ri++, i++) {
            float r = rewards[ri - 1];
            value = value + (to_play[index - 1] == to_play[index + i - 1] ? r : -r) * P.disc_pow[i];
        }
        return value;
    }
    return 0.0f;
}
