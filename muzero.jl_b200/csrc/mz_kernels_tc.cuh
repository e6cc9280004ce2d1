// mz_kernels_tc.cuh -- mz_k_search_tc: the fused search kernel of mz_kernels.cuh with the network phase on the
// tcgen05 tensor cores (mz_tc.cuh).  Tree phases, epilogue and data layout are identical to mz_k_search; only the
// network arithmetic (bf16 operands, fp32 accumulate) and the staging of its inputs differ, so results agree with the
// exact path to bf16 tolerance (not bit-exactly): tests report value/policy tolerance and the visit-count match rate.
#pragma once
#include "mz_kernels.cuh"
#include "mz_tc.cuh"

struct mz_search_tc_args {
    mz_search_args base;
    const unsigned char *w_image;   // bf16 pre-swizzled weight image (global)
    const float *bias;              // fp32 bias block (global)
};

template <int MODE>
__global__ void __launch_bounds__(MZ_THREADS) mz_k_search_tc(const __grid_constant__ mz_params P, const mz_search_tc_args ta) {
    extern __shared__ __align__(1024) unsigned char mz_smem_tc[];
    const mz_search_args &a = ta.base;
    if (mz_cta_idle<MODE>(P, a, MZ_ROWS)) return;
    const mz_tc_plan sp = mz_tc_carve(mz_smem_tc, P.tc_net_off[3], P.tc_bias_floats, P.hidden_pad, P.S);
    const int tid = threadIdx.x;
    const int r = tid >> 3, ln = tid & (MZ_LANES - 1);
    const uint32_t segmask = 0xffu << ((tid & 31) & ~7);
    const int64_t g = (int64_t)blockIdx.x * MZ_ROWS + r;

    // ---- one-time setup: barriers, TMEM, weights (TMA bulk copies), zeroed operand tiles ----
    if (tid == 0) {
        mz_mbar_init(sp.mbar_w, 1); mz_mbar_init(sp.mbar_mma[0], 1); mz_mbar_init(sp.mbar_mma[1], 1);
        mz_fence_mbar_init();
    }
    __syncwarp();
    if (tid < 32) mz_tc_alloc(sp.tmem_slot);
    for (int i = tid; i < 9 * MZ_TC_TILE_BYTES / 4; i += MZ_THREADS) reinterpret_cast<uint32_t *>(sp.tiles_ptr)[i] = 0u;
    mz_fence_proxy_async();
    mz_tc_fence_before();
    __syncthreads();
    mz_tc_fence_after();
    const uint32_t tmem_base = *sp.tmem_slot;
    if (tid == 0) {
        const uint32_t wbytes = (uint32_t)P.tc_net_off[3], bbytes = (uint32_t)P.tc_bias_floats * 4u;
        mz_mbar_expect_tx(sp.mbar_w, wbytes + bbytes);
        for (int n = 0; n < 3; n++) {
            uint32_t off = (uint32_t)P.tc_net_off[n], len = (uint32_t)(P.tc_net_off[n + 1] - P.tc_net_off[n]);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(sp.w_base + off), "l"(ta.w_image + off), "r"(len), "r"(mz_smem_u32(sp.mbar_w)) : "memory");
        }
        mz_bulk_g2s((void *)sp.bias, ta.bias, bbytes, sp.mbar_w);
    }
    // compile the three networks into the round table (one thread, once per kernel)
    int *rounds = reinterpret_cast<int *>(sp.tmem_slot) + 4;            // [0] representation, [1] prediction, [2] dynamics round counts
    if (tid == 0) {
        mz_tc_builder B; B.prog = sp.prog; B.n = 0; B.w_base = sp.w_base; B.bias_base = mz_smem_u32(sp.bias);
        rounds[0] = mz_tc_build_net(B, P, 0, sp.inS, sp.bufT[0], mz_smem_u32(sp.outH), 0u, sp.t0[0], sp.t1[0], 0u);
        rounds[1] = mz_tc_build_net(B, P, 1, sp.in1, sp.bufT[0], mz_smem_u32(sp.outV), mz_smem_u32(sp.outL), sp.t0[0], sp.t1[0], sp.t1[0]);
        rounds[2] = mz_tc_build_net(B, P, 2, sp.in0, sp.bufT[1], mz_smem_u32(sp.outH), mz_smem_u32(sp.outR), sp.t0[1], sp.t1[1], sp.inS);
    }
    const int grp = tid >> 7, gtid = tid & (MZ_GROUP - 1);
    const uint32_t tmem_d = tmem_base + (uint32_t)(64 * grp), mbar_mma = mz_smem_u32(sp.mbar_mma[grp]);
    uint32_t q = 0;                                                     // rounds executed by this group (mbarrier parity)
    long long *tk = nullptr;
#ifdef MZ_PHASE_TIMERS
    long long rt[6] = {0, 0, 0, 0, 0, 0};
    if (tid == 0 || tid == MZ_GROUP + 32) tk = rt;                      // observers: the issuing thread of group 0, a plain epilogue thread of group 1
#endif
    uint16_t *path = sp.path + (size_t)r * (P.S + 2);

    // ---- per-tree state, replicated in the 8 lanes of the tree ----
    mz_tree tree; tree.A = nullptr; tree.hidden = nullptr;
    if (g < a.n) tree = mz_tree_at(P, a.tree_pool, g);
    const mz_root root = mz_root_begin<MODE>(P, a, g, g < a.n);
    const bool active = root.active;

    // ---- stage the stacked observations as a bf16 B tile (values are 0/1 and raw action indices: exact in bf16) ----
    for (int i = tid; i < MZ_ROWS * P.stack_size; i += MZ_THREADS) {
        int rr, k;
        if (MODE == MZ_MODE_API) { rr = i / P.stack_size; k = i % P.stack_size; }   // the caller's rows are contiguous
        else { k = i / MZ_ROWS; rr = i % MZ_ROWS; }                                  // slots, replay positions: every entry is computed
        mz_tc_store_bf16(sp.inS, rr, k, mz_root_obs<MODE>(P, a, (int64_t)blockIdx.x * MZ_ROWS + rr, k));
    }
    mz_fence_proxy_async();
    mz_mbar_wait(sp.mbar_w, 0);          // weights + biases have landed
    __syncthreads();

    // ---- root: representation -> h0 (fp32 in outH); prediction(h0) -> (v0, p0) ----
    const int n_repr = rounds[0], n_pred = rounds[1], n_dyn = rounds[2];
    if (grp == 0) q = mz_tc_run(sp.prog, 0, n_repr, tmem_d, mbar_mma, q, grp, gtid, tk);
    __syncthreads();
    for (int i = tid; i < MZ_ROWS * P.hidden; i += MZ_THREADS) { int k = i / MZ_ROWS, rr = i % MZ_ROWS; mz_tc_store_bf16(sp.in1, rr, k, sp.outH[k * MZ_ROWS + rr]); }
    mz_fence_proxy_async();
    __syncthreads();
    if (grp == 0) q = mz_tc_run(sp.prog, n_repr, n_pred, tmem_d, mbar_mma, q, grp, gtid, tk);
    __syncthreads();

    mz_minmax mm; mm.mn = INFINITY; mm.mx = -INFINITY;
    unsigned long long depth_sum = 0;
    MZ_TIMER_DECL;
    if (active) {
        for (int k = ln; k < P.hidden; k += MZ_LANES) tree.hidden[k] = sp.outH[k * MZ_ROWS + r];
        mz_root_init(P, tree, root, a.exploration, sp.outL + r, MZ_ROWS, ln, segmask);
    }

    // ---- simulations ----
    for (int sim = 1; sim <= P.S; sim++) {
        mz_leaf leaf; leaf.node = 0; leaf.parent = 0; leaf.action = 1; leaf.depth = 0; leaf.prior = 0.0f; leaf.parent_x = 0;
        MZ_TIMER(0);
        if (active) {
            leaf = mz_tree_select_lanes(P, tree, a.pbc0, a.sqrtN, root.legal, root.posmask, mm, root.game, root.move, (uint32_t)sim, ln, segmask, path);
            depth_sum += (unsigned long long)leaf.depth;
            MZ_TIMER(1);
            const int pe = mz_nx_exp(leaf.parent_x), dbl = mz_nx_dbl(leaf.parent_x);
            const float *h = tree.hidden + (size_t)pe * P.hidden_pad;
            const float sc = mz_bits2f((uint32_t)(127 + dbl) << 23);
            for (int k = ln; k < P.hidden; k += MZ_LANES) {
                float v = h[k] * sc;
                mz_tc_store_bf16(sp.in1, r, k, v);                 // prediction(parent.hidden_state) (Q5)
                mz_tc_store_bf16(sp.in0, r, k, v * 2.0f);          // make_state_action: state .*= 2 (Q6)
            }
            const float plane = P.act_plane_play[leaf.action];
            for (int k = P.obs_size + ln; k < P.sa_size; k += MZ_LANES) mz_tc_store_bf16(sp.in0, r, k, plane);
            __syncwarp(segmask);
            if (ln == 0) reinterpret_cast<uint32_t *>(&tree.A[leaf.parent])[0] = leaf.parent_x + (1u << 24);   // one more doubling (Q6)
        }
        mz_fence_proxy_async();
        MZ_TIMER(2);
        __syncthreads();
        MZ_TIMER(3);
        if (grp == 0) q = mz_tc_run(sp.prog, n_repr, n_pred, tmem_d, mbar_mma, q, grp, gtid, tk);
        else          q = mz_tc_run(sp.prog, n_repr + n_pred, n_dyn, tmem_d, mbar_mma, q, grp, gtid, tk);
        MZ_TIMER(4);
        __syncthreads();
        MZ_TIMER(5);
        if (active) {
            float *nh = tree.hidden + (size_t)sim * P.hidden_pad;
            for (int k = ln; k < P.hidden; k += MZ_LANES) nh[k] = sp.outH[k * MZ_ROWS + r];
            MZ_TIMER(6);
            mz_tree_expand_lanes(P, tree, leaf.node, sim, root.legal, sp.outL + r, sp.outR[r], leaf.prior, ln, segmask);
            MZ_TIMER(7);
            mz_tree_backup_lanes(P, tree, path, leaf.depth, sp.outV[r], mm, ln, segmask);
        }
        MZ_TIMER(8);
    }

    MZ_TIMER_FLUSH(a.stats);
#ifdef MZ_PHASE_TIMERS
    if (a.stats && tk) { int o_ = tid == 0 ? 16 : 24; for (int i_ = 0; i_ < 6; i_++) atomicAdd(&a.stats[o_ + i_], (unsigned long long)rt[i_]); atomicAdd(&a.stats[o_ + 6], (unsigned long long)q); }
#endif
    if (active && ln == 0) mz_root_finish<MODE>(P, a, g, tree, root, depth_sum);
    // ---- teardown: every tcgen05 operation has completed (all layers were waited on) ----
    mz_tc_fence_before();
    __syncthreads();
    if (tid < 32) mz_tc_dealloc(tmem_base);
}

// batched network callable on the tensor cores (parity / tolerance tests of the TC layers in isolation)
struct mz_nn_tc_args { const unsigned char *w_image; const float *bias; int32_t B, net; const float *in; float *out1; float *out2; };
__global__ void __launch_bounds__(MZ_THREADS) mz_k_nn_forward_tc(const __grid_constant__ mz_params P, const mz_nn_tc_args a) {
    extern __shared__ __align__(1024) unsigned char mz_smem_tc[];
    const mz_tc_plan sp = mz_tc_carve(mz_smem_tc, P.tc_net_off[3], P.tc_bias_floats, P.hidden_pad, P.S);
    const int tid = threadIdx.x;
    if (tid == 0) { mz_mbar_init(sp.mbar_w, 1); mz_mbar_init(sp.mbar_mma[0], 1); mz_mbar_init(sp.mbar_mma[1], 1); mz_fence_mbar_init(); }
    __syncwarp();
    if (tid < 32) mz_tc_alloc(sp.tmem_slot);
    for (int i = tid; i < 9 * MZ_TC_TILE_BYTES / 4; i += MZ_THREADS) reinterpret_cast<uint32_t *>(sp.tiles_ptr)[i] = 0u;
    mz_fence_proxy_async();
    mz_tc_fence_before();
    __syncthreads();
    mz_tc_fence_after();
    const uint32_t tmem_base = *sp.tmem_slot;
    if (tid == 0) {
        const uint32_t wbytes = (uint32_t)P.tc_net_off[3], bbytes = (uint32_t)P.tc_bias_floats * 4u;
        mz_mbar_expect_tx(sp.mbar_w, wbytes + bbytes);
        for (int n = 0; n < 3; n++) {
            uint32_t off = (uint32_t)P.tc_net_off[n], len = (uint32_t)(P.tc_net_off[n + 1] - P.tc_net_off[n]);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(sp.w_base + off), "l"(a.w_image + off), "r"(len), "r"(mz_smem_u32(sp.mbar_w)) : "memory");
        }
        mz_bulk_g2s((void *)sp.bias, a.bias, bbytes, sp.mbar_w);
    }
    float *h1 = a.net == 1 ? sp.outV : sp.outH, *h2 = a.net == 1 ? sp.outL : sp.outR;
    int *rounds = reinterpret_cast<int *>(sp.tmem_slot) + 4;
    if (tid == 0) {
        mz_tc_builder B; B.prog = sp.prog; B.n = 0; B.w_base = sp.w_base; B.bias_base = mz_smem_u32(sp.bias);
        rounds[0] = mz_tc_build_net(B, P, a.net, sp.inS, sp.bufT[0], mz_smem_u32(h1), mz_smem_u32(h2), sp.t0[0], sp.t1[0], sp.in1);
    }
    const int grp = tid >> 7, gtid = tid & (MZ_GROUP - 1);
    const int in = P.layers[P.nets[a.net].first].in;
    for (int i = tid; i < MZ_ROWS * in; i += MZ_THREADS) {
        int rr = i / in, k = i % in;
        int64_t gg = (int64_t)blockIdx.x * MZ_ROWS + rr;
        mz_tc_store_bf16(sp.inS, rr, k, gg < a.B ? a.in[gg * in + k] : 0.0f);
    }
    mz_fence_proxy_async();
    mz_mbar_wait(sp.mbar_w, 0);
    __syncthreads();
    if (grp == 0) mz_tc_run(sp.prog, 0, rounds[0], tmem_base, mz_smem_u32(sp.mbar_mma[0]), 0u, grp, gtid, nullptr);
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
    mz_tc_fence_before();
    __syncthreads();
    if (tid < 32) mz_tc_dealloc(tmem_base);
}
