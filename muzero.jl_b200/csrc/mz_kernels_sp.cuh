// mz_kernels_sp.cuh -- mz_k_search_sp: the fused search kernel of mz_kernels.cuh with the network phase on the tcgen05 tensor cores at
// near-Float32 accuracy (nn_mode = MZ_NN_SPLIT_MMA, mz_sp.cuh: bf16 hi / lo split of both operands, fp32 accumulation in TMEM).  Tree
// phases, move epilogue and data layout are the ones of mz_k_search; group 0 (threads 0..127) runs prediction(parent), group 1 the
// representation (at the root) and dynamics(parent, a), concurrently (SURVEY Q5), each with its own weight sets and TMEM columns.
// The dynamics rounds after the reward is final (the state head alone) and the hidden-state write run on a tail team of warps beside
// expand, backup and the next selection (DESIGN.md 2.1c).
#pragma once
#include "mz_kernels.cuh"
#include "mz_sp.cuh"

struct mz_search_sp_args { mz_search_args base; mz_sp_args sp; };

// profiling build: thread 0 stamps the stages of the whole kernel (set-up, staging, representation, root prediction, root expansion,
// simulation loop, move epilogue + teardown) into stats[50 ..]
#ifdef MZ_PHASE_TIMERS
#define MZ_KSTAMP_DECL long long mz_ks[8]; mz_ks[7] = clock64()
#define MZ_KSTAMP(i) mz_ks[i] = clock64()
#define MZ_KSTAMP_FLUSH(stats) do { if ((stats) && threadIdx.x == 0) { long long p_ = mz_ks[7]; for (int i_ = 0; i_ < 7; i_++) { atomicAdd(&(stats)[50 + i_], (unsigned long long)(mz_ks[i_] - p_)); p_ = mz_ks[i_]; } atomicAdd(&(stats)[57], 1ull); atomicMax(&(stats)[58], (unsigned long long)(mz_ks[6] - mz_ks[7])); } } while (0)
#else
#define MZ_KSTAMP_DECL
#define MZ_KSTAMP(i)
#define MZ_KSTAMP_FLUSH(stats)
#endif

// one thread: all rounds [first, first + count) share ONE set (the representation): a single expect_tx for the sum, then the copies
__device__ __forceinline__ void mz_sp_fill_many(const mz_sp_ctx &C, int first, int count) {
    uint32_t total = 0;
    for (int r = first; r < first + count; r++) total += mz_lds_u4(C.prog + (uint32_t)r * MZ_SP_RDESC_BYTES + 96).x;
    const int set = (int)(short)(mz_lds_u4(C.prog + (uint32_t)first * MZ_SP_RDESC_BYTES + 80).w & 0xffffu);
    const uint32_t bar = C.bars + 8u * (uint32_t)set;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
    for (int r = first; r < first + count; r++) {
        const uint32_t R = C.prog + (uint32_t)r * MZ_SP_RDESC_BYTES;
        const uint4 m = mz_lds_u4(R + 80), c0 = mz_lds_u4(R + 96), c1 = mz_lds_u4(R + 112);
        const int ncopy = (int)(short)(m.z >> 16);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(c0.z), "l"(C.image + (int32_t)c1.z), "r"(c1.x), "r"(bar) : "memory");
        if (ncopy > 1)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(c0.w), "l"(C.image + (int32_t)c1.w), "r"(c1.y), "r"(bar) : "memory");
    }
}
// one thread: the first round of every weight set of a network
__device__ __forceinline__ void mz_sp_prime(const mz_sp_ctx &C, const mz_sp_args &A, int net) {
    for (int s = 0; s < A.n_sets[net] && s < A.n_rounds[net]; s++) mz_sp_fill(C, C.prog + (uint32_t)(A.first[net] + s) * MZ_SP_RDESC_BYTES);
}
// one thread, before the CTA ends: the refills issued after the last pass must have landed (passes = passes over the network so far)
__device__ __forceinline__ void mz_sp_drain(const mz_sp_ctx &C, const mz_sp_args &A, int net, uint32_t passes, uint32_t bias = 0) {
    for (int s = 0; s < A.n_sets[net] && s < A.n_rounds[net]; s++) {
        const uint32_t R = C.prog + (uint32_t)(A.first[net] + s) * MZ_SP_RDESC_BYTES;
        const uint32_t per_pass = mz_lds_u4(R + 96).y & 0xffffu;
        if (per_pass) mz_sp_wait_weights(C, (int)(short)(mz_lds_u4(R + 80).w & 0xffffu), passes * per_pass + bias);
    }
}
__device__ __forceinline__ uint32_t mz_sp_group_tile(const mz_sp_plan_s &sp, int grp, int tile) { return sp.tiles + (uint32_t)((grp * MZ_SP_TILES_PER_GROUP + tile) * 2 * MZ_SP_TILE_BYTES); }

// the tail team, once per simulation: the tail rounds (mz_sp_run_tail), then the new hidden state of every active tree -> tree.hidden[sim]
// (8 threads per tree, as the tree phases; two trees per thread), then the "tail done" arrival that the workers wait for before staging
__device__ __forceinline__ uint32_t mz_sp_tail(const mz_params &P, const mz_search_args &a, const float *outH, const uint8_t *active, const mz_sp_ctx C, int first, int count,
                                            uint32_t tmem_d, uint32_t mbar, uint32_t q, uint32_t pass, uint32_t bias, int ttid, int sim, uint32_t mbar_tail) {
#ifdef MZ_PHASE_TIMERS
    const long long t0_ = clock64();
#endif
    q = mz_sp_run_tail(C, first, count, tmem_d, mbar, q, pass, bias, ttid);
    mz_named_sync(MZ_SP_BAR_TAIL, MZ_SP_TAIL_THREADS);                  // all four quadrants of the last round's outputs are in outH
    for (int rr = ttid / MZ_LANES; rr < MZ_ROWS; rr += MZ_SP_TAIL_THREADS / MZ_LANES) {
        if (!active[rr]) continue;
        float *nh = mz_tree_at(P, a.tree_pool, (int64_t)blockIdx.x * MZ_ROWS + rr).hidden + (size_t)sim * P.hidden_pad;
        for (int k = ttid & (MZ_LANES - 1); k < P.hidden; k += MZ_LANES) nh[k] = outH[k * MZ_SP_OS + rr];
    }
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar_tail) : "memory");
#ifdef MZ_PHASE_TIMERS
    // profiling build: the dynamics issuer's lane 0 times the tail from the end of its chain rounds' issue to "tail done"
    if (a.stats && ttid == 32) { atomicAdd(&a.stats[59], (unsigned long long)(clock64() - t0_)); atomicAdd(&a.stats[60], 1ull); }
#endif
    return q;
}

template <int MODE>
__global__ void __launch_bounds__(MZ_SP_SEARCH_THREADS) mz_k_search_sp(const __grid_constant__ mz_params P, const __grid_constant__ mz_search_sp_args sa) {
    extern __shared__ __align__(1024) unsigned char mz_smem_sp[];
    const mz_search_args &a = sa.base;
    const mz_sp_args &A = sa.sp;
    if (mz_cta_idle<MODE>(P, a, MZ_ROWS)) return;
    const mz_sp_plan_s sp = mz_sp_carve(mz_smem_sp, A.warea_bytes, A.bias_floats, A.total_rounds, P.hidden_pad, P.S, A.pbc_smem);
    const int tid = threadIdx.x;
    const int r = tid >> 3, ln = tid & (MZ_LANES - 1);
    const uint32_t segmask = 0xffu << ((tid & 31) & ~7);
    const int64_t g = (int64_t)blockIdx.x * MZ_ROWS + r;
    MZ_KSTAMP_DECL;
    const uint32_t tmem_base = mz_sp_setup(sp, A, MZ_SP_SEARCH_THREADS);
    MZ_KSTAMP(0);
    mz_sp_ctx C; C.prog = mz_smem_u32(sp.prog); C.image = A.image; C.bars = mz_smem_u32(sp.bars);
    const double *pbc = a.pbc0;
    if (A.pbc_smem) {                                                   // compact copy of ucb_score's table: row N holds n = 0..N
        for (int N = tid; N < P.S + 2; N += MZ_SP_SEARCH_THREADS) for (int n = 0; n <= N; n++) sp.pbc[(N * (N + 1)) / 2 + n] = a.pbc0[N * (P.S + 2) + n];
        pbc = sp.pbc;
    }
    // warps 0..7: tree phases + epilogues; warp 8 / 9: issuer of group 0 / 1; warps 8..11: the tail team (TMEM lane quadrants 0..3), which
    // runs the last `tail` dynamics rounds and the hidden-state write beside the tree phases (warps 10, 11 do nothing else)
    const bool worker = tid < MZ_THREADS, issuer = !worker && tid < MZ_THREADS + 64;
    const int grp = worker ? tid >> 7 : (tid < MZ_THREADS + 32 ? 0 : 1), gtid = tid & (MZ_GROUP - 1);
    const bool issuer0 = issuer && (tid & 31) == 0;                     // lane 0 of an issuer warp: one-off TMA work
    if (issuer0) {
        if (grp == 0) mz_sp_prime(C, A, 1);
        else mz_sp_fill_many(C, A.first[0], A.n_rounds[0]);
    }
    const uint32_t tmem_d = tmem_base + (uint32_t)(128 * grp), mbar_mma = mz_smem_u32(sp.mbar_mma[grp]);
    const uint32_t in_pred = mz_sp_group_tile(sp, 0, 0), in_dyn = mz_sp_group_tile(sp, 1, 0);
    const bool tanh_v = P.layers[P.nets[1].first + P.nets[1].n_trunk + P.nets[1].n_h1 - 1].act == MZ_ACT_TANH;
    const bool tanh_r = P.layers[P.nets[2].first + P.nets[2].n_trunk + P.nets[2].n_h1 + P.nets[2].n_h2 - 1].act == MZ_ACT_TANH;
    uint32_t q = 0, pass = 0;                                           // rounds / passes over its per-simulation network executed by this group
    long long *tk = nullptr;
#ifdef MZ_PHASE_TIMERS
    long long rt[6] = {0, 0, 0, 0, 0, 0};
    if (tid == 0 || tid == MZ_GROUP + 32) tk = rt;                      // observers: the issuing thread of group 0, a plain epilogue thread of group 1
#endif
    uint16_t *path = sp.path + (size_t)r * (P.S + 2);

    mz_tree tree; tree.A = nullptr; tree.hidden = nullptr;
    if (worker && g < a.n) tree = mz_tree_at(P, a.tree_pool, g);
    const bool persist = MODE == MZ_MODE_SLOTS && a.persist != 0 && P.arena_player == 0;
    uint32_t ply = 0;                                                   // moves played by this launch so far (persist: one launch plays the games to the end)
  for (;; ply++) {
    // the representation's weights lie over the dynamics sets: at every further ply they are fetched again (after the refills issued behind
    // the last dynamics pass have landed) and the dynamics sets are primed again after the representation -- one extra fill per set and ply,
    // which is the `bias` of the weight waits
    if (ply > 0 && issuer0 && grp == 1) { mz_sp_drain(C, A, 2, pass, ply - 1); mz_sp_fill_many(C, A.first[0], A.n_rounds[0]); }
    // ---- per-tree state, replicated in the 8 lanes of the tree ----
    const mz_root root = mz_root_begin<MODE>(P, a, g, worker && g < a.n);
    const bool active = root.active;

    // ---- stage the stacked observations (hi / lo operand tiles of group 1) ----
    if (worker && ln == 0) sp.active[r] = active;                       // for the tail team's hidden-state write
    for (int i = tid; i < MZ_ROWS * P.stack_size; i += MZ_SP_SEARCH_THREADS) {
        int rr, k;
        if (MODE == MZ_MODE_API) { rr = i / P.stack_size; k = i % P.stack_size; }   // the caller's rows are contiguous
        else { k = i / MZ_ROWS; rr = i % MZ_ROWS; }                                  // slots, replay positions: every entry is computed
        mz_sp_stage(in_dyn, k, rr, mz_root_obs<MODE>(P, a, (int64_t)blockIdx.x * MZ_ROWS + rr, k));
    }
    mz_fence_proxy_async();
    __syncthreads();
    MZ_KSTAMP(1);

    // ---- root: representation -> h0 (group 1, its weights lie over the dynamics area); then the dynamics sets are primed while
    //      group 0 runs prediction(h0) -> (v0, p0) ----
    if (grp == 1) {
        if (worker) q = mz_sp_run(C, A.first[0], A.n_rounds[0], tmem_d, mbar_mma, q, grp, gtid, nullptr);
        else if (issuer) { q = mz_sp_run_issuer(C, A.first[0], A.n_rounds[0], tmem_d, mbar_mma, q, 0u, grp, nullptr, 0u, ply); if (issuer0) mz_sp_prime(C, A, 2); }
    }
    __syncthreads();
    MZ_KSTAMP(2);
    for (int i = tid; i < MZ_ROWS * P.hidden; i += MZ_SP_SEARCH_THREADS) { const int k = i / MZ_ROWS, rr = i % MZ_ROWS; mz_sp_stage(in_pred, k, rr, sp.outH[k * MZ_SP_OS + rr]); }
    mz_fence_proxy_async();
    __syncthreads();
    if (grp == 0) {
        if (worker) q = mz_sp_run(C, A.first[1], A.n_rounds[1], tmem_d, mbar_mma, q, grp, gtid, nullptr);
        else q = mz_sp_run_issuer(C, A.first[1], A.n_rounds[1], tmem_d, mbar_mma, q, pass, grp);
        pass++;
    }
    __syncthreads();
    MZ_KSTAMP(3);

    mz_minmax mm; mm.mn = INFINITY; mm.mx = -INFINITY;
    unsigned long long depth_sum = 0;
    MZ_TIMER_DECL;
    if (active) {
        for (int k = ln; k < P.hidden; k += MZ_LANES) tree.hidden[k] = sp.outH[k * MZ_SP_OS + r];
        mz_root_init(P, tree, root, a.exploration, sp.outL + r, MZ_SP_OS, ln, segmask);
    }

    MZ_KSTAMP(4);
    // ---- simulations: the worker warps and the others (issuers, tail team) run separate loops that meet at named barriers ----
    if (worker) {
    // byte offsets of this lane's staging positions (k = ln + 8 i, tree r) inside an operand tile: the same in every simulation
    uint32_t soff[8];
#pragma unroll
    for (int i = 0; i < 8; i++) soff[i] = mz_sp_tile_offset(ln + MZ_LANES * i, r & (MZ_ROWS - 1));
    for (int sim = 1; sim <= P.S; sim++) {
        mz_leaf leaf; leaf.node = 0; leaf.parent = 0; leaf.action = 1; leaf.depth = 0; leaf.prior = 0.0f; leaf.parent_x = 0;
        MZ_TIMER(0);
        if (active) {
            leaf = mz_tree_select_lanes(P, tree, pbc, a.sqrtN, root.legal, root.posmask, mm, root.game, root.move, (uint32_t)sim, ln, segmask, path, A.pbc_smem != 0);
            depth_sum += (unsigned long long)leaf.depth;
        }
        MZ_TIMER(1);
        // The tail of the previous simulation (its last dynamics rounds and its hidden-state write) must be done before staging: staging
        // reads tree.hidden[pe], where pe may be the node that simulation expanded, and overwrites group 1's input tile, which the tail's
        // rounds may still read.  The next pass's MMAs (TMEM, operand tiles) start after the barrier behind staging, so after this wait
        // too.  The tail team arrives after tcgen05.wait::ld + tcgen05.fence::before_thread_sync of its last round.  The first
        // simulation of a move follows CTA-wide barriers that the team joins when its last tail is done.
        if (A.tail && sim > 1) mz_sp_wait_mma(mz_smem_u32(sp.mbar_tail), (uint32_t)(ply * P.S + sim - 2));
        MZ_TIMER(6);
        if (active) {
            const int pe = mz_nx_exp(leaf.parent_x), dbl = mz_nx_dbl(leaf.parent_x);
            const float *h = tree.hidden + (size_t)pe * P.hidden_pad;
            const float sc = mz_bits2f((uint32_t)(127 + dbl) << 23);
            float hv[8];                                           // all loads first: the staging stores are volatile asm, loads do not move across them
#pragma unroll
            for (int i = 0; i < 8; i++) { const int k = ln + MZ_LANES * i; hv[i] = k < P.hidden ? h[k] : 0.0f; }
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int k = ln + MZ_LANES * i;
                if (k < P.hidden) {
                    const float v = hv[i] * sc;
                    mz_sp_stage_at(in_pred + soff[i], v);          // prediction(parent.hidden_state) (Q5)
                    mz_sp_stage_at(in_dyn + soff[i], v * 2.0f);    // make_state_action: state .*= 2 (Q6)
                }
            }
            const float plane = P.act_plane_play[leaf.action];
#pragma unroll
            for (int i = 0; i < 8; i++) { const int k = ln + MZ_LANES * i; if (k >= P.obs_size && k < P.sa_size) mz_sp_stage_at(in_dyn + soff[i], plane); }
            __syncwarp(segmask);
            if (ln == 0) reinterpret_cast<uint32_t *>(&tree.A[leaf.parent])[0] = leaf.parent_x + (1u << 24);   // one more doubling (Q6)
        }
        mz_fence_proxy_async();
        MZ_TIMER(2);
        mz_named_sync(MZ_SP_BAR_SIM, MZ_THREADS + 64);                 // workers + issuers
        MZ_TIMER(3);
        q = mz_sp_run(C, A.first[grp + 1], grp == 0 ? A.n_rounds[1] : A.n_rounds[2] - A.tail, tmem_d, mbar_mma, q, grp, gtid, tk);
        if (grp == 1 && A.tail) { mz_sp_bar_arrive(1); q += (uint32_t)A.tail; }     // the issuer syncs on it before the tail's first round
        pass++;
        MZ_TIMER(4);
        mz_named_sync(MZ_SP_BAR_WORK, MZ_THREADS);                     // both networks' outputs but the tail's are in place
        MZ_TIMER(5);
        if (active) {
            if (!A.tail) {
                float *nh = tree.hidden + (size_t)sim * P.hidden_pad;
                for (int k = ln; k < P.hidden; k += MZ_LANES) nh[k] = sp.outH[k * MZ_SP_OS + r];
            }
            MZ_TIMER(6);
            float rw = sp.outR[r], vl = sp.outV[r];
            if (tanh_r || tanh_v) {                                // both tanh side by side: even lanes the value, odd lanes the reward
                float x = (ln & 1) ? rw : vl;
                if ((ln & 1) ? tanh_r : tanh_v) x = mz_tanhf(x);
                vl = __shfl_sync(segmask, x, 0, MZ_LANES); rw = __shfl_sync(segmask, x, 1, MZ_LANES);
            }
            mz_tree_expand_lanes(P, tree, leaf.node, sim, root.legal, sp.outL + r, rw, leaf.prior, ln, segmask, MZ_SP_OS);
            MZ_TIMER(7);
            mz_tree_backup_lanes(P, tree, path, leaf.depth, vl, mm, ln, segmask);
        }
        MZ_TIMER(8);
    }

    MZ_KSTAMP(5);
    MZ_TIMER_FLUSH(a.stats);
#ifdef MZ_PHASE_TIMERS
    // rounds timed: the tail's rounds run on the tail team
    if (a.stats && tk) { int o_ = tid == 0 ? 16 : 24; for (int i_ = 0; i_ < 6; i_++) atomicAdd(&a.stats[o_ + i_], (unsigned long long)rt[i_]); atomicAdd(&a.stats[o_ + 6], (unsigned long long)(q - (tid == 0 ? 0u : (uint32_t)A.tail * pass))); }
#endif
    if (active && ln == 0) mz_root_finish<MODE>(P, a, g, tree, root, depth_sum);
    } else {
    for (int sim = 1; sim <= P.S; sim++) {
        if (issuer) {
            mz_named_sync(MZ_SP_BAR_SIM, MZ_THREADS + 64);
            q = mz_sp_run_issuer(C, A.first[grp + 1], grp == 0 ? A.n_rounds[1] : A.n_rounds[2] - A.tail, tmem_d, mbar_mma, q, pass, grp, nullptr, 0u, grp == 1 ? ply : 0u);
            pass++;
        }
        if (A.tail) {               // the tail team: warp 8 is done with prediction, warp 9 goes on issuing, warps 10, 11 only run tails
            const uint32_t qt = mz_sp_tail(P, a, sp.outH, sp.active, C, A.first[2] + A.n_rounds[2] - A.tail, A.tail, tmem_base + 128u, mz_smem_u32(sp.mbar_mma[1]),
                                           issuer && grp == 1 ? q : (uint32_t)((ply + 1) * A.n_rounds[0] + (ply * P.S + sim - 1) * A.n_rounds[2] + A.n_rounds[2] - A.tail),
                                           pass - 1u, ply, gtid, sim, mz_smem_u32(sp.mbar_tail));
            if (issuer && grp == 1) q = qt;
        }
    }
    }
    if (!persist) break;
    __syncthreads();                                                    // the epilogues' slot updates are visible to the CTA: the next ply starts from them
    {
        int more = 0;
        const int64_t gg = (int64_t)blockIdx.x * MZ_ROWS + tid;
        if (tid < MZ_ROWS && gg < a.n) more = a.slots.status[gg] == MZ_SLOT_ACTIVE;
        if (!__syncthreads_or(more)) break;
    }
  }
    // ---- teardown: every MMA has been waited on; weight copies still in flight (the refills after the last pass) must land before the
    //      CTA's shared memory is released ----
    if (issuer0) mz_sp_drain(C, A, grp == 0 ? 1 : 2, pass, grp == 0 ? 0u : ply);
    mz_tc_fence_before();
    __syncthreads();
    MZ_KSTAMP(6);
    MZ_KSTAMP_FLUSH(a.stats);
    if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)MZ_SP_TMEM_COLS) : "memory");
}

// batched network callable on this path (network outputs against the Float32 oracle and the oracle's emulation of the operand split)
struct mz_nn_sp_args { mz_sp_args sp; int32_t B, net; const float *in; float *out1; float *out2; };
__global__ void __launch_bounds__(MZ_SP_THREADS) mz_k_nn_forward_sp(const __grid_constant__ mz_params P, const __grid_constant__ mz_nn_sp_args a) {
    extern __shared__ __align__(1024) unsigned char mz_smem_sp[];
    const mz_sp_args &A = a.sp;
    const mz_sp_plan_s sp = mz_sp_carve(mz_smem_sp, A.warea_bytes, A.bias_floats, A.total_rounds, P.hidden_pad, P.S, A.pbc_smem);
    const int tid = threadIdx.x;
    const uint32_t tmem_base = mz_sp_setup(sp, A, MZ_SP_THREADS);
    mz_sp_ctx C; C.prog = mz_smem_u32(sp.prog); C.image = A.image; C.bars = mz_smem_u32(sp.bars);
    const bool worker = tid < MZ_THREADS;
    const int grp = worker ? tid >> 7 : (tid - MZ_THREADS) >> 5, gtid = tid & (MZ_GROUP - 1);
    const bool issuer0 = !worker && (tid & 31) == 0;
    const int rg = a.net == 1 ? 0 : 1;                                   // the group that runs this network
    if (grp == rg && issuer0) { if (a.net == 0) mz_sp_fill_many(C, A.first[0], A.n_rounds[0]); else mz_sp_prime(C, A, a.net); }
    const int in = P.layers[P.nets[a.net].first].in;
    const uint32_t tile = mz_sp_group_tile(sp, rg, 0);
    for (int i = tid; i < MZ_ROWS * in; i += MZ_SP_THREADS) {
        const int rr = i / in, k = i % in;
        const int64_t gg = (int64_t)blockIdx.x * MZ_ROWS + rr;
        mz_sp_stage(tile, k, rr, gg < a.B ? a.in[gg * in + k] : 0.0f);
    }
    mz_fence_proxy_async();
    __syncthreads();
    if (grp == rg) {
        if (worker) mz_sp_run(C, A.first[a.net], A.n_rounds[a.net], tmem_base + (uint32_t)(128 * grp), mz_smem_u32(sp.mbar_mma[grp]), 0u, grp, gtid, nullptr);
        else mz_sp_run_issuer(C, A.first[a.net], A.n_rounds[a.net], tmem_base + (uint32_t)(128 * grp), mz_smem_u32(sp.mbar_mma[grp]), 0u, 0u, grp);
    }
    __syncthreads();
    const int64_t g = (int64_t)blockIdx.x * MZ_ROWS + tid;
    if (tid < MZ_ROWS && g < a.B) {
        if (a.net == 1) {
            float logits[MZ_MAX_A], policy[MZ_MAX_A];
            for (int i = 0; i < P.A; i++) logits[i] = sp.outL[i * MZ_SP_OS + tid];
            mz_softmax(logits, P.A, policy);
            const bool th = P.layers[P.nets[1].first + P.nets[1].n_trunk + P.nets[1].n_h1 - 1].act == MZ_ACT_TANH;
            a.out1[g] = th ? mz_tanhf(sp.outV[tid]) : sp.outV[tid];
            for (int i = 0; i < P.A; i++) a.out2[g * P.A + i] = policy[i];
        } else {
            for (int k = 0; k < P.hidden; k++) a.out1[g * P.hidden + k] = sp.outH[k * MZ_SP_OS + tid];
            if (a.net == 2) {
                const bool th = P.layers[P.nets[2].first + P.nets[2].n_trunk + P.nets[2].n_h1 + P.nets[2].n_h2 - 1].act == MZ_ACT_TANH;
                a.out2[g] = th ? mz_tanhf(sp.outR[tid]) : sp.outR[tid];
            }
        }
    }
    if (grp == rg && issuer0 && a.net != 0) mz_sp_drain(C, A, a.net, 1u);
    mz_tc_fence_before();
    __syncthreads();
    if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)MZ_SP_TMEM_COLS) : "memory");
}

// ---- tensor-core weight images from the device weights (after every update of d_w: set_weights, ADAM) ----------------------------
// mode 1: MZ_NN_BF16_TC image (one bf16 block per layer), mode 2: MZ_NN_SPLIT_MMA image (hi block, lo block).  Grid = (layers, slices).
struct mz_pack_args { const float *w; unsigned char *image; float *bias; int32_t mode; int32_t off[MZ_MAX_LAYERS], bytes[MZ_MAX_LAYERS], bias_off[MZ_MAX_LAYERS]; };
__global__ void __launch_bounds__(256) mz_k_pack_images(const __grid_constant__ mz_params P, const __grid_constant__ mz_pack_args a) {
    const mz_layer &l = P.layers[blockIdx.x];
    const int L = blockIdx.x;
    // FeedForwardHP.use_batch_norm (Learning.jl:70-79): BatchNorm runs in test mode everywhere (mz_common.h: mz_batchnorm), i.e. it is the affine map
    // y = s * (W x + b - mu) + beta with s = gamma / sqrt(sigma2 + 1f-5) in front of the relu: folded into the image as W' = diag(s) W, b' = s * (b - mu) + beta
    const float *bnp = l.bn ? a.w + l.b_off + l.out_pad : nullptr;      // beta | gamma | mu | sigma2, out_pad floats each
    for (int i = blockIdx.y * 256 + threadIdx.x; i < l.in * l.out; i += 256 * gridDim.y) {
        const int k = i / l.out, o = i - k * l.out;
        float w = a.w[l.w_off + k * l.out_pad + o];
        if (bnp) w = w * (bnp[l.out_pad + o] / sqrtf(bnp[3 * l.out_pad + o] + 1e-5f));
        const uint32_t off = (uint32_t)a.off[L] + mz_tc_tile_offset(o, k);
        if (a.mode == 2) {
            unsigned short hi, lo; mz_sp_split(w, hi, lo);
            *reinterpret_cast<unsigned short *>(a.image + off) = hi;
            *reinterpret_cast<unsigned short *>(a.image + off + a.bytes[L]) = lo;
        } else *reinterpret_cast<unsigned short *>(a.image + off) = __bfloat16_as_ushort(__float2bfloat16_rn(w));
    }
    if (blockIdx.y == 0) for (int o = threadIdx.x; o < l.out; o += 256) {
        float b = a.w[l.b_off + o];
        if (bnp) b = (bnp[l.out_pad + o] / sqrtf(bnp[3 * l.out_pad + o] + 1e-5f)) * (b - bnp[2 * l.out_pad + o]) + bnp[o];
        a.bias[a.bias_off[L] + o] = b;
    }
}

// ---- learner: the K-step unroll forward (src/Learning.jl:347-370, Q19) with the networks on this path ------------------------------
// Same schedule as mz_k_learn_forward (32 samples per CTA, prediction(h_i) || dynamics(h_i, a_i) on the two groups), the layers as
// split-precision tcgen05 rounds.  Used when the context's nn_mode is MZ_NN_SPLIT_MMA and grad_mode = MZ_GRAD_REFERENCE_L2: the
// reference's gradient does not depend on the forward pass (Q20: 2 * theta), so the update stays bit-identical to the exact path
// and only the reported losses carry the ~1e-6 of the tensor-core arithmetic.
struct mz_learn_sp_args { mz_sp_args sp; int32_t B; mz_batch batch; float *pred_values, *pred_rewards, *pred_policies; };
__global__ void __launch_bounds__(MZ_SP_THREADS) mz_k_learn_forward_sp(const __grid_constant__ mz_params P, const __grid_constant__ mz_learn_sp_args a) {
    extern __shared__ __align__(1024) unsigned char mz_smem_sp[];
    const mz_sp_args &A = a.sp;
    const mz_sp_plan_s sp = mz_sp_carve(mz_smem_sp, A.warea_bytes, A.bias_floats, A.total_rounds, P.hidden_pad, P.S, A.pbc_smem);
    const int tid = threadIdx.x, K1 = P.K + 1;
    const uint32_t tmem_base = mz_sp_setup(sp, A, MZ_SP_THREADS);
    mz_sp_ctx C; C.prog = mz_smem_u32(sp.prog); C.image = A.image; C.bars = mz_smem_u32(sp.bars);
    const bool worker = tid < MZ_THREADS;
    const int grp = worker ? tid >> 7 : (tid - MZ_THREADS) >> 5, gtid = tid & (MZ_GROUP - 1);
    const bool issuer0 = !worker && (tid & 31) == 0;
    if (issuer0) { if (grp == 0) mz_sp_prime(C, A, 1); else mz_sp_fill_many(C, A.first[0], A.n_rounds[0]); }
    const uint32_t tmem_d = tmem_base + (uint32_t)(128 * grp), mbar_mma = mz_smem_u32(sp.mbar_mma[grp]);
    const uint32_t in_pred = mz_sp_group_tile(sp, 0, 0), in_dyn = mz_sp_group_tile(sp, 1, 0);
    const bool tanh_v = P.layers[P.nets[1].first + P.nets[1].n_trunk + P.nets[1].n_h1 - 1].act == MZ_ACT_TANH;
    const bool tanh_r = P.layers[P.nets[2].first + P.nets[2].n_trunk + P.nets[2].n_h1 + P.nets[2].n_h2 - 1].act == MZ_ACT_TANH;
    const int64_t g = (int64_t)blockIdx.x * MZ_ROWS + tid;
    const bool row_ok = tid < MZ_ROWS && g < a.B;
    uint32_t q = 0, pass = 0;
    for (int i = tid; i < MZ_ROWS * P.stack_size; i += MZ_SP_THREADS) {
        const int rr = i / P.stack_size, k = i % P.stack_size;
        const int64_t gg = (int64_t)blockIdx.x * MZ_ROWS + rr;
        mz_sp_stage(in_dyn, k, rr, gg < a.B ? a.batch.obs[gg * P.stack_size + k] : 0.0f);
    }
    mz_fence_proxy_async();
    __syncthreads();
    if (grp == 1) {                                                     // representation (:347); then the dynamics weights take its place
        if (worker) q = mz_sp_run(C, A.first[0], A.n_rounds[0], tmem_d, mbar_mma, q, grp, gtid, nullptr);
        else { q = mz_sp_run_issuer(C, A.first[0], A.n_rounds[0], tmem_d, mbar_mma, q, 0u, grp); if (issuer0 && P.K > 0) mz_sp_prime(C, A, 2); }
    }
    __syncthreads();
    const int n_eval = P.K > 0 ? P.K : 1;
    const bool dyn = P.K > 0;
    for (int e = 0; e < n_eval; e++) {                                  // evaluation e: prediction(h_e) || dynamics(h_e, a_e)
        for (int i = tid; i < MZ_ROWS * P.hidden; i += MZ_SP_THREADS) {
            const int k = i / MZ_ROWS, rr = i % MZ_ROWS;
            const float h = sp.outH[k * MZ_SP_OS + rr];
            mz_sp_stage(in_pred, k, rr, h);
            if (dyn) mz_sp_stage(in_dyn, k, rr, h * 2.0f);             // make_dynamics_input (:293-304): state * 2 (a copy), action plane = Float32(a) / A
        }
        if (dyn && tid < MZ_ROWS) {
            const float plane = row_ok ? a.batch.actions[g * K1 + e] / (float)P.A : 0.0f;
            for (int k = P.obs_size; k < P.sa_size; k++) mz_sp_stage(in_dyn, k, tid, plane);
        }
        mz_fence_proxy_async();
        __syncthreads();
        if (grp == 0 || dyn) {
            const int net = grp == 0 ? 1 : 2;
            if (worker) q = mz_sp_run(C, A.first[net], A.n_rounds[net], tmem_d, mbar_mma, q, grp, gtid, nullptr);
            else q = mz_sp_run_issuer(C, A.first[net], A.n_rounds[net], tmem_d, mbar_mma, q, pass, grp);
            pass++;
        }
        __syncthreads();
        if (row_ok) {   // evaluation e is row e + 1, and also row 0 when e == 0 (Q19: row i >= 1 = prediction(h_{i-1})); rewards: row 0 = 0 (:352)
            float logits[MZ_MAX_A], policy[MZ_MAX_A];
            for (int k = 0; k < P.A; k++) logits[k] = sp.outL[k * MZ_SP_OS + tid];
            mz_softmax(logits, P.A, policy);
            const float v = tanh_v ? mz_tanhf(sp.outV[tid]) : sp.outV[tid];
            const float rw = dyn ? (tanh_r ? mz_tanhf(sp.outR[tid]) : sp.outR[tid]) : 0.0f;
            for (int rr = (e == 0 ? 0 : e + 1); rr <= (dyn ? e + 1 : 0); rr++) {
                a.pred_values[g * K1 + rr] = v;
                for (int k = 0; k < P.A; k++) a.pred_policies[(g * K1 + rr) * P.A + k] = policy[k];
                a.pred_rewards[g * K1 + rr] = rr == 0 ? 0.0f : rw;
            }
        }
        __syncthreads();                                                // outH = h_{e+1} is staged at the top of the next evaluation
    }
    if (issuer0) mz_sp_drain(C, A, grp == 0 ? 1 : 2, pass);
    mz_tc_fence_before();
    __syncthreads();
    if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)MZ_SP_TMEM_COLS) : "memory");
}
