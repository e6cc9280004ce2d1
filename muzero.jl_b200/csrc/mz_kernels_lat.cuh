// mz_kernels_lat.cuh -- mz_k_search_lat: run_mcts / play_game for FEW roots (src/SelfPlay.jl:230-285, 330-382).
//
// The batched search kernels put 32 trees on one SM and stream the weights through shared memory layer by layer; one move costs them the
// same ~0.9-1.7 ms whether 1 or 4096 trees are searched, which made the call the reference makes -- one root at a time -- slower on the
// GPU than on a CPU core.  This kernel is the opposite trade: ONE tree per thread-block CLUSTER of two SMs, everything resident.
//   * CTA 0 keeps the representation + prediction networks (fp32, TMA bulk copies at kernel start), the whole tree (node records and
//     hidden states, tree_stride_bytes) and the compact PUCT table in its shared memory: a selection level is a shared-memory access,
//     not an L2 round trip;
//   * CTA 1 keeps the dynamics network; the two run prediction(parent) and dynamics(parent, a) concurrently (SURVEY Q5).  The staged
//     dynamics input travels CTA 0 -> CTA 1 and (next hidden state, reward) CTA 1 -> CTA 0 through distributed shared memory, ordered
//     by the cluster barrier (barrier.cluster arrive.release / wait.acquire), twice per simulation.
//   * a Dense layer is one output feature per thread with the arithmetic contract's sequential-k fmaf chain (DESIGN.md 3.1), so the
//     results are BIT-IDENTICAL to mz_k_search and the Float32 oracle; trunk layers use 64 threads, the two heads of a network the two
//     halves of the CTA.
//   * the tree phases are the lane-parallel routines of mz_kernels.cuh (8 lanes), pointed at shared memory.
// Grid = 2 x roots; up to 74 roots run concurrently on a B200.
#pragma once
#include <cooperative_groups.h>
#include "mz_kernels.cuh"

#define MZ_LAT_THREADS 128
#define MZ_LAT_HALF 64

struct mz_lat_plan {
    float *w;                                       // this CTA's networks, layer l at w + loc[l]
    float *xin, *xdyn, *bufT, *tb; int md;          // staged inputs (CTA 0: representation / prediction, CTA 1: dynamics), trunk output, ping / pong per half:
                                                    // buffer (half, i) = tb + (2 * half + i) * md -- arithmetic, not a pointer table (which lands in local memory)
    float *outV, *outL, *outR, *outH;               // CTA 0: value, logits, reward, hidden state of the evaluated leaf
    unsigned char *tree; double *pbc; uint16_t *path; int4 *lay; int32_t *gofs; uint64_t *mbar, *lbar;
};
MZ_HD size_t mz_lat_smem_bytes(int w_floats, int max_dim, int hidden_pad, int tree_bytes, int S, int pbc_smem) {
    size_t w = ((size_t)w_floats * 4 + 256 + 127) & ~(size_t)127;   // + slack: a row fetch reads 64 floats whatever `in` is
    size_t md = ((size_t)(max_dim > 64 ? max_dim : 64) * 4 + 15) & ~(size_t)15;
    size_t out = ((size_t)(4 + 16 + 4 + (hidden_pad > 64 ? hidden_pad : 64)) * 4 + 127) & ~(size_t)127;   // outH is also a layer INPUT (root prediction): 64 readable floats
    size_t tree = ((size_t)tree_bytes + 127) & ~(size_t)127;
    size_t tab = pbc_smem ? ((((size_t)S + 2) * ((size_t)S + 3) / 2) * 8 + 127) & ~(size_t)127 : 0;
    size_t path = (((size_t)S + 2) * 2 + 127) & ~(size_t)127;
    return 128 + w + 7 * md + out + tree + tab + path + MZ_MAX_LAYERS * 20 + 128;
}
__device__ __forceinline__ mz_lat_plan mz_lat_carve(unsigned char *c, int w_floats, int max_dim, int hidden_pad, int tree_bytes, int S, int pbc_smem) {
    mz_lat_plan p;
    const size_t md = ((size_t)(max_dim > 64 ? max_dim : 64) * 4 + 15) & ~(size_t)15;
    p.w = (float *)c; c += ((size_t)w_floats * 4 + 256 + 127) & ~(size_t)127;
    p.xin = (float *)c; c += md; p.xdyn = (float *)c; c += md; p.bufT = (float *)c; c += md;
    p.tb = (float *)c; p.md = (int)(md / 4); c += 4 * md;
    p.outV = (float *)c; p.outL = p.outV + 4; p.outR = p.outV + 20; p.outH = p.outV + 24; c += ((size_t)(24 + (hidden_pad > 64 ? hidden_pad : 64)) * 4 + 127) & ~(size_t)127;
    p.tree = c; c += ((size_t)tree_bytes + 127) & ~(size_t)127;
    p.pbc = (double *)c; c += pbc_smem ? ((((size_t)S + 2) * ((size_t)S + 3) / 2) * 8 + 127) & ~(size_t)127 : 0;
    p.path = (uint16_t *)c; c += (((size_t)S + 2) * 2 + 127) & ~(size_t)127;
    p.lay = (int4 *)c; p.gofs = (int32_t *)(c + MZ_MAX_LAYERS * 16); p.mbar = (uint64_t *)(c + MZ_MAX_LAYERS * 20); p.lbar = p.mbar + 1;
    return p;
}

// ---- weight image of this kernel (built on the device from the padded blob by mz_k_pack_lat whenever the weights change) ----------
// layer l = [out][RS] floats, row o = the weights of output o over its inputs (W[k][o] transposed, zero beyond `in`), followed by the
// biases (out rounded up to 4).  RS = 4 * odd >= in rounded up to 4: a thread reads its row with 16-byte loads and the rows of a
// quarter-warp fall into different banks.
MZ_HD int mz_lat_rs(int in) { int q = (in + 3) / 4; if ((q & 1) == 0) q++; return 4 * q; }
MZ_HD int mz_lat_layer_floats(int in, int out) { return out * mz_lat_rs(in) + ((out + 3) & ~3); }
struct mz_pack_lat_args { const float *w; float *image; int32_t off[MZ_MAX_LAYERS]; };
__global__ void __launch_bounds__(256) mz_k_pack_lat(const __grid_constant__ mz_params P, const __grid_constant__ mz_pack_lat_args a) {
    const mz_layer &l = P.layers[blockIdx.x];
    const int rs = mz_lat_rs(l.in);
    float *img = a.image + a.off[blockIdx.x];
    for (int i = blockIdx.y * 256 + threadIdx.x; i < l.out * rs; i += 256 * gridDim.y) {
        const int o = i / rs, k = i - o * rs;
        img[i] = k < l.in ? a.w[l.w_off + k * l.out_pad + o] : 0.0f;
    }
    if (blockIdx.y == 0) for (int o = threadIdx.x; o < ((l.out + 3) & ~3); o += 256) img[l.out * rs + o] = o < l.out ? a.w[l.b_off + o] : 0.0f;
}

// y[t] = act(sum_k fmaf(W[k][t], x[k]) + b[t]) for one sample, thread t = output feature: the accumulation order of mz_dense_tile.
// The weights of a layer do not depend on its input, so a thread fetches its row into registers while it waits for the input
// (mz_lat_preload); what is left on the critical path of a layer is the broadcast loads of x and the dependent fmaf chain.
#define MZ_LAT_KMAX 64
struct mz_lat_col { float4 w[MZ_LAT_KMAX / 4]; float b; int in, out, act; };
__device__ __forceinline__ void mz_lat_preload(mz_lat_col &c, const mz_lat_plan &sp, int l, int t) {
    const int4 L = sp.lay[l];                                            // x = in, y = RS, z = out | act << 16, w = float offset of the block
    c.in = L.x; c.out = L.z & 0xffff; c.act = L.z >> 16;
    if (t < c.out) {
        const uint32_t row = mz_smem_u32(sp.w + L.w) + 4u * (uint32_t)(t * L.y);
#pragma unroll
        for (int k4 = 0; k4 < MZ_LAT_KMAX / 4; k4++) c.w[k4] = (4 * k4 < L.y) ? mz_lds128(row + 16u * (uint32_t)k4) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);   // rows are RS floats long, zero beyond `in`
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(c.b) : "r"(mz_smem_u32(sp.w + L.w) + 4u * (uint32_t)(c.out * L.y + t)));
    }
}
// `fetch_next` runs between the loads of the input vector and the fmaf chain: the fetch of the next layer's weight row (64 shared-memory
// wavefronts per warp) must not be queued in FRONT of the 16 broadcast loads the chain waits for
template <typename F>
__device__ __forceinline__ void mz_lat_apply(const mz_lat_col &c, const float *x, float *y, int t, F fetch_next) {
    const uint32_t xa = mz_smem_u32(x);
    float4 xv[MZ_LAT_KMAX / 4];                                           // every activation buffer holds at least MZ_LAT_KMAX readable floats
#pragma unroll
    for (int k4 = 0; k4 < MZ_LAT_KMAX / 4; k4++) xv[k4] = mz_lds128(xa + 16u * (uint32_t)k4);
    fetch_next();
    if (t >= c.out) return;
    float acc = 0.0f;
    // One straight chain of 64 fmaf for every layer: the image's rows are zero beyond `in` and the activation buffers hold finite values
    // there (zeroed at kernel start, later only layer outputs), so the extra links add +-0 to the sum.  That leaves the sum unchanged
    // bit for bit (x + (+-0) = x for every x but -0, and a sum that starts at +0 only becomes -0 through an fp32 underflow).
#pragma unroll
    for (int k4 = 0; k4 < MZ_LAT_KMAX / 4; k4++) {
        acc = fmaf(c.w[k4].x, xv[k4].x, acc); acc = fmaf(c.w[k4].y, xv[k4].y, acc);
        acc = fmaf(c.w[k4].z, xv[k4].z, acc); acc = fmaf(c.w[k4].w, xv[k4].w, acc);
    }
    float r = acc + c.b;
    if (c.act == MZ_ACT_RELU) r = fmaxf(r, 0.0f);
    else if (c.act == MZ_ACT_TANH) r = mz_tanhf_ni(r);
    y[t] = r;
}
// layers wider than MZ_LAT_KMAX inputs (the representation's first layer with a deep observation stack; root only)
__device__ __noinline__ void mz_lat_dense_wide(const float *w, int in, int rs, int out, int act, const float *x, float *y, int t) {
    if (t >= out) return;
    float acc = 0.0f;
    const float *wp = w + t * rs;
    for (int k = 0; k < in; k++) acc = fmaf(wp[k], x[k], acc);
    float r = acc + w[out * rs + t];
    if (act == MZ_ACT_RELU) r = fmaxf(r, 0.0f);
    else if (act == MZ_ACT_TANH) r = mz_tanhf_ni(r);
    y[t] = r;
}
// one network on the 128 threads of the CTA: trunk on the first half, then head 1 on the first half and head 2 on the second (Split,
// src/Learning.jl:60-68).  The layer descriptors come from the shared-memory copy sp.lay: reading mz_params through a reference costs an
// L2 round trip per field, which is most of a layer's time at this size.
// A thread keeps TWO weight rows in registers: the fetch of its next layer's row is issued before the fmaf chain of the current one, so
// it costs nothing.  The layers of a chain are separated by a named barrier of the 64 threads that run it (bar.sync 1 + half, 64); the
// hand-off trunk -> heads is one barrier of all 128 threads (bar.sync 3).  The barrier that publishes the network's outputs (and the one
// that makes its input visible when `cluster_sync_first`) is the caller's: a cluster barrier during the simulations.
struct mz_lat_net_s { int first, n_trunk, n_h1, n_h2; };
__device__ __forceinline__ void mz_lat_net(const mz_lat_plan &sp, const mz_lat_net_s N, const float *src, float *h1dst, float *h2dst, bool cluster_sync_first) {
    const int half = threadIdx.x >> 6, t = threadIdx.x & (MZ_LAT_HALF - 1);
    const bool heads = N.n_h1 > 0;
    const int my_n = half == 0 ? N.n_trunk + N.n_h1 : N.n_h2;                        // my layers: half 0 = trunk then head 1, half 1 = head 2
    const int lbase = half == 0 ? N.first : N.first + N.n_trunk + N.n_h1;
    mz_lat_col c0, c1; c0.in = c0.out = c0.act = 0; c0.b = 0.0f; c1 = c0;
    const bool wide = my_n > 0 && sp.lay[lbase].x > MZ_LAT_KMAX;                     // only a network's first layer may be wider than 64 inputs
    if (my_n > 0 && !wide) mz_lat_preload(c0, sp, lbase, t);
    if (cluster_sync_first) cooperative_groups::this_cluster().sync();
    if (half == 1 && my_n > 0) asm volatile("bar.sync 3, 128;" ::: "memory");        // the trunk's output
    const float *cur = half == 0 ? src : sp.bufT;
    int i = 0;
    auto layer = [&](mz_lat_col &c, mz_lat_col &n) {
        const bool trunk = half == 0 && i < N.n_trunk;
        const bool last_of_chain = trunk ? i == N.n_trunk - 1 : i == my_n - 1;
        float *d = trunk ? (last_of_chain ? (heads ? sp.bufT : h1dst) : sp.tb + (i & 1) * sp.md) : (last_of_chain ? (half == 0 ? h1dst : h2dst) : sp.tb + (2 * half + (i & 1)) * sp.md);
        auto fetch_next = [&] { if (i + 1 < my_n) mz_lat_preload(n, sp, lbase + i + 1, t); };
        if (i == 0 && wide) { fetch_next(); const int4 L = sp.lay[lbase]; mz_lat_dense_wide(sp.w + L.w, L.x, L.y, L.z & 0xffff, L.z >> 16, cur, d, t); }
        else mz_lat_apply(c, cur, d, t, fetch_next);
        cur = d;
        if (trunk && last_of_chain && heads) asm volatile("bar.sync 3, 128;" ::: "memory");
        else if (i + 1 < my_n) asm volatile("bar.sync %0, 64;" ::"r"(half + 1) : "memory");
        i++;
    };
    while (i < my_n) {
        layer(c0, c1);
        if (i >= my_n) break;
        layer(c1, c0);
    }
}

// rarely executed, large: kept out of the simulation loop's instruction footprint
__device__ __noinline__ void mz_lat_add_noise(const mz_params &P, mz_f4 *A, float *hidden, uint32_t legal, uint32_t game, uint32_t move) { mz_tree t; t.A = A; t.hidden = hidden; mz_tree_add_noise(P, t, legal, game, move); }
struct mz_lat_args { mz_search_args base; const float *image; int32_t w_floats, pbc_smem; };

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MZ_LAT_THREADS) mz_k_search_lat(const __grid_constant__ mz_params P, const __grid_constant__ mz_lat_args la) {
    static_assert(MODE != MZ_MODE_REPLAY, "stored positions are reanalysed in bulk by the batched kernels");
    extern __shared__ __align__(128) unsigned char mz_smem_lat[];
    namespace cg = cooperative_groups;
    const mz_search_args &a = la.base;
    const int64_t g = (int64_t)(blockIdx.x >> 1);
    const int rank = (int)(blockIdx.x & 1u);
    const int tid = threadIdx.x;
    if (MODE == MZ_MODE_SLOTS) {      // both CTAs of the cluster read the same word; it changes only in the epilogue, after the last cluster barrier
        if (!(a.slots.status[g] == MZ_SLOT_ACTIVE && (P.arena_player == 0 || a.slots.player[g] == P.arena_player))) return;
    }
    const mz_lat_plan sp = mz_lat_carve(mz_smem_lat, la.w_floats, a.max_dim, P.hidden_pad, P.tree_stride_bytes, P.S, la.pbc_smem);
    cg::cluster_group cluster = cg::this_cluster();

    // ---- this CTA's networks -> shared memory (TMA bulk copies on one mbarrier) ----
    const int net_lo = rank == 0 ? 0 : 2, net_hi = rank == 0 ? 1 : 2;
    const mz_lat_net_s net_rep = {P.nets[0].first, P.nets[0].n_trunk, P.nets[0].n_h1, P.nets[0].n_h2}, net_pre = {P.nets[1].first, P.nets[1].n_trunk, P.nets[1].n_h1, P.nets[1].n_h2},
                       net_dyn = {P.nets[2].first, P.nets[2].n_trunk, P.nets[2].n_h1, P.nets[2].n_h2};
    if (tid == 0) {
        mz_mbar_init(sp.mbar, 1); mz_fence_mbar_init();
        int goff = 0, off = 0;                                            // float offsets: in the global image (all layers in order), in this CTA's area
        for (int n = 0; n < 3; n++) {
            const mz_net &N = P.nets[n];
            for (int l = N.first; l < N.first + N.n_trunk + N.n_h1 + N.n_h2; l++) {
                const mz_layer &L = P.layers[l];
                const int fl = mz_lat_layer_floats(L.in, L.out);
                if (n >= net_lo && n <= net_hi) { sp.lay[l] = make_int4(L.in, mz_lat_rs(L.in), L.out | (L.act << 16), off); sp.gofs[l] = goff; off += fl; }
                goff += fl;
            }
        }
        mz_mbar_expect_tx(sp.mbar, (uint32_t)off * 4u);
        for (int n = net_lo; n <= net_hi; n++) {
            const mz_net &N = P.nets[n];
            for (int l = N.first; l < N.first + N.n_trunk + N.n_h1 + N.n_h2; l++)
                mz_bulk_g2s(sp.w + sp.lay[l].w, la.image + sp.gofs[l], (uint32_t)mz_lat_layer_floats(P.layers[l].in, P.layers[l].out) * 4u, sp.mbar);
        }
    }
    // every buffer a layer reads its input from holds 64 readable floats, finite beyond the layer's `in` (zero weights meet them there):
    // xin, xdyn, bufT, the ping / pong buffers and the output block (outH is the root prediction's input)
    for (int i = tid; i < (int)((float *)sp.tree - sp.xin); i += MZ_LAT_THREADS) sp.xin[i] = 0.0f;
    __syncthreads();
    const int ln = tid & (MZ_LANES - 1);
    const uint32_t segmask = 0xffu;
    const bool lanes = rank == 0 && tid < MZ_LANES;                     // the 8 lanes that own the tree
    const mz_root root = mz_root_begin<MODE>(P, a, g, rank == 0);
    mz_tree tree; tree.A = (mz_f4 *)sp.tree; tree.hidden = (float *)(sp.tree + P.hidden_off_bytes);
    const double *pbc = a.pbc0;
    if (rank == 0) {
        if (la.pbc_smem) {                                              // compact copy of ucb_score's table: row N holds n = 0..N
            for (int N = tid; N < P.S + 2; N += MZ_LAT_THREADS) for (int n = 0; n <= N; n++) sp.pbc[(N * (N + 1)) / 2 + n] = a.pbc0[N * (P.S + 2) + n];
            pbc = sp.pbc;
        }
        // stacked observations (get_stacked_observations, SelfPlay.jl:128-149)
        for (int k = tid; k < P.stack_size; k += MZ_LAT_THREADS) sp.xin[k] = mz_root_obs<MODE>(P, a, g, k);
    }
    const bool active = root.active;
    __syncthreads();
    mz_mbar_wait(sp.mbar, 0);
    cluster.sync();                                                     // both CTAs are resident: distributed shared memory may be written

    // One loop for both CTAs of the cluster (one call site per routine keeps the kernel's code small: with one warp per scheduler an
    // instruction-cache miss is not hidden by anything).  Iteration -1: representation -> h0; 0: prediction(h0) -> (v0, p0), root
    // expansion + noise (SelfPlay.jl:233-249); 1..S: the simulations (:254-283).  CTA 1 only takes part in the simulations: dynamics.
    float *r_outH = cluster.map_shared_rank(sp.outH, 0), *r_outR = cluster.map_shared_rank(sp.outR, 0), *r_xdyn = cluster.map_shared_rank(sp.xdyn, 1);
    mz_minmax mm; mm.mn = INFINITY; mm.mx = -INFINITY;
    unsigned long long depth_sum = 0;
    mz_leaf leaf; leaf.node = 0; leaf.parent = 0; leaf.action = 1; leaf.depth = 0; leaf.prior = 0.0f; leaf.parent_x = 0;
#ifdef MZ_LAT_TIMERS
    long long lt[8] = {0, 0, 0, 0, 0, 0, 0, 0}, lt0 = clock64();
#define MZ_LT(i) do { long long c_ = clock64(); lt[i] += c_ - lt0; lt0 = c_; } while (0)
#else
#define MZ_LT(i)
#endif
    for (int it = rank == 0 ? -1 : 1; it <= P.S; it++) {
        MZ_LT(7);
        if (lanes && active && it >= 1) {
            leaf = mz_tree_select_lanes(P, tree, pbc, a.sqrtN, root.legal, root.posmask, mm, root.game, root.move, (uint32_t)it, ln, segmask, sp.path, la.pbc_smem != 0);
            depth_sum += (unsigned long long)leaf.depth;
            MZ_LT(0);
            const int pe = mz_nx_exp(leaf.parent_x), dbl = mz_nx_dbl(leaf.parent_x);
            const float *h = tree.hidden + (size_t)pe * P.hidden_pad;
            const float sc = mz_bits2f((uint32_t)(127 + dbl) << 23);                         // 2^dbl: state after dbl in-place doublings (Q6)
            for (int k = ln; k < P.hidden; k += MZ_LANES) {
                const float v = h[k] * sc;
                sp.xin[k] = v;                                                               // prediction(parent.hidden_state), :271 (Q5)
                r_xdyn[k] = v * 2.0f;                                                        // make_state_action: state .*= 2, :11
            }
            const float plane = P.act_plane_play[leaf.action];                               // :8-9
            for (int k = P.obs_size + ln; k < P.sa_size; k += MZ_LANES) r_xdyn[k] = plane;
            __syncwarp(segmask);
            if (ln == 0) reinterpret_cast<uint32_t *>(&tree.A[leaf.parent])[0] = leaf.parent_x + (1u << 24);   // one more doubling (Q6)
        }
        MZ_LT(1);
        {
            const mz_lat_net_s N = rank == 1 ? net_dyn : it < 0 ? net_rep : net_pre;
            const float *src = rank == 1 ? sp.xdyn : it == 0 ? sp.outH : sp.xin;
            float *d1 = rank == 1 ? r_outH : it < 0 ? sp.outH : sp.outV, *d2 = rank == 1 ? r_outR : sp.outL;
            mz_lat_net(sp, N, src, d1, d2, it >= 1);
        }
        MZ_LT(3);
        if (it >= 1) cluster.sync();                                                         // both networks' outputs are visible; dynamics' have landed in CTA 0
        else __syncthreads();
        MZ_LT(4);
        if (lanes && active && it >= 0) {
            float *nh = tree.hidden + (size_t)it * P.hidden_pad;
            for (int k = ln; k < P.hidden; k += MZ_LANES) nh[k] = sp.outH[k];
            // the root's expansion shares the simulations' call site instead of calling mz_root_init: with a second inlined expansion this
            // kernel compiled (sm_100a, -Xptxas -v, cuobjdump -sass) to 6680 instead of 6008 SASS instructions and 241 instead of 239 registers
            // in MODE_API, 8000 instead of 7320 instructions in MODE_SLOTS
            if (it == 0 && ln == 0) { mz_f4 node; node.x = mz_bits2f(mz_nx_pack(0, -1, 0)); node.y = 0.0f; node.z = 0.0f; node.w = 0.0f; tree.A[0] = node; }   // Node(prior=0), :232
            __syncwarp(segmask);
            mz_tree_expand_lanes(P, tree, it == 0 ? 0 : leaf.node, it, root.legal, sp.outL, it == 0 ? 0.0f : sp.outR[0], it == 0 ? 0.0f : leaf.prior, ln, segmask, 1);   // :245, :280 (Q7)
            MZ_LT(5);
            if (it == 0) {
                if (ln == 0 && a.exploration && P.exploration_eps != 0.0f) mz_lat_add_noise(P, tree.A, tree.hidden, root.legal, root.game, root.move);   // :247-249
                __syncwarp(segmask);
            } else mz_tree_backup_lanes(P, tree, sp.path, leaf.depth, sp.outV[0], mm, ln, segmask);                         // :281
        }
        MZ_LT(6);
    }
    if (rank == 1) return;
#ifdef MZ_LAT_TIMERS
    if (tid == 0 && g == 0) printf("lat timers (cycles / simulation): select %lld stage %lld sync1 %lld pred %lld sync2(wait dyn) %lld expand %lld backup %lld loop %lld\n",
                                   lt[0] / P.S, lt[1] / P.S, lt[2] / P.S, lt[3] / P.S, lt[4] / P.S, lt[5] / P.S, lt[6] / P.S, lt[7] / P.S);
#endif
    if (lanes && active && ln == 0) mz_root_finish<MODE>(P, a, g, tree, root, depth_sum);
}
