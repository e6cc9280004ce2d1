// mz_device.cuh -- sm_100a device machinery shared by the kernels of libmuzero_b200:
//   * mbarrier + cp.async.bulk (TMA 1-D bulk copy) weight pipeline: each Dense layer's padded {W,b} block is
//     staged global -> shared by one elected thread while the previous layer computes;
//   * the exact-fp32 Dense tile: 32 rows x out_pad columns per 128-thread group, 4x4 register tiles,
//     sequential-k fmaf (bit-identical to the arithmetic contract in DESIGN.md);
//   * two independent 128-thread groups per CTA (named barriers), so prediction(parent) and dynamics(parent, a)
//     -- which are data-independent (SURVEY Q5) -- run concurrently, each with its own weight pipeline.
#pragma once
#include <cuda_runtime.h>
#include "mz_common.h"

#define MZ_ROWS 32          // rows (trees / samples) per CTA
#define MZ_GROUP 128        // threads per network group
#define MZ_THREADS 256      // two groups
#ifndef MZ_KUNROLL
#define MZ_KUNROLL 4     // k-steps unrolled in the exact dense tile (measured: 4 beats 2 and 8 on B200)
#endif
#define MZ_PRAGMA_(x) _Pragma(#x)
#define MZ_PRAGMA(x) MZ_PRAGMA_(x)
#define MZ_UNROLL_K MZ_PRAGMA(unroll MZ_KUNROLL)
#define MZ_LANES 8          // lanes cooperating on one tree in the tree phases (MZ_THREADS / MZ_ROWS)

__device__ __forceinline__ uint32_t mz_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mz_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mz_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mz_fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mz_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mz_smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void mz_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(mz_smem_u32(dst)), "l"(src), "r"(bytes), "r"(mz_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mz_mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(mz_smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a lost bulk copy must fault the kernel, never hang the GPU
__device__ __forceinline__ void mz_mbar_wait(uint64_t *bar, uint32_t parity) {
    for (uint32_t spin = 0; !mz_mbar_try_wait(bar, parity); spin++)
        if (spin > (1u << 24)) __trap();
}
__device__ __forceinline__ void mz_fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// named barrier over one 128-thread group (ids 1 and 2; 0 is __syncthreads)
__device__ __forceinline__ void mz_group_sync(int grp) { asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(MZ_GROUP) : "memory"); }

__device__ __forceinline__ float4 mz_lds128(uint32_t addr) {
    float4 v;
    asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void mz_sts128(uint32_t addr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

struct mz_nn_pipe {          // one per group
    float *wbuf[2];
    uint64_t *mbar;          // [2]
    const float *wglob;      // padded device blob
    uint32_t q;              // layers executed so far by this group (uniform within the group)
    int grp, gtid;
};

__device__ __forceinline__ void mz_nn_issue(const mz_nn_pipe &s, const mz_params &P, int layer, uint32_t slot) {
    const mz_layer &L = P.layers[layer];
    uint32_t bytes = (uint32_t)L.floats * 4u;
    mz_mbar_expect_tx(&s.mbar[slot], bytes);
    mz_bulk_g2s(s.wbuf[slot], s.wglob + L.w_off, bytes, &s.mbar[slot]);
}

__device__ __noinline__ float mz_tanhf_ni(float x) { return mz_tanhf(x); }

// one k-step of the 4x4 register tile with packed fp32 FMA (fma.rn.f32x2, sm_100+): two IEEE round-to-nearest FMAs per
// instruction, bit-identical to 16 scalar fmaf: acc[i][j] = fmaf(w[j], x[i], acc[i][j])
__device__ __forceinline__ void mz_fma_step(unsigned long long (&acc2)[4][2], const float4 wv, const float4 xv) {
    unsigned long long w01, w23;
    asm("mov.b64 %0, {%1, %2};" : "=l"(w01) : "f"(wv.x), "f"(wv.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(w23) : "f"(wv.z), "f"(wv.w));
    const float xi[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        unsigned long long xx;
        asm("mov.b64 %0, {%1, %1};" : "=l"(xx) : "f"(xi[i]));
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][0]) : "l"(w01), "l"(xx));
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[i][1]) : "l"(w23), "l"(xx));
    }
}   // keeps the (rare) tanh out of the hot epilogue code

// y[o][row] = act( sum_k fmaf(W[k][o], x[k][row]) + b[o] ),  activations k-major: x[k*32 + row].
// SAVE also streams the outputs to global memory in the same k-major [o][32] layout (the learner's backward pass reads
// them back as the next layer's input activations).
// bn: the layer is followed by BatchNorm in test mode (FeedForwardHP.use_batch_norm, Learning.jl:70-79); beta | gamma | mu | sigma2 lie behind the bias
template <bool SAVE>
__device__ __forceinline__ void mz_dense_tile_body(int in, int out_pad, int act, uint32_t w_smem, uint32_t src_smem, uint32_t dst_smem, int gtid, float *gsave, int bn = 0) {
    const int lane = gtid & 31, warp = gtid >> 5;
    const int rg = lane & 7;
    const int opq = out_pad >> 2;
    const uint32_t wstride = (uint32_t)out_pad * 4u;
    for (int g = (warp << 2) | (lane >> 3); g < opq; g += 16) {
        // packed fp32 FMA (fma.rn.f32x2, sm_100+): two IEEE round-to-nearest FMAs per instruction, so the result is
        // bit-identical to 16 scalar fmaf per k while the FMA pipe sees half the instructions
        unsigned long long acc2[4][2];
#pragma unroll
        for (int i = 0; i < 4; i++) { acc2[i][0] = 0ull; acc2[i][1] = 0ull; }
        uint32_t wa = w_smem + (uint32_t)g * 16u;
        uint32_t xa = src_smem + (uint32_t)rg * 16u;
MZ_UNROLL_K
        for (int k = 0; k < in; k++) {
            mz_fma_step(acc2, mz_lds128(wa), mz_lds128(xa));
            wa += wstride; xa += MZ_ROWS * 4;
        }
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            asm("mov.b64 {%0, %1}, %2;" : "=f"(acc[i][0]), "=f"(acc[i][1]) : "l"(acc2[i][0]));
            asm("mov.b64 {%0, %1}, %2;" : "=f"(acc[i][2]), "=f"(acc[i][3]) : "l"(acc2[i][1]));
        }
        const float4 bv = mz_lds128(w_smem + (uint32_t)in * wstride + (uint32_t)g * 16u);
        const float bj[4] = {bv.x, bv.y, bv.z, bv.w};
        float bnp[4][4];                                           // [beta, gamma, mu, sigma2][j]
        if (bn) {
#pragma unroll
            for (int q = 0; q < 4; q++) { const float4 t = mz_lds128(w_smem + (uint32_t)(in + 1 + q) * wstride + (uint32_t)g * 16u); bnp[q][0] = t.x; bnp[q][1] = t.y; bnp[q][2] = t.z; bnp[q][3] = t.w; }
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            float4 r;
            r.x = acc[0][j] + bj[j]; r.y = acc[1][j] + bj[j]; r.z = acc[2][j] + bj[j]; r.w = acc[3][j] + bj[j];
            if (bn) { r.x = mz_batchnorm(r.x, bnp[0][j], bnp[1][j], bnp[2][j], bnp[3][j]); r.y = mz_batchnorm(r.y, bnp[0][j], bnp[1][j], bnp[2][j], bnp[3][j]);
                      r.z = mz_batchnorm(r.z, bnp[0][j], bnp[1][j], bnp[2][j], bnp[3][j]); r.w = mz_batchnorm(r.w, bnp[0][j], bnp[1][j], bnp[2][j], bnp[3][j]); }
            if (act == MZ_ACT_RELU) { r.x = fmaxf(r.x, 0.0f); r.y = fmaxf(r.y, 0.0f); r.z = fmaxf(r.z, 0.0f); r.w = fmaxf(r.w, 0.0f); }
            else if (act == MZ_ACT_TANH) { r.x = mz_tanhf_ni(r.x); r.y = mz_tanhf_ni(r.y); r.z = mz_tanhf_ni(r.z); r.w = mz_tanhf_ni(r.w); }
            mz_sts128(dst_smem + (uint32_t)((4 * g + j) * MZ_ROWS * 4) + (uint32_t)rg * 16u, r);
            if (SAVE) *reinterpret_cast<float4 *>(gsave + (4 * g + j) * MZ_ROWS + rg * 4) = r;
        }
    }
}

// One copy of each in the binary (noinline): every layer of every network goes through them.
__device__ __noinline__ void mz_dense_tile(int in, int out_pad, int act, uint32_t w_smem, uint32_t src_smem, uint32_t dst_smem, int gtid) {
    mz_dense_tile_body<false>(in, out_pad, act, w_smem, src_smem, dst_smem, gtid, nullptr);
}
__device__ __noinline__ void mz_dense_tile_bn(int in, int out_pad, int act, uint32_t w_smem, uint32_t src_smem, uint32_t dst_smem, int gtid) {
    mz_dense_tile_body<false>(in, out_pad, act, w_smem, src_smem, dst_smem, gtid, nullptr, 1);
}
__device__ __noinline__ void mz_dense_tile_save(int in, int out_pad, int act, uint32_t w_smem, uint32_t src_smem, uint32_t dst_smem, int gtid, float *gsave) {
    mz_dense_tile_body<true>(in, out_pad, act, w_smem, src_smem, dst_smem, gtid, gsave);
}

// One layer for one group: prefetch `next` (or nothing when next < 0) into the other buffer, wait for this layer's
// weights, compute, group barrier.  Preconditions: this layer's copy was issued earlier; a barrier separates the last
// reads of the other buffer (layer q-1) and of `dst`'s previous contents from this call.
// BN: the kernel was instantiated for use_batch_norm networks.  A template parameter, not a run-time test: with the test (or the BatchNorm
// epilogue inside mz_dense_tile) the ordinary networks' search kernel ran 9 - 20 % slower (88 - 98 M instead of 107 M simulations/s).
template <bool BN = false>
__device__ __forceinline__ void mz_nn_layer(mz_nn_pipe &s, const mz_params &P, int layer, int next, const float *src, float *dst) {
    if (s.gtid == 0 && next >= 0) mz_nn_issue(s, P, next, (s.q + 1) & 1u);
    mz_mbar_wait(&s.mbar[s.q & 1u], (s.q >> 1) & 1u);
    const mz_layer &L = P.layers[layer];
    if (BN && L.bn) mz_dense_tile_bn(L.in, L.out_pad, L.act, mz_smem_u32(s.wbuf[s.q & 1u]), mz_smem_u32(src), mz_smem_u32(dst), s.gtid);
    else mz_dense_tile(L.in, L.out_pad, L.act, mz_smem_u32(s.wbuf[s.q & 1u]), mz_smem_u32(src), mz_smem_u32(dst), s.gtid);
    mz_group_sync(s.grp);
    s.q++;
}
template <bool BN = false>
__device__ __forceinline__ void mz_nn_chain(mz_nn_pipe &s, const mz_params &P, int first, int n, int after, const float *src,
                                            float *dst, float *t0, float *t1) {
    const float *cur = src;
    for (int i = 0; i < n; i++) {
        float *d = (i == n - 1) ? dst : ((i & 1) ? t1 : t0);
        mz_nn_layer<BN>(s, P, first + i, (i == n - 1) ? after : first + i + 1, cur, d);
        cur = d;
    }
}
// trunk -> bufT, head 1 -> h1dst, head 2 -> h2dst (Split, src/Learning.jl:60-68); `after` = layer prefetched last
template <bool BN = false>
__device__ __noinline__ void mz_nn_net(mz_nn_pipe &s, const mz_params &P, int net, int after, const float *src, float *bufT,
                                       float *h1dst, float *h2dst, float *t0, float *t1) {
    const mz_net &N = P.nets[net];
    int f = N.first;
    if (N.n_h1 == 0) { mz_nn_chain<BN>(s, P, f, N.n_trunk, after, src, h1dst, t0, t1); return; }
    mz_nn_chain<BN>(s, P, f, N.n_trunk, f + N.n_trunk, src, bufT, t0, t1);
    mz_nn_chain<BN>(s, P, f + N.n_trunk, N.n_h1, f + N.n_trunk + N.n_h1, bufT, h1dst, t0, t1);
    mz_nn_chain<BN>(s, P, f + N.n_trunk + N.n_h1, N.n_h2, after, bufT, h2dst, t0, t1);
}

// shared-memory carve-up used by every NN-running kernel
struct mz_smem_plan {
    float *wbuf[2][2]; uint64_t *mbar[2];        // per group
    float *bufT[2], *t0[2], *t1[2];              // per group scratch activations
    float *in0, *in1;                            // staged inputs: in0 = representation / dynamics input, in1 = prediction input
    float *outV, *outL, *outR, *outH;            // value (4 rows), policy logits (16), reward (4), hidden (hidden_pad)
    double *pbc0, *sqrtN;
    uint16_t *path;                              // [32][S+2] selection paths
};
__host__ __device__ inline size_t mz_smem_bytes(int max_dim, int max_layer_floats, int hidden_pad, int S) {
    size_t w = ((size_t)max_layer_floats * 4 + 127) & ~(size_t)127;
    size_t buf = (size_t)max_dim * MZ_ROWS * 4;
    size_t small = (size_t)(4 + 16 + 4) * MZ_ROWS * 4 + (size_t)hidden_pad * MZ_ROWS * 4;
    size_t tab = (((size_t)S + 2) * 8 * 2 + 127) & ~(size_t)127;
    size_t path = (((size_t)S + 2) * 2 * MZ_ROWS + 127) & ~(size_t)127;
    return 4 * w + 128 + 8 * buf + small + tab + path + 128;
}
__device__ __forceinline__ mz_smem_plan mz_smem_carve(unsigned char *base, int max_dim, int max_layer_floats, int hidden_pad, int S) {
    mz_smem_plan p;
    size_t w = ((size_t)max_layer_floats * 4 + 127) & ~(size_t)127;
    size_t buf = (size_t)max_dim * MZ_ROWS * 4;
    unsigned char *c = base;
    for (int g = 0; g < 2; g++) for (int i = 0; i < 2; i++) { p.wbuf[g][i] = (float *)c; c += w; }
    p.mbar[0] = (uint64_t *)c; p.mbar[1] = (uint64_t *)(c + 32); c += 128;
    p.in0 = (float *)c; c += buf;                // in0, in1, bufT[0..1], t0[0..1], t1[0..1] are contiguous (zeroed together)
    p.in1 = (float *)c; c += buf;
    for (int g = 0; g < 2; g++) { p.bufT[g] = (float *)c; c += buf; p.t0[g] = (float *)c; c += buf; p.t1[g] = (float *)c; c += buf; }
    p.outV = (float *)c; c += 4 * MZ_ROWS * 4;
    p.outL = (float *)c; c += 16 * MZ_ROWS * 4;
    p.outR = (float *)c; c += 4 * MZ_ROWS * 4;
    p.outH = (float *)c; c += (size_t)hidden_pad * MZ_ROWS * 4;
    p.pbc0 = (double *)c; p.sqrtN = p.pbc0 + (S + 2); c += (((size_t)S + 2) * 8 * 2 + 127) & ~(size_t)127;
    p.path = (uint16_t *)c;
    return p;
}
// both pipes are initialised by thread 0 of the CTA; every thread builds the descriptor of its own group
__device__ __forceinline__ void mz_pipe_init(mz_nn_pipe &s, const mz_smem_plan &sp, const float *wglob) {
    s.grp = threadIdx.x / MZ_GROUP; s.gtid = threadIdx.x & (MZ_GROUP - 1);
    s.wbuf[0] = sp.wbuf[s.grp][0]; s.wbuf[1] = sp.wbuf[s.grp][1]; s.mbar = sp.mbar[s.grp]; s.wglob = wglob; s.q = 0;
    if (threadIdx.x == 0) {
        mz_mbar_init(&sp.mbar[0][0], 1); mz_mbar_init(&sp.mbar[0][1], 1); mz_mbar_init(&sp.mbar[1][0], 1); mz_mbar_init(&sp.mbar[1][1], 1);
        mz_fence_mbar_init();
    }
}
__device__ __forceinline__ void mz_zero_activations(const mz_smem_plan &sp, int max_dim) {
    for (int i = threadIdx.x; i < 8 * max_dim * MZ_ROWS; i += MZ_THREADS) sp.in0[i] = 0.0f;
}
