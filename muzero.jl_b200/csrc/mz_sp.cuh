// mz_sp.cuh -- split-precision tensor-core network path (MZ_NN_SPLIT_MMA): the Dense layers of the three networks as tcgen05.mma with
// both operands split into bf16 hi + lo parts (x = hi + lo): D = W_hi X_hi + W_lo X_hi + W_hi X_lo, fp32 accumulation in TMEM, i.e. 16
// mantissa bits per operand instead of 8.  Results track the Float32 networks to ~1e-6 (tests/test_gpu_mma.py) and the search built on
// them reproduces the Float32 oracle's visit counts on > 99 % of roots, where plain bf16 operands reach 72 %.
//
// Orientation as in mz_tc.cuh: D[out feature m][tree n] = sum_k W[m][k] X[n][k]; weights = A operand (M = 64, K-major SWIZZLE_128B,
// pre-swizzled on the host), the CTA's 32 trees = N.  What is different:
//   * activations are N-MAJOR B tiles ([k][32 trees] bf16, 64 B per k row, SWIZZLE_64B): a thread of the epilogue holds one feature
//     (= one k row of the next layer) for eight trees, which is ONE 16-byte st.shared per tile (hi, lo) instead of eight 2-byte stores.
//     The eight columns a thread receives from tcgen05.ld.16x256b.x4 are {8q + 2c + e}; it writes them as chunk c = columns
//     {8c + 2q + e}.  That permutation of the tree order is an involution, so after an even number of hidden layers the order is
//     natural again, and the final layer of a chain (fp32 outputs) undoes whatever is left (`perm`).
//   * the hi and lo tile of an activation are adjacent, so [X_hi | X_lo] is ONE N = 64 operand: a k-step is W_hi [X_hi | X_lo] (N = 64, two
//     accumulator halves) + W_lo X_hi (N = 32, onto the first half) -- two instructions and 7 KB of operand reads instead of three and 9 KB
//     (these small MMAs are bound by the shared-memory reads of their operands); the epilogue adds the two halves.
//   * weight blocks (hi + lo = 4 bytes per weight: 240 KB for prediction + dynamics) live in WEIGHT SETS that alternate between two
//     rounds of a network (mz_common.h: mz_sp_plan).  A set is refilled by TMA bulk copy the moment the MMAs of the round that used it
//     are observed complete, and waited for only when its next round is about to issue;
//   * a dedicated issuer warp per group: MMA issue, weight waits and refills never sit on the warps that run the epilogues.
//   * final tanh layers (value, reward: one output row) store the pre-activation; the 32 trees apply tanh in parallel when they read it.
#pragma once
#include "mz_tc.cuh"

#define MZ_SP_IDESC32 (MZ_TC_IDESC | (1u << 16))                                          // M = 64, N = 32, B operand MN-major (cute::UMMA::InstrDescriptor::b_major_)
#define MZ_SP_IDESC64 ((MZ_TC_IDESC & ~(0x3fu << 17)) | ((64u >> 3) << 17) | (1u << 16))    // M = 64, N = 64
#define MZ_SP_TMEM_COLS 256            // two groups x two jobs x (32 + 32) fp32 columns
#define MZ_SP_TAIL_THREADS 128         // mz_k_search_sp's tail team: warps 8..11, one per TMEM lane quadrant

struct __align__(16) mz_sp_rdesc {                  // device form of mz_sp_round: everything a round needs, shared addresses resolved
    unsigned long long a_hi[2], a_lo[2], b_hi[2];   // words  0..11: UMMA descriptors at k-step 0
    uint32_t dst[2];                                // words 12..13: hi output tile (lo = + MZ_SP_TILE_BYTES) or 0
    uint32_t f32[2];                                // words 14..15: fp32 output [m * MZ_SP_OS + tree] or 0
    uint32_t bias[2];                               // words 16..17
    int16_t ks[2], out[2];                          // words 18, 19
    int16_t act[2], perm[2];                        // words 20, 21
    int16_t njobs, ncopy, set, next;                // words 22, 23
    uint32_t wbytes;                                // word  24
    uint16_t per_pass, ord;                         // word  25: fills of this round's set per network pass (0: never refilled); which of them this round consumes
    uint32_t copy_dst[2], copy_bytes[2]; int32_t copy_src[2];   // words 26..31
};
static_assert(sizeof(mz_sp_rdesc) == MZ_SP_RDESC_BYTES, "mz_sp_rdesc size");
__device__ __forceinline__ uint4 mz_lds_u4(uint32_t addr) { uint4 v; asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr)); return v; }
__device__ __forceinline__ uint64_t mz_u64(uint32_t lo, uint32_t hi) { return (uint64_t)lo | ((uint64_t)hi << 32); }

// K-major SWIZZLE_128B A descriptor = mz_tc_desc.  N-major SWIZZLE_64B B descriptor (cute::UMMA::make_umma_desc<Major::MN>, B64:
// ((4,n),(8,k)):((1,LBO),(4,SBO)) in 16-byte units): 64 contiguous bytes = 32 trees, 8 k rows per 512-byte swizzle atom -> SBO = 512 B;
// LBO = the distance to the next group of 32 columns = one tile: columns 32..63 of an N = 64 operand are the lo tile.
__device__ __forceinline__ uint64_t mz_sp_bdesc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3ffffu) >> 4) | ((uint64_t)(MZ_SP_TILE_BYTES >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)4 << 61);
}
__device__ __forceinline__ void mz_sp_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// byte offset of (k row, tree n) inside an N-major SWIZZLE_64B tile: Swizzle<2,4,3> = 16-byte chunk index ^ ((k >> 1) & 3)
__device__ __forceinline__ uint32_t mz_sp_tile_offset(int k, int n) { return (uint32_t)(k * 64 + ((((n >> 3) ^ (k >> 1)) & 3) << 4) + (n & 7) * 2); }
// x -> bf16 hi (round to nearest even) and bf16 lo = bf16(x - hi)
__device__ __forceinline__ void mz_sp_split(float x, unsigned short &hi, unsigned short &lo) {
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    hi = __bfloat16_as_ushort(h); lo = __bfloat16_as_ushort(__float2bfloat16_rn(x - __bfloat162float(h)));
}
__device__ __forceinline__ void mz_sp_stage(uint32_t tile_hi, int k, int n, float v) {
    unsigned short hi, lo; mz_sp_split(v, hi, lo);
    const uint32_t a = tile_hi + mz_sp_tile_offset(k, n);
    asm volatile("st.shared.b16 [%0], %1;" ::"r"(a), "h"(hi) : "memory");
    asm volatile("st.shared.b16 [%0], %1;" ::"r"(a + MZ_SP_TILE_BYTES), "h"(lo) : "memory");
}
__device__ __forceinline__ void mz_sp_stage_at(uint32_t addr_hi, float v) {
    unsigned short hi, lo; mz_sp_split(v, hi, lo);
    asm volatile("st.shared.b16 [%0], %1;" ::"r"(addr_hi), "h"(hi) : "memory");
    asm volatile("st.shared.b16 [%0], %1;" ::"r"(addr_hi + MZ_SP_TILE_BYTES), "h"(lo) : "memory");
}
// (x0, x1) -> packed bf16 hi parts (x0 in the low half) and packed bf16 lo parts
__device__ __forceinline__ void mz_sp_split2(float x0, float x1, uint32_t &h, uint32_t &l) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(x1), "f"(x0));
    const float h0 = __uint_as_float(h << 16), h1 = __uint_as_float(h & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(l) : "f"(x1 - h1), "f"(x0 - h0));
}

struct mz_sp_plan_s {                               // carve-up of the dynamic shared memory
    uint32_t w_base, tiles;                         // weight area, operand tiles (shared addresses); group g tile t: tiles + (3 g + t) * 2 * TILE (hi, lo)
    unsigned char *tiles_ptr;
    uint64_t *bars;                                 // [MZ_SP_MAX_SETS] weight-set barriers
    uint64_t *mbar_mma[2]; uint32_t *tmem_slot;
    uint64_t *mbar_tail; uint8_t *active;           // mz_k_search_sp: "tail done" barrier, per-tree active flags of the current move
    float *bias, *outV, *outL, *outR, *outH; double *pbc; uint16_t *path; mz_sp_rdesc *prog;
};
__device__ __forceinline__ mz_sp_plan_s mz_sp_carve(unsigned char *raw, int warea_bytes, int bias_floats, int total_rounds, int hidden_pad, int S, int pbc_smem) {
    mz_sp_plan_s p;
    const uint32_t a = mz_smem_u32(raw);
    unsigned char *c = raw + (((a + 1023u) & ~1023u) - a);              // swizzled tiles need 1024-byte alignment
    p.w_base = mz_smem_u32(c); c += warea_bytes;
    p.tiles = mz_smem_u32(c); p.tiles_ptr = c; c += 2 * MZ_SP_TILES_PER_GROUP * 2 * MZ_SP_TILE_BYTES;
    p.bars = (uint64_t *)c; p.mbar_mma[0] = (uint64_t *)(c + 8 * MZ_SP_MAX_SETS); p.mbar_mma[1] = p.mbar_mma[0] + 1; p.tmem_slot = (uint32_t *)(c + 8 * MZ_SP_MAX_SETS + 16);
    p.mbar_tail = (uint64_t *)(c + 8 * MZ_SP_MAX_SETS + 24); p.active = c + 8 * MZ_SP_MAX_SETS + 32;
    c += MZ_SP_CTRL_BYTES;
    p.bias = (float *)c; c += ((size_t)bias_floats * 4 + 127) & ~(size_t)127;
    p.outV = (float *)c; p.outL = p.outV + 4 * MZ_SP_OS; p.outR = p.outV + 20 * MZ_SP_OS; p.outH = p.outV + 24 * MZ_SP_OS; c += (size_t)(24 + hidden_pad) * MZ_SP_OS * 4;
    p.pbc = (double *)c; c += pbc_smem ? ((((size_t)S + 2) * ((size_t)S + 3) / 2) * 8 + 127) & ~(size_t)127 : 0;
    p.path = (uint16_t *)c; c += (((size_t)S + 2) * 2 * 32 + 127) & ~(size_t)127;
    p.prog = (mz_sp_rdesc *)c;
    (void)total_rounds;
    return p;
}

struct mz_sp_args {                                 // what a kernel on this path needs besides mz_params
    const unsigned char *image; const float *bias; const mz_sp_round *rounds;
    int32_t first[3], n_rounds[3], set_first[3], n_sets[3];
    int32_t total_rounds, total_sets, warea_bytes, bias_floats, pbc_smem;
    int32_t tail;                                   // mz_sp_plan::tail: trailing dynamics rounds that mz_k_search_sp runs off the simulation chain
};

// one-time set-up by all threads: barriers, TMEM, zeroed tiles, biases, the round table.  Ends with a CTA barrier.
__device__ __forceinline__ uint32_t mz_sp_setup(const mz_sp_plan_s &sp, const mz_sp_args &A, int nthreads) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int i = 0; i < A.total_sets; i++) mz_mbar_init(&sp.bars[i], 1);
        mz_mbar_init(sp.mbar_mma[0], 1); mz_mbar_init(sp.mbar_mma[1], 1); mz_mbar_init(sp.mbar_tail, MZ_SP_TAIL_THREADS);
        mz_fence_mbar_init();
    }
    __syncwarp();
    if (tid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(mz_smem_u32(sp.tmem_slot)), "r"((uint32_t)MZ_SP_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < 2 * MZ_SP_TILES_PER_GROUP * 2 * MZ_SP_TILE_BYTES / 16; i += nthreads) reinterpret_cast<uint4 *>(sp.tiles_ptr)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = tid; i < A.bias_floats; i += nthreads) sp.bias[i] = A.bias[i];
    if (tid < A.total_rounds) {
        const mz_sp_round G = A.rounds[tid];
        mz_sp_rdesc R;
        const int grp = (tid >= A.first[1] && tid < A.first[1] + A.n_rounds[1]) ? 0 : 1;      // prediction rounds run on group 0, the others on group 1
        const uint32_t tg = sp.tiles + (uint32_t)(grp * MZ_SP_TILES_PER_GROUP * 2 * MZ_SP_TILE_BYTES);
        R.wbytes = 0;
        for (int j = 0; j < 2; j++) {
            const mz_sp_job &J = G.job[j < G.njobs ? j : 0];
            R.a_hi[j] = mz_tc_desc(sp.w_base + (uint32_t)J.a_off); R.a_lo[j] = mz_tc_desc(sp.w_base + (uint32_t)(J.a_off + J.a_bytes));
            R.b_hi[j] = mz_sp_bdesc(tg + (uint32_t)(J.src_tile * 2 * MZ_SP_TILE_BYTES));
            R.dst[j] = J.dst_tile >= 0 ? tg + (uint32_t)(J.dst_tile * 2 * MZ_SP_TILE_BYTES) : 0u;
            R.f32[j] = J.f32_off >= 0 ? mz_smem_u32(sp.outV) + 4u * (uint32_t)J.f32_off : 0u;
            R.bias[j] = mz_smem_u32(sp.bias) + 4u * (uint32_t)J.bias_off;
            R.ks[j] = J.ks; R.out[j] = J.out; R.act[j] = J.act == MZ_ACT_TANH ? (int16_t)MZ_ACT_ID : J.act; R.perm[j] = J.perm;   // tanh (final layers only): applied by the reader
            const mz_sp_copy &Cp = G.copy[j < G.ncopy ? j : 0];
            R.copy_dst[j] = sp.w_base + (uint32_t)Cp.dst_off; R.copy_bytes[j] = j < G.ncopy ? (uint32_t)Cp.bytes : 0u; R.copy_src[j] = Cp.src_off;
            R.wbytes += R.copy_bytes[j];
        }
        R.njobs = G.njobs; R.ncopy = G.ncopy; R.set = G.set; R.next = G.next; R.per_pass = (uint16_t)G.per_pass; R.ord = (uint16_t)G.ord;
        sp.prog[tid] = R;
    }
    mz_fence_proxy_async();
    mz_tc_fence_before();
    __syncthreads();
    mz_tc_fence_after();
    return *sp.tmem_slot;
}

struct mz_sp_ctx { uint32_t prog; const unsigned char *image; uint32_t bars; };     // prog, bars: shared addresses

// one thread: starts the TMA copies of the round at shared address R into its weight set
__device__ __forceinline__ void mz_sp_fill(const mz_sp_ctx &C, uint32_t R) {
    const uint4 m = mz_lds_u4(R + 80), c0 = mz_lds_u4(R + 96), c1 = mz_lds_u4(R + 112);   // words 20..23 | 24..27 | 28..31
    const int set = (int)(short)(m.w & 0xffffu), ncopy = (int)(short)(m.z >> 16);
    const uint32_t bar = C.bars + 8u * (uint32_t)set;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(c0.x) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(c0.z), "l"(C.image + (int32_t)c1.z), "r"(c1.x), "r"(bar) : "memory");
    if (ncopy > 1)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(c0.w), "l"(C.image + (int32_t)c1.w), "r"(c1.y), "r"(bar) : "memory");
}
// one thread: waits until the weights for a round have landed: fill number pass * per_pass + ord of set `set`
__device__ __forceinline__ void mz_sp_wait_weights(const mz_sp_ctx &C, int set, uint32_t fill) {
    const uint32_t bar = C.bars + 8u * (uint32_t)set;
    uint32_t ok = 0, spin = 0;
    while (!ok) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(bar), "r"(fill & 1u) : "memory");
        if (++spin > (1u << 24)) __trap();
    }
}

// bias + activation + store of one job's accumulator fragment: thread t of warp w holds rows m = 16w + t/4 (+8), columns 8q + 2(t%4) + e;
// v = W_hi X_hi + W_lo X_hi, u = W_hi X_lo
__device__ __forceinline__ void mz_sp_epilogue(const uint32_t (&v)[16], const uint32_t (&u)[16], int out, int act, int perm, uint32_t bias, uint32_t dst, uint32_t f32, int w, int t) {
    const int c = t & 3;
    const float lo = act == MZ_ACT_RELU ? 0.0f : -INFINITY;
#pragma unroll
    for (int half = 0; half < 2; half++) {
        const int m = 16 * w + (t >> 2) + 8 * half;
        if (m < out) {
            const float b = mz_lds32(bias + (uint32_t)m * 4u);
            float x[8];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                x[2 * q] = fmaxf((__uint_as_float(v[4 * q + 2 * half]) + __uint_as_float(u[4 * q + 2 * half])) + b, lo);
                x[2 * q + 1] = fmaxf((__uint_as_float(v[4 * q + 2 * half + 1]) + __uint_as_float(u[4 * q + 2 * half + 1])) + b, lo);
            }
            if (dst) {                  // hidden layer: chunk c of k row m of the next operand tiles
                uint32_t h[4], l[4];
#pragma unroll
                for (int q = 0; q < 4; q++) mz_sp_split2(x[2 * q], x[2 * q + 1], h[q], l[q]);
                const uint32_t a = dst + (uint32_t)(m * 64 + ((c ^ (m >> 1)) & 3) * 16);
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + MZ_SP_TILE_BYTES), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
            } else if (perm) {          // final layer, permuted input order: column 8q + 2c + e is tree 8c + 2q + e
                const uint32_t a = f32 + (uint32_t)((m * MZ_SP_OS + 8 * c) * 4);
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x[0]), "f"(x[1]), "f"(x[2]), "f"(x[3]) : "memory");
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a + 16u), "f"(x[4]), "f"(x[5]), "f"(x[6]), "f"(x[7]) : "memory");
            } else {
#pragma unroll
                for (int q = 0; q < 4; q++)
                    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(f32 + (uint32_t)((m * MZ_SP_OS + 8 * q + 2 * c) * 4)), "f"(x[2 * q]), "f"(x[2 * q + 1]) : "memory");
            }
        }
    }
}

// ---- one pass over a network = rounds [first, first + count), run by the group's four EPILOGUE warps and its ISSUER warp ----
// Per round:   issuer: (weights of the round have landed) -> [rounds >= 1: wait until all 128 epilogue threads have written the operand
//                      tiles: named barrier, they arrive, it syncs] -> MMAs -> commit -> (MMAs complete) -> refill the round's weight set
//              epilogue warps: wait for the commit -> tcgen05.ld -> bias / activation / hi-lo split -> st.shared -> proxy fence -> arrive.
// The epilogue warps never wait for each other, and everything that is not on the chain MMA -> epilogue -> MMA (descriptor loads, weight
// waits, refills) sits on the issuer warp, which has a whole epilogue of slack per round.
#define MZ_SP_THREADS (MZ_THREADS + 64)             // 8 worker warps (tree phases + epilogues) + one issuer warp per group
#define MZ_SP_SEARCH_THREADS (MZ_THREADS + MZ_SP_TAIL_THREADS)   // mz_k_search_sp: + warps 10, 11, which with the two issuers form the tail team
// named barriers: 1, 2 = group 0 / 1 (epilogue warps + issuer); in mz_k_search_sp 3 = workers + issuers before a network pass, 4 = the
// workers after it, 5 = the tail team between its rounds, 6 = the gate of a tail's first round
enum { MZ_SP_BAR_SIM = 3, MZ_SP_BAR_WORK = 4, MZ_SP_BAR_TAIL = 5, MZ_SP_BAR_GATE = 6 };
__device__ __forceinline__ void mz_named_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void mz_named_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void mz_sp_bar_arrive(int grp) { asm volatile("bar.arrive %0, %1;" ::"r"(grp + 1), "n"(MZ_GROUP + 32) : "memory"); }
__device__ __forceinline__ void mz_sp_bar_sync(int grp) { asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(MZ_GROUP + 32) : "memory"); }
__device__ __forceinline__ void mz_sp_wait_mma(uint32_t mbar, uint32_t q) {
    uint32_t ok = 0, spin = 0;
    while (!ok) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(mbar), "r"(q & 1u) : "memory");
        if (++spin > (1u << 24)) __trap();
    }
}
// q = rounds executed by the group so far (parity of its MMA barrier), pass = passes over this network so far (which fill of a weight set a
// round consumes).  Both functions return the advanced q.
// TMA bulk store of one 4 KB operand tile to global memory (the learner saves every layer's input for the backward pass)
__device__ __forceinline__ void mz_sp_store_tile(unsigned char *gdst, uint32_t smem_tile) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_tile), "r"((uint32_t)MZ_SP_TILE_BYTES) : "memory");
}
__device__ __forceinline__ void mz_sp_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void mz_sp_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void mz_sp_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// one thread: the MMAs of a round (descriptor words 0..11 in d0..d2, k-steps in e1.z)
__device__ __forceinline__ void mz_sp_issue_mmas(uint4 d0, uint4 d1, uint4 d2, uint4 e1, int njobs, uint32_t tmem_d) {
#pragma unroll 1
    for (int j = 0; j < njobs; j++) {
        const uint64_t ah = j ? mz_u64(d0.z, d0.w) : mz_u64(d0.x, d0.y), al = j ? mz_u64(d1.z, d1.w) : mz_u64(d1.x, d1.y), bh = j ? mz_u64(d2.z, d2.w) : mz_u64(d2.x, d2.y);
        const uint32_t d = tmem_d + 64u * (uint32_t)j;
        const int ks = (int)(short)(j ? (e1.z >> 16) : (e1.z & 0xffffu));
#pragma unroll 1
        for (int k = 0; k < ks; k++) {           // A: +32 B per K = 16 step inside the 128-byte swizzle row; B: 16 k rows = 1024 B
            const uint64_t ka = (uint64_t)(2 * k), kb = (uint64_t)(64 * k);
            mz_sp_mma(d, ah + ka, bh + kb, MZ_SP_IDESC64, k > 0 ? 1u : 0u);          // W_hi [X_hi | X_lo] -> columns 0..31 | 32..63
            mz_sp_mma(d, al + ka, bh + kb, MZ_SP_IDESC32, 1u);                       // W_lo X_hi          -> columns 0..31
        }
    }
}
// save / fslot: learner only -- the hi tile of every job's input goes to save + fslot[2 * round + job] * 4 KB (fslot: shared address of an int16 table)
// bias: extra fills every weight set of this network has seen (a persistent self-play kernel primes the representation / dynamics sets anew at every ply)
__device__ __noinline__ uint32_t mz_sp_run_issuer(const mz_sp_ctx C, int first, int count, uint32_t tmem_d, uint32_t mbar, uint32_t q, uint32_t pass, int grp,
                                                  unsigned char *save = nullptr, uint32_t fslot = 0, uint32_t bias = 0) {
    uint32_t R = C.prog + (uint32_t)first * MZ_SP_RDESC_BYTES;
    for (int r = 0; r < count; r++, R += MZ_SP_RDESC_BYTES, q++) {
        const uint4 d0 = mz_lds_u4(R), d1 = mz_lds_u4(R + 16), d2 = mz_lds_u4(R + 32), e1 = mz_lds_u4(R + 64), e2 = mz_lds_u4(R + 80);
        const uint32_t fo = mz_lds_u4(R + 96).y;                        // per_pass | ord << 16
        const int njobs = (int)(short)(e2.z & 0xffffu), set = (int)(short)(e2.w & 0xffffu), next = (int)(short)(e2.w >> 16);
        if (mz_elect_one()) mz_sp_wait_weights(C, set, pass * (fo & 0xffffu) + (fo >> 16) + bias);
        if (r > 0) mz_sp_bar_sync(grp);                                 // the previous round's outputs are in the operand tiles, its accumulators have been read
        mz_tc_fence_after();
        if (mz_elect_one()) {
            mz_sp_issue_mmas(d0, d1, d2, e1, njobs, tmem_d);
            // learner: the commit releases this round's epilogue, which may overwrite tiles the previous round's stores still read
            if (save) mz_sp_store_wait_read();
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
            if (save) {                                                 // this round's input tiles -> global (they stay untouched until a later round's epilogue)
                for (int j = 0; j < njobs; j++) {
                    short sl; asm volatile("ld.shared.s16 %0, [%1];" : "=h"(sl) : "r"(fslot + 2u * (uint32_t)(2 * (first + r) + j)));
                    mz_sp_store_tile(save + (size_t)sl * MZ_SP_TILE_BYTES, (uint32_t)((j ? d2.z : d2.x) & 0x3fffu) << 4);
                }
                mz_sp_store_commit();
            }
            mz_sp_wait_mma(mbar, q);
            if (next >= 0) mz_sp_fill(C, C.prog + (uint32_t)next * MZ_SP_RDESC_BYTES);      // the round's weights are free: hand the set to its next user
        }
        __syncwarp();
    }
    return q;
}
__device__ __noinline__ uint32_t mz_sp_run(const mz_sp_ctx C, int first, int count, uint32_t tmem_d, uint32_t mbar, uint32_t q, int grp, int gtid, long long *tk) {
    long long tprev = 0; (void)tprev; (void)tk;
    const int w = gtid >> 5, t = gtid & 31;
    const uint32_t lane_base = tmem_d + ((uint32_t)(32 * w) << 16);     // M = 64: rows 16w..16w+15 live in lanes 32w..32w+15
    uint32_t R = C.prog + (uint32_t)first * MZ_SP_RDESC_BYTES;
    for (int r = 0; r < count; r++, R += MZ_SP_RDESC_BYTES, q++) {
        const uint4 e0 = mz_lds_u4(R + 48), e1 = mz_lds_u4(R + 64), e2 = mz_lds_u4(R + 80);   // words 12..15 | 16..19 | 20..23
        const int njobs = (int)(short)(e2.z & 0xffffu);
        MZ_RT(0);
        mz_sp_wait_mma(mbar, q);
        MZ_RT(1);
        mz_tc_fence_after();
        __syncwarp();
        uint32_t v0[16], u0[16], v1[16], u1[16];
        mz_tc_ld16x256(lane_base, v0); mz_tc_ld16x256(lane_base + 32u, u0);
        if (njobs > 1) { mz_tc_ld16x256(lane_base + 64u, v1); mz_tc_ld16x256(lane_base + 96u, u1); }
        mz_tc_wait_ld();
        MZ_RT(2);
        mz_sp_epilogue(v0, u0, (int)(short)(e1.w & 0xffffu), (int)(short)(e2.x & 0xffffu), (int)(short)(e2.y & 0xffffu), e1.x, e0.x, e0.z, w, t);
        if (njobs > 1) mz_sp_epilogue(v1, u1, (int)(short)(e1.w >> 16), (int)(short)(e2.x >> 16), (int)(short)(e2.y >> 16), e1.y, e0.y, e0.w, w, t);
        MZ_RT(3);
        mz_fence_proxy_async();
        mz_tc_fence_before();
        MZ_RT(4);
        if (r + 1 < count) mz_sp_bar_arrive(grp);
        MZ_RT(5);
    }
    return q;
}

// ---- the TAIL of a dynamics pass in mz_k_search_sp: its trailing rounds [first, first + count), which feed no reward job ----------------
// Run by the tail team (warps 8..11 = TMEM lane quadrants 0..3, ttid = thread index in the team) beside the tree phases of the worker
// warps.  Warp 9, the dynamics issuer, issues every round and runs quadrant 1 of its epilogue; warps 8, 10, 11 run quadrants 0, 2, 3.
// Round `first`: the issuer syncs on group 1's barrier (the worker warps arrive after their last round), issues, and opens the gate
// for the other three -- before it they could not tell round `first`'s phase of the MMA barrier from an earlier one with the same
// parity.  Later rounds: the team arrives on the tail barrier after its epilogue and the issuer syncs on it, as in mz_sp_run_issuer /
// mz_sp_run.  q = group 1's rounds before round `first`.  Issue and epilogue are separate calls: one function with both would need
// more registers than either.
__device__ __noinline__ void mz_sp_tail_issue(const mz_sp_ctx C, uint32_t R, uint32_t tmem_d, uint32_t mbar, uint32_t q, uint32_t pass, uint32_t bias, bool first) {
    const uint4 d0 = mz_lds_u4(R), d1 = mz_lds_u4(R + 16), d2 = mz_lds_u4(R + 32), e1 = mz_lds_u4(R + 64), e2 = mz_lds_u4(R + 80);
    const uint32_t fo = mz_lds_u4(R + 96).y;
    const int njobs = (int)(short)(e2.z & 0xffffu), set = (int)(short)(e2.w & 0xffffu), next = (int)(short)(e2.w >> 16);
    if (mz_elect_one()) mz_sp_wait_weights(C, set, pass * (fo & 0xffffu) + (fo >> 16) + bias);
    if (first) mz_sp_bar_sync(1); else mz_named_sync(MZ_SP_BAR_TAIL, MZ_SP_TAIL_THREADS);
    mz_tc_fence_after();
    if (mz_elect_one()) {
        mz_sp_issue_mmas(d0, d1, d2, e1, njobs, tmem_d);
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
    }
    __syncwarp();
    if (first) mz_named_arrive(MZ_SP_BAR_GATE, MZ_SP_TAIL_THREADS);
    if (mz_elect_one()) {
        mz_sp_wait_mma(mbar, q);
        if (next >= 0) mz_sp_fill(C, C.prog + (uint32_t)next * MZ_SP_RDESC_BYTES);      // the round's weights are free: hand the set to its next user
    }
    __syncwarp();
}
// one quadrant of a tail round's epilogue (as a round of mz_sp_run).  A tail round has one job, the state head's layer: the reward head
// has ended before the tail begins.  Reading one job's accumulators keeps this call 32 registers lighter than mz_sp_run, and the
// kernel has no registers to spare around it.
__device__ __noinline__ void mz_sp_tail_epilogue(uint32_t R, uint32_t lane_base, uint32_t mbar, uint32_t q, int w, int t) {
    const uint4 e0 = mz_lds_u4(R + 48), e1 = mz_lds_u4(R + 64), e2 = mz_lds_u4(R + 80);
    mz_sp_wait_mma(mbar, q);
    mz_tc_fence_after();
    __syncwarp();
    uint32_t v0[16], u0[16];
    mz_tc_ld16x256(lane_base, v0); mz_tc_ld16x256(lane_base + 32u, u0);
    mz_tc_wait_ld();
    mz_sp_epilogue(v0, u0, (int)(short)(e1.w & 0xffffu), (int)(short)(e2.x & 0xffffu), (int)(short)(e2.y & 0xffffu), e1.x, e0.x, e0.z, w, t);
    mz_fence_proxy_async();
    mz_tc_fence_before();
}
__device__ __forceinline__ uint32_t mz_sp_run_tail(const mz_sp_ctx C, int first, int count, uint32_t tmem_d, uint32_t mbar, uint32_t q, uint32_t pass, uint32_t bias, int ttid) {
    const int w = ttid >> 5;
    uint32_t R = C.prog + (uint32_t)first * MZ_SP_RDESC_BYTES;
    for (int r = 0; r < count; r++, R += MZ_SP_RDESC_BYTES, q++) {
        if (w == 1) mz_sp_tail_issue(C, R, tmem_d, mbar, q, pass, bias, r == 0);
        else if (r == 0) mz_named_sync(MZ_SP_BAR_GATE, MZ_SP_TAIL_THREADS);
        mz_sp_tail_epilogue(R, tmem_d + ((uint32_t)(32 * w) << 16), mbar, q, w, ttid & 31);
        if (w != 1 && r + 1 < count) mz_named_arrive(MZ_SP_BAR_TAIL, MZ_SP_TAIL_THREADS);
    }
    return q;
}
