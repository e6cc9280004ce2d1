// mz_kernels_rn.cuh -- the ResNet networks (net_type = MZ_NET_RESNET, repaired src/Learning.jl:148-255) on the tcgen05
// tensor cores, and the fused search kernel that uses them.
//
// Orientation (the opposite of the feed-forward tensor path): the ACTIVATIONS are the A operand.  A 1x1 convolution
// does not mix board cells, so every (tree, cell) pair is an independent row of a [rows x 64 channels] x [64 x 64] GEMM:
//   D[row = (tree, cell)][co] = sum_ci X[row][ci] * W[co][ci]         M = 128 rows per tile, N = 64, K = 64
// One CTA owns 4 tiles (TicTacToe: 14 trees x 9 cells = 126 rows per tile, 56 trees per CTA; a 6x7 board: 3 trees per
// tile).  Accumulators live in TMEM (lane = row, 64 fp32 columns per tile), so an epilogue thread owns one row: it reads
// its 64 channels with tcgen05.ld, applies the BatchNorm shift (its scale is folded into the bf16 weights; + action-plane term, + residual), relu, and
// writes the bf16 row of the next layer's A tile with eight 16-byte swizzled stores (and, for the last layer of the
// dynamics state head / the representation, the same row to the tree's hidden-state slot in HBM).  Weights stream
// through a two-slot shared-memory ring by TMA bulk copies, one block per step, prefetched one step ahead.
// The k x k convolutions of the representation network (root only) run as k*k accumulating tap-steps over shifted
// copies of the source tile; its first convolution is a single im2col tile built from the boards.
// The dense heads run on the same machinery with rows = trees.
// Execution is lock-step: all 256 threads walk the host-built step program; thread 0 issues the MMAs of a step's jobs
// back to back (each committed to its own mbarrier), warpgroup w runs the epilogues of jobs w and w + 2, so the tensor
// core works on the later jobs while the earlier ones are in their epilogue.
#pragma once
#include "mz_kernels_tc.cuh"

#define MZ_RN_TMEM_COLS 256
#define MZ_RN_TILE_BYTES 16384
#define MZ_RN_AUX_BYTES 32768
#define MZ_RN_OUT_ROWS 64          // trees per CTA in the fp32 head outputs / per-tree tables
#define MZ_RN_THREADS 512         // 16 warps: one warpgroup per tile job in the epilogues, 8 lanes per tree for 64 trees in the tree phases
#define MZ_RN_NPASS 1

struct mz_rn_plan {
    uint32_t tiles;                // X0..X3, T0..T3 (shared address)
    uint32_t aux;                  // HV | HP (two K blocks) ; or the two scratch tiles of the tap-steps
    uint32_t wring;                // two weight slots
    unsigned char *tiles_ptr, *wring_ptr;
    uint64_t *w_bar, *mma_bar, *scr_bar, *e_bar; uint32_t *tmem_slot;
    float *out;                    // fp32 head outputs: V [4][64] | L [16][64] | R [4][64]
    float *plane; int32_t *pe, *dbl, *active; unsigned long long *tree_base;
    double *pbc0, *sqrtN; uint16_t *path;
    mz_rn_step *prog;              // steps [smem_first, n_steps) of the program (the simulation loop's)
};
__host__ __device__ inline size_t mz_rn_smem_bytes(int slot_bytes, int S, int ntrees, int smem_steps) {
    size_t tab = (((size_t)S + 2) * 8 * 2 + 127) & ~(size_t)127;
    size_t path = (((size_t)S + 2) * 2 * ntrees + 127) & ~(size_t)127;
    return 1024 + 8 * MZ_RN_TILE_BYTES + MZ_RN_AUX_BYTES + 2 * (size_t)slot_bytes + 256 + 24 * MZ_RN_OUT_ROWS * 4 + 5 * MZ_RN_OUT_ROWS * 8 + tab + path + (size_t)smem_steps * sizeof(mz_rn_step) + 128;
}
__device__ __forceinline__ mz_rn_plan mz_rn_carve(unsigned char *raw, int slot_bytes, int S, int ntrees, int smem_steps) {
    mz_rn_plan p;
    uint32_t a = mz_smem_u32(raw);
    unsigned char *c = raw + (((a + 1023u) & ~1023u) - a);
    p.tiles_ptr = c; p.tiles = mz_smem_u32(c); c += 8 * MZ_RN_TILE_BYTES;
    p.aux = mz_smem_u32(c); c += MZ_RN_AUX_BYTES;
    p.wring_ptr = c; p.wring = mz_smem_u32(c); c += 2 * (size_t)slot_bytes;
    p.w_bar = (uint64_t *)c; p.mma_bar = p.w_bar + 2; p.scr_bar = p.w_bar + 6; p.e_bar = p.w_bar + 8; p.tmem_slot = (uint32_t *)(c + 128); c += 256;
    p.out = (float *)c; c += 24 * MZ_RN_OUT_ROWS * 4;
    p.tree_base = (unsigned long long *)c; c += MZ_RN_OUT_ROWS * 8;
    p.plane = (float *)c; c += MZ_RN_OUT_ROWS * 4; p.pe = (int32_t *)c; c += MZ_RN_OUT_ROWS * 4; p.dbl = (int32_t *)c; c += MZ_RN_OUT_ROWS * 4;
    p.active = (int32_t *)c; c += MZ_RN_OUT_ROWS * 4; c += MZ_RN_OUT_ROWS * 16;   // (spare)
    p.pbc0 = (double *)c; p.sqrtN = p.pbc0 + (S + 2); c += (((size_t)S + 2) * 8 * 2 + 127) & ~(size_t)127;
    p.path = (uint16_t *)c; c += (((size_t)S + 2) * 2 * ntrees + 127) & ~(size_t)127;
    p.prog = (mz_rn_step *)c;
    return p;
}
__device__ __forceinline__ uint32_t mz_rn_buf(const mz_rn_plan &sp, int id) {
    if (id < 8) return sp.tiles + (uint32_t)id * MZ_RN_TILE_BYTES;
    if (id == MZ_RN_BUF_HV) return sp.aux;
    if (id == MZ_RN_BUF_HP) return sp.aux + 8192u;
    return sp.aux + (uint32_t)(id - MZ_RN_BUF_S0) * MZ_RN_TILE_BYTES;
}
__device__ __forceinline__ int mz_rn_out_base(int out_id) { return out_id == MZ_RN_OUT_V ? 0 : out_id == MZ_RN_OUT_L ? 4 * MZ_RN_OUT_ROWS : 20 * MZ_RN_OUT_ROWS; }

__device__ __forceinline__ void mz_rn_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// kind::f16, D = F32, A = B = BF16, K-major, M = 128, N = 16 * n16
__device__ __forceinline__ uint32_t mz_rn_idesc(int n16) { return (1u << 4) | (1u << 7) | (1u << 10) | (((uint32_t)(n16 * 16) >> 3) << 17) | ((128u >> 4) << 24); }
__device__ __forceinline__ void mz_rn_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                   "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                   "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void mz_rn_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ uint4 mz_lds128u(uint32_t addr) { uint4 v; asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr)); return v; }
__device__ __forceinline__ void mz_sts128u(uint32_t addr, uint4 v) { asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory"); }
__device__ __forceinline__ float mz_bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float mz_bf16hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ uint32_t mz_pack_bf16(float lo, float hi) {   // round to nearest even, two values per instruction
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t mz_pack_bf16_relu(float lo, float hi) {   // max(x, 0) fused into the conversion
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ unsigned long long mz_f2pack(float a, float b) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void mz_f2unpack(unsigned long long p, float &a, float &b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(p)); }
__device__ __forceinline__ unsigned long long mz_fma2(unsigned long long a, unsigned long long b, unsigned long long c) {   // two IEEE fmaf per instruction
    unsigned long long d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d;
}
__device__ __forceinline__ unsigned long long mz_add2(unsigned long long a, unsigned long long b) {
    unsigned long long d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d;
}
__device__ __forceinline__ void mz_mbar_wait_u32(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0, spin = 0;
    while (!ok) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (++spin > (1u << 24)) __trap();
    }
}

// ---- executor state (uniform across the CTA) ----------------------------------------------------------------------
struct mz_rn_exec {
    mz_rn_plan sp; const mz_rn_step *steps; const unsigned char *image;
    uint32_t tmem; int slot_bytes;
    uint32_t wq;            // weight blocks consumed
    int pf;                 // step whose block is in (or on its way to) slot wq & 1, or -1
    uint32_t mqw;           // commits this thread's warpgroup has waited for on its barrier mma_bar[wg]
    uint32_t sq[2];         // commits seen per scratch barrier
    uint32_t eq0, eq1, ew0, ew1;  // per weight slot: row-local steps that released it through e_bar / releases thread 0 has waited for
    int pool_slot;          // hidden-state slot written by MZ_RN_F_POOL epilogues
    int W, H;
    int my_tree, my_cell;   // (tree, cell) of this thread's TMEM lane in its warpgroup's convolution tile
    uint32_t rowoff;        // byte offset of this thread's row inside a swizzled tile
    bool row_valid, tree_valid;   // this thread's row holds a (tree, cell) of an active tree / (rows = trees jobs) an active tree; set by mz_rn_bind_rows
    int st_tl[2], st_cell[2]; // hidden staging: this thread copies one 16-byte chunk of rows (tid >> 3) and (tid >> 3) + 64 of every tile
#ifdef MZ_PHASE_TIMERS
    long long st_t[6]; long long st_c;
#endif
};
__device__ __forceinline__ void mz_rn_issue_weights(const mz_rn_exec &X, const mz_rn_params &R, int s, uint32_t slot) {
    const mz_rn_step *st = s >= R.smem_first ? X.sp.prog + (s - R.smem_first) : X.steps + s;
    const int off = st->w_off, bytes = st->w_bytes;
    const uint32_t bar = mz_smem_u32(&X.sp.w_bar[slot]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(X.sp.wring + slot * (uint32_t)X.slot_bytes), "l"(X.image + off), "r"((uint32_t)bytes), "r"(bar) : "memory");
}

// a job descriptor as seven 32-bit loads (its fields are bytes: a member-wise copy would load them one by one)
__device__ __forceinline__ mz_rn_job mz_rn_load_job(const mz_rn_job *p) {
    static_assert(sizeof(mz_rn_job) == 28, "mz_rn_job layout");
    union { mz_rn_job j; uint32_t w[7]; } u;
#pragma unroll
    for (int i = 0; i < 7; i++) u.w[i] = reinterpret_cast<const uint32_t *>(p)[i];
    return u.j;
}
__device__ __forceinline__ void mz_rn_slot_free(mz_rn_exec &X, uint32_t sl) {
    if (sl == 0) { while (X.ew0 < X.eq0) { mz_mbar_wait_u32(mz_smem_u32(&X.sp.e_bar[0]), X.ew0 & 1u); X.ew0++; } }
    else { while (X.ew1 < X.eq1) { mz_mbar_wait_u32(mz_smem_u32(&X.sp.e_bar[1]), X.ew1 & 1u); X.ew1++; } }
}

struct mz_rn_tile_ctx { uint32_t taddr, pT, pE, dst, skp, r7x; unsigned char *pool; unsigned long long rv2; bool store; };
template <bool RELU, bool SKIP, bool PLANE, bool POOL>
__device__ __forceinline__ void mz_rn_tile_rows(const mz_rn_tile_ctx &c) {
#pragma unroll 1
    for (int half = 0; half < 2; half++) {
        uint32_t v[32];
        mz_rn_ld32(c.taddr + 32u * half, v);
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int c8 = 4 * half + q;
            const float4 t0 = mz_lds128(c.pT + c8 * 32), t1 = mz_lds128(c.pT + c8 * 32 + 16);
            unsigned long long T[4] = {mz_f2pack(t0.x, t0.y), mz_f2pack(t0.z, t0.w), mz_f2pack(t1.x, t1.y), mz_f2pack(t1.z, t1.w)};
            if (PLANE) {   // + action plane * (w_plane * s): y = acc + fmaf(plane, E, T)   (the BatchNorm scale is folded into the weights)
                const float4 e0 = mz_lds128(c.pE + c8 * 32), e1 = mz_lds128(c.pE + c8 * 32 + 16);
                T[0] = mz_fma2(c.rv2, mz_f2pack(e0.x, e0.y), T[0]); T[1] = mz_fma2(c.rv2, mz_f2pack(e0.z, e0.w), T[1]);
                T[2] = mz_fma2(c.rv2, mz_f2pack(e1.x, e1.y), T[2]); T[3] = mz_fma2(c.rv2, mz_f2pack(e1.z, e1.w), T[3]);
            }
            unsigned long long y[4];
#pragma unroll
            for (int i = 0; i < 4; i++) y[i] = mz_add2(mz_f2pack(__uint_as_float(v[8 * q + 2 * i]), __uint_as_float(v[8 * q + 2 * i + 1])), T[i]);
            const uint32_t chunk = (uint32_t)(c8 << 4) ^ c.r7x;
            if (SKIP) {
                const uint4 k = mz_lds128u(c.skp + chunk);
                y[0] = mz_add2(y[0], mz_f2pack(mz_bf16lo(k.x), mz_bf16hi(k.x))); y[1] = mz_add2(y[1], mz_f2pack(mz_bf16lo(k.y), mz_bf16hi(k.y)));
                y[2] = mz_add2(y[2], mz_f2pack(mz_bf16lo(k.z), mz_bf16hi(k.z))); y[3] = mz_add2(y[3], mz_f2pack(mz_bf16lo(k.w), mz_bf16hi(k.w)));
            }
            uint32_t o[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                float a0, a1; mz_f2unpack(y[i], a0, a1);
                o[i] = RELU ? mz_pack_bf16_relu(a0, a1) : mz_pack_bf16(a0, a1);
            }
            const uint4 ov = make_uint4(o[0], o[1], o[2], o[3]);
            if (c.store) mz_sts128u(c.dst + chunk, ov);
            if (POOL) { if (c.pool) *reinterpret_cast<uint4 *>(c.pool + c8 * 16) = ov; }
        }
    }
}

// epilogue of one job for one warpgroup thread (row = TMEM lane)
__device__ __forceinline__ void mz_rn_epilogue(const mz_rn_exec &X, const mz_rn_params &R, const mz_rn_job J, uint32_t wslot, int wgt) {
    const int warp4 = wgt >> 5, lane = wgt & 31, row = 32 * warp4 + lane;
    const uint32_t taddr = X.tmem + ((uint32_t)(32 * warp4) << 16) + 64u * J.acc;
    const uint32_t pS = wslot + (uint32_t)J.p_sub, pT = pS + 256u, pE = pS + 512u;
    const bool trees = (J.flags & MZ_RN_F_TREES) != 0;
    int tree, cell;
    if (trees) { tree = row; cell = 0; } else { tree = X.my_tree; cell = X.my_cell; }   // convolution job j is always run by warpgroup j
    const bool valid = trees ? X.tree_valid : X.row_valid;
    const int jflags = J.flags, jact = J.act;
    if (J.epi == MZ_RN_EPI_TILE) {
        const uint32_t rowoff = X.rowoff;
        // destination and residual source of a tile epilogue are always X/T tiles (buffer ids < 8; checked by the host builder)
        const uint32_t dst = X.sp.tiles + (uint32_t)J.dst_buf * MZ_RN_TILE_BYTES + rowoff;
        const uint32_t skp = J.skip_buf != 0xff ? X.sp.tiles + (uint32_t)J.skip_buf * MZ_RN_TILE_BYTES + rowoff : 0u;
        const float rowval = (J.flags & MZ_RN_F_PLANE) ? X.sp.plane[tree < MZ_RN_OUT_ROWS ? tree : 0] : 0.0f;
        unsigned char *pool = nullptr;
        if ((J.flags & MZ_RN_F_POOL) && valid)
            pool = reinterpret_cast<unsigned char *>(X.sp.tree_base[tree]) + R.hidden_off_bytes + (size_t)X.pool_slot * R.node_bytes + (size_t)cell * 128;
        // the inner loop is compiled per (relu, skip, plane) combination: no uniform branches or per-element selects inside it; rows
        // that are not valid (the two pad rows of a tile, idle trees) are computed like the others and zeroed afterwards
        const mz_rn_tile_ctx tc{taddr, pT, pE, dst, skp, (uint32_t)((row & 7) << 4), pool, mz_f2pack(rowval, rowval), !trees || row < MZ_RN_OUT_ROWS};
        const int combo = (jact == MZ_ACT_RELU ? 4 : 0) | (skp ? 2 : 0) | ((jflags & MZ_RN_F_PLANE) ? 1 : 0);
#define MZ_RN_TILE_DISPATCH(POOL_) \
        switch (combo) { \
            case 4: mz_rn_tile_rows<true, false, false, POOL_>(tc); break;      /* ConvBN + relu, dense + relu */ \
            case 6: mz_rn_tile_rows<true, true, false, POOL_>(tc); break;       /* second convolution of a residual block */ \
            case 5: mz_rn_tile_rows<true, false, true, POOL_>(tc); break;       /* first dynamics convolution (action plane) */ \
            case 0: mz_rn_tile_rows<false, false, false, POOL_>(tc); break;     /* first dense layer of the policy head (no activation) */ \
            case 2: mz_rn_tile_rows<false, true, false, POOL_>(tc); break; \
            case 1: mz_rn_tile_rows<false, false, true, POOL_>(tc); break; \
            case 3: mz_rn_tile_rows<false, true, true, POOL_>(tc); break; \
            default: mz_rn_tile_rows<true, true, true, POOL_>(tc); break; \
        }
        if (jflags & MZ_RN_F_POOL) { MZ_RN_TILE_DISPATCH(true) } else { MZ_RN_TILE_DISPATCH(false) }
#undef MZ_RN_TILE_DISPATCH
        if (!valid && tc.store) {
#pragma unroll
            for (int c8 = 0; c8 < 8; c8++) mz_sts128u(dst + (uint32_t)(c8 << 4), make_uint4(0u, 0u, 0u, 0u));
        }
    } else if (J.epi == MZ_RN_EPI_HEAD) {
        uint32_t v[16];
        mz_rn_ld16(taddr, v);
        if (valid) {
            const int nf = J.nfa + J.nfb;
            for (int f = 0; f < nf; f++) {
                const float y = fmaxf(__uint_as_float(v[f]) + mz_lds32(pT + f * 4), 0.0f);
                const bool second = f >= J.nfa;
                const int k = cell + R.cells * (second ? f - J.nfa : f);
                const uint32_t tile = mz_rn_buf(X.sp, second ? J.dst2_buf : J.dst_buf) + (uint32_t)(k >> 6) * 8192u;
                mz_tc_store_bf16(tile, tree, k & 63, y);
            }
        }
    } else {
        uint32_t v[16];
        mz_rn_ld16(taddr, v);
        if (row < R.ntrees) {
            float *o = X.sp.out + mz_rn_out_base(J.out_id);
            for (int k = 0; k < J.out; k++) {
                float y = __uint_as_float(v[k]) + mz_lds32(pT + k * 4);
                if (J.act == MZ_ACT_TANH) y = mz_tanhf_noinline(y); else if (J.act == MZ_ACT_RELU) y = fmaxf(y, 0.0f);
                o[k * MZ_RN_OUT_ROWS + row] = y;
            }
        }
    }
}

// Runs steps [first, last) of the program; next_first = the step that will run after this range (its weights are
// prefetched during the last step), or -1.  Inlined at its (single) call site per kernel so that the executor state
// stays in registers; the steps of the simulation loop are read from shared memory.
#ifdef MZ_PHASE_TIMERS
#define MZ_RN_ST(i) do { long long c_ = clock64(); X.st_t[i] += c_ - X.st_c; X.st_c = c_; } while (0)
#else
#define MZ_RN_ST(i)
#endif
__device__ __forceinline__ void mz_rn_run(mz_rn_exec &X, const mz_rn_params &R, int first, int last, int next_first) {
    const int tid = threadIdx.x, wg = tid >> 7, wgt = tid & 127;
    // a range lies entirely in the shared-memory copy of the program (the simulation loop's) or entirely in global memory (the root's)
    const mz_rn_step *const prog = first >= R.smem_first ? X.sp.prog - R.smem_first : X.steps;
    for (int s = first; s < last; s++) {
        MZ_RN_ST(5);
        const mz_rn_step *st = prog + s;
        const uint32_t slot = X.wq & 1u;
        const int next = s + 1 < last ? s + 1 : next_first;
        const uint32_t hdr = reinterpret_cast<const uint32_t *>(st)[2], hdr2 = reinterpret_cast<const uint32_t *>(st)[3];   // njobs, ntaps, tap, last | dx, dy, accumulate, rowlocal
        const int njobs = (int)(hdr & 0xffu), ntaps = (int)((hdr >> 8) & 0xffu), is_last = (int)(hdr >> 24), st_rowlocal = (int)(hdr2 >> 24);
        const int mine = (int)(int8_t)((reinterpret_cast<const uint32_t *>(st->wgjob)[0] >> (8 * wg)) & 0xffu);   // this warpgroup's job in the step, or -1
        if (tid == 0) {
            // a slot last used by a row-local step is free once all four warpgroups have finished that step's epilogue (it reads the
            // BatchNorm shifts from the slot): each of them arrives on e_bar[slot] after its own barrier
            if (X.pf != s) { mz_rn_slot_free(X, slot); mz_rn_issue_weights(X, R, s, slot); }
            if (next >= 0) { mz_rn_slot_free(X, slot ^ 1u); mz_rn_issue_weights(X, R, next, slot ^ 1u); }
        }
        mz_mbar_wait_u32(mz_smem_u32(&X.sp.w_bar[slot]), (X.wq >> 1) & 1u);
        const uint32_t wslot = X.sp.wring + slot * (uint32_t)X.slot_bytes;
        MZ_RN_ST(0);
        if (ntaps > 1) {
            // tap-step: per tile, A = copy of the source tile shifted by (dx, dy) cells, built in one of two scratch tiles
            const int dx = st->dx, dy = st->dy, accumulate = st->accumulate;
#pragma unroll
            for (int j = 0; j < MZ_RN_TILES; j++) {
                if (j >= njobs) break;
                const uint32_t sl = (uint32_t)(j & 1);
                if (j >= 2) mz_mbar_wait_u32(mz_smem_u32(&X.sp.scr_bar[sl]), (X.sq[sl] - 1u) & 1u);   // the MMA that read this scratch tile is done
                const uint32_t src = mz_rn_buf(X.sp, st->jobs[j].a_buf), dst = mz_rn_buf(X.sp, MZ_RN_BUF_S0 + (int)sl);
                for (int i = tid; i < 128 * 8; i += MZ_RN_THREADS) {
                    const int row = i >> 3, ch = i & 7;
                    uint4 v; v.x = v.y = v.z = v.w = 0u;
                    if (row < R.rows_valid) {
                        const int t = row / R.cells, cell = row % R.cells, x = cell % X.W + dx, y = cell / X.W + dy;
                        if (x >= 0 && x < X.W && y >= 0 && y < X.H) {
                            const int sr = t * R.cells + x + X.W * y;
                            v = mz_lds128u(src + (uint32_t)((sr >> 3) * 1024 + (sr & 7) * 128 + ((ch ^ (sr & 7)) << 4)));
                        }
                    }
                    mz_sts128u(dst + (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((ch ^ (row & 7)) << 4)), v);
                }
                mz_fence_proxy_async();
                mz_tc_fence_before();
                __syncthreads();
                if (tid < 32) {
                    mz_tc_fence_after();
                    if (mz_elect_one()) {
                        const uint64_t ad = mz_tc_desc(dst), bd = mz_tc_desc(wslot + (uint32_t)st->jobs[j].w_sub);
                        const uint32_t idesc = mz_rn_idesc(st->jobs[j].n16), acc = st->jobs[j].acc;
#pragma unroll
                        for (int k = 0; k < 4; k++) mz_rn_mma(X.tmem + 64u * acc, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (accumulate || k > 0) ? 1u : 0u);
                        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mz_smem_u32(&X.sp.scr_bar[sl])) : "memory");
                        if (is_last) asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mz_smem_u32(&X.sp.mma_bar[st->jobs[j].wg])) : "memory");
                    }
                    __syncwarp();
                }
                X.sq[sl]++;
            }
            // every MMA of the step is complete before its weight slot / scratch tiles are reused
#pragma unroll
            for (uint32_t sl = 0; sl < 2; sl++) if (X.sq[sl] > 0) mz_mbar_wait_u32(mz_smem_u32(&X.sp.scr_bar[sl]), (X.sq[sl] - 1u) & 1u);
        } else {
            // every warpgroup's first warp issues the MMAs of the job that warpgroup will run the epilogue of (tcgen05.mma may be issued
            // from any warp): the four issues run in parallel instead of one thread issuing 16 MMAs ahead of its own epilogue
            if ((tid & 127) < 32) {
                mz_tc_fence_after();
                if (mine >= 0 && mz_elect_one()) {
                    const mz_rn_job J = mz_rn_load_job(&st->jobs[mine]);
                    const uint32_t a = mz_rn_buf(X.sp, J.a_buf), idesc = mz_rn_idesc(J.n16);
                    for (int kb = 0; kb < J.kblocks; kb++) {
                        const uint64_t ad = mz_tc_desc(a + (uint32_t)kb * 8192u), bd = mz_tc_desc(wslot + (uint32_t)J.w_sub + (uint32_t)(kb * J.n16 * 2048));
#pragma unroll
                        for (int k = 0; k < 4; k++) mz_rn_mma(X.tmem + 64u * J.acc, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
                    }
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mz_smem_u32(&X.sp.mma_bar[wg])) : "memory");
                }
                __syncwarp();
            }
        }
        MZ_RN_ST(1);
        if (is_last) {
            // a warpgroup runs at most one epilogue per step (convolution job j <-> warpgroup j; dense heads: one job per warpgroup),
            // so the epilogue code exists once
            if (mine >= 0) {
                const mz_rn_job J = mz_rn_load_job(&st->jobs[mine]);
                mz_mbar_wait_u32(mz_smem_u32(&X.sp.mma_bar[wg]), X.mqw & 1u);
                X.mqw++;
                mz_tc_fence_after();
                __syncwarp();
                MZ_RN_ST(2);
                mz_rn_epilogue(X, R, J, wslot, wgt);
                MZ_RN_ST(3);
            }
        }
        mz_fence_proxy_async();
        mz_tc_fence_before();
        if (st_rowlocal == 1 && s + 1 < last) {
            // the next step reads only what this warpgroup wrote: meet inside the warpgroup, release the weight slot, run on
            asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory");
            if (wgt == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mz_smem_u32(&X.sp.e_bar[slot])) : "memory");
            if (slot == 0) X.eq0++; else X.eq1++;
        } else {
            __syncthreads();
        }
        mz_tc_fence_after();
        MZ_RN_ST(4);
        X.wq++; X.pf = next;
    }
}

// parent hidden states (bf16 rows in the tree pools) -> X tiles, scaled by 2^doublings (Q6); rows of idle trees are zero
__device__ __forceinline__ void mz_rn_stage_hidden(const mz_rn_exec &X, const mz_rn_params &R) {
    constexpr int NIT = MZ_RN_TILES * 128 * 8 / MZ_RN_THREADS;   // 16-byte chunks per thread; all loads are issued before the first store
    static_assert(NIT == 2 * MZ_RN_TILES, "staging layout assumes 512 threads");
    const int ch = threadIdx.x & 7, r0 = threadIdx.x >> 3;
    uint4 v[NIT]; float sc[NIT];
#pragma unroll
    for (int it = 0; it < NIT; it++) {
        const int h = it & 1, tile = it >> 1;
        v[it] = make_uint4(0u, 0u, 0u, 0u); sc[it] = 1.0f;
        if (X.st_tl[h] >= 0) {
            const int tree = tile * R.tpt + X.st_tl[h];
            if (X.sp.active[tree]) {
                const unsigned char *src = reinterpret_cast<const unsigned char *>(X.sp.tree_base[tree]) + R.hidden_off_bytes + (size_t)X.sp.pe[tree] * R.node_bytes + (size_t)(X.st_cell[h] * 128 + ch * 16);
                v[it] = *reinterpret_cast<const uint4 *>(src);
                sc[it] = __uint_as_float((uint32_t)(127 + X.sp.dbl[tree]) << 23);
            }
        }
    }
#pragma unroll
    for (int it = 0; it < NIT; it++) {
        const int row = r0 + 64 * (it & 1), tile = it >> 1;
        uint4 o = v[it];
        if (sc[it] != 1.0f) {
            const float f = sc[it];
            o.x = mz_pack_bf16(mz_bf16lo(o.x) * f, mz_bf16hi(o.x) * f); o.y = mz_pack_bf16(mz_bf16lo(o.y) * f, mz_bf16hi(o.y) * f);
            o.z = mz_pack_bf16(mz_bf16lo(o.z) * f, mz_bf16hi(o.z) * f); o.w = mz_pack_bf16(mz_bf16lo(o.w) * f, mz_bf16hi(o.w) * f);
        }
        mz_sts128u(X.sp.tiles + (uint32_t)(tile * MZ_RN_TILE_BYTES + (row >> 3) * 1024 + (row & 7) * 128 + ((ch ^ (row & 7)) << 4)), o);
    }
    mz_fence_proxy_async();
    __syncthreads();
}

struct mz_search_rn_args {
    mz_search_args base;
    const unsigned char *image; const mz_rn_step *steps;
    // mz_k_rn_forward only
    int32_t net, B; const float *in; float *out1, *out2; unsigned char *scratch_pool;
};

// common prologue: barriers, TMEM, zeroed tiles, executor state
__device__ __forceinline__ void mz_rn_setup(mz_rn_exec &X, const mz_params &P, const mz_rn_params &R, const mz_search_rn_args &ta, unsigned char *smem) {
    X.sp = mz_rn_carve(smem, R.slot_bytes, P.S, R.ntrees, R.n_steps - R.smem_first);
    X.steps = ta.steps; X.image = ta.image; X.slot_bytes = R.slot_bytes; X.wq = 0; X.pf = -1; X.pool_slot = 0; X.W = P.W; X.H = P.H;
    X.mqw = 0;
    X.sq[0] = X.sq[1] = 0; X.eq0 = X.eq1 = X.ew0 = X.ew1 = 0;
    for (int h = 0; h < 2; h++) { const int row = (int)(threadIdx.x >> 3) + 64 * h; X.st_tl[h] = row < R.rows_valid ? row / R.cells : -1; X.st_cell[h] = row % R.cells; }
    { const int row = (int)(threadIdx.x & 127); X.my_tree = (int)(threadIdx.x >> 7) * R.tpt + row / R.cells; X.my_cell = row % R.cells; }
#ifdef MZ_PHASE_TIMERS
    for (int i = 0; i < 6; i++) X.st_t[i] = 0;
    X.st_c = clock64();
#endif
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int i = 0; i < 2; i++) mz_mbar_init(&X.sp.w_bar[i], 1);
        for (int i = 0; i < 4; i++) mz_mbar_init(&X.sp.mma_bar[i], 1);
        for (int i = 0; i < 2; i++) mz_mbar_init(&X.sp.scr_bar[i], 1);
        for (int i = 0; i < 2; i++) mz_mbar_init(&X.sp.e_bar[i], MZ_RN_TILES);
        mz_fence_mbar_init();
    }
    __syncwarp();
    if (tid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(mz_smem_u32(X.sp.tmem_slot)), "r"((uint32_t)MZ_RN_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < (8 * MZ_RN_TILE_BYTES + MZ_RN_AUX_BYTES) / 16; i += MZ_RN_THREADS) reinterpret_cast<uint4 *>(X.sp.tiles_ptr)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = tid; i < 24 * MZ_RN_OUT_ROWS; i += MZ_RN_THREADS) X.sp.out[i] = 0.0f;
    for (int i = tid; i < (R.n_steps - R.smem_first) * (int)(sizeof(mz_rn_step) / 4); i += MZ_RN_THREADS)
        reinterpret_cast<uint32_t *>(X.sp.prog)[i] = reinterpret_cast<const uint32_t *>(ta.steps + R.smem_first)[i];
    for (int i = tid; i < MZ_RN_OUT_ROWS; i += MZ_RN_THREADS) { X.sp.active[i] = 0; X.sp.pe[i] = 0; X.sp.dbl[i] = 0; X.sp.plane[i] = 0.0f; X.sp.tree_base[i] = 0ull; }
    mz_fence_proxy_async();
    mz_tc_fence_before();
    __syncthreads();
    mz_tc_fence_after();
    X.tmem = *X.sp.tmem_slot;
}
// binds this thread's row: call once the active flags of the launch are in shared memory
__device__ __forceinline__ void mz_rn_bind_rows(mz_rn_exec &X, const mz_rn_params &R) {
    const int row = (int)(threadIdx.x & 127);
    X.rowoff = (uint32_t)((row >> 3) * 1024 + (row & 7) * 128);
    X.row_valid = row < R.rows_valid && X.sp.active[X.my_tree < MZ_RN_OUT_ROWS ? X.my_tree : 0] != 0;
    X.tree_valid = row < R.ntrees && X.sp.active[row < MZ_RN_OUT_ROWS ? row : 0] != 0;
}
__device__ __forceinline__ void mz_rn_teardown(const mz_rn_exec &X) {
    mz_tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(X.tmem), "r"((uint32_t)MZ_RN_TMEM_COLS) : "memory");
}
// im2col tiles of the first representation convolution: element (row = (tree, cell), kk = tap * planes + plane)
template <typename F>
__device__ __forceinline__ void mz_rn_im2col(const mz_rn_exec &X, const mz_params &P, const mz_rn_params &R, F &&stacked /* (tree, plane, cell) -> float */) {
    const int k = R.ksize, pad = k / 2, kk_n = k * k * R.planes;
    for (int i = threadIdx.x; i < MZ_RN_TILES * 128 * kk_n; i += MZ_RN_THREADS) {
        const int kk = i % kk_n, row = (i / kk_n) & 127, tile = i / (kk_n * 128);
        float v = 0.0f;
        if (row < R.rows_valid) {
            const int tree = tile * R.tpt + row / R.cells, cell = row % R.cells;
            const int t = kk / R.planes, pl = kk % R.planes, x = cell % P.W + pad - (t % k), y = cell / P.W + pad - (t / k);
            if (X.sp.active[tree] && x >= 0 && x < P.W && y >= 0 && y < P.H) v = stacked(tree, pl, x + P.W * y);
        }
        mz_tc_store_bf16(X.sp.tiles + (uint32_t)(tile * MZ_RN_TILE_BYTES), row, kk, v);
    }
    mz_fence_proxy_async();
    __syncthreads();
}

template <int MODE>
__global__ void __launch_bounds__(MZ_RN_THREADS) mz_k_search_rn(const __grid_constant__ mz_params P, const __grid_constant__ mz_rn_params R, const mz_search_rn_args ta) {
    extern __shared__ __align__(1024) unsigned char mz_smem_rn[];
    const mz_search_args &a = ta.base;
    if (mz_cta_idle<MODE>(P, a, R.ntrees)) return;
    mz_rn_exec X;
    mz_rn_setup(X, P, R, ta, mz_smem_rn);
    const mz_rn_plan &sp = X.sp;
    const int tid = threadIdx.x, ln = tid & (MZ_LANES - 1);
    const uint32_t segmask = 0xffu << ((tid & 31) & ~7);

    // ---- per-tree state: 64 trees x 8 lanes, replicated in the lanes of each tree ----
    mz_root root[MZ_RN_NPASS]; mz_tree tree[MZ_RN_NPASS]; mz_minmax mm[MZ_RN_NPASS]; int ts[MZ_RN_NPASS]; int64_t gidx[MZ_RN_NPASS];
#pragma unroll
    for (int p = 0; p < MZ_RN_NPASS; p++) {
        ts[p] = 64 * p + (tid >> 3); gidx[p] = (int64_t)blockIdx.x * R.ntrees + ts[p];
        root[p] = mz_root{}; tree[p].A = nullptr; tree[p].hidden = nullptr;
        if (ts[p] < R.ntrees && gidx[p] < a.n) {
            tree[p] = mz_tree_at(P, a.tree_pool, gidx[p]);
            root[p] = mz_root_begin<MODE>(P, a, gidx[p], true);
            if (ln == 0) { sp.active[ts[p]] = root[p].active ? 1 : 0; sp.tree_base[ts[p]] = (unsigned long long)(uintptr_t)tree[p].A; }
        }
        mm[p].mn = INFINITY; mm[p].mx = -INFINITY;
    }
    __syncthreads();
    mz_rn_bind_rows(X, R);

    // ---- root: representation (im2col of the stacked observation) -> h0 in the pool; prediction(h0) ----
    mz_rn_im2col(X, P, R, [&](int t, int pl, int cell) { return mz_root_obs<MODE>(P, a, (int64_t)blockIdx.x * R.ntrees + t, cell + P.cells * pl); });
    // ---- phases: 0 = representation (root), 1 = prediction(h0), then per simulation 2 = prediction(parent), 3 = dynamics.
    //      One loop so that the step executor is inlined exactly once. ----
    const float *outV = sp.out, *outL = sp.out + 4 * MZ_RN_OUT_ROWS, *outR = sp.out + 20 * MZ_RN_OUT_ROWS;
    unsigned long long depth_sum = 0;
    mz_leaf leaf[MZ_RN_NPASS];
    int sim = 0;
#ifdef MZ_PHASE_TIMERS
    long long rn_t[8] = {0, 0, 0, 0, 0, 0, 0, 0}, rn_c = clock64();
#define MZ_RN_T(i) do { long long c_ = clock64(); rn_t[i] += c_ - rn_c; rn_c = c_; } while (0)
#else
#define MZ_RN_T(i)
#endif
    for (int phase = 0; ; phase = phase == 3 ? 2 : phase + 1) {
        MZ_RN_T(7);
        if (phase == 2) {
            if (++sim > P.S) break;
            // select (SelfPlay.jl:261-268); the parent's hidden state will be staged for both networks
#pragma unroll
            for (int p = 0; p < MZ_RN_NPASS; p++) {
                leaf[p].node = 0; leaf[p].parent = 0; leaf[p].action = 1; leaf[p].depth = 0; leaf[p].prior = 0.0f; leaf[p].parent_x = 0;
                if (root[p].active) {
                    uint16_t *path = sp.path + (size_t)ts[p] * (P.S + 2);
                    leaf[p] = mz_tree_select_lanes(P, tree[p], a.pbc0, a.sqrtN, root[p].legal, root[p].posmask, mm[p], root[p].game, root[p].move, (uint32_t)sim, ln, segmask, path);
                    depth_sum += (unsigned long long)leaf[p].depth;
                    if (ln == 0) {
                        sp.pe[ts[p]] = mz_nx_exp(leaf[p].parent_x); sp.dbl[ts[p]] = mz_nx_dbl(leaf[p].parent_x);
                        sp.plane[ts[p]] = P.act_plane_play[leaf[p].action];
                        reinterpret_cast<uint32_t *>(&tree[p].A[leaf[p].parent])[0] = leaf[p].parent_x + (1u << 24);   // one more doubling (Q6)
                    }
                }
            }
            __syncthreads();
            MZ_RN_T(0);
        }
        if (phase >= 1) mz_rn_stage_hidden(X, R);
        MZ_RN_T(1);      // root: h0 (pe = 0, dbl = 0); simulations: the parent's state (Q5), for prediction and again for dynamics
        int first, last, next;
        if (phase == 0) { first = R.prog_repr[0]; last = R.prog_repr[1]; next = R.prog_pred[0]; X.pool_slot = 0; }
        else if (phase == 1) { first = R.prog_pred[0]; last = R.prog_pred[1]; next = R.prog_pred[0]; }
        else if (phase == 2) { first = R.prog_pred[0]; last = R.prog_pred[1]; next = R.prog_dyn[0]; }
        else { first = R.prog_dyn[0]; last = R.prog_dyn[1]; next = sim < P.S ? R.prog_pred[0] : -1; X.pool_slot = sim; }
        mz_rn_run(X, R, first, last, next);
        MZ_RN_T(phase == 0 ? 2 : phase == 3 ? 4 : 3);
        if (phase == 0 || phase == 3) { __threadfence_block(); __syncthreads(); }   // hidden states written to the pool are read back by the next staging
        if (phase == 1) {
#pragma unroll
            for (int p = 0; p < MZ_RN_NPASS; p++) {
                if (root[p].active) mz_root_init(P, tree[p], root[p], a.exploration, outL + ts[p], MZ_RN_OUT_ROWS, ln, segmask);
            }
        } else if (phase == 3) {
#pragma unroll
            for (int p = 0; p < MZ_RN_NPASS; p++) {
                if (root[p].active) {
                    const uint16_t *path = sp.path + (size_t)ts[p] * (P.S + 2);
                    mz_tree_expand_lanes(P, tree[p], leaf[p].node, sim, root[p].legal, outL + ts[p], outR[ts[p]], leaf[p].prior, ln, segmask, MZ_RN_OUT_ROWS);
                    mz_tree_backup_lanes(P, tree[p], path, leaf[p].depth, outV[ts[p]], mm[p], ln, segmask);
                }
            }
            MZ_RN_T(5);
        }
    }
#ifdef MZ_PHASE_TIMERS
    if (a.stats && tid == 0) { for (int i = 0; i < 8; i++) atomicAdd(&a.stats[32 + i], (unsigned long long)rn_t[i]); atomicAdd(&a.stats[40], 1ull); }
    if (a.stats && (tid == 0 || tid == 128)) { for (int i = 0; i < 6; i++) atomicAdd(&a.stats[41 + 7 * (tid >> 7) + i], (unsigned long long)X.st_t[i]); atomicAdd(&a.stats[47 + 7 * (tid >> 7)], (unsigned long long)X.wq); }
#endif

    // ---- results (lane 0 of each tree): the trees' leaf depths are summed over the passes, so only the first pass adds them ----
#pragma unroll
    for (int p = 0; p < MZ_RN_NPASS; p++) {
        if (!(root[p].active && ln == 0)) continue;
        mz_root_finish<MODE>(P, a, gidx[p], tree[p], root[p], depth_sum);
        depth_sum = 0;
    }
    mz_rn_teardown(X);
}

// batched network callables (init_*(hyper::ResNetHP) callables): net 0 representation(stacked), 1 prediction(hidden),
// 2 dynamics(state_action).  Hidden states go through a scratch pool of one slot per tree (bf16, like the real pool).
__global__ void __launch_bounds__(MZ_RN_THREADS) mz_k_rn_forward(const __grid_constant__ mz_params P, const __grid_constant__ mz_rn_params R, const mz_search_rn_args ta) {
    extern __shared__ __align__(1024) unsigned char mz_smem_rn[];
    mz_rn_exec X;
    mz_rn_setup(X, P, R, ta, mz_smem_rn);
    const mz_rn_plan &sp = X.sp;
    const int tid = threadIdx.x;
    const int64_t g0 = (int64_t)blockIdx.x * R.ntrees;
    // scratch pool: per tree one hidden slot, addressed as tree_base + hidden_off + 0 * node_bytes
    for (int t = tid; t < R.ntrees; t += MZ_RN_THREADS) {
        sp.active[t] = g0 + t < ta.B ? 1 : 0;
        sp.tree_base[t] = (unsigned long long)(uintptr_t)(ta.scratch_pool + (size_t)(g0 + t) * R.node_bytes) - (unsigned long long)R.hidden_off_bytes;
    }
    __syncthreads();
    mz_rn_bind_rows(X, R);
    if (ta.net == 0) {
        mz_rn_im2col(X, P, R, [&](int t, int pl, int cell) { return ta.in[(g0 + t) * P.stack_size + cell + P.cells * pl]; });
    } else {
        // stage the fp32 input states as bf16 rows (dynamics: the caller's state is already doubled; the kernel multiplies the accumulator by 2)
        const float mul = ta.net == 2 ? 0.5f : 1.0f;
        const int in_dim = ta.net == 2 ? P.sa_size : P.hidden;
        for (int i = tid; i < MZ_RN_TILES * 128 * 64; i += MZ_RN_THREADS) {
            const int c = i & 63, row = (i >> 6) & 127, tile = i >> 13;
            float v = 0.0f;
            if (row < R.rows_valid && c < R.nf) {
                const int t = tile * R.tpt + row / R.cells, cell = row % R.cells;
                if (sp.active[t]) v = ta.in[(g0 + t) * in_dim + cell + P.cells * c] * mul;
            }
            mz_tc_store_bf16(sp.tiles + (uint32_t)(tile * MZ_RN_TILE_BYTES), row, c, v);
        }
        if (ta.net == 2) for (int t = tid; t < R.ntrees; t += MZ_RN_THREADS) sp.plane[t] = sp.active[t] ? ta.in[(g0 + t) * in_dim + P.hidden] : 0.0f;
        mz_fence_proxy_async();
        __syncthreads();
    }
    mz_rn_run(X, R, ta.net == 0 ? R.prog_repr[0] : ta.net == 1 ? R.prog_pred[0] : R.prog_dyn[0], ta.net == 0 ? R.prog_repr[1] : ta.net == 1 ? R.prog_pred[1] : R.prog_dyn[1], -1);
    __threadfence_block();
    __syncthreads();
    if (ta.net != 1) {   // hidden state out: Julia (W,H,nf) order, from the bf16 scratch pool
        for (int i = tid; i < R.ntrees * P.hidden; i += MZ_RN_THREADS) {
            const int t = i / P.hidden, k = i % P.hidden, cell = k % P.cells, c = k / P.cells;
            if (g0 + t < ta.B) {
                const unsigned short h = *reinterpret_cast<const unsigned short *>(ta.scratch_pool + (size_t)(g0 + t) * R.node_bytes + (size_t)cell * 128 + c * 2);
                ta.out1[(g0 + t) * P.hidden + k] = __uint_as_float((uint32_t)h << 16);
            }
        }
        if (ta.net == 2) for (int t = tid; t < R.ntrees; t += MZ_RN_THREADS) if (g0 + t < ta.B) ta.out2[g0 + t] = sp.out[20 * MZ_RN_OUT_ROWS + t];
    } else {
        for (int t = tid; t < R.ntrees; t += MZ_RN_THREADS) if (g0 + t < ta.B) {
            float logits[MZ_MAX_A], policy[MZ_MAX_A];
            for (int i = 0; i < P.A; i++) logits[i] = sp.out[4 * MZ_RN_OUT_ROWS + i * MZ_RN_OUT_ROWS + t];
            mz_softmax(logits, P.A, policy);
            ta.out1[g0 + t] = sp.out[t];
            for (int i = 0; i < P.A; i++) ta.out2[(g0 + t) * P.A + i] = policy[i];
        }
    }
    mz_rn_teardown(X);
}
