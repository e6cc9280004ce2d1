// mz_api.cu -- the C ABI of libmuzero_b200 (include/muzero_b200.h): context management, host<->device staging
// and kernel launches.  No torch types, no CPU fallback: every compute entry point launches sm_100a kernels.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <cstdarg>
#include <cstdio>
#include <memory>
#include <string>
#include <vector>
#include "mz_host.h"
#include "mz_learner_bptt.cuh"
#include "mz_rn_host.h"
#include "mz_kernels_rn.cuh"
#include "mz_kernels_sp.cuh"
#include "mz_kernels_lat.cuh"
#include "mz_learner_tc.cuh"

namespace {

thread_local std::string tl_error;

struct dev_buf {   // grow-only device scratch
    void *p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = (bytes + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct timed_launch { cudaEvent_t a, b; int family; };

struct nccl_api {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool load() {
        if (handle) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) { handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (handle) break; }
        if (!handle) return false;
        GetUniqueId = (decltype(GetUniqueId))dlsym(handle, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(handle, "ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))dlsym(handle, "ncclCommDestroy");
        AllReduce = (decltype(AllReduce))dlsym(handle, "ncclAllReduce");
        AllGather = (decltype(AllGather))dlsym(handle, "ncclAllGather");
        GetErrorString = (decltype(GetErrorString))dlsym(handle, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && CommDestroy && AllReduce && AllGather && GetErrorString;
    }
} g_nccl;

}  // namespace

extern "C" { static void p2p_teardown(mz_ctx *c); }

// One set of network weights (store_floats floats in the parameter store's layout) and the images the search kernels read, each rebuilt
// from w before its next use when version has moved past the image's (ensure_images, ensure_lat_image).  mz_ctx::own holds the context's
// networks; mz_ctx::opp the opponent networks of MZ_OPP_NETWORK, allocated on the first mz_set_opponent_weights / mz_snapshot_opponent with
// the images of the context's path only.
struct mz_wstore {
    float *w = nullptr; uint64_t version = 1, img_version = 0, lat_version = 0;
    unsigned char *tc = nullptr; float *tc_bias = nullptr;   // MZ_NN_BF16_TC: bf16 image and bias
    unsigned char *sp = nullptr; float *sp_bias = nullptr;   // MZ_NN_SPLIT_MMA: bf16 hi + lo image and bias
    float *lat = nullptr;                                    // mz_k_search_lat: fp32, rows = outputs
    unsigned char *rn = nullptr;                             // ResNet: bf16 image, BatchNorm folded
};

struct mz_ctx {
    mz_config cfg; mzh::model M; int device = 0;
    cudaStream_t stream = nullptr; bool own_stream = false;
    cudaStream_t stream2 = nullptr; cudaEvent_t ev_search[2] = {nullptr, nullptr};   // save / refill of move k beside the search of move k + 1 (run_wave)
    std::string err;
    size_t smem_bytes = 0; int sm_count = 0;
    // the learner's parameter store: fp32 parameters, ADAM moments and gradient, store_floats each; packed: in the padded device layout of the
    // FeedForwardHP kernels (mzh::pack_weights), else (ResNet) in blob order.  d_mask (use_batch_norm, ResNet): 1 = Flux parameter, 0 = BatchNorm
    // running statistic; net_bounds: where each network starts in the store, and its end
    mz_wstore own;   // the context's networks: own.w is the store's parameter array
    mz_wstore opp; bool opp_full = false;   // MZ_OPP_NETWORK's opponent networks (opp.w == NULL until first set); opp_full: a whole set is loaded
    float *d_m = nullptr, *d_v = nullptr, *d_grad = nullptr; int store_floats = 0; bool packed = true;
    unsigned char *d_mask = nullptr; int net_bounds[4] = {0, 0, 0, 0};
    size_t smem_bytes_tc = 0;   // tensor-core path (image: own.tc)
    // data-parallel learner over peer memory (mz_k_dp_adam): gradient exchange buffers (double-buffered) and arrival flags of every rank
    float *d_xgrad = nullptr; uint32_t *d_xflags = nullptr; float *peer_grad[MZ_DP_MAX_RANKS] = {}; uint32_t *peer_flags[MZ_DP_MAX_RANKS] = {};
    bool p2p = false; uint32_t dp_step = 0;
    // the learner's scratch: the ResNet unroll (h, h', state-action input, value, policy, reward, node pool); MZ_GRAD_BPTT on the SIMT kernel
    // (activations, per-tile partial gradients) and on the tensor cores (saved activation / gradient tiles, per-chunk partial gradients)
    dev_buf rn_buf[7], bptt_act, bptt_gpart, lr_xsave, lr_dzsave, lr_gpart;
    // MZ_GRAD_BPTT on the tensor cores (mz_learner_tc.cuh): backward rounds
    mz_lr_plan lrp{}; mz_lr_bround *d_brounds = nullptr; size_t smem_bytes_lr = 0;
    // mz_k_search_lat (one tree per 2-CTA cluster, networks and tree resident in shared memory): calls with at most lat_max_roots roots
    int lat_image_floats = 0;
    unsigned char *h_lat_stage = nullptr, *d_lat_stage = nullptr; size_t lat_stage_cap = 0;   // one pinned / device block for all inputs and outputs of a small run_mcts call
    bool lat_ok = false; int lat_w_floats = 0, lat_pbc_smem = 0, lat_max_roots = 0, lat_max_slots = 0; size_t smem_bytes_lat = 0;
    bool persist_ok = true;     // MUZERO_B200_PERSIST=0: one search launch per move also for single-wave self-play on the split-precision path
    bool slots_dirty = false;   // a wave is in progress or ended with an error: the slots are reset before the next one
    int refill_wave_sync = 1;   // 1: mz_k_save_refill starts new games only when every slot is free (default; MUZERO_B200_REFILL=immediate refills at once)
    mz_sp_plan spp{}; mz_sp_args spa{}; mz_sp_round *d_rounds_sp = nullptr; size_t smem_bytes_sp = 0;   // split-precision tensor-core path
    double *d_pbc0 = nullptr, *d_sqrtN = nullptr;
    void *d_trees = nullptr;
    mz_slots slots{}; mz_ring ring{};
    mz_ring play_ring{};   // mz_play_games: a ring of its own, so that play_game's histories go to the caller and not into the replay buffer
    unsigned long long *d_stats = nullptr;
    mz_batch batch{}; int batch_cap = 0;
    float *d_pv = nullptr, *d_pr = nullptr, *d_pp = nullptr, *d_rowv = nullptr, *d_rowp = nullptr, *d_rowinvg = nullptr;
    double *d_rowr = nullptr, *d_lossout = nullptr;
    int64_t *h_counters = nullptr; double *h_lossout = nullptr; unsigned long long *h_stats = nullptr;   // pinned
    int64_t *h_wave = nullptr, *d_wave = nullptr; cudaEvent_t ev_wave[2] = {nullptr, nullptr};   // pinned: two snapshots of the counters, self-play runs one iteration ahead of the host
    dev_buf scratch[12];
    int64_t adam_t = 1; double bp1 = 0.9, bp2 = 0.999;   // Flux.ADAM: the next update's step number and beta powers (adam_seek)
    ncclComm_t comm = nullptr; int rank = 0, nranks = 1;
    // net_type = MZ_NET_RESNET
    mzh::rn_model rn; mz_rn_step *d_rn_steps = nullptr; size_t smem_bytes_rn = 0;
    // grad_mode = MZ_GRAD_BPTT
    mzh::bptt_program bptt; mz_bstage *d_bstages[2] = {nullptr, nullptr}; size_t smem_bytes_bptt = 0;
    float *d_w_fold = nullptr;   // use_batch_norm + MZ_GRAD_BPTT: the weights with every BatchNorm folded into its Dense layer
    int bptt_dims[4] = {0, 0, 0, 0};   // mz_bptt_args: dim_wide, dim_narrow, wfloats[2]
    int64_t launches = 0; bool timing = false; std::vector<timed_launch> timed; double fam_ms[8] = {0}; int64_t fam_n[8] = {0};
    double last_mean_legal = 0, last_mean_depth = 0;
};

namespace {

int fail(mz_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
    tl_error = buf;
    if (c) c->err = buf;
    return code;
}
#define MZ_CUDA(c, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail((c), MZ_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
#define MZ_CHECK_CTX(c) do { if (!(c)) return fail(nullptr, MZ_E_ARG, "ctx is NULL"); MZ_CUDA((c), cudaSetDevice((c)->device)); } while (0)

struct launch_scope {   // counts launches and, when enabled, brackets them with events on the stream they go to (default: the ctx stream)
    mz_ctx *c; int family; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr;
    launch_scope(mz_ctx *c_, int fam, cudaStream_t st_ = nullptr) : c(c_), family(fam), st(st_ ? st_ : c_->stream) {
        c->launches++;
        if (c->timing) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, st); }
    }
    ~launch_scope() { if (c->timing) { cudaEventRecord(b, st); c->timed.push_back({a, b, family}); } }
};

void collect_timings(mz_ctx *c) {
    if (c->timed.empty()) return;
    cudaStreamSynchronize(c->stream);
    if (c->stream2) cudaStreamSynchronize(c->stream2);
    for (auto &t : c->timed) {
        float ms = 0; cudaEventElapsedTime(&ms, t.a, t.b);
        c->fam_ms[t.family] += ms; c->fam_n[t.family]++;
        cudaEventDestroy(t.a); cudaEventDestroy(t.b);
    }
    c->timed.clear();
}

// The dynamic shared memory limit of a kernel is a per-function (process-wide) attribute: contexts with different network /
// tree sizes share it, so it is always raised to everything the device allows (the launch itself asks for what it needs).
template <typename F> cudaError_t allow_max_smem(F *func, const cudaDeviceProp &prop) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, func);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(prop.sharedMemPerBlockOptin - fa.sharedSizeBytes));
}
template <typename T> cudaError_t dmalloc(T **p, size_t n) { return cudaMalloc((void **)p, n * sizeof(T) > 0 ? n * sizeof(T) : 16); }

void free_ring(mz_ring &r) {
    void *ptrs[] = {r.game_id, r.T, r.h_p1, r.h_p2, r.h_action, r.h_reward, r.h_to_play, r.h_cv, r.h_rv, r.h_rrv, r.reanalysed, r.q_pos, r.q_game, r.prefix, r.upd, r.counters};
    for (void *p : ptrs) if (p) cudaFree(p);
    r = mz_ring{};
}
int alloc_ring(mz_ctx *c, mz_ring &r, size_t R) {
    const mz_params &P = c->M.P; const size_t Tm = (size_t)P.Tmax;
    free_ring(r);
    r.capacity = (int64_t)R;
    MZ_CUDA(c, dmalloc(&r.game_id, R)); MZ_CUDA(c, dmalloc(&r.T, R));
    MZ_CUDA(c, dmalloc(&r.h_p1, R * Tm)); MZ_CUDA(c, dmalloc(&r.h_p2, R * Tm)); MZ_CUDA(c, dmalloc(&r.h_action, R * Tm));
    MZ_CUDA(c, dmalloc(&r.h_reward, R * Tm)); MZ_CUDA(c, dmalloc(&r.h_to_play, R * Tm)); MZ_CUDA(c, dmalloc(&r.h_cv, R * Tm * P.A)); MZ_CUDA(c, dmalloc(&r.h_rv, R * Tm));
    MZ_CUDA(c, dmalloc(&r.q_pos, R * Tm)); MZ_CUDA(c, dmalloc(&r.q_game, R)); MZ_CUDA(c, dmalloc(&r.prefix, R)); MZ_CUDA(c, dmalloc(&r.upd, R * Tm));
    MZ_CUDA(c, cudaMemset(r.q_pos, 0, R * Tm * 4)); MZ_CUDA(c, cudaMemset(r.q_game, 0, R * 4)); MZ_CUDA(c, cudaMemset(r.upd, 0, R * Tm * 8));
    MZ_CUDA(c, dmalloc(&r.h_rrv, R * Tm)); MZ_CUDA(c, dmalloc(&r.reanalysed, R)); MZ_CUDA(c, cudaMemset(r.reanalysed, 0, R)); MZ_CUDA(c, cudaMemset(r.h_rrv, 0, R * Tm * sizeof(float)));
    MZ_CUDA(c, dmalloc(&r.counters, 8)); MZ_CUDA(c, cudaMemset(r.counters, 0, 8 * sizeof(int64_t)));
    MZ_CUDA(c, cudaMemset(r.T, 0, R * sizeof(int32_t)));
    return MZ_OK;
}

int alloc_batch(mz_ctx *c, int B) {
    if (B <= c->batch_cap) return MZ_OK;
    const mz_params &P = c->M.P; int K1 = P.K + 1;
    // free + null first: if a later allocation fails the ctx holds no dangling pointer (batch_cap = 0 forces a clean retry)
    void **ptrs[] = {(void **)&c->batch.weights, (void **)&c->batch.index, (void **)&c->batch.obs, (void **)&c->batch.actions, (void **)&c->batch.values,
                     (void **)&c->batch.rewards, (void **)&c->batch.policies, (void **)&c->batch.gscale, (void **)&c->d_pv, (void **)&c->d_pr, (void **)&c->d_pp,
                     (void **)&c->d_rowv, (void **)&c->d_rowp, (void **)&c->d_rowinvg, (void **)&c->d_rowr};
    for (void **p : ptrs) { if (*p) cudaFree(*p); *p = nullptr; }
    c->batch_cap = 0;
    MZ_CUDA(c, dmalloc(&c->batch.index, (size_t)B * 2)); MZ_CUDA(c, dmalloc(&c->batch.obs, (size_t)B * P.stack_size));
    MZ_CUDA(c, dmalloc(&c->batch.actions, (size_t)B * K1)); MZ_CUDA(c, dmalloc(&c->batch.values, (size_t)B * K1));
    MZ_CUDA(c, dmalloc(&c->batch.rewards, (size_t)B * K1)); MZ_CUDA(c, dmalloc(&c->batch.policies, (size_t)B * K1 * P.A));
    MZ_CUDA(c, dmalloc(&c->batch.gscale, (size_t)B)); MZ_CUDA(c, dmalloc(&c->batch.weights, (size_t)B));
    MZ_CUDA(c, dmalloc(&c->d_pv, (size_t)B * K1)); MZ_CUDA(c, dmalloc(&c->d_pr, (size_t)B * K1)); MZ_CUDA(c, dmalloc(&c->d_pp, (size_t)B * K1 * P.A));
    MZ_CUDA(c, dmalloc(&c->d_rowv, (size_t)B)); MZ_CUDA(c, dmalloc(&c->d_rowp, (size_t)B)); MZ_CUDA(c, dmalloc(&c->d_rowinvg, (size_t)B));
    MZ_CUDA(c, dmalloc(&c->d_rowr, (size_t)B));
    c->batch_cap = B;
    return MZ_OK;
}

// one array of the parameter store (d_w, d_m, d_v, d_grad) to / from the caller's blob order (n_params floats)
int store_to_host(mz_ctx *c, const float *d, float *blob) {
    std::vector<float> dev(c->packed ? (size_t)c->store_floats : 0);
    MZ_CUDA(c, cudaMemcpyAsync(c->packed ? dev.data() : blob, d, (size_t)c->store_floats * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->packed) mzh::unpack_weights(c->M.P, dev.data(), blob);
    return MZ_OK;
}
int store_from_host(mz_ctx *c, float *d, const float *blob) {
    std::vector<float> dev(c->packed ? (size_t)c->store_floats : 0);
    if (c->packed) mzh::pack_weights(c->M.P, blob, dev.data());
    MZ_CUDA(c, cudaMemcpyAsync(d, c->packed ? dev.data() : blob, (size_t)c->store_floats * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
int upload_weights(mz_ctx *c, const std::vector<float> &src) {
    const int r = store_from_host(c, c->own.w, src.data());
    c->own.version++;                                      // the images are rebuilt before their next use (ensure_images)
    return r;
}
int download_weights(mz_ctx *c, std::vector<float> &src) {
    src.resize((size_t)c->M.P.n_params);
    return store_to_host(c, c->own.w, src.data());
}

int read_counters(mz_ctx *c) {
    MZ_CUDA(c, cudaMemcpyAsync(c->h_counters, c->ring.counters, 8 * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
int write_counters(mz_ctx *c) {
    MZ_CUDA(c, cudaMemcpyAsync(c->ring.counters, c->h_counters, 8 * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}

int ctx_net_params(const mz_ctx *c, int net) {
    if (c->cfg.net_type == MZ_NET_RESNET) return net == MZ_NET_ALL ? mzh::rn_total_params(c->rn) : c->rn.n_params[net];
    return mzh::net_params(c->M.P, net);
}
int ctx_net_offset(const mz_ctx *c, int net) {
    if (c->cfg.net_type == MZ_NET_RESNET) return net == MZ_NET_ALL ? 0 : c->rn.base[net];
    return mzh::net_src_offset(c->M.P, net);
}
template <typename T> int h2d(mz_ctx *c, dev_buf &b, const T *host, size_t n, T **out) {
    MZ_CUDA(c, b.ensure(n * sizeof(T) + 16));
    if (host && n) MZ_CUDA(c, cudaMemcpyAsync(b.p, host, n * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    *out = (T *)b.p;
    return MZ_OK;
}
template <typename T> int d2h(mz_ctx *c, T *host, const T *dev, size_t n) {
    if (host && n) MZ_CUDA(c, cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    return MZ_OK;
}
#define MZ_TRY(x) do { int r_ = (x); if (r_ != MZ_OK) return r_; } while (0)
// h2d's allocation for scratch that a kernel may read before it writes it: zeroed whenever it grows
template <typename T> int alloc_zeroed(mz_ctx *c, dev_buf &b, size_t n, T **out) {
    const size_t cap = b.cap;
    MZ_TRY(h2d<T>(c, b, nullptr, n, out));
    if (b.cap != cap) MZ_CUDA(c, cudaMemsetAsync(b.p, 0, b.cap, c->stream));
    return MZ_OK;
}

// Flux.ADAM's state after `steps_done` updates: the next update is step adam_t = steps_done + 1 with the beta powers beta^adam_t, by repeated
// product as the running state builds them
void adam_seek(mz_ctx *c, int64_t steps_done) {
    c->adam_t = steps_done + 1; c->bp1 = 0.9; c->bp2 = 0.999;
    for (int64_t i = 0; i < steps_done; i++) { c->bp1 *= 0.9; c->bp2 *= 0.999; }
}

// which kernels a learner step of `grad_mode` runs on in this context: 0 = fp32 SIMT (mz_k_learn_forward / mz_k_learn_bptt), 1 = the unroll forward
// on the tensor cores (mz_k_learn_forward_sp), 2 = forward and backward on the tensor cores (mz_k_learn_bptt_tc + mz_k_learn_dw), 3 = ResNet: unroll
// through the bf16 inference kernel (mz_k_rn_forward), -1 = not available (ResNet with MZ_GRAD_BPTT).  MUZERO_B200_BPTT_SIMT (set to anything) keeps
// MZ_GRAD_BPTT on the SIMT kernel.
int learner_path(const mz_ctx *c, int grad_mode) {
    if (c->cfg.net_type == MZ_NET_RESNET) return grad_mode == MZ_GRAD_REFERENCE_L2 ? 3 : -1;
    if (c->cfg.nn_mode != MZ_NN_SPLIT_MMA) return 0;
    if (grad_mode == MZ_GRAD_BPTT) return (c->lrp.ok && !getenv("MUZERO_B200_BPTT_SIMT")) ? 2 : 0;
    return 1;
}

// where this step's local gradient goes: d_grad, or -- data-parallel over peer memory -- the half of the exchange buffer the next
// update reads (the other half may still be read by a peer that is one step behind)
float *grad_out(mz_ctx *c) { return c->p2p ? c->d_xgrad + (size_t)((c->dp_step + 1u) & 1u) * (size_t)c->M.P.total_floats : c->d_grad; }

// ResNet: fetch the parameters, fold BatchNorm and pack the bf16 B-operand images on the host (rn_pack, one block per program step), upload
// the image.  (A device-side packer would save the round trip; the ResNet learner is a functional path, not a tuned one.)
int rn_sync_image(mz_ctx *c, mz_wstore &s) {
    std::unique_ptr<float[]> blob(new float[(size_t)c->store_floats]);   // not zero-filled: the copy overwrites all of it
    MZ_TRY(store_to_host(c, s.w, blob.get()));
    std::vector<unsigned char> image;
    mzh::rn_pack(c->rn, blob.get(), image);
    MZ_CUDA(c, cudaMemcpyAsync(s.rn, image.data(), (size_t)c->rn.image_bytes, cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    s.img_version = s.version;
    return MZ_OK;
}

// The tensor-core and ResNet paths read bf16 images of the weights; whenever a store's weights have changed (set_weights, an ADAM step,
// mz_set_opponent_weights, mz_snapshot_opponent) its image is rebuilt before the next kernel that reads it (FeedForwardHP: on the device).
int ensure_images(mz_ctx *c, mz_wstore &s) {
    if (s.img_version == s.version) return MZ_OK;
    if (c->cfg.net_type == MZ_NET_RESNET) return rn_sync_image(c, s);
    const mz_params &P = c->M.P;
    mz_pack_args a{}; a.w = s.w;
    if (c->cfg.nn_mode == MZ_NN_SPLIT_MMA && s.sp) {
        a.mode = 2; a.image = s.sp; a.bias = s.sp_bias;
        for (int i = 0; i < P.n_layers; i++) { a.off[i] = c->spp.w_off[i]; a.bytes[i] = c->spp.w_bytes[i]; a.bias_off[i] = i * 64; }
    } else if (c->cfg.nn_mode == MZ_NN_BF16_TC && s.tc) {
        a.mode = 1; a.image = s.tc; a.bias = s.tc_bias;
        for (int i = 0; i < P.n_layers; i++) { a.off[i] = P.tc_a_off[i]; a.bytes[i] = 0; a.bias_off[i] = P.tc_bias_off[i]; }
    } else { s.img_version = s.version; return MZ_OK; }
    { launch_scope ls(c, 5); mz_k_pack_images<<<dim3((unsigned)P.n_layers, 4), 256, 0, c->stream>>>(P, a); }
    MZ_CUDA(c, cudaGetLastError());
    s.img_version = s.version;
    return MZ_OK;
}
int ensure_images(mz_ctx *c) { return ensure_images(c, c->own); }

// the weight image of mz_k_search_lat (rows = outputs), rebuilt from the store's weights when they have changed since it was last used
int ensure_lat_image(mz_ctx *c, mz_wstore &s) {
    if (s.lat_version == s.version) return MZ_OK;
    const mz_params &P = c->M.P;
    mz_pack_lat_args a{}; a.w = s.w; a.image = s.lat;
    int off = 0;
    for (int n = 0; n < 3; n++) for (int l = P.nets[n].first; l < P.nets[n].first + P.nets[n].n_trunk + P.nets[n].n_h1 + P.nets[n].n_h2; l++) { a.off[l] = off; off += mz_lat_layer_floats(P.layers[l].in, P.layers[l].out); }
    { launch_scope ls(c, 5); mz_k_pack_lat<<<dim3((unsigned)P.n_layers, 4), 256, 0, c->stream>>>(P, a); }
    MZ_CUDA(c, cudaGetLastError());
    s.lat_version = s.version;
    return MZ_OK;
}

// ---- ResNet learner (grad_mode = MZ_GRAD_REFERENCE_L2: the reference's actual update, Q20) ---------------------------------------------
// The K-step unroll (Learning.jl:347-370) as a sequence of the batched network kernel mz_k_rn_forward on device buffers (bf16 inference
// arithmetic, BatchNorm with its stored statistics: the reference computes the predictions outside the pullback, i.e. in test mode), then
// the loss tail; the update is ADAM on 2 * theta over Flux.params (launch_update), after which the bf16 image is rebuilt (ensure_images).
int rn_forward_dev(mz_ctx *c, int net, int B, const float *d_in, float *d_o1, float *d_o2, unsigned char *pool) {
    mz_search_rn_args t{}; t.image = c->own.rn; t.steps = c->d_rn_steps; t.net = net; t.B = B; t.in = d_in; t.out1 = d_o1; t.out2 = d_o2; t.scratch_pool = pool;
    const int nt = c->rn.R.ntrees;
    launch_scope ls(c, 3); mz_k_rn_forward<<<(B + nt - 1) / nt, MZ_RN_THREADS, c->smem_bytes_rn, c->stream>>>(c->M.P, c->rn.R, t);
    return MZ_OK;
}
int rn_learn_forward(mz_ctx *c, int B) {
    const mz_params &P = c->M.P;
    MZ_TRY(ensure_images(c));
    float *h, *nh, *sa, *o1, *o2, *r; unsigned char *pool;
    MZ_TRY(h2d<float>(c, c->rn_buf[0], nullptr, (size_t)B * P.hidden, &h)); MZ_TRY(h2d<float>(c, c->rn_buf[1], nullptr, (size_t)B * P.hidden, &nh));
    MZ_TRY(h2d<float>(c, c->rn_buf[2], nullptr, (size_t)B * P.sa_size, &sa)); MZ_TRY(h2d<float>(c, c->rn_buf[3], nullptr, (size_t)B, &o1));
    MZ_TRY(h2d<float>(c, c->rn_buf[4], nullptr, (size_t)B * P.A, &o2)); MZ_TRY(h2d<float>(c, c->rn_buf[5], nullptr, (size_t)B, &r));
    MZ_TRY(h2d<unsigned char>(c, c->rn_buf[6], nullptr, (size_t)B * c->rn.R.node_bytes + 256, &pool));
    const int K1 = P.K + 1, tb = (B + 127) / 128;
    MZ_TRY(rn_forward_dev(c, 0, B, c->batch.obs, h, nullptr, pool));                                      // :347
    MZ_TRY(rn_forward_dev(c, 1, B, h, o1, o2, pool));                                                      // :351 (= row 1's prediction, Q19)
    { launch_scope ls(c, 3); mz_k_rn_scatter<<<tb, 128, 0, c->stream>>>(B, P.A, K1, 0, P.K > 0 ? 1 : -1, o1, o2, nullptr, 1, c->d_pv, c->d_pp, c->d_pr); }
    for (int i = 1; i <= P.K; i++) {                                                                       // :355-370
        if (i > 1) {
            MZ_TRY(rn_forward_dev(c, 1, B, h, o1, o2, pool));
            launch_scope ls(c, 3); mz_k_rn_scatter<<<tb, 128, 0, c->stream>>>(B, P.A, K1, i, -1, o1, o2, nullptr, 0, c->d_pv, c->d_pp, c->d_pr);
        }
        { launch_scope ls(c, 3); mz_k_rn_make_sa<<<(B * P.sa_size + 255) / 256, 256, 0, c->stream>>>(B, P.hidden, P.cells, P.A, K1, i - 1, h, c->batch.actions, sa); }
        MZ_TRY(rn_forward_dev(c, 2, B, sa, nh, r, pool));
        { launch_scope ls(c, 3); mz_k_rn_scatter<<<tb, 128, 0, c->stream>>>(B, P.A, K1, i, -1, nullptr, nullptr, r, 0, c->d_pv, c->d_pp, c->d_pr); }
        float *t = h; h = nh; nh = t;
    }
    return MZ_OK;
}

// the loss (Learning.jl:261-288) from the unroll's predictions: per-sample partial sums, then the data terms and each network's sum(theta^2).
// Without a mask, the 7-CTA reduce sums theta^2 layer by layer over the padded store (the FeedForwardHP losses' summation order); with one,
// the data terms and then the masked sums over net_bounds (Flux.params leave out the BatchNorm statistics)
void launch_loss(mz_ctx *c, int B) {
    const mz_params &P = c->M.P;
    { launch_scope ls(c, 3); const int ry = P.K + 1 < MZ_LOSS_RY ? P.K + 1 : MZ_LOSS_RY;
      mz_k_loss_rows<<<(B + 31) / 32, dim3(32, (unsigned)ry), 0, c->stream>>>(P, B, c->batch, c->d_pv, c->d_pr, c->d_pp, c->d_rowv, c->d_rowr, c->d_rowp, c->d_rowinvg); }
    if (c->d_mask) {
        { launch_scope ls(c, 3); mz_k_loss_reduce<<<4, 1024, 0, c->stream>>>(P, B, c->d_rowv, c->d_rowr, c->d_rowp, c->d_rowinvg, c->own.w, c->d_lossout, 4); }
        { launch_scope ls(c, 3); mz_k_sqnorm_masked<<<3, 1024, 0, c->stream>>>(c->net_bounds[0], c->net_bounds[1], c->net_bounds[2], c->net_bounds[3], c->own.w, c->d_mask, c->d_lossout); }
    } else { launch_scope ls(c, 3); mz_k_loss_reduce<<<7, 1024, 0, c->stream>>>(P, B, c->d_rowv, c->d_rowr, c->d_rowp, c->d_rowinvg, c->own.w, c->d_lossout); }
}

int launch_learn_forward(mz_ctx *c, int B, int grad_mode = MZ_GRAD_REFERENCE_L2) {
    const mz_params &P = c->M.P;
    const int path = learner_path(c, grad_mode);
    if (path == -1) return fail(c, MZ_E_UNSUPPORTED, "the ResNet learner implements MZ_GRAD_REFERENCE_L2 (the reference's update); the backward pass through the convolution towers is not built");
    if (path != 3 && grad_mode != MZ_GRAD_REFERENCE_L2 && grad_mode != MZ_GRAD_BPTT) return fail(c, MZ_E_ARG, "unknown grad_mode %d", grad_mode);
    mz_learn_args a{}; a.wglob = c->own.w; a.B = B; a.max_dim = c->M.max_dim; a.max_layer_floats = c->M.max_layer_floats; a.batch = c->batch;
    a.pred_values = c->d_pv; a.pred_rewards = c->d_pr; a.pred_policies = c->d_pp;
    const int tiles = (B + MZ_ROWS - 1) / MZ_ROWS;
    if (path == 3) MZ_TRY(rn_learn_forward(c, B));
    else if (path == 2) {
        // forward + backward on the tensor cores (mz_learner_tc.cuh): kernel 1 = unroll forward + dX chain with saved tiles, kernel 2 = dW / db
        MZ_TRY(ensure_images(c));
        const mz_lr_plan &L = c->lrp;
        const int chunks = tiles < 16 ? tiles : 16;
        const size_t bytes = (size_t)tiles * L.slots_per_cta * MZ_SP_TILE_BYTES;
        unsigned char *xsave, *dzsave; float *gpart;
        MZ_TRY(alloc_zeroed(c, c->lr_xsave, bytes, &xsave)); MZ_TRY(alloc_zeroed(c, c->lr_dzsave, bytes, &dzsave));
        MZ_TRY(alloc_zeroed(c, c->lr_gpart, (size_t)chunks * P.total_floats, &gpart));
        mz_lr_args t{}; t.sp = c->spa; t.sp.pbc_smem = 0; t.brounds = c->d_brounds;
        for (int n = 0; n < 3; n++) {
            t.bfirst[n] = L.bfirst[n]; t.bn_rounds[n] = L.bn_rounds[n]; t.slot_base[n] = L.slot_base[n]; t.layers_in_net[n] = L.layers_in_net[n]; t.first_layer[n] = P.nets[n].first;
            for (int h = 0; h < 2; h++) { t.start_tile[n][h] = L.start_tile[n][h]; t.start_layer[n][h] = L.start_layer[n][h]; t.start_perm[n][h] = L.start_perm[n][h]; }
        }
        t.btotal_rounds = L.btotal_rounds; t.slots_per_cta = L.slots_per_cta; t.n_eval = L.n_eval; t.lg_off = (L.bwarea_bytes + 127) & ~127; t.dh_extra = mz_lr_alias_fits(c->spp.bias_floats, P.hidden_pad) ? 0 : 1;
        t.f.f = a; t.xsave = xsave; t.dzsave = dzsave; t.dbg = getenv("MUZERO_B200_LR_STAMPS") ? c->d_stats + 4 : nullptr;
        t.inv_g_sum = c->d_lossout + 7;                                    // (slot 7 of the loss scratch is free)
        { launch_scope ls(c, 3); mz_k_inv_g_sum<<<1, 1024, 0, c->stream>>>(B, c->batch.gscale, (P.per && c->batch.weights) ? c->batch.weights : nullptr, c->d_lossout + 7); }
        { launch_scope ls(c, 3); mz_k_learn_bptt_tc<<<tiles, MZ_SP_THREADS, c->smem_bytes_lr, c->stream>>>(P, t); }
        mz_dw_args d{}; d.xsave = xsave; d.dzsave = dzsave; d.gpart = gpart; d.tiles = tiles; d.chunks = chunks; d.slots_per_cta = L.slots_per_cta; d.n_eval = L.n_eval;
        for (int n = 0; n < 3; n++) { d.slot_base[n] = L.slot_base[n]; d.layers_in_net[n] = L.layers_in_net[n]; d.first_layer[n] = P.nets[n].first; }
        { launch_scope ls(c, 3); mz_k_learn_dw<<<dim3((unsigned)P.n_layers, (unsigned)chunks), 128, MZ_DW_STAGES * 2 * MZ_SP_TILE_BYTES + 1024, c->stream>>>(P, d); }
        // (use_batch_norm: the images these kernels read are the folded layers (mz_k_pack_images), so the sums are dW', db': same chain rule as below)
        if (c->cfg.use_batch_norm) { launch_scope ls(c, 4); mz_k_grad_reduce_bn<<<dim3((unsigned)P.n_layers, 16), 256, 0, c->stream>>>(P, chunks, gpart, c->own.w, grad_out(c)); }
        else { launch_scope ls(c, 4); mz_k_grad_reduce<<<(P.total_floats + 255) / 256, 256, 0, c->stream>>>(P.total_floats, chunks, gpart, c->own.w, grad_out(c)); }
    } else if (grad_mode == MZ_GRAD_BPTT) {   // forward + backward through the unroll in one kernel; per-tile partial gradients
        if (!c->smem_bytes_bptt) return fail(c, MZ_E_UNSUPPORTED, "MZ_GRAD_BPTT is not built for this network: it needs every layer output and every layer input other than the observation stack to be at most 64 wide, and its buffers to fit one CTA's shared memory");
        float *act, *gpart;
        MZ_TRY(h2d<float>(c, c->bptt_act, nullptr, (size_t)tiles * c->bptt.plan.tile_floats, &act));
        MZ_TRY(h2d<float>(c, c->bptt_gpart, nullptr, (size_t)tiles * P.total_floats, &gpart));
        mz_bptt_args b{}; b.f = a; b.act = act; b.gpart = gpart; b.stages[0] = c->d_bstages[0]; b.stages[1] = c->d_bstages[1];
        b.dim_wide = c->bptt_dims[0]; b.dim_narrow = c->bptt_dims[1]; b.wfloats[0] = c->bptt_dims[2]; b.wfloats[1] = c->bptt_dims[3];
        if (c->cfg.use_batch_norm) {   // BatchNorm in test mode = a Dense layer with folded weights: the kernel runs on the folded copy, the reduce applies the chain rule
            if (!c->d_w_fold) MZ_CUDA(c, dmalloc(&c->d_w_fold, (size_t)P.total_floats));
            { launch_scope ls(c, 5); mz_k_bn_fold<<<dim3((unsigned)P.n_layers, 4), 256, 0, c->stream>>>(P, c->own.w, c->d_w_fold); }
            b.f.wglob = c->d_w_fold;
        }
        { launch_scope ls(c, 3); mz_k_learn_bptt<<<tiles, MZ_THREADS, c->smem_bytes_bptt, c->stream>>>(P, c->bptt.plan, b); }
        if (c->cfg.use_batch_norm) { launch_scope ls(c, 4); mz_k_grad_reduce_bn<<<dim3((unsigned)P.n_layers, 16), 256, 0, c->stream>>>(P, tiles, gpart, c->own.w, grad_out(c)); }
        else { launch_scope ls(c, 4); mz_k_grad_reduce<<<(P.total_floats + 255) / 256, 256, 0, c->stream>>>(P.total_floats, tiles, gpart, c->own.w, grad_out(c)); }
    } else if (path == 1) {   // the unroll on the tensor cores (mz_kernels_sp.cuh)
        MZ_TRY(ensure_images(c));
        mz_learn_sp_args t{}; t.sp = c->spa; t.B = B; t.batch = c->batch; t.pred_values = c->d_pv; t.pred_rewards = c->d_pr; t.pred_policies = c->d_pp;
        launch_scope ls(c, 3); mz_k_learn_forward_sp<<<tiles, MZ_SP_THREADS, c->smem_bytes_sp, c->stream>>>(P, t);
    } else {
        launch_scope ls(c, 3);
        if (c->cfg.use_batch_norm) mz_k_learn_forward<true><<<tiles, MZ_THREADS, c->smem_bytes, c->stream>>>(P, a);
        else mz_k_learn_forward<false><<<tiles, MZ_THREADS, c->smem_bytes, c->stream>>>(P, a);
    }
    launch_loss(c, B);
    MZ_CUDA(c, cudaGetLastError());
    return MZ_OK;
}
// losses (Learning.jl:283-287): data loss = value_loss + reward_loss + policy_loss; each net adds its own sum(theta^2)
int finish_losses(mz_ctx *c, int B, float *losses) {
    MZ_CUDA(c, cudaMemcpyAsync(c->h_lossout, c->d_lossout, 8 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    const double *o = c->h_lossout;
    float value_loss = (float)(o[0] / (double)B);
    float policy_loss = (float)((o[1] / (double)B) * (o[2] / (double)B));   // mean_j(s_j) * mean_i(1/g_i), Q21
    float data;
    if (c->cfg.intermediate_rewards) data = (float)(((double)value_loss + o[3] / (double)B) + (double)policy_loss);
    else data = (value_loss + 0.0f) + policy_loss;
    for (int n = 0; n < 3; n++) losses[n] = data + (float)o[4 + n];
    return MZ_OK;
}
// one learning! update of the parameter store.  The BatchNorm statistics (d_mask = 0) have zero gradient and stay put.
int launch_update(mz_ctx *c, int64_t t, int grad_mode) {
    const int n = c->store_floats;
    if (t == 1) {   // learning! builds a fresh optimiser (Learning.jl:318): restarting at step 1 clears the moments too
        if (c->adam_t > 1) { MZ_CUDA(c, cudaMemsetAsync(c->d_m, 0, (size_t)n * 4, c->stream)); MZ_CUDA(c, cudaMemsetAsync(c->d_v, 0, (size_t)n * 4, c->stream)); }
        adam_seek(c, 0);
    }
    // MZ_GRAD_BPTT: d_grad was produced by launch_learn_forward (mz_k_learn_bptt + mz_k_grad_reduce)
    if (grad_mode == MZ_GRAD_REFERENCE_L2 && !c->p2p && !c->comm) {   // one GPU: gradient (2 * theta) and update in one launch
        launch_scope ls(c, 4); mz_k_adam_l2<<<(n + 255) / 256, 256, 0, c->stream>>>(n, c->own.w, c->d_m, c->d_v, c->d_grad, c->d_mask, mzh::cos_schedule(t), c->bp1, c->bp2);
    } else {
        if (grad_mode == MZ_GRAD_REFERENCE_L2) { launch_scope ls(c, 4); mz_k_l2_grad<<<(n + 255) / 256, 256, 0, c->stream>>>(n, c->own.w, c->d_mask, grad_out(c)); }
        if (c->p2p) {    // data-parallel over peer memory: ONE kernel waits for the peers' gradients, sums them in rank order over NVLink and applies ADAM
            mz_dp_args d{}; d.rank = c->rank; d.nranks = c->nranks; d.step = ++c->dp_step; d.n = n; d.flags_local = c->d_xflags;
            for (int r = 0; r < c->nranks; r++) { d.peer_grad[r] = c->peer_grad[r] + (size_t)(d.step & 1u) * (size_t)n; d.peer_flags[r] = c->peer_flags[r]; }
            launch_scope ls(c, 4); mz_k_dp_adam<<<(n + 255) / 256, 256, 0, c->stream>>>(c->own.w, c->d_m, c->d_v, d, mzh::cos_schedule(t), c->bp1, c->bp2, 1.0f / (float)c->nranks);
        } else {
            float scale = 1.0f;
            if (c->comm) {   // data-parallel through NCCL: sum gradients over ranks, average in the update
                ncclResult_t r = g_nccl.AllReduce(c->d_grad, c->d_grad, (size_t)n, ncclFloat, ncclSum, c->comm, c->stream);
                if (r != ncclSuccess) return fail(c, MZ_E_NCCL, "ncclAllReduce: %s", g_nccl.GetErrorString(r));
                scale = 1.0f / (float)c->nranks;
            }
            launch_scope ls(c, 4); mz_k_adam<<<(n + 255) / 256, 256, 0, c->stream>>>(n, c->own.w, c->d_m, c->d_v, c->d_grad, mzh::cos_schedule(t), c->bp1, c->bp2, scale);
        }
    }
    MZ_CUDA(c, cudaGetLastError());
    c->bp1 *= 0.9; c->bp2 *= 0.999; c->adam_t++;
    c->own.version++;
    return MZ_OK;
}

// the fields of a search launch that do not depend on where its roots come from
static mz_search_args search_args(const mz_ctx *c, int n, int exploration) {
    mz_search_args a{}; a.pbc0 = c->d_pbc0; a.sqrtN = c->d_sqrtN; a.tree_pool = c->d_trees; a.n = n; a.max_dim = c->M.max_dim;
    a.max_layer_floats = c->M.max_layer_floats; a.exploration = exploration;
    return a;
}
// One search over the roots of `a` (MODE_API: the caller's a.n roots; MODE_SLOTS: the a.n game slots; MODE_REPLAY: a.n stored positions)
// in ONE launch of kernel family 0 (run_wave_body relabels those of an idle iteration), with the weights and images of store `ws` (NULL:
// the context's own networks).  lat > 0: the low-latency kernel (mz_kernels_lat.cuh) on roots [0, lat), one 2-CTA cluster each; otherwise
// the batched kernel of the context's networks.  MODE_REPLAY always takes the batched kernel: the latency kernel has no instantiation for it.
template <int MODE>
static void launch_search(mz_ctx *c, const mz_params &P, const mz_search_args &args, int lat, const mz_wstore *ws = nullptr) {
    const mz_wstore &s = ws ? *ws : c->own;
    mz_search_args a = args; a.wglob = s.w;
    const unsigned ctas = (unsigned)((a.n + MZ_ROWS - 1) / MZ_ROWS);
    launch_scope ls(c, 0);
    if constexpr (MODE != MZ_MODE_REPLAY) {
        if (lat > 0) {
            mz_lat_args t{}; t.base = a; t.image = s.lat; t.w_floats = c->lat_w_floats; t.pbc_smem = c->lat_pbc_smem;
            mz_k_search_lat<MODE><<<2 * lat, MZ_LAT_THREADS, c->smem_bytes_lat, c->stream>>>(P, t);
            return;
        }
    }
    if (c->cfg.net_type == MZ_NET_RESNET) {
        mz_search_rn_args t{}; t.base = a; t.image = s.rn; t.steps = c->d_rn_steps;
        const int nt = c->rn.R.ntrees;
        mz_k_search_rn<MODE><<<(a.n + nt - 1) / nt, MZ_RN_THREADS, c->smem_bytes_rn, c->stream>>>(P, c->rn.R, t);
    } else if (c->cfg.nn_mode == MZ_NN_SPLIT_MMA) {
        mz_search_sp_args t{}; t.base = a; t.sp = c->spa; t.sp.image = s.sp; t.sp.bias = s.sp_bias;
        mz_k_search_sp<MODE><<<ctas, MZ_SP_SEARCH_THREADS, c->smem_bytes_sp, c->stream>>>(P, t);
    } else if (c->cfg.nn_mode == MZ_NN_BF16_TC) {
        mz_search_tc_args t{}; t.base = a; t.w_image = s.tc; t.bias = s.tc_bias;
        mz_k_search_tc<MODE><<<ctas, MZ_THREADS, c->smem_bytes_tc, c->stream>>>(P, t);
    } else if (c->cfg.use_batch_norm) mz_k_search<MODE, true><<<ctas, MZ_THREADS, c->smem_bytes, c->stream>>>(P, a);
    else mz_k_search<MODE><<<ctas, MZ_THREADS, c->smem_bytes, c->stream>>>(P, a);
}

}  // namespace

extern "C" {

int mz_abi_version(void) { return MZ_ABI_VERSION; }
int mz_default_config(mz_config *cfg) { if (!cfg) return fail(nullptr, MZ_E_ARG, "cfg is NULL"); mzh::default_config(cfg); return MZ_OK; }
int mz_julia_dict_order(int A, int32_t *order) { if (A < 1 || A > MZ_MAX_A || !order) return fail(nullptr, MZ_E_ARG, "bad arguments"); mzh::julia_dict_order(A, order); return MZ_OK; }
const char *mz_last_error(mz_ctx *ctx) { return ctx ? ctx->err.c_str() : tl_error.c_str(); }

int mz_num_params(const mz_config *cfg, int net) {
    if (!cfg || net < 0 || net > 3) return fail(nullptr, MZ_E_ARG, "bad arguments");
    mzh::model M; if (const char *e = mzh::build_model(*cfg, M)) return fail(nullptr, MZ_E_ARG, "%s", e);
    if (cfg->net_type == MZ_NET_RESNET) {
        mzh::rn_model R; mzh::rn_units_build(*cfg, R);
        return net == MZ_NET_ALL ? mzh::rn_total_params(R) : R.n_params[net];
    }
    return mzh::net_params(M.P, net);
}

int mz_create(const mz_config *cfg, int device, mz_ctx **out) {
    if (!cfg || !out) return fail(nullptr, MZ_E_ARG, "cfg/out is NULL");
    *out = nullptr;
    mz_ctx *c = new mz_ctx();
    c->cfg = *cfg; c->device = device;
    if (const char *e = mzh::build_model(*cfg, c->M)) { int r = fail(nullptr, MZ_E_ARG, "%s", e); delete c; return r; }
    if (cfg->replay_buffer_size < cfg->num_slots) { int r = fail(nullptr, MZ_E_ARG, "replay_buffer_size must be >= num_slots"); delete c; return r; }
    if (cfg->nn_mode != MZ_NN_FP32_EXACT && cfg->nn_mode != MZ_NN_BF16_TC && cfg->nn_mode != MZ_NN_SPLIT_MMA) { int r = fail(nullptr, MZ_E_ARG, "unknown nn_mode %d", cfg->nn_mode); delete c; return r; }
    if (cfg->net_type == MZ_NET_FEEDFORWARD && cfg->nn_mode == MZ_NN_BF16_TC && !c->M.P.tc_ok) { int r = fail(nullptr, MZ_E_UNSUPPORTED, "MZ_NN_BF16_TC needs every layer to have in <= 64 and out <= 64"); delete c; return r; }
    if (cfg->nn_mode == MZ_NN_SPLIT_MMA && (cfg->net_type != MZ_NET_FEEDFORWARD || !c->M.P.tc_ok)) { int r = fail(nullptr, MZ_E_UNSUPPORTED, "MZ_NN_SPLIT_MMA needs the FeedForwardHP networks with every layer in <= 64 and out <= 64"); delete c; return r; }
    if (cfg->net_type == MZ_NET_FEEDFORWARD && cfg->use_batch_norm && cfg->nn_mode == MZ_NN_BF16_TC) { int r = fail(nullptr, MZ_E_UNSUPPORTED, "use_batch_norm runs on the exact fp32 path (MZ_NN_FP32_EXACT) and, folded into the weight image, on the split-precision path (MZ_NN_SPLIT_MMA); not in MZ_NN_BF16_TC"); delete c; return r; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { int r = fail(nullptr, MZ_E_CUDA, "no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e)); delete c; return r; }
#define MZ_CREATE(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { int r_ = fail(nullptr, MZ_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); mz_destroy(c); return r_; } } while (0)
    MZ_CREATE(cudaSetDevice(device));
    cudaDeviceProp prop; MZ_CREATE(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { int r = fail(nullptr, MZ_E_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); mz_destroy(c); return r; }
    c->sm_count = prop.multiProcessorCount;
    if (const char *rf = getenv("MUZERO_B200_REFILL")) c->refill_wave_sync = !strcmp(rf, "wave") ? 1 : 0;
    if (const char *pe = getenv("MUZERO_B200_PERSIST")) c->persist_ok = atoi(pe) != 0;
    const bool resnet = cfg->net_type == MZ_NET_RESNET;
    if (resnet) {
        if (const char *er = mzh::rn_build(*cfg, c->M.P, c->rn)) { int r = fail(nullptr, MZ_E_ARG, "%s", er); mz_destroy(c); return r; }
        c->M.P.tree_stride_bytes = c->rn.R.tree_stride_bytes; c->M.P.hidden_off_bytes = c->rn.R.hidden_off_bytes;
        c->M.P.n_params = mzh::rn_total_params(c->rn); c->M.P.total_floats = 4;
        c->smem_bytes_rn = mz_rn_smem_bytes(c->rn.R.slot_bytes, c->M.P.S, c->rn.R.ntrees, c->rn.R.n_steps - c->rn.R.smem_first);
        if (c->smem_bytes_rn + 1024 > (size_t)prop.sharedMemPerBlockOptin) { int r = fail(nullptr, MZ_E_UNSUPPORTED, "the ResNet search kernel needs %zu B of shared memory per CTA, device allows %zu", c->smem_bytes_rn, (size_t)prop.sharedMemPerBlockOptin); mz_destroy(c); return r; }
        MZ_CREATE(allow_max_smem(mz_k_search_rn<MZ_MODE_API>, prop)); MZ_CREATE(allow_max_smem(mz_k_search_rn<MZ_MODE_SLOTS>, prop)); MZ_CREATE(allow_max_smem(mz_k_rn_forward, prop));
        MZ_CREATE(allow_max_smem(mz_k_search_rn<MZ_MODE_REPLAY>, prop));
        MZ_CREATE(cudaMalloc((void **)&c->own.rn, (size_t)c->rn.image_bytes + 4096));
        MZ_CREATE(dmalloc(&c->d_rn_steps, c->rn.steps.size() + 1));
        MZ_CREATE(cudaMemcpy(c->d_rn_steps, c->rn.steps.data(), c->rn.steps.size() * sizeof(mz_rn_step), cudaMemcpyHostToDevice));
    }
    const mz_params &P = c->M.P;
    c->smem_bytes = resnet ? 0 : mz_smem_bytes(c->M.max_dim, c->M.max_layer_floats, P.hidden_pad, P.S);
    if (c->smem_bytes > (size_t)prop.sharedMemPerBlockOptin) { int r = fail(nullptr, MZ_E_UNSUPPORTED, "network needs %zu B of shared memory per CTA, device allows %zu", c->smem_bytes, (size_t)prop.sharedMemPerBlockOptin); mz_destroy(c); return r; }
    MZ_CREATE(allow_max_smem(mz_k_search<MZ_MODE_API>, prop));
    MZ_CREATE(allow_max_smem(mz_k_search<MZ_MODE_SLOTS>, prop));
    MZ_CREATE(allow_max_smem(mz_k_search<MZ_MODE_REPLAY>, prop));
    MZ_CREATE(allow_max_smem(mz_k_nn_forward<false>, prop));
    MZ_CREATE(allow_max_smem(mz_k_reanalyse<false>, prop));
    MZ_CREATE(allow_max_smem(mz_k_learn_forward<false>, prop));
    if (!resnet && cfg->use_batch_norm) {   // the same kernels instantiated with the BatchNorm epilogue
        MZ_CREATE(allow_max_smem(mz_k_search<MZ_MODE_API, true>, prop)); MZ_CREATE(allow_max_smem(mz_k_search<MZ_MODE_SLOTS, true>, prop));
        MZ_CREATE(allow_max_smem(mz_k_search<MZ_MODE_REPLAY, true>, prop));
        MZ_CREATE(allow_max_smem(mz_k_nn_forward<true>, prop)); MZ_CREATE(allow_max_smem(mz_k_reanalyse<true>, prop)); MZ_CREATE(allow_max_smem(mz_k_learn_forward<true>, prop));
    }
    if (!resnet) {   // the low-latency search kernel for few roots: does a network pair fit one SM's shared memory in fp32?
        int nf[3] = {0, 0, 0}; bool narrow = true;
        for (int n = 0; n < 3; n++) for (int l = P.nets[n].first; l < P.nets[n].first + P.nets[n].n_trunk + P.nets[n].n_h1 + P.nets[n].n_h2; l++) {
            nf[n] += mz_lat_layer_floats(P.layers[l].in, P.layers[l].out); if (P.layers[l].out > MZ_LAT_HALF) narrow = false;
            if (P.layers[l].in > MZ_LAT_KMAX && l != P.nets[n].first) narrow = false;   // only a network's first layer may be wider than 64 inputs
        }
        c->lat_image_floats = nf[0] + nf[1] + nf[2];
        c->lat_w_floats = nf[0] + nf[1] > nf[2] ? nf[0] + nf[1] : nf[2];
        c->lat_pbc_smem = 1;
        c->smem_bytes_lat = mz_lat_smem_bytes(c->lat_w_floats, c->M.max_dim, P.hidden_pad, P.tree_stride_bytes, P.S, 1);
        if (c->smem_bytes_lat + 1024 > (size_t)prop.sharedMemPerBlockOptin) { c->lat_pbc_smem = 0; c->smem_bytes_lat = mz_lat_smem_bytes(c->lat_w_floats, c->M.max_dim, P.hidden_pad, P.tree_stride_bytes, P.S, 0); }
        c->lat_ok = narrow && !cfg->use_batch_norm && P.A <= 16 && c->smem_bytes_lat + 1024 <= (size_t)prop.sharedMemPerBlockOptin && (size_t)c->lat_w_floats * 4 < (1u << 20);
        // run_mcts: two SMs per root.  Measured (profiles/r2j_run_mcts_latency.log): against the exact batched kernel it wins up to two rounds of
        // clusters, against the split-precision one up to one round
        c->lat_max_roots = cfg->nn_mode == MZ_NN_FP32_EXACT ? c->sm_count : c->sm_count / 2;
        c->lat_max_slots = 16;                                           // self-play: contexts built for one or a few games at a time (play_game)
        if (const char *el = getenv("MUZERO_B200_LAT")) c->lat_max_roots = c->lat_max_slots = atoi(el);   // measurement / test switch; 0 = off
        if (c->lat_ok) { MZ_CREATE(allow_max_smem(mz_k_search_lat<MZ_MODE_API>, prop)); MZ_CREATE(allow_max_smem(mz_k_search_lat<MZ_MODE_SLOTS>, prop)); MZ_CREATE(dmalloc(&c->own.lat, (size_t)c->lat_image_floats + 64)); }
    }
    if (!resnet) { if (const char *eb = mzh::build_bptt(P, c->bptt)) { int r = fail(nullptr, MZ_E_ARG, "%s", eb); mz_destroy(c); return r; } }
    bool bptt_fits = !resnet;
    if (!resnet) {
        // mz_k_learn_bptt's own carve-up (mz_bptt_carve): only in0 and group 0's staged-input slots are as wide as the observation stack.
        // The backward tile covers 64 outputs (bias sums: 4 warps x 16) and 64 inputs wherever an input gradient is needed, i.e. everywhere
        // except the representation's first layer (dx_mode = NONE)
        int narrow = 4, wf[2] = {0, 0};
        for (int n = 0; n < 3; n++) {
            const mz_net &N = P.nets[n];
            for (int i = 0; i < N.n_trunk + N.n_h1 + N.n_h2; i++) {
                const mz_layer &L = P.layers[N.first + i];
                if (L.out_pad > narrow) narrow = L.out_pad;
                if (!(n == 0 && i == 0) && L.in > narrow) narrow = L.in;
                if (L.floats > wf[n == 2]) wf[n == 2] = L.floats;
            }
        }
        narrow = (narrow + 3) & ~3;
        c->bptt_dims[0] = c->M.max_dim; c->bptt_dims[1] = narrow; c->bptt_dims[2] = wf[0]; c->bptt_dims[3] = wf[1];
        c->smem_bytes_bptt = mz_bptt_smem_bytes(c->M.max_dim, narrow, wf[0], wf[1], P.hidden_pad);
        bptt_fits = narrow <= 64 && c->smem_bytes_bptt + 4096 <= (size_t)prop.sharedMemPerBlockOptin;   // 4 KB head-room for the kernel's static shared memory
    }
    if (bptt_fits) {
        MZ_CREATE(allow_max_smem(mz_k_learn_bptt, prop));
        for (int g = 0; g < 2; g++) {
            MZ_CREATE(dmalloc(&c->d_bstages[g], c->bptt.stages[g].size() + 1));
            if (!c->bptt.stages[g].empty()) MZ_CREATE(cudaMemcpy(c->d_bstages[g], c->bptt.stages[g].data(), c->bptt.stages[g].size() * sizeof(mz_bstage), cudaMemcpyHostToDevice));
        }
    } else c->smem_bytes_bptt = 0;  // MZ_GRAD_BPTT reports MZ_E_UNSUPPORTED for this configuration
    if (c->M.P.tc_ok) {
        c->smem_bytes_tc = mz_tc_smem_bytes(P.tc_net_off[3], P.tc_bias_floats, P.hidden_pad, P.S);
        if (c->smem_bytes_tc <= (size_t)prop.sharedMemPerBlockOptin) {
            MZ_CREATE(allow_max_smem(mz_k_search_tc<MZ_MODE_API>, prop));
            MZ_CREATE(allow_max_smem(mz_k_search_tc<MZ_MODE_SLOTS>, prop));
            MZ_CREATE(allow_max_smem(mz_k_search_tc<MZ_MODE_REPLAY>, prop));
            MZ_CREATE(allow_max_smem(mz_k_nn_forward_tc, prop));
            MZ_CREATE(cudaMalloc((void **)&c->own.tc, (size_t)P.tc_net_off[3] + 8192));
            MZ_CREATE(cudaMemset(c->own.tc, 0, (size_t)P.tc_net_off[3] + 8192));
            MZ_CREATE(dmalloc(&c->own.tc_bias, (size_t)P.tc_bias_floats));
        } else if (cfg->nn_mode == MZ_NN_BF16_TC) {
            int r = fail(nullptr, MZ_E_UNSUPPORTED, "MZ_NN_BF16_TC needs %zu B of shared memory per CTA, device allows %zu", c->smem_bytes_tc, (size_t)prop.sharedMemPerBlockOptin);
            mz_destroy(c); return r;
        }
    }
    if (!resnet && P.tc_ok) {
        // rounds + weight sets for this device's shared memory (mz_host.h: build_sp_plan); the table of rounds lives in global memory
        mzh::build_sp_plan(P, (size_t)prop.sharedMemPerBlockOptin, c->spp);
        if (c->spp.ok) {
            const mz_sp_plan &S = c->spp;
            c->smem_bytes_sp = mz_sp_smem_bytes(S.warea_bytes, S.bias_floats, S.total_rounds, P.hidden_pad, P.S, S.pbc_smem);
            MZ_CREATE(allow_max_smem(mz_k_search_sp<MZ_MODE_API>, prop));
            MZ_CREATE(allow_max_smem(mz_k_search_sp<MZ_MODE_SLOTS>, prop));
            MZ_CREATE(allow_max_smem(mz_k_search_sp<MZ_MODE_REPLAY>, prop));
            MZ_CREATE(allow_max_smem(mz_k_nn_forward_sp, prop));
            MZ_CREATE(allow_max_smem(mz_k_learn_forward_sp, prop));
            MZ_CREATE(cudaMalloc((void **)&c->own.sp, (size_t)S.image_bytes + 256));
            MZ_CREATE(cudaMemset(c->own.sp, 0, (size_t)S.image_bytes + 256));
            MZ_CREATE(dmalloc(&c->own.sp_bias, (size_t)S.bias_floats));
            MZ_CREATE(cudaMalloc((void **)&c->d_rounds_sp, sizeof(mz_sp_round) * MZ_SP_MAX_ROUNDS));
            MZ_CREATE(cudaMemcpy(c->d_rounds_sp, S.round, sizeof(mz_sp_round) * MZ_SP_MAX_ROUNDS, cudaMemcpyHostToDevice));
            mz_sp_args &A = c->spa;
            A.image = c->own.sp; A.bias = c->own.sp_bias; A.rounds = c->d_rounds_sp;
            for (int n = 0; n < 3; n++) { A.first[n] = S.first[n]; A.n_rounds[n] = S.n_rounds[n]; A.set_first[n] = S.set_first[n]; A.n_sets[n] = S.n_sets[n]; }
            A.total_rounds = S.total_rounds; A.total_sets = S.total_sets; A.warea_bytes = S.warea_bytes; A.bias_floats = S.bias_floats; A.pbc_smem = S.pbc_smem; A.tail = S.tail;
            // the learner's backward rounds on the same machinery
            mzh::build_lr_plan(P, S, c->lrp);
            c->smem_bytes_lr = mz_lr_smem_bytes(S.warea_bytes, S.bias_floats, S.total_rounds, c->lrp.btotal_rounds, P.hidden_pad);
            if (c->lrp.ok && (c->smem_bytes_lr + 64 > (size_t)prop.sharedMemPerBlockOptin ||
                              ((c->lrp.bwarea_bytes + 127) & ~127) + c->lrp.n_eval * MZ_LR_LG_ROWS * MZ_ROWS * 4 > S.warea_bytes || P.A > 16)) c->lrp.ok = 0;
            if (c->lrp.ok) {
                MZ_CREATE(allow_max_smem(mz_k_learn_bptt_tc, prop));
                MZ_CREATE(allow_max_smem(mz_k_learn_dw, prop));
                MZ_CREATE(cudaMalloc((void **)&c->d_brounds, sizeof(mz_lr_bround) * MZ_LR_MAX_ROUNDS));
                MZ_CREATE(cudaMemcpy(c->d_brounds, c->lrp.bround, sizeof(mz_lr_bround) * MZ_LR_MAX_ROUNDS, cudaMemcpyHostToDevice));
            }
        } else if (cfg->nn_mode == MZ_NN_SPLIT_MMA) {
            int r = fail(nullptr, MZ_E_UNSUPPORTED, "MZ_NN_SPLIT_MMA: the networks do not fit the shared memory of this device (%zu B per CTA)", (size_t)prop.sharedMemPerBlockOptin);
            mz_destroy(c); return r;
        }
    }
    MZ_CREATE(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true;
    MZ_CREATE(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) MZ_CREATE(cudaEventCreateWithFlags(&c->ev_search[i], cudaEventDisableTiming));
    c->packed = !resnet;
    c->store_floats = resnet ? P.n_params : P.total_floats;
    const size_t nf = (size_t)c->store_floats;
    MZ_CREATE(dmalloc(&c->own.w, nf)); MZ_CREATE(dmalloc(&c->d_m, nf)); MZ_CREATE(dmalloc(&c->d_v, nf)); MZ_CREATE(dmalloc(&c->d_grad, nf));
    MZ_CREATE(cudaMemset(c->own.w, 0, nf * 4)); MZ_CREATE(cudaMemset(c->d_m, 0, nf * 4)); MZ_CREATE(cudaMemset(c->d_v, 0, nf * 4));
    if (resnet || cfg->use_batch_norm) {   // Flux.params of a BatchNorm are beta and gamma: the running statistics take no part in sum(abs2, theta), its gradient or ADAM
        std::vector<unsigned char> mask(nf + 16, 1);
        if (resnet) {
            for (int n = 0; n < 3; n++) for (const mzh::rn_unit &u : c->rn.units[n]) if (u.kind == 0) for (int i = 0; i < u.cout; i++) { mask[(size_t)u.mu_off + i] = 0; mask[(size_t)u.var_off + i] = 0; }
        } else {
            for (int i = 0; i < P.n_layers; i++) if (P.layers[i].bn) for (int o = 0; o < 2 * P.layers[i].out_pad; o++) mask[(size_t)P.layers[i].b_off + 3 * P.layers[i].out_pad + o] = 0;
        }
        MZ_CREATE(cudaMalloc((void **)&c->d_mask, nf + 16)); MZ_CREATE(cudaMemcpy(c->d_mask, mask.data(), nf + 16, cudaMemcpyHostToDevice));
        for (int n = 0; n < 3; n++) c->net_bounds[n] = resnet ? c->rn.base[n] : P.layers[P.nets[n].first].w_off;
        c->net_bounds[3] = (int)nf;
    }
    MZ_CREATE(dmalloc(&c->d_pbc0, c->M.pbc0.size())); MZ_CREATE(dmalloc(&c->d_sqrtN, c->M.sqrtN.size()));
    MZ_CREATE(cudaMemcpy(c->d_pbc0, c->M.pbc0.data(), c->M.pbc0.size() * 8, cudaMemcpyHostToDevice));
    MZ_CREATE(cudaMemcpy(c->d_sqrtN, c->M.sqrtN.data(), c->M.sqrtN.size() * 8, cudaMemcpyHostToDevice));
    const size_t G = (size_t)cfg->num_slots, Tm = (size_t)P.Tmax, R = (size_t)cfg->replay_buffer_size;
    MZ_CREATE(cudaMalloc(&c->d_trees, G * (size_t)P.tree_stride_bytes));
    mz_slots &s = c->slots;
    MZ_CREATE(dmalloc(&s.p1, G)); MZ_CREATE(dmalloc(&s.p2, G)); MZ_CREATE(dmalloc(&s.player, G)); MZ_CREATE(dmalloc(&s.T, G));
    MZ_CREATE(dmalloc(&s.status, G)); MZ_CREATE(dmalloc(&s.game_id, G));
    MZ_CREATE(dmalloc(&s.fin_list, G + 6));
    MZ_CREATE(dmalloc(&s.h_p1, G * Tm)); MZ_CREATE(dmalloc(&s.h_p2, G * Tm)); MZ_CREATE(dmalloc(&s.h_action, G * Tm));
    MZ_CREATE(dmalloc(&s.h_reward, G * Tm)); MZ_CREATE(dmalloc(&s.h_to_play, G * Tm)); MZ_CREATE(dmalloc(&s.h_cv, G * Tm * P.A)); MZ_CREATE(dmalloc(&s.h_rv, G * Tm));
    MZ_CREATE(cudaMemset(s.status, 0, G * sizeof(int32_t)));
    MZ_CREATE(cudaMemset(s.h_p1, 0, G * Tm * sizeof(uint64_t))); MZ_CREATE(cudaMemset(s.h_p2, 0, G * Tm * sizeof(uint64_t)));   // the board before move 0 is empty
    if (const int rr = alloc_ring(c, c->ring, R)) { mz_destroy(c); return rr; }
    MZ_CREATE(dmalloc(&c->d_stats, 64)); MZ_CREATE(cudaMemset(c->d_stats, 0, 64 * sizeof(unsigned long long)));
    MZ_CREATE(dmalloc(&c->d_lossout, 8));
    MZ_CREATE(cudaMallocHost((void **)&c->h_counters, 8 * sizeof(int64_t)));
    MZ_CREATE(cudaHostAlloc((void **)&c->h_wave, 16 * sizeof(int64_t), cudaHostAllocMapped));   // mz_k_save_refill writes its counter snapshot straight into it
    MZ_CREATE(cudaHostGetDevicePointer((void **)&c->d_wave, c->h_wave, 0));
    for (int i = 0; i < 2; i++) MZ_CREATE(cudaEventCreateWithFlags(&c->ev_wave[i], cudaEventDisableTiming));
    MZ_CREATE(cudaMallocHost((void **)&c->h_lossout, 8 * sizeof(double)));
    MZ_CREATE(cudaMallocHost((void **)&c->h_stats, 64 * sizeof(unsigned long long)));
    MZ_CREATE(cudaDeviceSynchronize());
#undef MZ_CREATE
    *out = c;
    return MZ_OK;
}

int mz_destroy(mz_ctx *c) {
    if (!c) return MZ_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    collect_timings(c);
    if (c->comm && g_nccl.CommDestroy) { p2p_teardown(c); g_nccl.CommDestroy(c->comm); }
    void *ptrs[] = {c->opp.w, c->opp.tc, c->opp.tc_bias, c->opp.sp, c->opp.sp_bias, c->opp.lat, c->opp.rn, c->d_mask, c->d_w_fold, c->own.lat, c->d_brounds, c->own.sp, c->own.sp_bias, c->d_rounds_sp, c->own.rn, c->d_rn_steps, c->d_bstages[0], c->d_bstages[1], c->own.tc, c->own.tc_bias, c->own.w, c->d_m, c->d_v, c->d_grad, c->d_pbc0, c->d_sqrtN, c->d_trees, c->slots.p1, c->slots.p2, c->slots.player, c->slots.T,
                    c->slots.status, c->slots.game_id, c->slots.fin_list, c->slots.h_p1, c->slots.h_p2, c->slots.h_action, c->slots.h_reward, c->slots.h_to_play,
                    c->slots.h_cv, c->slots.h_rv, c->d_stats, c->d_lossout, c->batch.index, c->batch.obs,
                    c->batch.actions, c->batch.values, c->batch.rewards, c->batch.policies, c->batch.gscale, c->batch.weights, c->d_pv, c->d_pr, c->d_pp,
                    c->d_rowv, c->d_rowp, c->d_rowinvg, c->d_rowr};
    for (void *p : ptrs) if (p) cudaFree(p);
    for (auto &b : c->scratch) b.release();
    for (auto &b : c->rn_buf) b.release();
    for (dev_buf *b : {&c->bptt_act, &c->bptt_gpart, &c->lr_xsave, &c->lr_dzsave, &c->lr_gpart}) b->release();
    free_ring(c->ring);
    free_ring(c->play_ring);
    if (c->h_lat_stage) cudaFreeHost(c->h_lat_stage);
    if (c->d_lat_stage) cudaFree(c->d_lat_stage);
    if (c->h_counters) cudaFreeHost(c->h_counters);
    if (c->h_wave) cudaFreeHost(c->h_wave);
    for (int i = 0; i < 2; i++) if (c->ev_wave[i]) cudaEventDestroy(c->ev_wave[i]);
    if (c->h_lossout) cudaFreeHost(c->h_lossout);
    if (c->h_stats) cudaFreeHost(c->h_stats);
    if (c->stream2) { cudaStreamSynchronize(c->stream2); cudaStreamDestroy(c->stream2); }
    for (int i = 0; i < 2; i++) if (c->ev_search[i]) cudaEventDestroy(c->ev_search[i]);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return MZ_OK;
}

int mz_set_stream(mz_ctx *c, void *cuda_stream) {
    MZ_CHECK_CTX(c);
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->own_stream) { cudaStreamDestroy(c->stream); c->own_stream = false; }
    c->stream = (cudaStream_t)cuda_stream;
    return MZ_OK;
}
int mz_synchronize(mz_ctx *c) { MZ_CHECK_CTX(c); MZ_CUDA(c, cudaStreamSynchronize(c->stream)); return MZ_OK; }
int mz_device_info(mz_ctx *c, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor, int64_t *free_bytes) {
    MZ_CHECK_CTX(c);
    cudaDeviceProp prop; MZ_CUDA(c, cudaGetDeviceProperties(&prop, c->device));
    size_t fr = 0, tot = 0; MZ_CUDA(c, cudaMemGetInfo(&fr, &tot));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (free_bytes) *free_bytes = (int64_t)fr;
    return MZ_OK;
}

// ---- weights ----------------------------------------------------------------------------------------
int mz_init_weights(mz_ctx *c, uint64_t seed) {
    MZ_CHECK_CTX(c);
    std::vector<float> src((size_t)c->M.P.n_params);
    if (c->cfg.net_type == MZ_NET_RESNET) mzh::rn_init_weights(c->rn, seed, src.data());
    else mzh::init_weights(c->M.P, seed, src.data());
    return upload_weights(c, src);
}
int mz_set_weights(mz_ctx *c, int net, const float *blob, int64_t n) {
    MZ_CHECK_CTX(c);
    if (net < 0 || net > 3 || !blob) return fail(c, MZ_E_ARG, "bad net id or NULL blob");
    if (n != ctx_net_params(c, net)) return fail(c, MZ_E_ARG, "weight blob has %lld floats, net %d needs %d", (long long)n, net, ctx_net_params(c, net));
    std::vector<float> src;
    if (net == MZ_NET_ALL) src.assign(blob, blob + n);                    // whole model: nothing to merge with
    else { MZ_TRY(download_weights(c, src)); memcpy(src.data() + ctx_net_offset(c, net), blob, (size_t)n * sizeof(float)); }
    return upload_weights(c, src);
}
// the opponent store, with the images of the context's path only; on failure nothing is left half-allocated
static int alloc_opponent(mz_ctx *c) {
    if (c->opp.w) return MZ_OK;
    const mz_params &P = c->M.P;
    mz_wstore s;
    cudaError_t e = dmalloc(&s.w, (size_t)c->store_floats);
    if (e == cudaSuccess && c->cfg.nn_mode == MZ_NN_SPLIT_MMA && c->own.sp) {
        e = cudaMalloc((void **)&s.sp, (size_t)c->spp.image_bytes + 256);
        if (e == cudaSuccess) e = cudaMemsetAsync(s.sp, 0, (size_t)c->spp.image_bytes + 256, c->stream);
        if (e == cudaSuccess) e = dmalloc(&s.sp_bias, (size_t)c->spp.bias_floats);
    }
    if (e == cudaSuccess && c->cfg.nn_mode == MZ_NN_BF16_TC && c->own.tc) {
        e = cudaMalloc((void **)&s.tc, (size_t)P.tc_net_off[3] + 8192);
        if (e == cudaSuccess) e = cudaMemsetAsync(s.tc, 0, (size_t)P.tc_net_off[3] + 8192, c->stream);
        if (e == cudaSuccess) e = dmalloc(&s.tc_bias, (size_t)P.tc_bias_floats);
    }
    if (e == cudaSuccess && c->own.lat) e = dmalloc(&s.lat, (size_t)c->lat_image_floats + 64);
    if (e == cudaSuccess && c->own.rn) e = cudaMalloc((void **)&s.rn, (size_t)c->rn.image_bytes + 4096);
    if (e != cudaSuccess) {
        for (void *p : {(void *)s.w, (void *)s.sp, (void *)s.sp_bias, (void *)s.tc, (void *)s.tc_bias, (void *)s.lat, (void *)s.rn}) if (p) cudaFree(p);
        return fail(c, MZ_E_CUDA, "allocating the opponent networks: %s", cudaGetErrorString(e));
    }
    c->opp = s;
    return MZ_OK;
}
int mz_set_opponent_weights(mz_ctx *c, int net, const float *blob, int64_t n) {
    MZ_CHECK_CTX(c);
    if (net < 0 || net > 3 || !blob) return fail(c, MZ_E_ARG, "bad net id or NULL blob");
    if (n != ctx_net_params(c, net)) return fail(c, MZ_E_ARG, "weight blob has %lld floats, net %d needs %d", (long long)n, net, ctx_net_params(c, net));
    if (net != MZ_NET_ALL && !c->opp_full)
        return fail(c, MZ_E_STATE, "replacing one opponent network needs a full opponent set first (mz_set_opponent_weights with MZ_NET_ALL, or mz_snapshot_opponent)");
    MZ_TRY(alloc_opponent(c));
    std::vector<float> src((size_t)c->M.P.n_params);
    if (net == MZ_NET_ALL) memcpy(src.data(), blob, (size_t)n * sizeof(float));
    else { MZ_TRY(store_to_host(c, c->opp.w, src.data())); memcpy(src.data() + ctx_net_offset(c, net), blob, (size_t)n * sizeof(float)); }
    MZ_TRY(store_from_host(c, c->opp.w, src.data()));
    c->opp.version++;
    c->opp_full = true;
    return MZ_OK;
}
int mz_snapshot_opponent(mz_ctx *c) {
    MZ_CHECK_CTX(c);
    MZ_TRY(alloc_opponent(c));
    MZ_CUDA(c, cudaMemcpyAsync(c->opp.w, c->own.w, (size_t)c->store_floats * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
    c->opp.version++;
    c->opp_full = true;
    return MZ_OK;
}
int mz_get_weights(mz_ctx *c, int net, float *blob, int64_t n) {
    MZ_CHECK_CTX(c);
    if (net < 0 || net > 3 || !blob) return fail(c, MZ_E_ARG, "bad net id or NULL blob");
    if (n != ctx_net_params(c, net)) return fail(c, MZ_E_ARG, "weight blob has %lld floats, net %d needs %d", (long long)n, net, ctx_net_params(c, net));
    std::vector<float> src;
    MZ_TRY(download_weights(c, src));
    memcpy(blob, src.data() + ctx_net_offset(c, net), (size_t)n * sizeof(float));
    return MZ_OK;
}

// ---- batched network callables -------------------------------------------------------------------------
static int nn_forward(mz_ctx *c, int net, int B, const float *in, float *out1, size_t n1, float *out2, size_t n2) {
    MZ_CHECK_CTX(c);
    if (B < 0 || (B > 0 && (!in || !out1))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (B == 0) return MZ_OK;
    MZ_TRY(ensure_images(c));
    const mz_params &P = c->M.P;
    const bool resnet = c->cfg.net_type == MZ_NET_RESNET;
    const int in_dim = resnet ? (net == 0 ? P.stack_size : net == 1 ? P.hidden : P.sa_size) : P.layers[P.nets[net].first].in;
    float *d_in, *d_o1, *d_o2;
    MZ_TRY(h2d(c, c->scratch[0], in, (size_t)B * in_dim, &d_in));
    MZ_TRY(h2d<float>(c, c->scratch[1], nullptr, (size_t)B * n1, &d_o1));
    MZ_TRY(h2d<float>(c, c->scratch[2], nullptr, (size_t)B * (n2 ? n2 : 1), &d_o2));
    mz_nn_args a{}; a.wglob = c->own.w; a.B = B; a.max_dim = c->M.max_dim; a.max_layer_floats = c->M.max_layer_floats; a.net = net; a.in = d_in; a.out1 = d_o1; a.out2 = d_o2;
    if (resnet) {
        unsigned char *d_pool;
        MZ_TRY(h2d<unsigned char>(c, c->scratch[3], nullptr, (size_t)B * c->rn.R.node_bytes, &d_pool));
        mz_search_rn_args t{}; t.image = c->own.rn; t.steps = c->d_rn_steps; t.net = net; t.B = B; t.in = d_in; t.out1 = d_o1; t.out2 = d_o2; t.scratch_pool = d_pool;
        const int nt = c->rn.R.ntrees;
        launch_scope ls(c, 5); mz_k_rn_forward<<<(B + nt - 1) / nt, MZ_RN_THREADS, c->smem_bytes_rn, c->stream>>>(P, c->rn.R, t);
    } else if (c->cfg.nn_mode == MZ_NN_SPLIT_MMA) {
        mz_nn_sp_args t{}; t.sp = c->spa; t.B = B; t.net = net; t.in = d_in; t.out1 = d_o1; t.out2 = d_o2;
        launch_scope ls(c, 5); mz_k_nn_forward_sp<<<(B + MZ_ROWS - 1) / MZ_ROWS, MZ_SP_THREADS, c->smem_bytes_sp, c->stream>>>(P, t);
    } else if (c->cfg.nn_mode == MZ_NN_BF16_TC) {
        mz_nn_tc_args t{}; t.w_image = c->own.tc; t.bias = c->own.tc_bias; t.B = B; t.net = net; t.in = d_in; t.out1 = d_o1; t.out2 = d_o2;
        launch_scope ls(c, 5); mz_k_nn_forward_tc<<<(B + MZ_ROWS - 1) / MZ_ROWS, MZ_THREADS, c->smem_bytes_tc, c->stream>>>(P, t);
    } else if (c->cfg.use_batch_norm) { launch_scope ls(c, 5); mz_k_nn_forward<true><<<(B + MZ_ROWS - 1) / MZ_ROWS, MZ_THREADS, c->smem_bytes, c->stream>>>(P, a); }
    else { launch_scope ls(c, 5); mz_k_nn_forward<false><<<(B + MZ_ROWS - 1) / MZ_ROWS, MZ_THREADS, c->smem_bytes, c->stream>>>(P, a); }
    MZ_CUDA(c, cudaGetLastError());
    MZ_TRY(d2h(c, out1, d_o1, (size_t)B * n1));
    if (n2 && out2) MZ_TRY(d2h(c, out2, d_o2, (size_t)B * n2));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
int mz_representation(mz_ctx *c, int B, const float *stacked_obs, float *hidden) {
    if (!c) return fail(nullptr, MZ_E_ARG, "ctx is NULL");
    return nn_forward(c, 0, B, stacked_obs, hidden, (size_t)c->M.P.hidden, nullptr, 0);
}
int mz_prediction(mz_ctx *c, int B, const float *hidden, float *value, float *policy) {
    if (!c) return fail(nullptr, MZ_E_ARG, "ctx is NULL");
    if (B > 0 && !policy) return fail(c, MZ_E_ARG, "NULL buffer");
    return nn_forward(c, 1, B, hidden, value, 1, policy, (size_t)c->M.P.A);
}
int mz_dynamics(mz_ctx *c, int B, const float *state_action, float *next_hidden, float *reward) {
    if (!c) return fail(nullptr, MZ_E_ARG, "ctx is NULL");
    if (B > 0 && !reward) return fail(c, MZ_E_ARG, "NULL buffer");
    return nn_forward(c, 2, B, state_action, next_hidden, (size_t)c->M.P.hidden, reward, 1);
}

// ---- environment -----------------------------------------------------------------------------------------
int mz_env_reset(mz_ctx *c, int n, uint64_t *p1, uint64_t *p2, int32_t *player) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!p1 || !p2 || !player))) return fail(c, MZ_E_ARG, "NULL buffer");
    for (int i = 0; i < n; i++) { p1[i] = 0; p2[i] = 0; player[i] = 1; }   // reset! (game.jl:15-20): a constant fill, no kernel needed
    return MZ_OK;
}
static int env_call(mz_ctx *c, int n, uint64_t *p1, uint64_t *p2, int32_t *player, const int32_t *action, float *reward, int32_t *done, uint32_t *legal, bool writeback) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!p1 || !p2 || !player))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    const mz_params &P = c->M.P;
    if (action) for (int i = 0; i < n; i++) if (action[i] < 1 || action[i] > P.A) return fail(c, MZ_E_ARG, "action %d out of range at %d", action[i], i);
    uint64_t *d1, *d2; int32_t *dp, *da = nullptr, *dd; float *dr; uint32_t *dl;
    MZ_TRY(h2d(c, c->scratch[0], p1, (size_t)n, &d1)); MZ_TRY(h2d(c, c->scratch[1], p2, (size_t)n, &d2)); MZ_TRY(h2d(c, c->scratch[2], player, (size_t)n, &dp));
    if (action) MZ_TRY(h2d(c, c->scratch[3], action, (size_t)n, &da));
    MZ_TRY(h2d<float>(c, c->scratch[4], nullptr, (size_t)n, &dr)); MZ_TRY(h2d<int32_t>(c, c->scratch[5], nullptr, (size_t)n, &dd)); MZ_TRY(h2d<uint32_t>(c, c->scratch[6], nullptr, (size_t)n, &dl));
    { launch_scope ls(c, 6); mz_k_env_step<<<(n + 255) / 256, 256, 0, c->stream>>>(P, n, d1, d2, dp, da, dr, dd, dl); }
    MZ_CUDA(c, cudaGetLastError());
    if (writeback) { MZ_TRY(d2h(c, p1, d1, (size_t)n)); MZ_TRY(d2h(c, p2, d2, (size_t)n)); MZ_TRY(d2h(c, player, dp, (size_t)n)); }
    MZ_TRY(d2h(c, reward, dr, (size_t)n)); MZ_TRY(d2h(c, done, dd, (size_t)n)); MZ_TRY(d2h(c, legal, dl, (size_t)n));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
int mz_env_step(mz_ctx *c, int n, uint64_t *p1, uint64_t *p2, int32_t *player, const int32_t *action, float *reward, int32_t *done, uint32_t *legal_mask) {
    if (!c) return fail(nullptr, MZ_E_ARG, "ctx is NULL");
    if (n > 0 && !action) return fail(c, MZ_E_ARG, "NULL action buffer");
    return env_call(c, n, p1, p2, player, action, reward, done, legal_mask, true);
}
int mz_env_legal(mz_ctx *c, int n, const uint64_t *p1, const uint64_t *p2, const int32_t *player, uint32_t *legal_mask) {
    if (!c) return fail(nullptr, MZ_E_ARG, "ctx is NULL");
    return env_call(c, n, (uint64_t *)p1, (uint64_t *)p2, (int32_t *)player, nullptr, nullptr, nullptr, legal_mask, false);
}
int mz_env_observation(mz_ctx *c, int n, const uint64_t *p1, const uint64_t *p2, float *obs) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!p1 || !p2 || !obs))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    const mz_params &P = c->M.P;
    uint64_t *d1, *d2; float *dobs;
    MZ_TRY(h2d(c, c->scratch[0], p1, (size_t)n, &d1)); MZ_TRY(h2d(c, c->scratch[1], p2, (size_t)n, &d2));
    MZ_TRY(h2d<float>(c, c->scratch[2], nullptr, (size_t)n * P.obs_size, &dobs));
    size_t tot = (size_t)n * P.obs_size;
    { launch_scope ls(c, 6); mz_k_env_obs<<<(unsigned)((tot + 255) / 256), 256, 0, c->stream>>>(P, n, d1, d2, dobs); }
    MZ_CUDA(c, cudaGetLastError());
    MZ_TRY(d2h(c, obs, dobs, tot));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}

// ---- MCTS ------------------------------------------------------------------------------------------------
int mz_run_mcts(mz_ctx *c, int n, const float *stacked_obs, const uint32_t *legal_mask, const int32_t *to_play, int exploration,
                const uint64_t *game_id, const int32_t *move_idx, int32_t *visit_counts, float *root_value, float *root_priors) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!stacked_obs || !legal_mask || !to_play || !game_id || !move_idx || !visit_counts || !root_value))) return fail(c, MZ_E_ARG, "NULL buffer");
    const mz_params &P = c->M.P;
    for (int i = 0; i < n; i++) {
        if (legal_mask[i] == 0 || (legal_mask[i] >> P.A) != 0) return fail(c, MZ_E_ARG, "legal actions of root %d must be a non-empty subset of the action space (SelfPlay.jl:243-244)", i);
        if (to_play[i] < 1 || to_play[i] > P.P) return fail(c, MZ_E_ARG, "to_play of root %d out of range", i);   // the search itself does not read it
    }
    if (c->lat_ok && n > 0 && n <= c->lat_max_roots && c->cfg.nn_mode != MZ_NN_BF16_TC) {
        // few roots: one tree per cluster in exact fp32 (mz_kernels_lat.cuh); every input in ONE pinned block and one copy each way -- at
        // this size the call's latency is what the caller sees (the reference calls run_mcts with one root at a time).  No game can be in
        // flight here: a wave ends with every slot idle or resets the slots.
        MZ_TRY(ensure_lat_image(c, c->own));
        auto al = [](size_t x) { return (x + 15) & ~(size_t)15; };
        const size_t o_st = 0, o_legal = al(o_st + (size_t)n * P.stack_size * 4), o_gid = al(o_legal + (size_t)n * 4), o_mv = al(o_gid + (size_t)n * 8),
                     o_vc = al(o_mv + (size_t)n * 4), o_rv = al(o_vc + (size_t)n * P.A * 4), o_pri = al(o_rv + (size_t)n * 4), total = al(o_pri + (size_t)n * P.A * 4);
        if (total > c->lat_stage_cap) {
            if (c->h_lat_stage) cudaFreeHost(c->h_lat_stage);
            if (c->d_lat_stage) cudaFree(c->d_lat_stage);
            c->h_lat_stage = nullptr; c->d_lat_stage = nullptr; c->lat_stage_cap = 0;
            const size_t want = (total + 65535) & ~(size_t)65535;
            MZ_CUDA(c, cudaMallocHost((void **)&c->h_lat_stage, want)); MZ_CUDA(c, cudaMalloc((void **)&c->d_lat_stage, want));
            c->lat_stage_cap = want;
        }
        unsigned char *h = c->h_lat_stage, *d = c->d_lat_stage;
        memcpy(h + o_st, stacked_obs, (size_t)n * P.stack_size * 4); memcpy(h + o_legal, legal_mask, (size_t)n * 4);
        memcpy(h + o_gid, game_id, (size_t)n * 8); memcpy(h + o_mv, move_idx, (size_t)n * 4);
        MZ_CUDA(c, cudaMemcpyAsync(d, h, o_vc, cudaMemcpyHostToDevice, c->stream));
        mz_search_args a = search_args(c, n, exploration);
        a.stacked = (const float *)(d + o_st); a.legal = (const uint32_t *)(d + o_legal); a.game_id = (const uint64_t *)(d + o_gid); a.move_idx = (const int32_t *)(d + o_mv);
        a.visit_counts = (int32_t *)(d + o_vc); a.root_value = (float *)(d + o_rv); a.root_priors = (float *)(d + o_pri);
        launch_search<MZ_MODE_API>(c, P, a, n);
        MZ_CUDA(c, cudaGetLastError());
        MZ_CUDA(c, cudaMemcpyAsync(h + o_vc, d + o_vc, total - o_vc, cudaMemcpyDeviceToHost, c->stream));
        MZ_CUDA(c, cudaStreamSynchronize(c->stream));
        memcpy(visit_counts, h + o_vc, (size_t)n * P.A * 4); memcpy(root_value, h + o_rv, (size_t)n * 4);
        if (root_priors) memcpy(root_priors, h + o_pri, (size_t)n * P.A * 4);
        return MZ_OK;
    }
    read_counters(c);
    if (c->h_counters[5] != 0) return fail(c, MZ_E_STATE, "self-play in progress");
    const int cap = c->cfg.num_slots;
    MZ_TRY(ensure_images(c));
    for (int off = 0; off < n; off += cap) {
        int m = n - off < cap ? n - off : cap;
        float *d_st, *d_rv, *d_pri; uint32_t *d_legal; int32_t *d_mv, *d_vc; uint64_t *d_gid;
        MZ_TRY(h2d(c, c->scratch[0], stacked_obs + (size_t)off * P.stack_size, (size_t)m * P.stack_size, &d_st));
        MZ_TRY(h2d(c, c->scratch[1], legal_mask + off, (size_t)m, &d_legal));
        MZ_TRY(h2d(c, c->scratch[3], game_id + off, (size_t)m, &d_gid)); MZ_TRY(h2d(c, c->scratch[4], move_idx + off, (size_t)m, &d_mv));
        MZ_TRY(h2d<int32_t>(c, c->scratch[5], nullptr, (size_t)m * P.A, &d_vc)); MZ_TRY(h2d<float>(c, c->scratch[6], nullptr, (size_t)m, &d_rv));
        MZ_TRY(h2d<float>(c, c->scratch[7], nullptr, (size_t)m * P.A, &d_pri));
        mz_search_args a = search_args(c, m, exploration);
        a.stacked = d_st; a.legal = d_legal; a.game_id = d_gid; a.move_idx = d_mv; a.visit_counts = d_vc; a.root_value = d_rv; a.root_priors = d_pri;
        launch_search<MZ_MODE_API>(c, P, a, 0);
        MZ_CUDA(c, cudaGetLastError());
        MZ_TRY(d2h(c, visit_counts + (size_t)off * P.A, d_vc, (size_t)m * P.A)); MZ_TRY(d2h(c, root_value + off, d_rv, (size_t)m));
        if (root_priors) MZ_TRY(d2h(c, root_priors + (size_t)off * P.A, d_pri, (size_t)m * P.A));
        MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return MZ_OK;
}

int mz_select_action(mz_ctx *c, int n, const int32_t *visit_counts, const uint32_t *legal_mask, float temperature, const uint64_t *game_id,
                     const int32_t *move_idx, int32_t *action) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!visit_counts || !legal_mask || !game_id || !move_idx || !action))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    const mz_params &P = c->M.P;
    int32_t *d_vc, *d_mv, *d_act; uint32_t *d_legal; uint64_t *d_gid;
    MZ_TRY(h2d(c, c->scratch[0], visit_counts, (size_t)n * P.A, &d_vc)); MZ_TRY(h2d(c, c->scratch[1], legal_mask, (size_t)n, &d_legal));
    MZ_TRY(h2d(c, c->scratch[2], game_id, (size_t)n, &d_gid)); MZ_TRY(h2d(c, c->scratch[3], move_idx, (size_t)n, &d_mv));
    MZ_TRY(h2d<int32_t>(c, c->scratch[4], nullptr, (size_t)n, &d_act));
    { launch_scope ls(c, 6); mz_k_select_action<<<(n + 127) / 128, 128, 0, c->stream>>>(P, n, d_vc, d_legal, temperature, d_gid, d_mv, d_act); }
    MZ_CUDA(c, cudaGetLastError());
    MZ_TRY(d2h(c, action, d_act, (size_t)n));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}

// ---- self-play ---------------------------------------------------------------------------------------------
// save_game + refill: number the finished games and hand out new ones (one CTA, ordered), copy their histories (many CTAs), priorities
static int launch_save_refill(mz_ctx *c, const mz_params &P, int G, unsigned long long *tally, int64_t *snap = nullptr, cudaStream_t st = nullptr) {
    if (!st) st = c->stream;
    { launch_scope ls(c, 1, st); mz_k_save_refill<<<1, 1024, 0, st>>>(P, c->slots, c->ring, G, tally, c->refill_wave_sync, snap); }
    { launch_scope ls(c, 1, st); mz_k_save_copy<<<c->sm_count, 256, 0, st>>>(P, c->slots, c->ring, G); }
    if (P.per) { launch_scope ls(c, 1, st); mz_k_save_per<<<(G + 255) / 256 < c->sm_count ? (G + 255) / 256 : c->sm_count, 256, 0, st>>>(P, c->slots, c->ring, G); }
    return MZ_OK;
}
// one wave of games on the slots; arena_player != 0: competitive play, `arena_opponent` moves for the other side
// every slot idle, no game in flight: the state a wave starts from (also the recovery after a wave that ended with an error)
static int slots_reset(mz_ctx *c) {
    if (c->stream2) cudaStreamSynchronize(c->stream2);
    c->slots_dirty = false;
    MZ_CUDA(c, cudaMemsetAsync(c->slots.status, 0, (size_t)c->cfg.num_slots * sizeof(int32_t), c->stream));
    MZ_CUDA(c, cudaMemsetAsync(c->ring.counters + 5, 0, sizeof(int64_t), c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
static int run_wave_body(mz_ctx *c, uint64_t first_game, int64_t n_games, float temperature, int arena_player, int arena_opponent, int tally_player, int64_t *simulations, int64_t *moves, bool allow_lat = true);
static int run_wave(mz_ctx *c, uint64_t first_game, int64_t n_games, float temperature, int arena_player, int arena_opponent, int tally_player, int64_t *simulations, int64_t *moves) {
    int rc = MZ_OK;
    const int64_t G = c->cfg.num_slots;
    if (n_games > G && c->refill_wave_sync && arena_player == 0 && c->cfg.net_type == MZ_NET_FEEDFORWARD && c->stream2 &&
        !getenv("MUZERO_B200_NO_OVERLAP") && first_game + (uint64_t)n_games <= 0xffffffffull) {
        // wave-synchronous refill hands out games num_slots at a time, in slot order: a call for more games than slots is a sequence of
        // single-wave calls, each of which the headline path plays in one launch (the other feed-forward paths: one launch per move with the
        // save / refill beside the next search)
        unsigned long long acc[4] = {0, 0, 0, 0}, tally[3] = {0, 0, 0};   // search statistics; wins / draws / losses of mz_arena(MZ_OPP_SELF)
        for (int64_t off = 0; off < n_games && rc == MZ_OK; off += G) {
            rc = run_wave_body(c, first_game + (uint64_t)off, n_games - off < G ? n_games - off : G, temperature, arena_player, arena_opponent, tally_player, nullptr, nullptr,
                               false /* a short last wave stays on this path's arithmetic: one call, one kernel family */);
            for (int i = 0; i < 4; i++) acc[i] += c->h_stats[i];
            for (int i = 0; i < 3; i++) tally[i] += c->h_stats[61 + i];
        }
        if (rc == MZ_OK) {
            for (int i = 0; i < 4; i++) c->h_stats[i] = acc[i];
            for (int i = 0; i < 3; i++) c->h_stats[61 + i] = tally[i];
            if (simulations) *simulations = (int64_t)acc[1];
            if (moves) *moves = (int64_t)acc[3];
            c->last_mean_depth = acc[1] ? (double)acc[0] / (double)acc[1] : 0.0;
            c->last_mean_legal = acc[3] ? (double)acc[2] / (double)acc[3] : 0.0;
        }
    } else rc = run_wave_body(c, first_game, n_games, temperature, arena_player, arena_opponent, tally_player, simulations, moves);
    if (rc != MZ_OK && rc != MZ_E_ARG) {   // a wave that failed half-way must not leave games in flight: later calls would answer MZ_E_STATE for ever
        const std::string keep = c->err;
        slots_reset(c);
        c->err = keep; tl_error = keep;
    }
    return rc;
}
static int run_wave_body(mz_ctx *c, uint64_t first_game, int64_t n_games, float temperature, int arena_player, int arena_opponent, int tally_player, int64_t *simulations, int64_t *moves, bool allow_lat) {
    if (n_games < 0) return fail(c, MZ_E_ARG, "n_games < 0");
    if (first_game + (uint64_t)n_games > 0xffffffffull) return fail(c, MZ_E_ARG, "game ids must fit in 32 bits (Philox counter)");
    mz_params P = c->M.P;
    P.arena_player = arena_player; P.arena_opponent = arena_opponent; P.arena_tally = tally_player;
    unsigned long long *tally = c->d_stats + 61;   // wins, draws, losses (the last three of the 64 counters)
    const int G = c->cfg.num_slots;
    // A wave starts from idle slots: a successful wave ends with every slot idle, a failed one is followed by slots_reset (run_wave), so the
    // device counters need not be read back here (two stream synchronisations per wave): only {next game id, end id, active games} go down,
    // in stream order, from pinned memory
    if (c->slots_dirty) MZ_TRY(slots_reset(c));
    c->slots_dirty = true;
    c->h_counters[3] = (int64_t)first_game; c->h_counters[4] = (int64_t)first_game + n_games; c->h_counters[5] = 0;
    MZ_CUDA(c, cudaMemcpyAsync(c->ring.counters + 3, c->h_counters + 3, 3 * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaMemsetAsync(c->d_stats, 0, 64 * sizeof(unsigned long long), c->stream));
    // MZ_OPP_NETWORK: the other side's plies are searched like MuZero's, by the same kernels reading the opponent store
    const bool vs_net = arena_player != 0 && arena_opponent == MZ_OPP_NETWORK;
    MZ_TRY(ensure_images(c));
    if (vs_net) MZ_TRY(ensure_images(c, c->opp));
    mz_search_args a = search_args(c, G, 1 /* play_game hard-codes exploration=true, SelfPlay.jl:359 */);
    a.slots = c->slots; a.temperature = temperature; a.stats = c->d_stats;
    // A wave starts with every slot idle and games are handed out in slot order, so a call for n_games <= num_slots games only ever uses the
    // slots [0, n_games): few games go to the low-latency kernel whatever the context's size (the bf16 mode keeps its own arithmetic)
    const int G_lat = (int64_t)G < n_games ? G : (int)n_games;
    const bool use_lat = allow_lat && c->lat_ok && G_lat >= 1 && G_lat <= c->lat_max_slots && c->cfg.nn_mode != MZ_NN_BF16_TC;
    if (use_lat) MZ_TRY(ensure_lat_image(c, c->own));
    if (use_lat && vs_net) MZ_TRY(ensure_lat_image(c, c->opp));
    int64_t total_moves = 0; int last_snap = 0;
    // The host runs one iteration behind the device: iteration k (opponent plies, search, save/refill, counter snapshot) is queued before
    // the snapshot of iteration k - 1 is read, so the GPU never waits for a launch.  When that snapshot says no game is active any more,
    // the iteration already queued finds every slot idle: each search CTA returns at its first instruction.
    // Single-wave calls (n_games <= num_slots: every game is handed out by the first refill): the save / refill kernels of move k only touch
    // slots that finished in move k (status tag P.fin_tag) and the ring, the search of move k + 1 only active slots -- so they run side by
    // side: save / refill on a second stream behind an event of search k, the searches back to back on the main stream.  The 128 search CTAs
    // leave 20 SMs free, which is where the small kernels go.
    const bool overlap = n_games <= (int64_t)G && c->stream2 != nullptr && !getenv("MUZERO_B200_NO_OVERLAP");
    cudaStream_t sB = overlap ? c->stream2 : c->stream;
    auto snapshot = [&](int i) -> int {
        MZ_CUDA(c, cudaEventRecord(c->ev_wave[i], sB));
        return MZ_OK;
    };
    P.fin_tag = 0;
    MZ_TRY(launch_save_refill(c, P, G, tally, c->d_wave));
    MZ_CUDA(c, cudaEventRecord(c->ev_wave[0], c->stream));
    // Single-wave self-play on the split-precision path: ONE launch plays the games to the end (mz_k_search_sp, a.persist).  CTA i of move
    // k + 1 depends only on CTA i of move k, while a launch per move lasts as long as its slowest CTA (12 % above the mean) and every move
    // pays launch gaps: here a CTA starts its next move when its own trees are done.  All finished games are saved by one save / refill at
    // the end, in slot order (= game id order).  MUZERO_B200_PERSIST=0 keeps one launch per move.
    if (overlap && !use_lat && arena_player == 0 && c->cfg.net_type == MZ_NET_FEEDFORWARD && c->cfg.nn_mode == MZ_NN_SPLIT_MMA && c->persist_ok) {
        mz_search_args ap = a; ap.persist = 1;
        launch_search<MZ_MODE_SLOTS>(c, P, ap, 0);
        MZ_TRY(launch_save_refill(c, P, G, tally, c->d_wave + 8));
        MZ_CUDA(c, cudaGetLastError());
        MZ_CUDA(c, cudaMemcpyAsync(c->h_stats, c->d_stats, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
        MZ_CUDA(c, cudaStreamSynchronize(c->stream));
        if (c->h_wave[8 + 5] != 0) return fail(c, MZ_E_STATE, "self-play did not terminate");
        c->slots_dirty = false;
        if (simulations) *simulations = (int64_t)c->h_stats[1];
        if (moves) *moves = (int64_t)c->h_stats[3];
        c->last_mean_depth = c->h_stats[1] ? (double)c->h_stats[0] / (double)c->h_stats[1] : 0.0;
        c->last_mean_legal = c->h_stats[3] ? (double)c->h_stats[2] / (double)c->h_stats[3] : 0.0;
        return MZ_OK;
    }
    for (int64_t k = 0;; k++) {
        if (k > n_games * (int64_t)(P.max_moves + 2) + 8) return fail(c, MZ_E_STATE, "self-play did not terminate");
        P.fin_tag = (int32_t)(k & 1);
        const size_t iter_entry = c->timed.size();
        if (vs_net) {   // the opponent's plies: slots whose side to move is the other one, then MuZero's below (a game may make both)
            mz_params Po = P; Po.arena_player = 3 - arena_player;
            launch_search<MZ_MODE_SLOTS>(c, Po, a, use_lat ? G_lat : 0, &c->opp);
        } else if (arena_player != 0) { launch_scope ls(c, 6); mz_k_opponent_move<<<(G + 127) / 128, 128, 0, c->stream>>>(P, c->slots, G); }
        launch_search<MZ_MODE_SLOTS>(c, P, a, use_lat ? G_lat : 0);   // few games (play_game one game at a time): one tree per cluster, exact fp32
        const size_t search_entry = c->timed.size();                       // (timing builds) index just past this iteration's search launch
        if (overlap) { MZ_CUDA(c, cudaEventRecord(c->ev_search[k & 1], c->stream)); MZ_CUDA(c, cudaStreamWaitEvent(sB, c->ev_search[k & 1], 0)); }
        MZ_TRY(launch_save_refill(c, P, G, tally, c->d_wave + 8 * ((k + 1) & 1), sB));
        MZ_TRY(snapshot((int)((k + 1) & 1)));
        last_snap = (int)((k + 1) & 1);
        MZ_CUDA(c, cudaGetLastError());
        MZ_CUDA(c, cudaEventSynchronize(c->ev_wave[k & 1]));
        const int64_t active = c->h_wave[8 * (k & 1) + 5];                 // games active when iteration k started
        if (active == 0) {
            // the iteration just queued is the idle one: keep its searches out of the per-family kernel statistics (family 7 = idle)
            for (size_t i = iter_entry; i < search_entry; i++) if (c->timed[i].family == 0) c->timed[i].family = 7;
            if (c->timed.size() > search_entry) c->timed[search_entry].family = 7;
            break;
        }
        total_moves += active;
    }
    if (overlap) MZ_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_wave[last_snap], 0));   // the last save / refill (tallies, counters) before anything else runs on the main stream
    MZ_CUDA(c, cudaMemcpyAsync(c->h_stats, c->d_stats, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    c->slots_dirty = false;
    if (simulations) *simulations = (int64_t)c->h_stats[1];
    if (moves) *moves = total_moves;
    c->last_mean_depth = c->h_stats[1] ? (double)c->h_stats[0] / (double)c->h_stats[1] : 0.0;
    c->last_mean_legal = c->h_stats[3] ? (double)c->h_stats[2] / (double)c->h_stats[3] : 0.0;
    return MZ_OK;
}

int mz_self_play(mz_ctx *c, uint64_t first_game, int64_t n_games, float temperature, int64_t *simulations, int64_t *moves) {
    MZ_CHECK_CTX(c);
    return run_wave(c, first_game, n_games, temperature, 0, MZ_OPP_SELF, 0, simulations, moves);
}
static int check_opponent_set(mz_ctx *c, int opponent) {
    if (opponent == MZ_OPP_NETWORK && !c->opp_full)
        return fail(c, MZ_E_STATE, "MZ_OPP_NETWORK needs opponent networks: set them with mz_set_opponent_weights or mz_snapshot_opponent");
    return MZ_OK;
}
// competitive_play! (src/SelfPlay.jl:421-435) for n_games games at once
int mz_arena(mz_ctx *c, uint64_t first_game, int64_t n_games, int opponent, int muzero_player, float temperature, int64_t *wins, int64_t *draws,
             int64_t *losses, int64_t *simulations) {
    MZ_CHECK_CTX(c);
    if (opponent != MZ_OPP_SELF && opponent != MZ_OPP_RANDOM && opponent != MZ_OPP_EXPERT && opponent != MZ_OPP_NETWORK)
        return fail(c, MZ_E_ARG, "opponent must be MZ_OPP_SELF, MZ_OPP_RANDOM, MZ_OPP_EXPERT or MZ_OPP_NETWORK (\"human\" has no batched meaning)");
    if (c->M.P.P != 2 && opponent != MZ_OPP_SELF) return fail(c, MZ_E_ARG, "an opponent needs a two-player game");
    if (muzero_player < 1 || muzero_player > c->M.P.P) return fail(c, MZ_E_ARG, "muzero_player %d out of range 1..%d", muzero_player, c->M.P.P);
    MZ_TRY(check_opponent_set(c, opponent));
    // length(conf.players) == 1 ? "self" : conf.opponent (:428); "self": every ply is searched, outcomes still tallied for muzero_player
    MZ_TRY(run_wave(c, first_game, n_games, temperature, opponent == MZ_OPP_SELF ? 0 : muzero_player, opponent, muzero_player, simulations, nullptr));
    if (wins) *wins = (int64_t)c->h_stats[61];
    if (draws) *draws = (int64_t)c->h_stats[62];
    if (losses) *losses = (int64_t)c->h_stats[63];
    return MZ_OK;
}
int mz_opponent_action(mz_ctx *c, int n, const uint64_t *p1, const uint64_t *p2, const int32_t *player, int opponent, const uint64_t *game_id,
                       const int32_t *move_idx, int32_t *action) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!p1 || !p2 || !player || !game_id || !move_idx || !action))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (opponent != MZ_OPP_RANDOM && opponent != MZ_OPP_EXPERT) return fail(c, MZ_E_ARG, "opponent must be MZ_OPP_RANDOM or MZ_OPP_EXPERT");
    if (n == 0) return MZ_OK;
    const mz_params &P = c->M.P;
    uint64_t *d_p1, *d_p2, *d_gid; int32_t *d_pl, *d_mv, *d_act;
    MZ_TRY(h2d(c, c->scratch[0], p1, (size_t)n, &d_p1)); MZ_TRY(h2d(c, c->scratch[1], p2, (size_t)n, &d_p2));
    MZ_TRY(h2d(c, c->scratch[2], player, (size_t)n, &d_pl)); MZ_TRY(h2d(c, c->scratch[3], game_id, (size_t)n, &d_gid));
    MZ_TRY(h2d(c, c->scratch[4], move_idx, (size_t)n, &d_mv)); MZ_TRY(h2d<int32_t>(c, c->scratch[5], nullptr, (size_t)n, &d_act));
    { launch_scope ls(c, 6); mz_k_opponent_action<<<(n + 127) / 128, 128, 0, c->stream>>>(P, n, d_p1, d_p2, d_pl, opponent, d_gid, d_mv, d_act); }
    MZ_CUDA(c, cudaGetLastError());
    MZ_TRY(d2h(c, action, d_act, (size_t)n));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}

// play_game (src/SelfPlay.jl:330-382) for n_games games at once, histories returned to the caller (in the order the games finished; game_id
// says which is which) and NOT saved: the reference's self_play! calls save_game itself (:414).  The wave runs on a ring of its own.
int mz_play_games(mz_ctx *c, uint64_t first_game, int n_games, float temperature, int opponent, int muzero_player, int64_t *game_id, int32_t *T, float *obs,
                  int32_t *actions, float *rewards, int32_t *to_play, float *child_visits, float *root_values, int64_t *simulations) {
    MZ_CHECK_CTX(c);
    if (n_games < 0) return fail(c, MZ_E_ARG, "n_games < 0");
    if (opponent != MZ_OPP_SELF && opponent != MZ_OPP_RANDOM && opponent != MZ_OPP_EXPERT && opponent != MZ_OPP_NETWORK)
        return fail(c, MZ_E_ARG, "opponent must be MZ_OPP_SELF, MZ_OPP_RANDOM, MZ_OPP_EXPERT or MZ_OPP_NETWORK (\"human\" has no batched meaning)");
    if (opponent != MZ_OPP_SELF && (c->M.P.P != 2 || muzero_player < 1 || muzero_player > 2)) return fail(c, MZ_E_ARG, "an opponent needs a two-player game and muzero_player in 1..2");
    MZ_TRY(check_opponent_set(c, opponent));
    if (simulations) *simulations = 0;
    if (n_games == 0) return MZ_OK;
    MZ_TRY(read_counters(c));
    if (c->h_counters[5] != 0) MZ_TRY(slots_reset(c));
    if (c->play_ring.capacity < n_games) MZ_TRY(alloc_ring(c, c->play_ring, (size_t)(n_games < c->cfg.num_slots ? c->cfg.num_slots : n_games)));
    MZ_CUDA(c, cudaMemsetAsync(c->play_ring.counters, 0, 8 * sizeof(int64_t), c->stream));
    const int per = c->M.P.per; c->M.P.per = 0;                  // priorities belong to save_game
    std::swap(c->ring, c->play_ring);
    int rc = run_wave(c, first_game, n_games, temperature, opponent == MZ_OPP_SELF ? 0 : muzero_player, opponent, 0, simulations, nullptr);
    if (rc == MZ_OK) rc = mz_history_export(c, 1, n_games, game_id, T, obs, actions, rewards, to_play, child_visits, root_values);
    std::swap(c->ring, c->play_ring);
    c->M.P.per = per;
    return rc;
}

int mz_replay_info(mz_ctx *c, int64_t *n_games, int64_t *first_key, int64_t *total_samples) {
    MZ_CHECK_CTX(c);
    MZ_TRY(read_counters(c));
    int64_t played = c->h_counters[0], n = played < c->ring.capacity ? played : c->ring.capacity;
    if (n_games) *n_games = n;
    if (first_key) *first_key = played - n + 1;
    if (total_samples) *total_samples = c->h_counters[2];
    return MZ_OK;
}
int mz_replay_clear(mz_ctx *c) {
    MZ_CHECK_CTX(c);
    MZ_TRY(slots_reset(c));
    for (int i = 0; i < 8; i++) c->h_counters[i] = 0;
    MZ_TRY(write_counters(c));
    MZ_CUDA(c, cudaMemsetAsync(c->ring.T, 0, (size_t)c->ring.capacity * sizeof(int32_t), c->stream));
    MZ_CUDA(c, cudaMemsetAsync(c->ring.reanalysed, 0, (size_t)c->ring.capacity, c->stream));
    return MZ_OK;
}

int mz_history_export(mz_ctx *c, int64_t key0, int n, int64_t *game_id, int32_t *T, float *obs, int32_t *actions, float *rewards,
                      int32_t *to_play, float *child_visits, float *root_values) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!game_id || !T || !obs || !actions || !rewards || !to_play || !child_visits || !root_values))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    MZ_TRY(read_counters(c));
    int64_t played = c->h_counters[0], have = played < c->ring.capacity ? played : c->ring.capacity, first = played - have + 1;
    if (key0 < first || key0 + n - 1 > played) return fail(c, MZ_E_ARG, "keys %lld..%lld not in the buffer (holds %lld..%lld)", (long long)key0, (long long)(key0 + n - 1), (long long)first, (long long)played);
    const mz_params &P = c->M.P; const size_t Tm = (size_t)P.Tmax, N = (size_t)n;
    int64_t *d_gid; int32_t *d_T, *d_act, *d_tp; float *d_obs, *d_rew, *d_cv, *d_rv;
    MZ_TRY(h2d<int64_t>(c, c->scratch[0], nullptr, N, &d_gid)); MZ_TRY(h2d<int32_t>(c, c->scratch[1], nullptr, N, &d_T));
    MZ_TRY(h2d<float>(c, c->scratch[2], nullptr, N * Tm * P.obs_size, &d_obs)); MZ_TRY(h2d<int32_t>(c, c->scratch[3], nullptr, N * Tm, &d_act));
    MZ_TRY(h2d<float>(c, c->scratch[4], nullptr, N * Tm, &d_rew)); MZ_TRY(h2d<int32_t>(c, c->scratch[5], nullptr, N * Tm, &d_tp));
    MZ_TRY(h2d<float>(c, c->scratch[6], nullptr, N * Tm * P.A, &d_cv)); MZ_TRY(h2d<float>(c, c->scratch[7], nullptr, N * Tm, &d_rv));
    size_t tot = N * Tm * P.obs_size;
    { launch_scope ls(c, 2); mz_k_history_export<<<(unsigned)((tot + 255) / 256), 256, 0, c->stream>>>(P, c->ring, key0, n, d_gid, d_T, d_obs, d_act, d_rew, d_tp, d_cv, d_rv); }
    MZ_CUDA(c, cudaGetLastError());
    MZ_TRY(d2h(c, game_id, d_gid, N)); MZ_TRY(d2h(c, T, d_T, N)); MZ_TRY(d2h(c, obs, d_obs, tot)); MZ_TRY(d2h(c, actions, d_act, N * Tm));
    MZ_TRY(d2h(c, rewards, d_rew, N * Tm)); MZ_TRY(d2h(c, to_play, d_tp, N * Tm)); MZ_TRY(d2h(c, child_visits, d_cv, N * Tm * P.A)); MZ_TRY(d2h(c, root_values, d_rv, N * Tm));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}

int mz_history_import(mz_ctx *c, int n, const int64_t *game_id, const int32_t *T, const float *obs, const int32_t *actions, const float *rewards,
                      const int32_t *to_play, const float *child_visits, const float *root_values) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!game_id || !T || !obs || !actions || !rewards || !to_play || !child_visits || !root_values))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    if (n > c->ring.capacity) return fail(c, MZ_E_ARG, "more histories than replay_buffer_size");
    const mz_params &P = c->M.P; const size_t Tm = (size_t)P.Tmax, N = (size_t)n;
    for (int i = 0; i < n; i++) if (T[i] < 1 || T[i] > P.Tmax) return fail(c, MZ_E_ARG, "history %d has length %d outside 1..%d", i, T[i], P.Tmax);
    MZ_TRY(read_counters(c));
    if (c->h_counters[5] != 0) return fail(c, MZ_E_STATE, "self-play in progress");
    // save_game bookkeeping (ReplayBuffer.jl:147-160): counters + FIFO eviction accounting
    std::vector<int32_t> oldT((size_t)c->ring.capacity);
    MZ_CUDA(c, cudaMemcpyAsync(oldT.data(), c->ring.T, oldT.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    int64_t played = c->h_counters[0], key0 = played + 1;
    for (int i = 0; i < n; i++) {
        int64_t key = key0 + i, pos = (key - 1) % c->ring.capacity;
        c->h_counters[1] += T[i]; c->h_counters[2] += T[i];
        if (key > c->ring.capacity) c->h_counters[2] -= oldT[(size_t)pos];
    }
    c->h_counters[0] = played + n;
    int64_t *d_gid; int32_t *d_T, *d_act, *d_tp; float *d_obs, *d_rew, *d_cv, *d_rv;
    MZ_TRY(h2d(c, c->scratch[0], game_id, N, &d_gid)); MZ_TRY(h2d(c, c->scratch[1], T, N, &d_T));
    MZ_TRY(h2d(c, c->scratch[2], obs, N * Tm * P.obs_size, &d_obs)); MZ_TRY(h2d(c, c->scratch[3], actions, N * Tm, &d_act));
    MZ_TRY(h2d(c, c->scratch[4], rewards, N * Tm, &d_rew)); MZ_TRY(h2d(c, c->scratch[5], to_play, N * Tm, &d_tp));
    MZ_TRY(h2d(c, c->scratch[6], child_visits, N * Tm * P.A, &d_cv)); MZ_TRY(h2d(c, c->scratch[7], root_values, N * Tm, &d_rv));
    { launch_scope ls(c, 2); mz_k_history_import<<<(unsigned)((N * Tm + 127) / 128), 128, 0, c->stream>>>(P, c->ring, key0, n, d_gid, d_T, d_obs, d_act, d_rew, d_tp, d_cv, d_rv); }
    if (c->cfg.per) { launch_scope ls(c, 2); mz_k_per_init<<<(n + 127) / 128, 128, 0, c->stream>>>(P, c->ring, key0, n); }   // save_game's initial priorities
    MZ_CUDA(c, cudaGetLastError());
    return write_counters(c);
}

// ---- reanalyse (GameHistory.reanalysed_predicted_root_values, consumed by compute_target_value, ReplayBuffer.jl:8) ----
int mz_reanalyse(mz_ctx *c, int64_t key0, int n) {
    MZ_CHECK_CTX(c);
    if (c->cfg.net_type != MZ_NET_FEEDFORWARD) return fail(c, MZ_E_UNSUPPORTED, "reanalyse runs the exact feed-forward networks");
    if (n < 0) return fail(c, MZ_E_ARG, "n < 0");
    if (n == 0) return MZ_OK;
    MZ_TRY(read_counters(c));
    if (c->h_counters[5] != 0) return fail(c, MZ_E_STATE, "self-play in progress");
    int64_t played = c->h_counters[0], have = played < c->ring.capacity ? played : c->ring.capacity, first = played - have + 1;
    if (key0 < first || key0 + n - 1 > played) return fail(c, MZ_E_ARG, "keys %lld..%lld not in the buffer (holds %lld..%lld)", (long long)key0, (long long)(key0 + n - 1), (long long)first, (long long)played);
    const mz_params &P = c->M.P;
    mz_reanalyse_args a{}; a.wglob = c->own.w; a.max_dim = c->M.max_dim; a.max_layer_floats = c->M.max_layer_floats; a.n = n; a.key0 = key0; a.ring = c->ring;
    const int64_t total = (int64_t)n * P.Tmax;
    { launch_scope ls(c, 5);
      if (c->cfg.use_batch_norm) mz_k_reanalyse<true><<<(unsigned)((total + MZ_ROWS - 1) / MZ_ROWS), MZ_THREADS, c->smem_bytes, c->stream>>>(P, a);
      else mz_k_reanalyse<false><<<(unsigned)((total + MZ_ROWS - 1) / MZ_ROWS), MZ_THREADS, c->smem_bytes, c->stream>>>(P, a); }
    MZ_CUDA(c, cudaGetLastError());
    return MZ_OK;
}
// MuZero Reanalyze: run_mcts again at every stored position of games key0 .. key0+n-1, with the current networks and the root self-play
// searched there.  The dense root list (ring entry pos * Tmax + t for t < T) is built on the host from the games' lengths: one small copy
// each way, and the search launches then hold only real positions (Connect Four games fill far fewer than Tmax).  It is ordered by move
// t, then by key: the trees of a CTA search in lock step, so a CTA takes as long as its deepest tree, and late positions (fewer legal
// actions) search deeper -- the reason self-play keeps a wave at one ply (mz_k_save_refill's wave_sync).  The list is cut into launches
// of at most num_slots roots, the capacity of the tree pool; every root's result depends only on its own position and keys.
int mz_reanalyse_search(mz_ctx *c, int64_t key0, int n, int exploration, int64_t *simulations) {
    MZ_CHECK_CTX(c);
    if (simulations) *simulations = 0;
    if (n < 0) return fail(c, MZ_E_ARG, "n < 0");
    if (n == 0) return MZ_OK;
    MZ_TRY(read_counters(c));
    if (c->h_counters[5] != 0) return fail(c, MZ_E_STATE, "self-play in progress");
    int64_t played = c->h_counters[0], have = played < c->ring.capacity ? played : c->ring.capacity, first = played - have + 1;
    if (key0 < first || key0 + n - 1 > played) return fail(c, MZ_E_ARG, "keys %lld..%lld not in the buffer (holds %lld..%lld)", (long long)key0, (long long)(key0 + n - 1), (long long)first, (long long)played);
    const mz_params &P = c->M.P;
    const int64_t cap = c->ring.capacity, Tm = P.Tmax, pos0 = (key0 - 1) % cap, n1 = n < cap - pos0 ? n : cap - pos0;   // the range wraps after n1 games
    std::vector<int32_t> T((size_t)n);
    MZ_CUDA(c, cudaMemcpyAsync(T.data(), c->ring.T + pos0, (size_t)n1 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (n1 < n) MZ_CUDA(c, cudaMemcpyAsync(T.data() + n1, c->ring.T, (size_t)(n - n1) * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    std::vector<int64_t> roots;
    for (int t = 0; t < Tm; t++)
        for (int j = 0; j < n; j++) if (t < T[(size_t)j]) roots.push_back(((key0 + j - 1) % cap) * Tm + t);
    MZ_TRY(ensure_images(c));
    int64_t *d_roots;
    MZ_TRY(h2d(c, c->scratch[0], roots.data(), roots.size(), &d_roots));
    { launch_scope ls(c, 5); mz_k_reanalyse_mark<<<(unsigned)(((int64_t)n * Tm + 127) / 128), 128, 0, c->stream>>>(P, c->ring, key0, n); }
    MZ_CUDA(c, cudaGetLastError());
    const int64_t total = (int64_t)roots.size(), chunk = c->cfg.num_slots;
    for (int64_t off = 0; off < total; off += chunk) {
        mz_search_args a = search_args(c, (int)(total - off < chunk ? total - off : chunk), exploration);
        a.ring = c->ring; a.replay = d_roots + off;   // a.stats stays NULL: mz_search_stats describes self-play
        launch_search<MZ_MODE_REPLAY>(c, P, a, 0);
        MZ_CUDA(c, cudaGetLastError());
    }
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    if (simulations) *simulations = total * P.S;
    return MZ_OK;
}
int mz_reanalysed_export(mz_ctx *c, int64_t key0, int n, float *values, int32_t *flags) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!values || !flags))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    MZ_TRY(read_counters(c));
    int64_t played = c->h_counters[0], have = played < c->ring.capacity ? played : c->ring.capacity, first = played - have + 1;
    if (key0 < first || key0 + n - 1 > played) return fail(c, MZ_E_ARG, "keys not in the buffer");
    const size_t Tm = (size_t)c->M.P.Tmax;
    std::vector<uint8_t> fl((size_t)c->ring.capacity);
    MZ_CUDA(c, cudaMemcpyAsync(fl.data(), c->ring.reanalysed, fl.size(), cudaMemcpyDeviceToHost, c->stream));
    for (int j = 0; j < n; j++) {
        const int64_t pos = (key0 + j - 1) % c->ring.capacity;
        MZ_CUDA(c, cudaMemcpyAsync(values + (size_t)j * Tm, c->ring.h_rrv + (size_t)pos * Tm, Tm * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    }
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int j = 0; j < n; j++) flags[j] = fl[(size_t)((key0 + j - 1) % c->ring.capacity)];
    return MZ_OK;
}

// ---- replay state for checkpoint / resume: counters, priorities, reanalysed values ---------------------------
int mz_replay_counters(mz_ctx *c, int64_t out[3]) {
    MZ_CHECK_CTX(c);
    if (!out) return fail(c, MZ_E_ARG, "NULL buffer");
    MZ_TRY(read_counters(c));
    for (int i = 0; i < 3; i++) out[i] = c->h_counters[i];
    return MZ_OK;
}
int mz_replay_set_counters(mz_ctx *c, int64_t num_played_games, int64_t num_played_steps, int64_t total_samples) {
    MZ_CHECK_CTX(c);
    if (num_played_games < 0 || num_played_steps < 0 || total_samples < 0) return fail(c, MZ_E_ARG, "counters must be >= 0");
    MZ_TRY(read_counters(c));
    if (c->h_counters[5] != 0) return fail(c, MZ_E_STATE, "self-play in progress");
    c->h_counters[0] = num_played_games; c->h_counters[1] = num_played_steps; c->h_counters[2] = total_samples;
    return write_counters(c);
}
static int keys_in_buffer(mz_ctx *c, int64_t key0, int n) {
    MZ_TRY(read_counters(c));
    const int64_t played = c->h_counters[0], have = played < c->ring.capacity ? played : c->ring.capacity, first = played - have + 1;
    if (key0 < first || key0 + n - 1 > played) return fail(c, MZ_E_ARG, "keys %lld..%lld not in the buffer (holds %lld..%lld)", (long long)key0, (long long)(key0 + n - 1), (long long)first, (long long)played);
    return MZ_OK;
}
int mz_replay_set_priorities(mz_ctx *c, int64_t key0, int n, const uint32_t *q_pos, const uint32_t *q_game) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!q_pos || !q_game))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    MZ_TRY(keys_in_buffer(c, key0, n));
    const size_t Tm = (size_t)c->M.P.Tmax;
    for (int j = 0; j < n; j++) {
        const int64_t pos = (key0 + j - 1) % c->ring.capacity;
        MZ_CUDA(c, cudaMemcpyAsync(c->ring.q_pos + (size_t)pos * Tm, q_pos + (size_t)j * Tm, Tm * 4, cudaMemcpyHostToDevice, c->stream));
        MZ_CUDA(c, cudaMemcpyAsync(c->ring.q_game + pos, q_game + j, 4, cudaMemcpyHostToDevice, c->stream));
    }
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
int mz_reanalysed_import(mz_ctx *c, int64_t key0, int n, const float *values, const int32_t *flags) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!values || !flags))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    MZ_TRY(keys_in_buffer(c, key0, n));
    const size_t Tm = (size_t)c->M.P.Tmax;
    std::vector<uint8_t> fl((size_t)n);
    for (int j = 0; j < n; j++) fl[(size_t)j] = flags[j] ? 1 : 0;
    for (int j = 0; j < n; j++) {
        const int64_t pos = (key0 + j - 1) % c->ring.capacity;
        MZ_CUDA(c, cudaMemcpyAsync(c->ring.h_rrv + (size_t)pos * Tm, values + (size_t)j * Tm, Tm * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        MZ_CUDA(c, cudaMemcpyAsync(c->ring.reanalysed + pos, fl.data() + j, 1, cudaMemcpyHostToDevice, c->stream));
    }
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}

// ---- replay sampling / learner -----------------------------------------------------------------------------
// get_batch on the device ring; conf.PER: prefix scan of the game priorities first, weight normalisation after
static int launch_gather(mz_ctx *c, uint64_t step, int B) {
    if (c->cfg.per) { launch_scope ls(c, 2); mz_k_per_scan<<<1, 1024, 0, c->stream>>>(c->M.P, c->ring); }
    { launch_scope ls(c, 2); mz_k_replay_gather<<<B, 64, 0, c->stream>>>(c->M.P, c->ring, step, B, c->batch); }
    if (c->cfg.per) { launch_scope ls(c, 2); mz_k_per_normalise<<<1, 1024, 0, c->stream>>>(B, c->batch.weights); }
    MZ_CUDA(c, cudaGetLastError());
    return MZ_OK;
}
// update_priorities! after the optimiser step (Learning.jl:400-404)
static int launch_per_update(mz_ctx *c, int B) {
    if (!c->cfg.per) return MZ_OK;
    const int n = B * (c->M.P.K + 1);
    for (int phase = 0; phase < 3; phase++) { launch_scope ls(c, 2); mz_k_per_update<<<(n + 127) / 128, 128, 0, c->stream>>>(c->M.P, c->ring, B, c->batch.index, c->d_pv, c->batch.values, phase); }
    MZ_CUDA(c, cudaGetLastError());
    return MZ_OK;
}
static int gather_batch(mz_ctx *c, uint64_t step) {
    const int B = c->cfg.batch_size;
    MZ_TRY(alloc_batch(c, B));
    MZ_TRY(read_counters(c));
    if (c->h_counters[0] < 1) return fail(c, MZ_E_STATE, "replay buffer is empty (learning! waits for num_played_games >= 1, Learning.jl:311)");
    return launch_gather(c, step, B);
}
int mz_get_batch(mz_ctx *c, uint64_t step, int32_t *index_batch, float *obs_batch, float *action_batch, float *value_batch, float *reward_batch,
                 float *policy_batch, float *gscale) {
    MZ_CHECK_CTX(c);
    if (!index_batch || !obs_batch || !action_batch || !value_batch || !reward_batch || !policy_batch || !gscale) return fail(c, MZ_E_ARG, "NULL buffer");
    MZ_TRY(gather_batch(c, step));
    const mz_params &P = c->M.P; const size_t B = (size_t)c->cfg.batch_size, K1 = (size_t)P.K + 1;
    MZ_TRY(d2h(c, index_batch, c->batch.index, B * 2)); MZ_TRY(d2h(c, obs_batch, c->batch.obs, B * P.stack_size));
    MZ_TRY(d2h(c, action_batch, c->batch.actions, B * K1)); MZ_TRY(d2h(c, value_batch, c->batch.values, B * K1));
    MZ_TRY(d2h(c, reward_batch, c->batch.rewards, B * K1)); MZ_TRY(d2h(c, policy_batch, c->batch.policies, B * K1 * P.A));
    MZ_TRY(d2h(c, gscale, c->batch.gscale, B));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
int mz_get_batch_per(mz_ctx *c, uint64_t step, int32_t *index_batch, float *obs_batch, float *action_batch, float *value_batch, float *reward_batch,
                     float *policy_batch, float *gscale, float *weight_batch) {
    MZ_CHECK_CTX(c);
    if (!c->cfg.per) return fail(c, MZ_E_STATE, "conf.PER is false: use mz_get_batch");
    if (!weight_batch) return fail(c, MZ_E_ARG, "NULL buffer");
    int rc = mz_get_batch(c, step, index_batch, obs_batch, action_batch, value_batch, reward_batch, policy_batch, gscale);
    if (rc != MZ_OK) return rc;
    MZ_TRY(d2h(c, weight_batch, c->batch.weights, (size_t)c->cfg.batch_size));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
int mz_replay_priorities(mz_ctx *c, int64_t key0, int n, uint32_t *q_pos, uint32_t *q_game) {
    MZ_CHECK_CTX(c);
    if (n < 0 || (n > 0 && (!q_pos || !q_game))) return fail(c, MZ_E_ARG, "NULL buffer");
    if (n == 0) return MZ_OK;
    MZ_TRY(read_counters(c));
    int64_t played = c->h_counters[0], have = played < c->ring.capacity ? played : c->ring.capacity, first = played - have + 1;
    if (key0 < first || key0 + n - 1 > played) return fail(c, MZ_E_ARG, "keys not in the buffer");
    const size_t Tm = (size_t)c->M.P.Tmax;
    for (int j = 0; j < n; j++) {
        const int64_t pos = (key0 + j - 1) % c->ring.capacity;
        MZ_CUDA(c, cudaMemcpyAsync(q_pos + (size_t)j * Tm, c->ring.q_pos + (size_t)pos * Tm, Tm * 4, cudaMemcpyDeviceToHost, c->stream));
        MZ_CUDA(c, cudaMemcpyAsync(q_game + j, c->ring.q_game + pos, 4, cudaMemcpyDeviceToHost, c->stream));
    }
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    return MZ_OK;
}
static int upload_batch(mz_ctx *c, int B, const float *obs, const float *act, const float *val, const float *rew, const float *pol, const float *gs) {
    if (B < 1 || !obs || !act || !val || !rew || !pol || !gs) return fail(c, MZ_E_ARG, "bad batch");
    MZ_TRY(alloc_batch(c, B));
    const mz_params &P = c->M.P; const size_t K1 = (size_t)P.K + 1, b = (size_t)B;
    MZ_CUDA(c, cudaMemcpyAsync(c->batch.obs, obs, b * P.stack_size * 4, cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaMemcpyAsync(c->batch.actions, act, b * K1 * 4, cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaMemcpyAsync(c->batch.values, val, b * K1 * 4, cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaMemcpyAsync(c->batch.rewards, rew, b * K1 * 4, cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaMemcpyAsync(c->batch.policies, pol, b * K1 * P.A * 4, cudaMemcpyHostToDevice, c->stream));
    MZ_CUDA(c, cudaMemcpyAsync(c->batch.gscale, gs, b * 4, cudaMemcpyHostToDevice, c->stream));
    if (c->cfg.per) {   // caller-supplied batches carry no importance weights unless mz_learn_gradients_w provides them: weight_batch = 1
        std::vector<float> ones(b, 1.0f);
        MZ_CUDA(c, cudaMemcpyAsync(c->batch.weights, ones.data(), b * 4, cudaMemcpyHostToDevice, c->stream));
        MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return MZ_OK;
}
int mz_learn_forward(mz_ctx *c, int B, const float *obs_batch, const float *action_batch, const float *value_batch, const float *reward_batch,
                     const float *policy_batch, const float *gscale, float *pred_values, float *pred_rewards, float *pred_policies, float *losses) {
    MZ_CHECK_CTX(c);
    if (!losses) return fail(c, MZ_E_ARG, "NULL losses");
    MZ_TRY(upload_batch(c, B, obs_batch, action_batch, value_batch, reward_batch, policy_batch, gscale));
    MZ_TRY(launch_learn_forward(c, B));
    const mz_params &P = c->M.P; const size_t K1 = (size_t)P.K + 1, b = (size_t)B;
    MZ_TRY(d2h(c, pred_values, c->d_pv, b * K1)); MZ_TRY(d2h(c, pred_rewards, c->d_pr, b * K1)); MZ_TRY(d2h(c, pred_policies, c->d_pp, b * K1 * P.A));
    return finish_losses(c, B, losses);
}
int mz_learn_step_batch(mz_ctx *c, int64_t t, int grad_mode, int B, const float *obs_batch, const float *action_batch, const float *value_batch,
                        const float *reward_batch, const float *policy_batch, const float *gscale, float *losses) {
    MZ_CHECK_CTX(c);
    if (!losses || t < 1) return fail(c, MZ_E_ARG, "bad arguments");
    MZ_TRY(upload_batch(c, B, obs_batch, action_batch, value_batch, reward_batch, policy_batch, gscale));
    MZ_TRY(launch_learn_forward(c, B, grad_mode));
    MZ_TRY(launch_update(c, t, grad_mode));
    return finish_losses(c, B, losses);
}
// gradients of one batch without an update (parity entry point): grad in the reference blob order
int mz_learn_gradients(mz_ctx *c, int grad_mode, int B, const float *obs_batch, const float *action_batch, const float *value_batch,
                       const float *reward_batch, const float *policy_batch, const float *gscale, float *grad, float *losses) {
    return mz_learn_gradients_w(c, grad_mode, B, obs_batch, action_batch, value_batch, reward_batch, policy_batch, gscale, nullptr, grad, losses);
}
int mz_learn_gradients_w(mz_ctx *c, int grad_mode, int B, const float *obs_batch, const float *action_batch, const float *value_batch,
                         const float *reward_batch, const float *policy_batch, const float *gscale, const float *weight_batch, float *grad, float *losses) {
    MZ_CHECK_CTX(c);
    if (!losses || !grad) return fail(c, MZ_E_ARG, "bad arguments");
    if (weight_batch && !c->cfg.per) return fail(c, MZ_E_STATE, "importance weights need conf.PER = true");
    MZ_TRY(upload_batch(c, B, obs_batch, action_batch, value_batch, reward_batch, policy_batch, gscale));
    if (weight_batch) MZ_CUDA(c, cudaMemcpyAsync(c->batch.weights, weight_batch, (size_t)B * 4, cudaMemcpyHostToDevice, c->stream));
    MZ_TRY(launch_learn_forward(c, B, grad_mode));
    const int n = c->store_floats;
    if (grad_mode == MZ_GRAD_REFERENCE_L2) { launch_scope ls(c, 4); mz_k_l2_grad<<<(n + 255) / 256, 256, 0, c->stream>>>(n, c->own.w, c->d_mask, grad_out(c)); }
    MZ_TRY(store_to_host(c, grad_out(c), grad));
    return finish_losses(c, B, losses);
}
int mz_learn_step(mz_ctx *c, int64_t t, int grad_mode, float *losses) {
    MZ_CHECK_CTX(c);
    if (!losses || t < 1) return fail(c, MZ_E_ARG, "bad arguments");
    MZ_TRY(gather_batch(c, (uint64_t)t));
    MZ_TRY(launch_learn_forward(c, c->cfg.batch_size, grad_mode));
    MZ_TRY(launch_update(c, t, grad_mode));
    MZ_TRY(launch_per_update(c, c->cfg.batch_size));
    return finish_losses(c, c->cfg.batch_size, losses);
}
// n consecutive learning! iterations (steps t0 .. t0+n-1) without a host round trip in between: the replay gather of
// step t+1 is queued behind the ADAM update of step t on the same stream; only the last step's losses are read back
// (the reference logs them every checkpoint_interval steps, Learning.jl:416-424).
int mz_learn_steps(mz_ctx *c, int64_t t0, int n, int grad_mode, float *losses) {
    MZ_CHECK_CTX(c);
    if (!losses || t0 < 1 || n < 1) return fail(c, MZ_E_ARG, "bad arguments");
    const int B = c->cfg.batch_size;
    MZ_TRY(alloc_batch(c, B));
    MZ_TRY(read_counters(c));
    if (c->h_counters[0] < 1) return fail(c, MZ_E_STATE, "replay buffer is empty (learning! waits for num_played_games >= 1, Learning.jl:311)");
    for (int i = 0; i < n; i++) {
        MZ_TRY(launch_gather(c, (uint64_t)(t0 + i), B));
        MZ_TRY(launch_learn_forward(c, B, grad_mode));
        MZ_TRY(launch_update(c, t0 + i, grad_mode));
        MZ_TRY(launch_per_update(c, B));
    }
    return finish_losses(c, B, losses);
}
// ---- checkpoint / resume of the optimiser (weights: mz_get_weights / mz_set_weights; histories: mz_history_export / import) ----
// Flux.ADAM keeps (mt, vt, beta powers) per parameter array (Learning.jl:318, 395-397); m and v cross the ABI in the blob order.
int mz_get_optimizer_state(mz_ctx *c, float *m, float *v, int64_t n, int64_t *steps_done) {
    MZ_CHECK_CTX(c);
    if (!m || !v || !steps_done || n != c->M.P.n_params) return fail(c, MZ_E_ARG, "bad arguments (need %d floats per moment)", c->M.P.n_params);
    MZ_TRY(store_to_host(c, c->d_m, m));
    MZ_TRY(store_to_host(c, c->d_v, v));
    *steps_done = c->adam_t - 1;
    return MZ_OK;
}
int mz_set_optimizer_state(mz_ctx *c, const float *m, const float *v, int64_t n, int64_t steps_done) {
    MZ_CHECK_CTX(c);
    if (!m || !v || steps_done < 0 || n != c->M.P.n_params) return fail(c, MZ_E_ARG, "bad arguments (need %d floats per moment)", c->M.P.n_params);
    MZ_TRY(store_from_host(c, c->d_m, m));
    MZ_TRY(store_from_host(c, c->d_v, v));
    adam_seek(c, steps_done);
    return MZ_OK;
}
int mz_optimizer_reset(mz_ctx *c) {
    MZ_CHECK_CTX(c);
    MZ_CUDA(c, cudaMemsetAsync(c->d_m, 0, (size_t)c->store_floats * 4, c->stream));
    MZ_CUDA(c, cudaMemsetAsync(c->d_v, 0, (size_t)c->store_floats * 4, c->stream));
    adam_seek(c, 0);
    return MZ_OK;
}

// ---- multi-GPU -------------------------------------------------------------------------------------------------
int mz_comm_unique_id(uint8_t id[128]) {
    if (!id) return fail(nullptr, MZ_E_ARG, "id is NULL");
    if (!g_nccl.load()) return fail(nullptr, MZ_E_NCCL, "cannot load libnccl.so.2: %s", dlerror());
    ncclUniqueId u; ncclResult_t r = g_nccl.GetUniqueId(&u);
    if (r != ncclSuccess) return fail(nullptr, MZ_E_NCCL, "ncclGetUniqueId: %s", g_nccl.GetErrorString(r));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    memcpy(id, &u, 128);
    return MZ_OK;
}
// closes the peer mappings and frees the exchange buffers (after a barrier: a peer may still be reading them)
static void p2p_teardown(mz_ctx *c) {
    if (!c->d_xgrad) return;
    if (c->comm && c->d_xflags) {   // barrier through NCCL, then nobody touches anybody's buffers again
        g_nccl.AllReduce(c->d_xflags + MZ_DP_MAX_RANKS, c->d_xflags + MZ_DP_MAX_RANKS, 1, ncclInt32, ncclSum, c->comm, c->stream);
        cudaStreamSynchronize(c->stream);
    }
    for (int r = 0; r < MZ_DP_MAX_RANKS; r++) {
        if (r != c->rank && c->peer_grad[r]) cudaIpcCloseMemHandle(c->peer_grad[r]);
        if (r != c->rank && c->peer_flags[r]) cudaIpcCloseMemHandle(c->peer_flags[r]);
        c->peer_grad[r] = nullptr; c->peer_flags[r] = nullptr;
    }
    cudaFree(c->d_xgrad); cudaFree(c->d_xflags);
    c->d_xgrad = nullptr; c->d_xflags = nullptr; c->p2p = false; c->dp_step = 0;
}
// Maps every rank's gradient exchange buffer and flag block into this process (CUDA IPC; the 128 bytes of handles per rank travel through
// ncclAllGather).  Any failure leaves the NCCL allreduce in charge.  MUZERO_B200_DP=nccl forces that, too.
static void p2p_setup(mz_ctx *c) {
    const char *force = getenv("MUZERO_B200_DP");
    if ((force && !strcmp(force, "nccl")) || c->nranks < 2 || c->nranks > MZ_DP_MAX_RANKS || c->cfg.net_type != MZ_NET_FEEDFORWARD) return;
    const size_t n = (size_t)c->M.P.total_floats;
    unsigned char mine[128], *d_all = nullptr; std::vector<unsigned char> all((size_t)128 * c->nranks);
    bool ok = cudaMalloc((void **)&c->d_xgrad, 2 * n * sizeof(float)) == cudaSuccess && cudaMalloc((void **)&c->d_xflags, 2 * MZ_DP_MAX_RANKS * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMemset(c->d_xgrad, 0, 2 * n * sizeof(float)) == cudaSuccess && cudaMemset(c->d_xflags, 0, 2 * MZ_DP_MAX_RANKS * sizeof(uint32_t)) == cudaSuccess;
    memset(mine, 0, sizeof(mine));
    cudaIpcMemHandle_t hg, hf;
    ok = ok && cudaIpcGetMemHandle(&hg, c->d_xgrad) == cudaSuccess && cudaIpcGetMemHandle(&hf, c->d_xflags) == cudaSuccess;
    if (ok) { memcpy(mine, &hg, 64); memcpy(mine + 64, &hf, 64); }
    // every rank takes part in the gather even when its own set-up failed: a zeroed blob tells the others
    unsigned char flag_ok = ok ? 1 : 0;
    if (cudaMalloc((void **)&d_all, (size_t)129 * c->nranks + 129 + 16) != cudaSuccess) { cudaGetLastError(); return; }
    std::vector<unsigned char> sendv(129); memcpy(sendv.data(), mine, 128); sendv[128] = flag_ok;
    cudaMemcpyAsync(d_all + (size_t)129 * c->nranks, sendv.data(), 129, cudaMemcpyHostToDevice, c->stream);
    ncclResult_t r = g_nccl.AllGather(d_all + (size_t)129 * c->nranks, d_all, 129, ncclUint8, c->comm, c->stream);
    std::vector<unsigned char> recv((size_t)129 * c->nranks);
    cudaMemcpyAsync(recv.data(), d_all, recv.size(), cudaMemcpyDeviceToHost, c->stream);
    cudaStreamSynchronize(c->stream);
    bool all_ok = ok && r == ncclSuccess;
    for (int q = 0; q < c->nranks; q++) all_ok = all_ok && recv[(size_t)129 * q + 128] == 1;
    if (all_ok) {
        for (int q = 0; q < c->nranks && all_ok; q++) {
            if (q == c->rank) { c->peer_grad[q] = c->d_xgrad; c->peer_flags[q] = c->d_xflags; continue; }
            cudaIpcMemHandle_t pg, pf; memcpy(&pg, &recv[(size_t)129 * q], 64); memcpy(&pf, &recv[(size_t)129 * q + 64], 64);
            all_ok = cudaIpcOpenMemHandle((void **)&c->peer_grad[q], pg, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess &&
                     cudaIpcOpenMemHandle((void **)&c->peer_flags[q], pf, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
        }
    }
    // unanimous or not at all: a rank that could not map a peer must not leave the others waiting for its flags
    int32_t vote = all_ok ? 1 : 0, *d_vote = reinterpret_cast<int32_t *>(d_all + (((size_t)129 * c->nranks + 129 + 15) & ~(size_t)15) - 0);
    d_vote = reinterpret_cast<int32_t *>(d_all);     // the gather buffer is free again (cudaMalloc memory is 256-byte aligned)
    cudaMemcpyAsync(d_vote, &vote, 4, cudaMemcpyHostToDevice, c->stream);
    g_nccl.AllReduce(d_vote, d_vote, 1, ncclInt32, ncclMin, c->comm, c->stream);
    cudaMemcpyAsync(&vote, d_vote, 4, cudaMemcpyDeviceToHost, c->stream);
    cudaStreamSynchronize(c->stream);
    cudaFree(d_all);
    cudaGetLastError();
    if (vote == 1) { c->p2p = true; c->dp_step = 0; }
    else p2p_teardown(c);
}
int mz_comm_init(mz_ctx *c, int rank, int nranks, const uint8_t id[128]) {
    MZ_CHECK_CTX(c);
    if (!id || nranks < 1 || rank < 0 || rank >= nranks) return fail(c, MZ_E_ARG, "bad rank/nranks/id");
    if (!g_nccl.load()) return fail(c, MZ_E_NCCL, "cannot load libnccl.so.2: %s", dlerror());
    if (c->comm) { p2p_teardown(c); g_nccl.CommDestroy(c->comm); c->comm = nullptr; }
    ncclUniqueId u; memcpy(&u, id, 128);
    ncclResult_t r = g_nccl.CommInitRank(&c->comm, nranks, u, rank);
    if (r != ncclSuccess) { c->comm = nullptr; return fail(c, MZ_E_NCCL, "ncclCommInitRank: %s", g_nccl.GetErrorString(r)); }
    c->rank = rank; c->nranks = nranks;
    p2p_setup(c);
    return MZ_OK;
}
int mz_comm_destroy(mz_ctx *c) {
    MZ_CHECK_CTX(c);
    if (c->comm) { MZ_CUDA(c, cudaStreamSynchronize(c->stream)); p2p_teardown(c); g_nccl.CommDestroy(c->comm); c->comm = nullptr; }
    c->rank = 0; c->nranks = 1;
    return MZ_OK;
}
int mz_learner_path(mz_ctx *c, int grad_mode) { return c ? learner_path(c, grad_mode) : 0; }
// 0 = no communicator, 1 = ncclAllReduce + mz_k_adam, 2 = mz_k_dp_adam over peer memory (NVLink loads, fused with the update)
int mz_comm_mode(mz_ctx *c) { if (!c) return 0; return c->p2p ? 2 : c->comm ? 1 : 0; }

// ---- instrumentation ---------------------------------------------------------------------------------------------
int mz_launch_count(mz_ctx *c, int64_t *n) { if (!c || !n) return fail(c, MZ_E_ARG, "NULL"); *n = c->launches; return MZ_OK; }
int mz_kernel_time_reset(mz_ctx *c, int enable) {
    MZ_CHECK_CTX(c);
    collect_timings(c);
    for (int i = 0; i < 8; i++) { c->fam_ms[i] = 0; c->fam_n[i] = 0; }
    c->timing = enable != 0;
    return MZ_OK;
}
int mz_kernel_time(mz_ctx *c, int family, double *ms, int64_t *launches) {
    MZ_CHECK_CTX(c);
    if (family < 0 || family >= 8) return fail(c, MZ_E_ARG, "family out of range");
    collect_timings(c);
    if (ms) *ms = c->fam_ms[family];
    if (launches) *launches = c->fam_n[family];
    return MZ_OK;
}
int mz_phase_cycles(mz_ctx *c, uint64_t out[60]) {   // only meaningful in a -DMZ_PHASE_TIMERS build
    if (!c || !out) return fail(c, MZ_E_ARG, "NULL");
    MZ_CUDA(c, cudaMemcpyAsync(c->h_stats, c->d_stats, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    MZ_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 60; i++) out[i] = (uint64_t)c->h_stats[4 + i];
    return MZ_OK;
}
int mz_search_stats(mz_ctx *c, double *mean_legal, double *mean_depth) {
    if (!c) return fail(nullptr, MZ_E_ARG, "ctx is NULL");
    if (mean_legal) *mean_legal = c->last_mean_legal;
    if (mean_depth) *mean_depth = c->last_mean_depth;
    return MZ_OK;
}

}  // extern "C"
