// mz_learner.cuh -- replay sampling + target construction (get_batch, src/ReplayBuffer.jl:188-217) as a gather
// kernel, the K-step unroll forward (src/Learning.jl:347-374), the loss (:261-288) and the ADAM update (:382-397).
#pragma once
#include "mz_kernels.cuh"

struct mz_batch {   // get_batch's tuple (ReplayBuffer.jl:216), device arrays
    int32_t *index;   // [B][2] (game key, position)
    float *obs;       // [B][stack]
    float *actions;   // [B][K+1]
    float *values;    // [B][K+1]
    float *rewards;   // [B][K+1]
    float *policies;  // [B][K+1][A]
    float *gscale;    // [B]
    float *weights;   // [B] importance-sampling weights (conf.PER; ReplayBuffer.jl:213-215), else unused
};

// One CTA per batch element.  Thread 0 draws (game, position) (sample_n_games :102-104, sample_position :80;
// Philox(seed, REPLAY, step, b)) and builds the targets (make_target :25-50, Q17-Q18); all threads then gather
// the stacked observation and the policy rows.
__global__ void __launch_bounds__(64) mz_k_replay_gather(const __grid_constant__ mz_params P, mz_ring r, uint64_t step, int B, mz_batch out) {
    __shared__ int s_pos, s_T; __shared__ int64_t s_ring;
    const int b = blockIdx.x, tid = threadIdx.x, K1 = P.K + 1;
    if (b >= B) return;
    if (tid == 0) {
        int64_t played = r.counters[0];
        int64_t n_games = played < r.capacity ? played : r.capacity;
        int64_t first_key = played - n_games + 1;
        mz_u4 q = mz_philox(P.seed, MZ_STREAM_REPLAY, (uint32_t)step, (uint32_t)b, 0, 0);
        int64_t gi; int pos, T; int64_t key, ring;
        if (P.per) {   // sample_n_games :90-100 / sample_position :75-79 by priority: inverse CDF over the exact integer prefix sums
            const unsigned long long Q = (unsigned long long)r.counters[6];
            const unsigned long long t = __umul64hi(((unsigned long long)q.x << 32) | q.z, Q);
            int64_t lo = 0, hi = n_games - 1;
            while (lo < hi) { int64_t mid = (lo + hi) >> 1; if (r.prefix[mid] > t) hi = mid; else lo = mid + 1; }
            gi = lo; key = first_key + gi; ring = (key - 1) % r.capacity; T = r.T[ring];
            const uint32_t *qp = r.q_pos + (size_t)ring * P.Tmax;
            unsigned long long Qg = 0; for (int i = 0; i < T; i++) Qg += qp[i];
            const unsigned long long t2 = __umul64hi(((unsigned long long)q.y << 32) | q.w, Qg);
            unsigned long long a2 = 0;
            for (pos = 1; pos < T; pos++) { a2 += qp[pos - 1]; if (a2 > t2) break; }
            const float game_prob = (float)((double)r.q_game[ring] / (double)Q), pos_prob = (float)((double)qp[pos - 1] / (double)Qg);
            out.weights[b] = 1.0f / (((float)r.counters[2] * game_prob) * pos_prob);      // :213 (total_samples)
        } else {
            gi = (int64_t)mz_u32_below(q.x, (uint32_t)n_games);
            key = first_key + gi; ring = (key - 1) % r.capacity; T = r.T[ring];
            pos = 1 + (int)mz_u32_below(q.y, (uint32_t)T);
        }
        s_pos = pos; s_T = T; s_ring = ring;
        out.index[2 * b] = (int32_t)key; out.index[2 * b + 1] = pos;
        int gs = T + 1 - pos; if (P.K < gs) gs = P.K;                      // :212
        out.gscale[b] = (float)gs;
    }
    __syncthreads();
    const int pos = s_pos, T = s_T; const int64_t ring = s_ring;
    // make_target (:25-50, Q17-Q18): the K + 1 unroll positions are independent of each other: one thread each
    for (int k = tid; k < K1; k += 64) {
        const float *rew = r.h_reward + (size_t)ring * P.Tmax; const uint8_t *tp = r.h_to_play + (size_t)ring * P.Tmax;
        const float *rv = (r.reanalysed[ring] ? r.h_rrv : r.h_rv) + (size_t)ring * P.Tmax;   // ReplayBuffer.jl:8
        const int32_t *act = r.h_action + (size_t)ring * P.Tmax;
        int ci = pos + k; float tv, tr; int a;
        if (ci < T) { tv = mz_target_value(P, T, rew, tp, rv, ci); tr = rew[ci - 1]; a = act[ci - 1]; }
        else if (ci == T) { tv = 0.0f; tr = rew[ci - 1]; a = act[ci - 1]; }
        else { tv = 0.0f; tr = 0.0f; a = 1 + (int)mz_u32_below(mz_philox(P.seed, MZ_STREAM_ABSORB, (uint32_t)step, (uint32_t)b, (uint32_t)k, 0).x, (uint32_t)P.A); }
        out.values[(size_t)b * K1 + k] = tv; out.rewards[(size_t)b * K1 + k] = tr; out.actions[(size_t)b * K1 + k] = (float)a;
    }
    for (int k = tid; k < P.stack_size; k += 64)                            // :207
        out.obs[(size_t)b * P.stack_size + k] = mz_stacked_value(P, r.h_p1 + (size_t)ring * P.Tmax, r.h_p2 + (size_t)ring * P.Tmax,
                                                                 r.h_action + (size_t)ring * P.Tmax, pos, k);
    for (int i = tid; i < K1 * P.A; i += 64) {
        int k = i / P.A, a = i % P.A, ci = pos + k;
        out.policies[((size_t)b * K1 + k) * P.A + a] = ci < T ? r.h_cv[((size_t)ring * P.Tmax + ci - 1) * P.A + a] : 1.0f / (float)P.A;
    }
}

// weight_batch ./= maximum(weight_batch) (ReplayBuffer.jl:215); the maximum is order independent
__global__ void __launch_bounds__(1024) mz_k_per_normalise(int B, float *w) {
    __shared__ float red[1024];
    const int tid = threadIdx.x;
    float m = 0.0f;
    for (int i = tid; i < B; i += 1024) m = fmaxf(m, w[i]);
    red[tid] = m; __syncthreads();
    for (int s = 512; s > 0; s >>= 1) { if (tid < s) red[tid] = fmaxf(red[tid], red[tid + s]); __syncthreads(); }
    const float mx = red[0];
    for (int i = tid; i < B; i += 1024) w[i] = w[i] / mx;
}

// K-step unroll forward for 32 samples per CTA (src/Learning.jl:347-370, Q19): row 0 = prediction(h0); for
// i = 1..K: row i = prediction(h_{i-1}) evaluated BEFORE the dynamics step; rewards row 0 = 0.
struct mz_learn_args { const float *wglob; int32_t B, max_dim, max_layer_floats, pad_; mz_batch batch; float *pred_values, *pred_rewards, *pred_policies; };
template <bool BN = false>
__global__ void __launch_bounds__(MZ_THREADS) mz_k_learn_forward(const __grid_constant__ mz_params P, const mz_learn_args a) {
    extern __shared__ __align__(128) unsigned char mz_smem[];
    const mz_smem_plan sp = mz_smem_carve(mz_smem, a.max_dim, a.max_layer_floats, P.hidden_pad, P.S);
    const int tid = threadIdx.x, K1 = P.K + 1;
    const int64_t g = (int64_t)blockIdx.x * MZ_ROWS + tid;
    const bool row_ok = tid < MZ_ROWS && g < a.B;
    mz_nn_pipe pipe;
    mz_pipe_init(pipe, sp, a.wglob);
    mz_zero_activations(sp, a.max_dim);
    __syncthreads();
    const int pred_first = P.nets[1].first, dyn_first = P.nets[2].first;
    if (tid == 0) mz_nn_issue(pipe, P, P.nets[0].first, 0);
    if (tid == MZ_GROUP && P.K > 0) mz_nn_issue(pipe, P, dyn_first, 0);
    for (int i = tid; i < MZ_ROWS * P.stack_size; i += MZ_THREADS) {
        int r = i / P.stack_size, k = i % P.stack_size;
        int64_t gg = (int64_t)blockIdx.x * MZ_ROWS + r;
        sp.in0[k * MZ_ROWS + r] = gg < a.B ? a.batch.obs[gg * P.stack_size + k] : 0.0f;
    }
    __syncthreads();
    // representation (:347) then row 0 = prediction(h0) (:351) on group 0; in1 keeps the current hidden state
    if (pipe.grp == 0) {
        mz_nn_net<BN>(pipe, P, 0, pred_first, sp.in0, sp.bufT[0], sp.in1, nullptr, sp.t0[0], sp.t1[0]);
        mz_nn_net<BN>(pipe, P, 1, P.K > 0 ? pred_first : -1, sp.in1, sp.bufT[0], sp.outV, sp.outL, sp.t0[0], sp.t1[0]);
    }
    __syncthreads();
    for (int i = 0; i <= P.K; i++) {
        if (row_ok) {   // store row i of the predictions (value/policy from prediction, reward from the dynamics step before it)
            float logits[MZ_MAX_A], policy[MZ_MAX_A];
            for (int k = 0; k < P.A; k++) logits[k] = sp.outL[k * MZ_ROWS + tid];
            mz_softmax(logits, P.A, policy);
            a.pred_values[g * K1 + i] = sp.outV[tid];
            for (int k = 0; k < P.A; k++) a.pred_policies[(g * K1 + i) * P.A + k] = policy[k];
            a.pred_rewards[g * K1 + i] = i == 0 ? 0.0f : sp.outR[tid];                              // :352 zeros for row 0
        }
        if (i == P.K) break;
        // unroll step i+1 (:355-370, Q19): prediction(h_i) is evaluated BEFORE the dynamics step, on the same h_i that
        // dynamics consumes, so the two networks run concurrently on the two groups.
        // make_dynamics_input (:293-304): state * 2 (copy), action plane = Float32(a) / A
        if (row_ok) {
            float plane = a.batch.actions[g * K1 + i] / (float)P.A;
            for (int k = 0; k < P.hidden; k++) sp.in0[k * MZ_ROWS + tid] = sp.in1[k * MZ_ROWS + tid] * 2.0f;
            for (int k = P.obs_size; k < P.sa_size; k++) sp.in0[k * MZ_ROWS + tid] = plane;
        }
        __syncthreads();
        const bool more = i + 1 < P.K;
        if (pipe.grp == 0) mz_nn_net<BN>(pipe, P, 1, more ? pred_first : -1, sp.in1, sp.bufT[0], sp.outV, sp.outL, sp.t0[0], sp.t1[0]);   // :356
        else               mz_nn_net<BN>(pipe, P, 2, more ? dyn_first : -1, sp.in0, sp.bufT[1], sp.outH, sp.outR, sp.t0[1], sp.t1[1]);     // :362
        __syncthreads();
        for (int k = tid; k < P.hidden * MZ_ROWS; k += MZ_THREADS) sp.in1[k] = sp.outH[k];          // h_{i+1}
        __syncthreads();
    }
}

// loss (src/Learning.jl:261-288, Q21): per-sample partial sums.  Block = 32 samples x up to 16 unroll rows: every (sample, row) term is
// computed by its own thread, then the sample's thread adds the rows in row order (the same sums as a loop over the rows).
#define MZ_LOSS_RY 16
__global__ void __launch_bounds__(32 * MZ_LOSS_RY) mz_k_loss_rows(const __grid_constant__ mz_params P, int B, mz_batch batch, const float *pv, const float *pr, const float *pp,
                                                                 float *row_v, double *row_r, float *row_p, float *row_invg) {
    __shared__ float t_v[40][32], t_p[40][32];
    __shared__ double t_r[40][32];
    const int b = blockIdx.x * 32 + threadIdx.x;
    const int K1 = P.K + 1, A = P.A;
    if (b < B) {
        for (int k = threadIdx.y; k < K1; k += blockDim.y) {
            const float d = pv[(size_t)b * K1 + k] - batch.values[(size_t)b * K1 + k];
            t_v[k][threadIdx.x] = d * d;
            const double dr = (double)pr[(size_t)b * K1 + k] - (double)batch.rewards[(size_t)b * K1 + k];
            t_r[k][threadIdx.x] = dr * dr;
            const float *p = pp + ((size_t)b * K1 + k) * A, *y = batch.policies + ((size_t)b * K1 + k) * A;
            float mx = p[0];
            for (int i = 1; i < A; i++) mx = p[i] > mx ? p[i] : mx;
            float se = 0.0f;
            for (int i = 0; i < A; i++) se = se + mz_expf(p[i] - mx);
            float lse = mz_logf(se), acc = 0.0f;
            for (int i = 0; i < A; i++) acc = acc + y[i] * ((p[i] - mx) - lse);   // logitcrossentropy on ALREADY softmaxed P
            t_p[k][threadIdx.x] = -acc;
        }
    }
    __syncthreads();
    if (b >= B || threadIdx.y != 0) return;
    float sv = 0.0f, spol = 0.0f; double sr = 0.0;
    for (int k = 0; k < K1; k++) { sv = sv + t_v[k][threadIdx.x]; sr = sr + t_r[k][threadIdx.x]; spol = spol + t_p[k][threadIdx.x]; }
    float gs = batch.gscale[b];
    if (P.per && batch.weights) {   // (sum ./ gradient_scale) .* weight_batch (Learning.jl:272-281)
        const float w = batch.weights[b];
        row_v[b] = (sv / gs) * w; row_r[b] = (sr / (double)gs) * (double)w; row_p[b] = spol; row_invg[b] = (1.0f / gs) * w;
    } else { row_v[b] = sv / gs; row_r[b] = sr / (double)gs; row_p[b] = spol; row_invg[b] = 1.0f / gs; }
}
// deterministic single-CTA tree reductions: out[0] = sum row_v, out[1] = sum row_p, out[2] = sum row_invg, out[3] = sum row_r,
// out[4..6] = sum(theta^2) per net (double accumulation; compared against the oracle with a stated tolerance)
__global__ void __launch_bounds__(1024) mz_k_loss_reduce(const __grid_constant__ mz_params P, int B, const float *row_v, const double *row_r,
                                                          const float *row_p, const float *row_invg, const float *theta, double *out, int nwhat = 7) {
    __shared__ double red[1024];
    const int tid = threadIdx.x;
    // one CTA per quantity (grid = 7): the seven reductions are independent; each keeps its own fixed summation tree
    for (int what = blockIdx.x; what < nwhat; what += gridDim.x) {   // nwhat = 4: the data terms only (mz_k_sqnorm_masked adds the rest)
        double acc = 0.0;
        if (what < 4) {
            for (int i = tid; i < B; i += 1024) acc += what == 0 ? (double)row_v[i] : what == 1 ? (double)row_p[i] : what == 2 ? (double)row_invg[i] : row_r[i];
        } else {
            const mz_net &N = P.nets[what - 4];
            int l0 = N.first, l1 = N.first + N.n_trunk + N.n_h1 + N.n_h2;
            int lo = P.layers[l0].w_off, hi = P.layers[l1 - 1].b_off + P.layers[l1 - 1].out_pad;
            for (int i = lo + tid; i < hi; i += 1024) { double t = (double)theta[i]; acc += t * t; }   // pad entries are zero
        }
        red[tid] = acc; __syncthreads();
        for (int s = 512; s > 0; s >>= 1) { if (tid < s) red[tid] += red[tid + s]; __syncthreads(); }
        if (tid == 0) out[what] = red[0];
        __syncthreads();
    }
}

// Gradients.  MZ_GRAD_REFERENCE_L2: the reference computes its predictions outside Zygote.pullback
// (Learning.jl:347-374 vs 385-393), so the gradient of every parameter array is that of sum(abs2, theta): 2*theta (Q20) over Flux.params
// (dense / conv weights and biases, BatchNorm beta / gamma), 0 for the BatchNorm running statistics.  mask: 1 = Flux parameter (NULL = all).
__global__ void mz_k_l2_grad(int n, const float *theta, const unsigned char *mask, float *grad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) grad[i] = (!mask || mask[i]) ? theta[i] + theta[i] : 0.0f;
}
// out[4 + net] = sum of theta^2 over the Flux parameters of each network, net = [b_net, b_net+1) (one CTA per network, double accumulation)
__global__ void __launch_bounds__(1024) mz_k_sqnorm_masked(int b0, int b1, int b2, int b3, const float *theta, const unsigned char *mask, double *out) {
    __shared__ double red[1024];
    const int tid = threadIdx.x, lo = blockIdx.x == 0 ? b0 : blockIdx.x == 1 ? b1 : b2, hi = blockIdx.x == 0 ? b1 : blockIdx.x == 1 ? b2 : b3;
    double acc = 0.0;
    for (int i = lo + tid; i < hi; i += 1024) if (mask[i]) { const double t = (double)theta[i]; acc += t * t; }
    red[tid] = acc; __syncthreads();
    for (int s = 512; s > 0; s >>= 1) { if (tid < s) red[tid] += red[tid + s]; __syncthreads(); }
    if (tid == 0) out[4 + blockIdx.x] = red[0];
}
// Flux.ADAM apply! + update! (Q22): Float32 state, Float64 arithmetic inside the broadcast, beta powers beta^t.
__global__ void mz_k_adam(int n, float *theta, float *m, float *v, const float *grad, double eta, double bp1, double bp2, float grad_scale) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
    float g = grad[i] * grad_scale;
    float mi = (float)(b1 * (double)m[i] + (1.0 - b1) * (double)g);
    float vi = (float)(b2 * (double)v[i] + (1.0 - b2) * (double)(g * g));
    m[i] = mi; v[i] = vi;
    float delta = (float)((double)mi / (1.0 - bp1) / (sqrt((double)vi / (1.0 - bp2)) + eps) * eta);
    theta[i] = theta[i] - delta;
}

// MZ_GRAD_REFERENCE_L2 on one GPU: the gradient is 2 * theta over Flux.params (Q20), so mz_k_l2_grad + mz_k_adam are one kernel (a B = 32 step is
// bound by its launches).  Same arithmetic, same bits; the gradient is still written out.  mask: as in mz_k_l2_grad.
__global__ void mz_k_adam_l2(int n, float *theta, float *m, float *v, float *grad, const unsigned char *mask, double eta, double bp1, double bp2) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
    const float th = theta[i];
    const float g = (!mask || mask[i]) ? th + th : 0.0f;
    grad[i] = g;
    float mi = (float)(b1 * (double)m[i] + (1.0 - b1) * (double)g);
    float vi = (float)(b2 * (double)v[i] + (1.0 - b2) * (double)(g * g));
    m[i] = mi; v[i] = vi;
    float delta = (float)((double)mi / (1.0 - bp1) / (sqrt((double)vi / (1.0 - bp2)) + eps) * eta);
    theta[i] = th - delta;
}

// Data-parallel update over peer memory: every rank's gradient lies in a buffer that all ranks have mapped (CUDA IPC, NVLink / NVSwitch).
// One kernel: announce "my gradient of step s is complete" in every peer's flag block, wait until every peer has announced the same,
// then each thread sums its element over the ranks IN RANK ORDER (so all ranks compute bit-identical sums) with loads straight from the
// peers' memory and applies Flux.ADAM (mz_k_adam's arithmetic).  Replaces ncclAllReduce + mz_k_adam: the 300 KB exchange is latency
// bound, and here it costs one flag round trip plus nranks - 1 remote loads per thread instead of a ring of launches.
// Buffers are double-buffered by step parity: a rank can only be one barrier ahead of a peer, so the half it overwrites at step s + 2
// is no longer read by anyone.
#define MZ_DP_MAX_RANKS 8
struct mz_dp_args { int32_t rank, nranks, n; uint32_t step; const float *peer_grad[MZ_DP_MAX_RANKS]; uint32_t *peer_flags[MZ_DP_MAX_RANKS]; uint32_t *flags_local; };
__global__ void __launch_bounds__(256) mz_k_dp_adam(float *theta, float *m, float *v, const __grid_constant__ mz_dp_args a, double eta, double bp1, double bp2, float grad_scale) {
    if (blockIdx.x == 0 && (int)threadIdx.x < a.nranks) {              // the local gradient was written by earlier kernels of this stream
        __threadfence_system();
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.peer_flags[threadIdx.x] + a.rank), "r"(a.step) : "memory");
    }
    if ((int)threadIdx.x < a.nranks) {
        uint32_t seen = 0, spin = 0;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.flags_local + threadIdx.x) : "memory");
            if (++spin > (1u << 28)) __trap();                          // a rank that never arrives must fault the kernel, not hang the GPU
        } while ((int32_t)(seen - a.step) < 0);
    }
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    float pv[MZ_DP_MAX_RANKS];                                          // all remote loads in flight before the first add
#pragma unroll
    for (int r = 0; r < MZ_DP_MAX_RANKS; r++) pv[r] = r < a.nranks ? __ldcv(a.peer_grad[r] + i) : 0.0f;
    float g = 0.0f;
#pragma unroll
    for (int r = 0; r < MZ_DP_MAX_RANKS; r++) if (r < a.nranks) g = g + pv[r];
    g = g * grad_scale;
    const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
    const float mi = (float)(b1 * (double)m[i] + (1.0 - b1) * (double)g);
    const float vi = (float)(b2 * (double)v[i] + (1.0 - b2) * (double)(g * g));
    m[i] = mi; v[i] = vi;
    const float delta = (float)((double)mi / (1.0 - bp1) / (sqrt((double)vi / (1.0 - bp2)) + eps) * eta);
    theta[i] = theta[i] - delta;
}

// ---- ResNet learner (reference_l2): glue kernels around the batched network kernel mz_k_rn_forward --------------------------------
// make_dynamics_input (Learning.jl:293-304) for the (W,H,num_filters) state: sa[b] = [2 * h[b] | action plane = Float32(a) / A]
__global__ void mz_k_rn_make_sa(int B, int hidden, int cells, int A, int K1, int step, const float *h, const float *actions, float *sa) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, sz = hidden + cells;
    if (i >= B * sz) return;
    const int b = i / sz, j = i - b * sz;
    sa[i] = j < hidden ? h[(size_t)b * hidden + j] * 2.0f : actions[(size_t)b * K1 + step] / (float)A;
}
// one row of the unroll's predictions: value + policy of prediction(h) into rows `row` (and `row2` if >= 0: rows 0 and 1 share prediction(h_0),
// Q19) when v != nullptr; the reward of the dynamics step into row `row` when r != nullptr; rzero: rewards of row 0 are 0 (Learning.jl:352)
__global__ void mz_k_rn_scatter(int B, int A, int K1, int row, int row2, const float *v, const float *pol, const float *r, int rzero, float *pv, float *pp, float *pr) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (v) for (int q = 0; q < 2; q++) {
        const int rw = q == 0 ? row : row2;
        if (rw < 0) continue;
        pv[(size_t)b * K1 + rw] = v[b];
        for (int k = 0; k < A; k++) pp[((size_t)b * K1 + rw) * A + k] = pol[(size_t)b * A + k];
    }
    if (r) pr[(size_t)b * K1 + row] = r[b];
    if (rzero) pr[(size_t)b * K1] = 0.0f;
}
