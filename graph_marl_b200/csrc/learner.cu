// learner.cu -- the device pieces of the batched DQN learner's update (graph_marl_b200/learner.py) and of sl.py's
// supervised update (graph_marl_b200/sl_trainer.py):
//
//   gm_td_grad         one-step TD error of tools/train_simple.py:107-110 (the reference's main.py learner):
//                      y = r + (!done) * gamma * max_a q_next,  loss += scale * sum (q[a] - y)^2,  dq = 2 scale (q - y) at a
//   gm_sl_mse_grad     sl.py:395-400's MSE of the all-pairs prediction against the shortest-path weights:
//                      loss += scale * sum (pred - y)^2,  d_pred = 2 scale (pred - y)
//   gm_optimizer_step  clip_grad_value_ + clip_grad_norm_ + AdamW(foreach=False) + interpolate_model (main.py:1007-1020)
//
// All three reduce with fixed-order partials (no float atomics), so a replayed CUDA graph computes what an eager call computes,
// bit for bit, and they keep their scalars (loss, step count) in device memory, so the launches can be captured.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace gm {

constexpr int kRedThreads = 256;
constexpr int kTdMaxBlocks = GM_LEARNER_PARTIALS;

// fixed-order block sum: warp shuffles, then the warp totals in warp order
__device__ inline double block_sum(double v, double* sh) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(FULL, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += sh[i];
    __syncthreads();
    return t;  // valid in thread 0
}

__global__ void __launch_bounds__(kRedThreads) td_grad_kernel(const float* __restrict__ q, const float* __restrict__ q_next,
                                                               const int64_t* __restrict__ action, const float* __restrict__ reward,
                                                               const uint8_t* __restrict__ done, int64_t R, int nA, float gamma,
                                                               float scale, float* __restrict__ dq, double* __restrict__ partials) {
    __shared__ double sh[kRedThreads / 32];
    double acc = 0.0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        const float* qn = q_next + r * nA;
        // max over actions that propagates a NaN like torch.max (fmaxf would drop it)
        float m = qn[0];
        for (int a = 1; a < nA; a++) {
            const float v = qn[a];
            if (v > m || isnan(v)) m = isnan(m) ? m : v;
        }
        // torch: reward + ((~done) * gamma) * next_q_max, each operation rounded to fp32
        const float y = __fadd_rn(reward[r], __fmul_rn(done[r] ? 0.f : gamma, m));
        const int act = (int)action[r];
        for (int a = 0; a < nA; a++) {
            float g = 0.f;
            if (a == act) {
                const float d = __fsub_rn(q[r * nA + a], y);
                acc += (double)d * (double)d;
                g = __fmul_rn(__fmul_rn(2.f, scale), d);
            }
            dq[r * nA + a] = g;
        }
    }
    const double s = block_sum(acc, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

// sl.py's all-pairs distance loss (sl.py:395-400): row b*N + v of pred against targets_all[index[b], v, :], the targets
// read from the dataset through the sample index (no gathered target batch).  One thread per (row, column) element, so
// a warp reads consecutive columns of a prediction row and of a target row.  The element's (b, v, u) advance by the
// grid stride's digits in base N, so the loop divides nothing (a 64-bit division is a call that spills).
__global__ void __launch_bounds__(kRedThreads) sl_mse_grad_kernel(const float* __restrict__ pred, int64_t ldp,
                                                                   const int32_t* __restrict__ targets_all,
                                                                   const int64_t* __restrict__ index, int64_t total, int N,
                                                                   float scale, float* __restrict__ d_pred,
                                                                   double* __restrict__ partials) {
    __shared__ double sh[kRedThreads / 32];
    double acc = 0.0;
    const float g2 = __fmul_rn(2.f, scale);
    const int start = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;  // < 2^31: grid <= partials
    int u = start % N, v = (start / N) % N;
    int64_t b = start / N / N;
    const int du = stride % N, dv = (stride / N) % N, db = stride / N / N;
    for (int64_t i = start; i < total; i += stride) {
        const int64_t r = b * N + v;  // prediction row
        const int64_t s = index ? index[b] : b;
        const float y = (float)targets_all[(s * N + v) * N + u];
        const float d = __fsub_rn(pred[r * ldp + u], y);
        acc += (double)d * (double)d;
        if (d_pred) d_pred[r * ldp + u] = __fmul_rn(g2, d);
        u += du;
        int carry = 0;
        if (u >= N) u -= N, carry = 1;
        v += dv + carry;
        if (v >= N) v -= N, b++;
        b += db;
    }
    const double t = block_sum(acc, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = t;
}

__global__ void td_loss_kernel(const double* __restrict__ partials, int n, double scale, float* __restrict__ loss) {
    if (threadIdx.x) return;
    double s = 0.0;
    for (int i = 0; i < n; i++) s += partials[i];
    *loss = (float)((double)*loss + s * scale);
}

// ---- optimizer -------------------------------------------------------------------------------------------------------
// pass 1: clamp every gradient to +-clip_value in place (clip_grad_value_), per-block sums of squares of the result
__global__ void __launch_bounds__(kRedThreads) clip_value_kernel(const gm_opt_entry* __restrict__ table, int n, float clip,
                                                                  double* __restrict__ partials, int64_t* __restrict__ step) {
    __shared__ double sh[kRedThreads / 32];
    double acc = 0.0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int e = 0; e < n; e++) {
        float* g = table[e].grad;
        const int64_t numel = table[e].numel;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < numel; i += stride) {
            const float v = fminf(fmaxf(g[i], -clip), clip);
            g[i] = v;
            acc += (double)v * (double)v;
        }
    }
    const double s = block_sum(acc, sh);
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = s;
        if (blockIdx.x == 0) *step += 1;
    }
}

// pass 2: every block sums the partials in the same order (identical norm everywhere), then clip_grad_norm_'s scaling and
// the AdamW update of torch.optim.AdamW(foreach=False) (_single_tensor_adamw), operation by operation in fp32 with the
// Python-side scalars (bias corrections, step size) formed in double and rounded to fp32 where torch rounds them
__global__ void __launch_bounds__(kRedThreads) adamw_kernel(const gm_opt_entry* __restrict__ table, int n,
                                                             const double* __restrict__ partials, int n_partials,
                                                             const int64_t* __restrict__ step, gm_opt_hparams h) {
    __shared__ float coef_s;
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < n_partials; i++) s += partials[i];
        const float norm = (float)sqrt(s);
        const float c = __fdiv_rn(h.max_norm, __fadd_rn(norm, 1e-6f));
        coef_s = fminf(c, 1.f);
    }
    __syncthreads();
    const float coef = coef_s;
    const double t = (double)*step;
    const double bc1 = 1.0 - pow((double)h.beta1, t), bc2 = 1.0 - pow((double)h.beta2, t);
    const float step_size = (float)(h.lr / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const float decay = (float)(1.0 - h.lr * h.weight_decay);
    const float w1 = (float)(1.0 - h.beta1), b2 = (float)h.beta2, w2 = (float)(1.0 - h.beta2), eps = (float)h.eps;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int e = 0; e < n; e++) {
        const gm_opt_entry E = table[e];
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < E.numel; i += stride) {
            const float g = __fmul_rn(E.grad[i], coef);
            E.grad[i] = g;
            const float p = __fmul_rn(E.param[i], decay);
            // exp_avg.lerp_(grad, w1), w1 < 0.5: self + w1 * (end - self)
            float m = E.exp_avg[i];
            m = __fadd_rn(m, __fmul_rn(w1, __fsub_rn(g, m)));
            // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
            float v = __fmul_rn(E.exp_avg_sq[i], b2);
            v = __fadd_rn(v, __fmul_rn(w2, __fmul_rn(g, g)));
            const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), eps);
            E.param[i] = __fadd_rn(p, __fmul_rn(-step_size, __fdiv_rn(m, denom)));
            E.exp_avg[i] = m;
            E.exp_avg_sq[i] = v;
        }
    }
}

// pass 3: target <- tau * online + (1 - tau) * target (util.interpolate_model)
__global__ void polyak_kernel(const gm_opt_pair* __restrict__ pairs, int n, float tau, float one_minus_tau) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int e = 0; e < n; e++) {
        const gm_opt_pair P = pairs[e];
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P.numel; i += stride)
            P.target[i] = __fadd_rn(__fmul_rn(tau, P.online[i]), __fmul_rn(one_minus_tau, P.target[i]));
    }
}

}  // namespace gm

using namespace gm;

extern "C" {

int gm_td_grad(const float* q, const float* q_next, const int64_t* action, const float* reward, const uint8_t* done,
               int64_t rows, int32_t n_actions, float gamma, float scale, float* dq, float* loss, double* partials,
               void* stream) {
    GM_CHECK_ARG(q && q_next && action && reward && done && dq && loss && partials, "gm_td_grad: null pointer");
    GM_CHECK_ARG(rows > 0 && n_actions > 0, "gm_td_grad: %lld rows x %d actions", (long long)rows, n_actions);
    const int blocks = (int)std::min<int64_t>((rows + kRedThreads - 1) / kRedThreads, kTdMaxBlocks);
    td_grad_kernel<<<blocks, kRedThreads, 0, (cudaStream_t)stream>>>(q, q_next, action, reward, done, rows, n_actions, gamma,
                                                                     scale, dq, partials);
    GM_LAUNCH_CHECK();
    td_loss_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(partials, blocks, (double)scale, loss);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int gm_sl_mse_grad(const float* pred, int64_t ldp, const int32_t* targets_all, const int64_t* index, int32_t B, int32_t N,
                   float scale, float* d_pred, float* loss, double* partials, void* stream) {
    GM_CHECK_ARG(pred && targets_all && loss && partials, "gm_sl_mse_grad: null pointer");
    GM_CHECK_ARG(B >= 1 && N >= 1 && ldp >= N, "gm_sl_mse_grad: %d samples x %d nodes, row stride %lld", B, N,
                 (long long)ldp);
    const int64_t total = (int64_t)B * N * N;
    const int blocks = (int)std::min<int64_t>((total + kRedThreads - 1) / kRedThreads, kTdMaxBlocks);
    sl_mse_grad_kernel<<<blocks, kRedThreads, 0, (cudaStream_t)stream>>>(pred, ldp, targets_all, index, total, N, scale,
                                                                         d_pred, partials);
    GM_LAUNCH_CHECK();
    td_loss_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(partials, blocks, (double)scale, loss);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int gm_optimizer_step(const gm_opt_entry* table_dev, int32_t n_entries, const gm_opt_pair* pairs_dev, int32_t n_pairs,
                      int64_t* step_dev, const gm_opt_hparams* h, double* partials, void* stream) {
    GM_CHECK_ARG(table_dev && step_dev && h && partials && n_entries > 0 && n_pairs >= 0 && (pairs_dev || !n_pairs),
                 "gm_optimizer_step: bad arguments");
    GM_CHECK_ARG(h->clip_value >= 0.f && h->max_norm > 0.f, "gm_optimizer_step: clip value %g / max norm %g",
                 (double)h->clip_value, (double)h->max_norm);
    cudaStream_t s = (cudaStream_t)stream;
    const int blocks = GM_LEARNER_PARTIALS;
    clip_value_kernel<<<blocks, kRedThreads, 0, s>>>(table_dev, n_entries, h->clip_value, partials, step_dev);
    GM_LAUNCH_CHECK();
    adamw_kernel<<<blocks, kRedThreads, 0, s>>>(table_dev, n_entries, partials, blocks, step_dev, *h);
    GM_LAUNCH_CHECK();
    if (n_pairs) {
        polyak_kernel<<<kNumSMs, kRedThreads, 0, s>>>(pairs_dev, n_pairs, (float)h->tau, (float)(1.0 - h->tau));
        GM_LAUNCH_CHECK();
    }
    return GM_OK;
}

}  // extern "C"
