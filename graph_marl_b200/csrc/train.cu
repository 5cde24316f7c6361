// train.cu -- training path of the hot modules: forward with a tape + hand-written backward kernels (SURVEY 8f-1).
//
// Reference: the learner of src/main.py:830-1006 and src/sl.py:366-428 differentiates NetMon
// (src/model.py:451-631: MLP encoder :32-42, nn.LSTMCell :491/:543, SimpleAggregation :213-229, neighbour readout
// :582-622) and the DQN (:199-203) with torch autograd.  Here the same derivatives are explicit CUDA kernels driven
// by two C-ABI calls per module (gm_*_forward_train writes a tape of activations, gm_*_backward consumes it), which
// graph_marl_b200/model.py wraps as torch.autograd.Function so that `loss.backward()` of the unmodified drivers runs
// them; sequences (<= 16 steps, main.py:840-915) unroll as a chain of those nodes with the state gradient handed
// from step to step on the device.
//
// Arithmetic: forward GEMMs go through linear_dispatch (fp32 FFMA or tcgen05 bf16x3, as the module's math mode says);
// the backward GEMMs dX = dZ W and dW = dZ^T X are fp32 FFMA kernels of this file (no operand transposes), so
// gradients match torch autograd to summation-order noise (tests/test_gpu_backward.py, rtol 1e-4).
//
// Built for rnn_type lstm with carry-over, agg sum | mean, neighbour readout, no global readout; every other
// configuration is reported as GM_ERR_INVALID and differentiated by the torch-composed path of model.py.
#include <algorithm>

#include "common.cuh"
#include "linear_simt.cuh"
#include "netmon_rows.cuh"

namespace gm {

int linear_dispatch(const LinearArgs& a, int math, void* ws, int64_t ws_bytes, cudaStream_t s);  // gemm_dispatch.cu

// ---------------------------------------------------------------------------------------
// fp32 GEMMs of the backward pass (64 x 64 output tile, 256 threads, 4 x 4 per thread, 16-deep chunks)
// ---------------------------------------------------------------------------------------
constexpr int BT = 64, BKC = 16;

// C[M,K] (+)= A[M,N] W[N,K]          (dX = dZ W: W in its nn.Linear [out, in] layout, no transpose)
__global__ void __launch_bounds__(256) gemm_nn_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ W, int64_t ldw,
                                                      float* __restrict__ C, int64_t ldc, int64_t M, int N, int K, int accumulate) {
    __shared__ float As[BKC][BT + 1];
    __shared__ float Ws[BKC][BT];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t m0 = (int64_t)blockIdx.y * BT;
    const int k0 = blockIdx.x * BT;
    float acc[4][4] = {};
    for (int n0 = 0; n0 < N; n0 += BKC) {
        for (int t = threadIdx.x; t < BT * BKC; t += 256) {
            const int r = t / BKC, c = t % BKC;  // A tile: 64 rows x 16 cols
            const int64_t m = m0 + r;
            As[c][r] = (m < M && n0 + c < N) ? A[m * lda + n0 + c] : 0.f;
            const int wr = t / BT, wc = t % BT;  // W tile: 16 rows x 64 cols
            Ws[wr][wc] = (n0 + wr < N && k0 + wc < K) ? W[(int64_t)(n0 + wr) * ldw + k0 + wc] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int nn = 0; nn < BKC; nn++) {
            float a[4], w[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = As[nn][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; j++) w[j] = Ws[nn][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int64_t m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int k = k0 + tx * 4 + j;
            if (k < K) C[m * ldc + k] = accumulate ? C[m * ldc + k] + acc[i][j] : acc[i][j];
        }
    }
}

// G[N,K] (+)= A[M,N]^T X[M,K]        (dW = dZ^T X: the reduction runs over the rows, both operands row-major).
// gridDim.z row chunks; chunk z > 0 (or accumulate) adds with atomics onto chunk 0's store, so the host zeroes G
// first when it splits.
__global__ void __launch_bounds__(256) gemm_tn_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ X, int64_t ldx,
                                                      float* __restrict__ G, int64_t ldg, int64_t M, int N, int K, int64_t rows_per_chunk,
                                                      int atomic) {
    __shared__ float As[BKC][BT];
    __shared__ float Xs[BKC][BT];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int n0 = blockIdx.y * BT, k0 = blockIdx.x * BT;
    const int64_t mlo = (int64_t)blockIdx.z * rows_per_chunk, mhi = min(M, mlo + rows_per_chunk);
    float acc[4][4] = {};
    for (int64_t m0 = mlo; m0 < mhi; m0 += BKC) {
        for (int t = threadIdx.x; t < BT * BKC; t += 256) {
            const int r = t / BT, c = t % BT;
            const int64_t m = m0 + r;
            As[r][c] = (m < mhi && n0 + c < N) ? A[m * lda + n0 + c] : 0.f;
            Xs[r][c] = (m < mhi && k0 + c < K) ? X[m * ldx + k0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int mm = 0; mm < BKC; mm++) {
            float a[4], x[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = As[mm][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; j++) x[j] = Xs[mm][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], x[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int n = n0 + ty * 4 + i;
        if (n >= N) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int k = k0 + tx * 4 + j;
            if (k >= K) continue;
            if (atomic) atomicAdd(&G[(int64_t)n * ldg + k], acc[i][j]);
            else G[(int64_t)n * ldg + k] = acc[i][j];
        }
    }
}

// out[n] (+)= sum_m Z[m, n]   (bias gradients): block = 32 columns x 8 row lanes
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ Z, int64_t ldz, float* __restrict__ out, int64_t M, int N,
                                                     int accumulate) {
    __shared__ float part[8][33];
    const int c = threadIdx.x & 31, rl = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + c;
    float s = 0.f;
    if (n < N)
        for (int64_t m = rl; m < M; m += 8) s += Z[m * ldz + n];
    part[rl][c] = s;
    __syncthreads();
    if (rl == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < 8; q++) t += part[q][c];
        out[n] = accumulate ? out[n] + t : t;
    }
}

__device__ __forceinline__ float act_grad_from_output(float a, int act) {
    switch (act) {
        case GM_ACT_LEAKY_RELU: return a > 0.f ? 1.f : 0.01f;
        case GM_ACT_RELU: return a > 0.f ? 1.f : 0.f;
        case GM_ACT_TANH: return 1.f - a * a;
        case GM_ACT_SIGMOID: return a * (1.f - a);
        case GM_ACT_ELU: return a > 0.f ? 1.f : a + 1.f;
        default: return 1.f;
    }
}

// dz = dy * act'(.) from the layer's OUTPUT a (every built activation has a derivative that is a function of it)
__global__ void act_bwd_kernel(const float* __restrict__ a, const float* __restrict__ dy, int64_t lddy, float* __restrict__ dz, int64_t R,
                               int W, int act) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * W) return;
    const int64_t r = idx / W;
    const int j = (int)(idx - r * W);
    dz[idx] = dy[r * lddy + j] * act_grad_from_output(a[idx], act);
}

// LSTM cell, training forward: gates [R,4H] hold the pre-activations (x W_ih^T + b_ih + h W_hh^T + b_hh) and are
// overwritten with the ACTIVATED gates (i, f, g, o) for the tape
__global__ void lstm_train_fwd_kernel(float* __restrict__ gates, const float* __restrict__ c_prev, int64_t ldcp, float* __restrict__ h_new,
                                      float* __restrict__ c_new, int64_t R, int H) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * H) return;
    const int64_t r = idx / H;
    const int j = (int)(idx - r * H);
    float* g = gates + r * 4 * H;
    const float i_ = sigmoidf_(g[j]), f_ = sigmoidf_(g[H + j]), g_ = tanhf(g[2 * H + j]), o_ = sigmoidf_(g[3 * H + j]);
    const float c = f_ * (c_prev ? c_prev[r * ldcp + j] : 0.f) + i_ * g_;
    g[j] = i_; g[H + j] = f_; g[2 * H + j] = g_; g[3 * H + j] = o_;
    c_new[idx] = c;
    h_new[idx] = o_ * tanhf(c);
}

// LSTM cell backward: (dh, dc) of the cell outputs -> dZ [R,4H] (pre-activation gate gradients) and dc_prev
__global__ void lstm_bwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev, int64_t ldcp, const float* __restrict__ c_new,
                                const float* __restrict__ dh, int64_t lddh, const float* __restrict__ dc, int64_t lddc,
                                float* __restrict__ dZ, float* __restrict__ dc_prev, int64_t lddcp, int64_t R, int H) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * H) return;
    const int64_t r = idx / H;
    const int j = (int)(idx - r * H);
    const float* g = gates + r * 4 * H;
    const float i_ = g[j], f_ = g[H + j], g_ = g[2 * H + j], o_ = g[3 * H + j];
    const float tc = tanhf(c_new[idx]);
    const float dh_ = dh ? dh[r * lddh + j] : 0.f;
    const float dct = (dc ? dc[r * lddc + j] : 0.f) + dh_ * o_ * (1.f - tc * tc);
    const float cp = c_prev ? c_prev[r * ldcp + j] : 0.f;
    float* z = dZ + r * 4 * H;
    z[j] = dct * g_ * i_ * (1.f - i_);
    z[H + j] = dct * cp * f_ * (1.f - f_);
    z[2 * H + j] = dct * i_ * (1.f - g_ * g_);
    z[3 * H + j] = dh_ * tc * o_ * (1.f - o_);
    dc_prev[r * lddcp + j] = dct * f_;
}

// ---- LayerNormLSTM cell (layernormlstm.py:24-42), one warp per row -------------------------------------------
// training forward: gi / gh [R,4H] hold x W_ih^T and h W_hh^T and are overwritten with their NORMALISED values
// (the LayerNorm backward needs y_hat and 1/sigma, not the raw rows); gates <- activated (i,f,g,o);
// chat <- normalised pre-LN cell; stats[r] = (rstd_i, rstd_h, rstd_c)
__global__ void lnlstm_train_fwd_kernel(float* __restrict__ gi, float* __restrict__ gh, gm_cell_params cp, const float* __restrict__ c_prev,
                                        int64_t ldcp, float* __restrict__ gates, float* __restrict__ chat, float* __restrict__ stats,
                                        float* __restrict__ h_new, float* __restrict__ c_new, int64_t R, int H) {
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= R) return;
    const int G = 4 * H;
    float* a = gi + r * G;
    float* b = gh + r * G;
    float sa = 0.f, sb = 0.f;
    for (int c = lane; c < G; c += 32) { sa += a[c]; sb += b[c]; }
    const float ma = warp_sum(sa) / (float)G, mb = warp_sum(sb) / (float)G;
    float va = 0.f, vb = 0.f;
    for (int c = lane; c < G; c += 32) {
        const float da = a[c] - ma, db = b[c] - mb;
        va += da * da; vb += db * db;
    }
    const float ra = 1.f / sqrtf(warp_sum(va) / (float)G + 1e-5f), rb = 1.f / sqrtf(warp_sum(vb) / (float)G + 1e-5f);
    float* g = gates + r * G;
    for (int c = lane; c < G; c += 32) {
        const float ya = (a[c] - ma) * ra, yb = (b[c] - mb) * rb;
        a[c] = ya; b[c] = yb;
        g[c] = ya * cp.ln_in_w[c] + cp.ln_in_b[c] + (yb * cp.ln_hid_w[c] + cp.ln_hid_b[c]) + cp.b_ih[c];
    }
    __syncwarp();
    float sc = 0.f;
    for (int j = lane; j < H; j += 32) {
        const float i_ = sigmoidf_(g[j]), f_ = sigmoidf_(g[H + j]), g_ = tanhf(g[2 * H + j]), o_ = sigmoidf_(g[3 * H + j]);
        const float cpre = f_ * (c_prev ? c_prev[r * ldcp + j] : 0.f) + i_ * g_;
        g[j] = i_; g[H + j] = f_; g[2 * H + j] = g_; g[3 * H + j] = o_;
        chat[r * H + j] = cpre;
        sc += cpre;
    }
    const float mc = warp_sum(sc) / (float)H;
    float vc = 0.f;
    for (int j = lane; j < H; j += 32) { const float d = chat[r * H + j] - mc; vc += d * d; }
    const float rc = 1.f / sqrtf(warp_sum(vc) / (float)H + 1e-5f);
    for (int j = lane; j < H; j += 32) {
        const float yc = (chat[r * H + j] - mc) * rc;
        const float c = yc * cp.ln_cell_w[j] + cp.ln_cell_b[j];
        chat[r * H + j] = yc;
        c_new[r * H + j] = c;
        h_new[r * H + j] = g[3 * H + j] * tanhf(c);
    }
    if (lane == 0) { stats[r * 4] = ra; stats[r * 4 + 1] = rb; stats[r * 4 + 2] = rc; }
}

// backward: (dh, dc) of the cell outputs -> dZ [R,4H] (gradient of the summed gate pre-activations), dgi / dgh [R,4H]
// (gradients of x W_ih^T / h W_hh^T through their LayerNorms), dct [R,H] (gradient of the post-LN cell, for the
// ln_cell parameter gradients) and dc_prev
__global__ void lnlstm_bwd_kernel(const float* __restrict__ yi, const float* __restrict__ yh, const float* __restrict__ gates,
                                  const float* __restrict__ chat, const float* __restrict__ stats, const float* __restrict__ c_new,
                                  gm_cell_params cp, const float* __restrict__ c_prev, int64_t ldcp, const float* __restrict__ dh,
                                  int64_t lddh, const float* __restrict__ dc, int64_t lddc, float* __restrict__ dZ,
                                  float* __restrict__ dgi, float* __restrict__ dgh, float* __restrict__ dct,
                                  float* __restrict__ dc_prev, int64_t lddcp, int64_t R, int H) {
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= R) return;
    const int G = 4 * H;
    const float* g = gates + r * G;
    const float ra = stats[r * 4], rb = stats[r * 4 + 1], rc = stats[r * 4 + 2];
    float* z = dZ + r * G;
    // LN_c backward: d c_pre = rstd (dyhat - mean(dyhat) - yhat mean(dyhat yhat)), dyhat = dc' * gamma_c
    float s1 = 0.f, s2 = 0.f;
    for (int j = lane; j < H; j += 32) {
        const float tc = tanhf(c_new[r * H + j]);
        const float dh_ = dh ? dh[r * lddh + j] : 0.f;
        const float d = (dc ? dc[r * lddc + j] : 0.f) + dh_ * g[3 * H + j] * (1.f - tc * tc);
        dct[r * H + j] = d;
        const float dy = d * cp.ln_cell_w[j];
        s1 += dy;
        s2 += dy * chat[r * H + j];
        z[3 * H + j] = dh_ * tc * g[3 * H + j] * (1.f - g[3 * H + j]);
    }
    const float m1 = warp_sum(s1) / (float)H, m2 = warp_sum(s2) / (float)H;
    for (int j = lane; j < H; j += 32) {
        const float dy = dct[r * H + j] * cp.ln_cell_w[j];
        const float dcp = rc * (dy - m1 - chat[r * H + j] * m2);
        const float i_ = g[j], f_ = g[H + j], g_ = g[2 * H + j];
        const float cpv = c_prev ? c_prev[r * ldcp + j] : 0.f;
        z[j] = dcp * g_ * i_ * (1.f - i_);
        z[H + j] = dcp * cpv * f_ * (1.f - f_);
        z[2 * H + j] = dcp * i_ * (1.f - g_ * g_);
        dc_prev[r * lddcp + j] = dcp * f_;
    }
    __syncwarp();
    // the two gate LayerNorms: dyhat = dZ * gamma
    const float* a = yi + r * G;
    const float* b = yh + r * G;
    float a1 = 0.f, a2 = 0.f, b1 = 0.f, b2 = 0.f;
    for (int c = lane; c < G; c += 32) {
        const float da = z[c] * cp.ln_in_w[c], db = z[c] * cp.ln_hid_w[c];
        a1 += da; a2 += da * a[c];
        b1 += db; b2 += db * b[c];
    }
    a1 = warp_sum(a1) / (float)G; a2 = warp_sum(a2) / (float)G; b1 = warp_sum(b1) / (float)G; b2 = warp_sum(b2) / (float)G;
    for (int c = lane; c < G; c += 32) {
        dgi[r * G + c] = ra * (z[c] * cp.ln_in_w[c] - a1 - a[c] * a2);
        dgh[r * G + c] = rb * (z[c] * cp.ln_hid_w[c] - b1 - b[c] * b2);
    }
}

// out[n] (+)= sum_m Z[m,n] * Y[m,n]   (LayerNorm weight gradients)
__global__ void __launch_bounds__(256) colsum_prod_kernel(const float* __restrict__ Z, const float* __restrict__ Y, int64_t ld,
                                                          float* __restrict__ out, int64_t M, int N, int accumulate) {
    __shared__ float part[8][33];
    const int c = threadIdx.x & 31, rl = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + c;
    float s = 0.f;
    if (n < N)
        for (int64_t m = rl; m < M; m += 8) s += Z[m * ld + n] * Y[m * ld + n];
    part[rl][c] = s;
    __syncthreads();
    if (rl == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < 8; q++) t += part[q][c];
        out[n] = accumulate ? out[n] + t : t;
    }
}

// transpose of the neighbour sum / mean (netmon.cu aggregate_kernel) as a scatter (any adjacency):
// dh[u] += sum over rows v whose list holds u of dM[v] (/ deg_v for mean)
__global__ void agg_bwd_kernel(const float* __restrict__ dM, float* __restrict__ dh, int B, int N, int H, const int* __restrict__ nbr,
                               const int* __restrict__ deg, int DM, const int* __restrict__ list_index, int mean) {
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= (int64_t)B * N) return;
    const int b = (int)(row / N), v = (int)(row - (int64_t)b * N);
    const int li = list_index ? list_index[b] : b;
    const int* lst = nbr + ((size_t)li * N + v) * DM;
    const int dg = deg[(size_t)li * N + v];
    const float scale = mean ? 1.f / (float)max(dg, 1) : 1.f;
    float* db = dh + (size_t)b * N * H;
    for (int c = lane; c < H; c += 32) {
        const float g = dM[row * H + c] * scale;
        for (int q = 0; q < dg; q++) atomicAdd(&db[(size_t)lst[q] * H + c], g);
    }
}

// transpose of the node readout (model.py:582-622, netmon.cu readout_kernel):
// dh[v] = d_out[v, 0:H]; dlast[n_k(v)] += d_out[v, H(1+k) : H(2+k)]
__global__ void readout_bwd_kernel(const float* __restrict__ d_out, float* __restrict__ dh, float* __restrict__ dlast, int B, int N, int H,
                                   const int* __restrict__ nbr, const int* __restrict__ deg, int DM, const int* __restrict__ list_index,
                                   int use_nbr, int max_degree) {
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= (int64_t)B * N) return;
    const int b = (int)(row / N), v = (int)(row - (int64_t)b * N);
    const int O = H + (use_nbr ? max_degree * H : 0);
    const float* o = d_out + row * O;
    for (int c = lane; c < H; c += 32) dh[row * H + c] = o[c];
    if (!use_nbr) return;
    const int li = list_index ? list_index[b] : b;
    const int* lst = nbr + ((size_t)li * N + v) * DM;
    const int dg = deg[(size_t)li * N + v];
    int slot = 0;
    for (int q = 0; q < dg && slot < max_degree; q++) {
        const int u = lst[q];
        if (u == v) continue;
        float* lu = dlast + ((size_t)b * N + u) * H;
        for (int c = lane; c < H; c += 32) atomicAdd(&lu[c], o[H + slot * H + c]);
        slot++;
    }
}

__global__ void add_rows_kernel(float* __restrict__ dst, int64_t ldd, const float* __restrict__ src, int64_t lds, int64_t R, int W) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * W) return;
    const int64_t r = idx / W;
    const int j = (int)(idx - r * W);
    dst[r * ldd + j] += src[r * lds + j];
}

// ---------------------------------------------------------------------------------------
static inline unsigned nblk(int64_t n, int per = 256) { return (unsigned)((n + per - 1) / per); }

static int gemm_nn(const float* A, int64_t lda, const float* W, int64_t ldw, float* C, int64_t ldc, int64_t M, int N, int K, int acc,
                   cudaStream_t s) {
    dim3 grid((K + BT - 1) / BT, (unsigned)((M + BT - 1) / BT));
    gemm_nn_kernel<<<grid, 256, 0, s>>>(A, lda, W, ldw, C, ldc, M, N, K, acc);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

// G = A^T X (accumulate: G += A^T X); rows split over up to 32 chunks when there are few output tiles
static int gemm_tn(const float* A, int64_t lda, const float* X, int64_t ldx, float* G, int64_t ldg, int64_t M, int N, int K, int acc,
                   cudaStream_t s) {
    const int tiles = ((K + BT - 1) / BT) * ((N + BT - 1) / BT);
    int chunks = (int)std::min<int64_t>(32, std::max<int64_t>(1, std::min<int64_t>((2 * kNumSMs) / std::max(tiles, 1), M / 256)));
    const int64_t rpc = (((M + chunks - 1) / chunks) + BKC - 1) / BKC * BKC;
    chunks = (int)((M + rpc - 1) / rpc);
    const int atomic = (chunks > 1 || acc) ? 1 : 0;
    if (chunks > 1 && !acc) GM_CUDA(cudaMemset2DAsync(G, ldg * 4, 0, (size_t)K * 4, N, s));
    dim3 grid((K + BT - 1) / BT, (N + BT - 1) / BT, chunks);
    gemm_tn_kernel<<<grid, 256, 0, s>>>(A, lda, X, ldx, G, ldg, M, N, K, rpc, atomic);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

static int colsum(const float* Z, int64_t ldz, float* out, int64_t M, int N, int acc, cudaStream_t s) {
    colsum_kernel<<<(N + 31) / 32, 256, 0, s>>>(Z, ldz, out, M, N, acc);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

// ---- MLP ----------------------------------------------------------------------------------
static int64_t mlp_tape_off(const gm_mlp_desc* m, int64_t rows, int l) {
    int64_t off = 0;
    for (int j = 0; j < l; j++) off += rows * m->units[j];
    return off;
}

static int mlp_check(const gm_mlp_desc* m) {
    GM_CHECK_ARG(m && m->n_layers >= 1 && m->n_layers <= GM_MAX_LAYERS && m->in_features > 0, "bad MLP descriptor");
    GM_CHECK_ARG(m->math == GM_MATH_FP32 || m->math == GM_MATH_BF16X3, "training runs fp32 or bf16x3 arithmetic (math %d)", m->math);
    for (int l = 0; l < m->n_layers; l++) GM_CHECK_ARG(m->units[l] > 0 && m->w[l], "layer %d", l);
    return GM_OK;
}

static int mlp_forward(const gm_mlp_desc* m, int64_t rows, const float* x, int64_t ldx, float* tape, void* ws, int64_t ws_bytes,
                       cudaStream_t s) {
    const float* in = x;
    int64_t ld = ldx;
    int kin = m->in_features;
    for (int l = 0; l < m->n_layers; l++) {
        float* y = tape + mlp_tape_off(m, rows, l);
        LinearArgs a{in, ld, m->w[l], kin, m->b[l], nullptr, y, m->units[l], rows, m->units[l], kin, m->act[l], 0};
        int rc = linear_dispatch(a, m->math, ws, ws_bytes, s);
        if (rc) return rc;
        in = y; ld = m->units[l]; kin = m->units[l];
    }
    return GM_OK;
}

// scratch of the backward: two [rows, maxw] gradient buffers
static int64_t mlp_bwd_floats(const gm_mlp_desc* m, int64_t rows) {
    int maxw = m->in_features;
    for (int l = 0; l < m->n_layers; l++) maxw = std::max(maxw, m->units[l]);
    return 2 * rows * (int64_t)maxw;
}

static int mlp_backward(const gm_mlp_desc* m, int64_t rows, const float* x, int64_t ldx, const float* tape, const float* d_out, int64_t ldd,
                        float* d_x, int64_t lddx, const gm_mlp_grads* g, float* scratch, cudaStream_t s) {
    int maxw = m->in_features;
    for (int l = 0; l < m->n_layers; l++) maxw = std::max(maxw, m->units[l]);
    float* dz = scratch;                          // dz_l = dy_l * act'(out_l)
    float* da = scratch + rows * (int64_t)maxw;   // gradient handed to the layer below (read by its act_bwd)
    const float* dy = d_out;
    int64_t lddy = ldd;
    for (int l = m->n_layers - 1; l >= 0; l--) {
        const int U = m->units[l], kin = l ? m->units[l - 1] : m->in_features;
        const float* out_l = tape + mlp_tape_off(m, rows, l);
        const float* in_l = l ? tape + mlp_tape_off(m, rows, l - 1) : x;
        const int64_t ldin = l ? kin : ldx;
        act_bwd_kernel<<<nblk(rows * U), 256, 0, s>>>(out_l, dy, lddy, dz, rows, U, m->act[l]);
        GM_LAUNCH_CHECK();
        int rc;
        if (g && g->w[l] && (rc = gemm_tn(dz, U, in_l, ldin, g->w[l], kin, rows, U, kin, 0, s))) return rc;
        if (g && g->b[l] && (rc = colsum(dz, U, g->b[l], rows, U, 0, s))) return rc;
        if (l > 0) {
            if ((rc = gemm_nn(dz, U, m->w[l], kin, da, kin, rows, U, kin, 0, s))) return rc;
            dy = da;
            lddy = kin;
        } else if (d_x) {
            if ((rc = gemm_nn(dz, U, m->w[l], kin, d_x, lddx, rows, U, kin, 0, s))) return rc;
        }
    }
    return GM_OK;
}

// ---- NetMon -------------------------------------------------------------------------------
struct NmTape {
    // float offsets: enc tape | (K+1) x gates [R,4H] | (K+1) x c | (K+1) x h | K x M
    // LayerNormLSTM adds per cell: yi, yh [R,4H] (normalised gate rows), chat [R,H], stats [R,4]
    int64_t enc, gates, c, h, M, yi, yh, chat, stats, total;
};

static gm_mlp_desc enc_desc(const gm_netmon_params* p) {
    gm_mlp_desc m{};
    m.n_layers = p->n_enc_layers;
    m.in_features = p->in_features;
    m.math = p->math == GM_MATH_BF16 ? GM_MATH_BF16X3 : p->math;
    for (int l = 0; l < p->n_enc_layers; l++) {
        m.units[l] = p->enc_units[l];
        m.act[l] = p->activation;
        m.w[l] = p->enc_w[l];
        m.b[l] = p->enc_b[l];
    }
    return m;
}

static NmTape nm_tape(const gm_netmon_params* p, int64_t R) {
    NmTape t;
    const gm_mlp_desc m = enc_desc(p);
    const int H = p->hidden, K = p->iterations;
    t.enc = 0;
    t.gates = mlp_tape_off(&m, R, m.n_layers);
    t.c = t.gates + (int64_t)(K + 1) * R * 4 * H;
    t.h = t.c + (int64_t)(K + 1) * R * H;
    t.M = t.h + (int64_t)(K + 1) * R * H;
    t.total = t.M + (int64_t)K * R * H;
    t.yi = t.yh = t.chat = t.stats = t.total;
    if (p->rnn_type == GM_RNN_LNLSTM) {
        t.yi = t.total;
        t.yh = t.yi + (int64_t)(K + 1) * R * 4 * H;
        t.chat = t.yh + (int64_t)(K + 1) * R * 4 * H;
        t.stats = t.chat + (int64_t)(K + 1) * R * H;
        t.total = t.stats + (int64_t)(K + 1) * R * 4;
    }
    return t;
}

static int nm_train_check(const gm_netmon_params* p) {
    GM_CHECK_ARG(p && p->hidden > 0 && p->n_enc_layers >= 1 && p->n_enc_layers <= GM_MAX_LAYERS &&
                     p->enc_units[p->n_enc_layers - 1] == p->hidden,
                 "bad NetMon descriptor");
    GM_CHECK_ARG((p->rnn_type == GM_RNN_LSTM || p->rnn_type == GM_RNN_LNLSTM) && p->rnn_carryover && !p->output_global_hidden &&
                     p->iterations >= 1,
                 "the device backward is built for rnn_type lstm / lnlstm with carry-over, K >= 1, no global readout");
    return GM_OK;
}

// scratch floats of forward / backward: dh, dc, dM, dlast, tmp [R,H] each, dZ [R,4H], MLP scratch
static int64_t nm_scratch_floats(const gm_netmon_params* p, int64_t R) {
    const gm_mlp_desc m = enc_desc(p);
    return 6 * R * (int64_t)p->hidden + R * 4ll * p->hidden + mlp_bwd_floats(&m, R) +
           (p->rnn_type == GM_RNN_LNLSTM ? R * 9ll * p->hidden : 0);  // + dgi, dgh [R,4H], dct [R,H]
}

}  // namespace gm

using namespace gm;

extern "C" {

int64_t gm_linear_workspace_bytes(int64_t M, int32_t N, int32_t K, int32_t math);

int64_t gm_mlp_tape_floats(const gm_mlp_desc* m, int64_t rows) { return m ? mlp_tape_off(m, rows, m->n_layers) : 0; }

int64_t gm_mlp_train_workspace_bytes(const gm_mlp_desc* m, int64_t rows) {
    if (!m) return 0;
    int64_t lin = 0;
    int kin = m->in_features;
    for (int l = 0; l < m->n_layers; l++) {
        lin = std::max(lin, gm_linear_workspace_bytes(rows, m->units[l], kin, m->math));
        kin = m->units[l];
    }
    return round_up(mlp_bwd_floats(m, rows) * 4, 256) + round_up(lin, 256) + 512;
}

int gm_mlp_forward_train(const gm_mlp_desc* m, int64_t rows, const float* x, int64_t ldx, float* tape, void* workspace,
                         int64_t workspace_bytes, void* stream) {
    int rc = mlp_check(m);
    if (rc) return rc;
    GM_CHECK_ARG(x && tape && rows > 0 && workspace_bytes >= gm_mlp_train_workspace_bytes(m, rows), "bad MLP forward arguments");
    char* lin = (char*)workspace + round_up(mlp_bwd_floats(m, rows) * 4, 256);
    lin = (char*)round_up((int64_t)lin, 256);
    return mlp_forward(m, rows, x, ldx, tape, lin, (char*)workspace + workspace_bytes - lin, (cudaStream_t)stream);
}

int gm_mlp_backward(const gm_mlp_desc* m, int64_t rows, const float* x, int64_t ldx, const float* tape, const float* d_out, int64_t ldd,
                    float* d_x, const gm_mlp_grads* grads, void* workspace, int64_t workspace_bytes, void* stream) {
    int rc = mlp_check(m);
    if (rc) return rc;
    GM_CHECK_ARG(x && tape && d_out && rows > 0 && workspace_bytes >= gm_mlp_train_workspace_bytes(m, rows), "bad MLP backward arguments");
    return mlp_backward(m, rows, x, ldx, tape, d_out, ldd, d_x, m->in_features, grads, (float*)workspace, (cudaStream_t)stream);
}

int64_t gm_netmon_tape_floats(const gm_netmon_params* p, int64_t rows) { return p ? nm_tape(p, rows).total : 0; }

int64_t gm_netmon_train_workspace_bytes(const gm_netmon_params* p, int64_t rows) {
    if (!p) return 0;
    const gm_mlp_desc m = enc_desc(p);
    int64_t lin = gm_linear_workspace_bytes(rows, 4 * p->hidden, p->hidden, m.math);
    int kin = m.in_features;
    for (int l = 0; l < m.n_layers; l++) {
        lin = std::max(lin, gm_linear_workspace_bytes(rows, m.units[l], kin, m.math));
        kin = m.units[l];
    }
    return round_up(nm_scratch_floats(p, rows) * 4, 256) + round_up(lin, 256) + 512;
}

int gm_netmon_forward_train(const gm_netmon_params* p, int32_t B, int32_t N, const float* node_obs, const int32_t* nbr_all,
                            const int32_t* deg, int32_t DM, const int32_t* list_index, const float* state_in, float* state_out,
                            int32_t max_degree, float* node_out, float* tape, void* workspace, int64_t workspace_bytes, void* stream) {
    int rc = nm_train_check(p);
    if (rc) return rc;
    GM_CHECK_ARG(node_obs && nbr_all && deg && state_out && tape && workspace && B > 0 && N > 0 && DM > 0 && max_degree <= DM, "bad arguments");
    const int64_t R = (int64_t)B * N;
    GM_CHECK_ARG(workspace_bytes >= gm_netmon_train_workspace_bytes(p, R), "workspace too small");
    cudaStream_t s = (cudaStream_t)stream;
    const int H = p->hidden, K = p->iterations;
    const gm_mlp_desc m = enc_desc(p);
    const NmTape T = nm_tape(p, R);
    char* lin = (char*)round_up((int64_t)((char*)workspace + round_up(nm_scratch_floats(p, R) * 4, 256)), 256);
    const int64_t lin_bytes = (char*)workspace + workspace_bytes - lin;
    if ((rc = mlp_forward(&m, R, node_obs, p->in_features, tape + T.enc, lin, lin_bytes, s))) return rc;
    const float* e = tape + T.enc + mlp_tape_off(&m, R, m.n_layers - 1);
    const bool LN = p->rnn_type == GM_RNN_LNLSTM;
    auto cell = [&](const gm_cell_params& cp, const float* x, const float* hp, int64_t ldhp, const float* cprev, int64_t ldcp, int idx) -> int {
        float* gates = tape + T.gates + (int64_t)idx * R * 4 * H;
        if (LN) {  // layernormlstm.py:28-40: the two gate GEMMs are normalised separately, no bias inside
            float* yi = tape + T.yi + (int64_t)idx * R * 4 * H;
            float* yh = tape + T.yh + (int64_t)idx * R * 4 * H;
            LinearArgs a{x, H, cp.w_ih, H, nullptr, nullptr, yi, 4 * H, R, 4 * H, H, -1, 0};
            int r2 = linear_dispatch(a, m.math, lin, lin_bytes, s);
            if (r2) return r2;
            if (hp) {
                LinearArgs b{hp, ldhp, cp.w_hh, H, nullptr, nullptr, yh, 4 * H, R, 4 * H, H, -1, 0};
                if ((r2 = linear_dispatch(b, m.math, lin, lin_bytes, s))) return r2;
            } else {
                GM_CUDA(cudaMemsetAsync(yh, 0, (size_t)R * 4 * H * 4, s));
            }
            lnlstm_train_fwd_kernel<<<nblk(R, 4), 128, 0, s>>>(yi, yh, cp, cprev, ldcp, gates, tape + T.chat + (int64_t)idx * R * H,
                                                              tape + T.stats + (int64_t)idx * R * 4, tape + T.h + (int64_t)idx * R * H,
                                                              tape + T.c + (int64_t)idx * R * H, R, H);
            GM_LAUNCH_CHECK();
            return GM_OK;
        }
        LinearArgs a{x, H, cp.w_ih, H, cp.b_ih, cp.b_hh, gates, 4 * H, R, 4 * H, H, -1, 0};
        int r2 = linear_dispatch(a, m.math, lin, lin_bytes, s);
        if (r2) return r2;
        if (hp) {
            LinearArgs b{hp, ldhp, cp.w_hh, H, nullptr, nullptr, gates, 4 * H, R, 4 * H, H, -1, 1};
            if ((r2 = linear_dispatch(b, m.math, lin, lin_bytes, s))) return r2;
        }
        lstm_train_fwd_kernel<<<nblk(R * H), 256, 0, s>>>(gates, cprev, ldcp, tape + T.h + (int64_t)idx * R * H,
                                                         tape + T.c + (int64_t)idx * R * H, R, H);
        GM_LAUNCH_CHECK();
        return GM_OK;
    };
    // rnn_obs (:491); a missing state is zeros (:480-484): the h GEMM contributes nothing then
    if ((rc = cell(p->rnn_obs, e, state_in, 2 * H, state_in ? state_in + H : nullptr, 2 * H, 0))) return rc;
    for (int it = 0; it < K; it++) {  // :509-554
        const float* h = tape + T.h + (int64_t)it * R * H;
        float* M = tape + T.M + (int64_t)it * R * H;
        if ((rc = aggregate_rows(h, H, M, B, N, H, nbr_all, deg, DM, list_index, p->agg_type == GM_AGG_MEAN, s))) return rc;
        if ((rc = cell(p->rnn_update, M, h, H, tape + T.c + (int64_t)it * R * H, H, it + 1))) return rc;
    }
    const float* hK = tape + T.h + (int64_t)K * R * H;
    const float* cK = tape + T.c + (int64_t)K * R * H;
    if ((rc = copy_rows(hK, H, state_out, 2 * H, R, H, s))) return rc;
    if ((rc = copy_rows(cK, H, state_out + H, 2 * H, R, H, s))) return rc;
    if (!node_out) return GM_OK;
    const float* last = tape + T.h + (int64_t)(K - 1) * R * H;  // h before the final iteration's aggregation (:510-519)
    const int use_nbr = p->output_neighbor_hidden;
    return readout_rows(hK, H, last, H, nullptr, nbr_all, deg, DM, list_index, nullptr, N, B, N, H, use_nbr, 0, max_degree,
                        node_out, H + (use_nbr ? max_degree * H : 0), s);
}

int gm_netmon_backward(const gm_netmon_params* p, int32_t B, int32_t N, const float* node_obs, const int32_t* nbr_all, const int32_t* deg,
                       int32_t DM, const int32_t* list_index, const float* state_in, int32_t max_degree, const float* tape,
                       const float* d_node_out, const float* d_state_out, float* d_state_in, const gm_netmon_grads* grads, void* workspace,
                       int64_t workspace_bytes, void* stream) {
    int rc = nm_train_check(p);
    if (rc) return rc;
    GM_CHECK_ARG(node_obs && nbr_all && deg && tape && grads && workspace && B > 0 && N > 0, "bad arguments");
    const int64_t R = (int64_t)B * N;
    GM_CHECK_ARG(workspace_bytes >= gm_netmon_train_workspace_bytes(p, R), "workspace too small");
    cudaStream_t s = (cudaStream_t)stream;
    const int H = p->hidden, K = p->iterations;
    const gm_mlp_desc m = enc_desc(p);
    const NmTape T = nm_tape(p, R);
    float* w = (float*)workspace;
    float *dh = w, *dc = w + R * H, *dM = w + 2 * R * H, *dlast = w + 3 * R * H, *tmp = w + 4 * R * H, *dcn = w + 5 * R * H;
    float* dZ = w + 6 * R * H;
    float* mlp_scratch = dZ + R * 4 * H;
    // ---- readout backward: dh_K and the gradient of `last` = h_{K-1} -------------------------------------------
    GM_CUDA(cudaMemsetAsync(dlast, 0, (size_t)R * H * 4, s));
    if (d_node_out) {
        readout_bwd_kernel<<<nblk(R, 4), 128, 0, s>>>(d_node_out, dh, dlast, B, N, H, nbr_all, deg, DM, list_index,
                                                     p->output_neighbor_hidden, max_degree);
        GM_LAUNCH_CHECK();
    } else {
        GM_CUDA(cudaMemsetAsync(dh, 0, (size_t)R * H * 4, s));
    }
    if (d_state_out) {
        add_rows_kernel<<<nblk(R * H), 256, 0, s>>>(dh, H, d_state_out, 2 * H, R, H); GM_LAUNCH_CHECK();
        if ((rc = copy_rows(d_state_out + H, 2 * H, dc, H, R, H, s))) return rc;
    } else {
        GM_CUDA(cudaMemsetAsync(dc, 0, (size_t)R * H * 4, s));
    }
    // One cell backwards: (dh, dc) of its outputs -> gradients of its two GEMM outputs (dZx for x W_ih^T, dZh for
    // h W_hh^T: the same dZ for nn.LSTMCell, the two LayerNorm backwards for LayerNormLSTMCell), dc_prev, and the
    // cell's parameter gradients (acc: add to what is there -- the update cell is shared by the K iterations).
    const bool LN = p->rnn_type == GM_RNN_LNLSTM;
    float* dgi = mlp_scratch + mlp_bwd_floats(&m, R);
    float* dgh = dgi + R * 4 * H;
    float* dct = dgh + R * 4 * H;
    const float* dZx = dZ;
    const float* dZh = dZ;
    auto cell_bwd = [&](const gm_cell_params& cp, const gm_cell_grads& g, int idx, const float* x, const float* hp, int64_t ldhp,
                        const float* cprev, int64_t ldcp, float* dc_prev, int64_t lddcp, int acc) -> int {
        const float* gates = tape + T.gates + (int64_t)idx * R * 4 * H;
        const float* c_new = tape + T.c + (int64_t)idx * R * H;
        int r2;
        if (LN) {
            const float* yi = tape + T.yi + (int64_t)idx * R * 4 * H;
            const float* yh = tape + T.yh + (int64_t)idx * R * 4 * H;
            const float* chat = tape + T.chat + (int64_t)idx * R * H;
            lnlstm_bwd_kernel<<<nblk(R, 4), 128, 0, s>>>(yi, yh, gates, chat, tape + T.stats + (int64_t)idx * R * 4, c_new, cp, cprev, ldcp,
                                                        dh, H, dc, H, dZ, dgi, dgh, dct, dc_prev, lddcp, R, H);
            GM_LAUNCH_CHECK();
            dZx = dgi; dZh = dgh;
            if (g.ln_in_w) { colsum_prod_kernel<<<(4 * H + 31) / 32, 256, 0, s>>>(dZ, yi, 4 * H, g.ln_in_w, R, 4 * H, acc); GM_LAUNCH_CHECK(); }
            if (g.ln_hid_w) { colsum_prod_kernel<<<(4 * H + 31) / 32, 256, 0, s>>>(dZ, yh, 4 * H, g.ln_hid_w, R, 4 * H, acc); GM_LAUNCH_CHECK(); }
            if (g.ln_cell_w) { colsum_prod_kernel<<<(H + 31) / 32, 256, 0, s>>>(dct, chat, H, g.ln_cell_w, R, H, acc); GM_LAUNCH_CHECK(); }
            if (g.ln_in_b && (r2 = colsum(dZ, 4 * H, g.ln_in_b, R, 4 * H, acc, s))) return r2;
            if (g.ln_hid_b && (r2 = colsum(dZ, 4 * H, g.ln_hid_b, R, 4 * H, acc, s))) return r2;
            if (g.ln_cell_b && (r2 = colsum(dct, H, g.ln_cell_b, R, H, acc, s))) return r2;
        } else {
            lstm_bwd_kernel<<<nblk(R * H), 256, 0, s>>>(gates, cprev, ldcp, c_new, dh, H, dc, H, dZ, dc_prev, lddcp, R, H);
            GM_LAUNCH_CHECK();
            if (g.b_hh && (r2 = colsum(dZ, 4 * H, g.b_hh, R, 4 * H, acc, s))) return r2;
        }
        if (g.b_ih && (r2 = colsum(dZ, 4 * H, g.b_ih, R, 4 * H, acc, s))) return r2;
        if (g.w_ih && (r2 = gemm_tn(dZx, 4 * H, x, H, g.w_ih, H, R, 4 * H, H, acc, s))) return r2;
        if (g.w_hh) {
            if (hp) { if ((r2 = gemm_tn(dZh, 4 * H, hp, ldhp, g.w_hh, H, R, 4 * H, H, acc, s))) return r2; }
            else if (!acc) GM_CUDA(cudaMemsetAsync(g.w_hh, 0, (size_t)4 * H * H * 4, s));
        }
        return GM_OK;
    };
    // ---- K x (rnn_update cell, aggregation) backwards ---------------------------------------------------------------
    for (int it = K - 1; it >= 0; it--) {
        const float* h_prev = tape + T.h + (int64_t)it * R * H;
        const float* M = tape + T.M + (int64_t)it * R * H;
        if ((rc = cell_bwd(p->rnn_update, grads->rnn_update, it + 1, M, h_prev, H, tape + T.c + (int64_t)it * R * H, H, dcn, H, it != K - 1))) return rc;
        if ((rc = gemm_nn(dZx, 4 * H, p->rnn_update.w_ih, H, dM, H, R, 4 * H, H, 0, s))) return rc;   // dM  = dZx W_ih
        if ((rc = gemm_nn(dZh, 4 * H, p->rnn_update.w_hh, H, tmp, H, R, 4 * H, H, 0, s))) return rc;  // dh_prev (direct)
        agg_bwd_kernel<<<nblk(R, 4), 128, 0, s>>>(dM, tmp, B, N, H, nbr_all, deg, DM, list_index, p->agg_type == GM_AGG_MEAN);
        GM_LAUNCH_CHECK();
        if (it == K - 1) {  // h_{K-1} is also the `last` of the readout
            add_rows_kernel<<<nblk(R * H), 256, 0, s>>>(tmp, H, dlast, H, R, H); GM_LAUNCH_CHECK();
        }
        std::swap(dh, tmp);
        std::swap(dc, dcn);
    }
    // ---- rnn_obs cell backward ------------------------------------------------------------------------------------
    {
        const float* e = tape + T.enc + mlp_tape_off(&m, R, m.n_layers - 1);
        float* dcs = d_state_in ? d_state_in + H : dcn;
        if ((rc = cell_bwd(p->rnn_obs, grads->rnn_obs, 0, e, state_in, 2 * H, state_in ? state_in + H : nullptr, 2 * H, dcs,
                           d_state_in ? 2 * H : H, 0)))
            return rc;
        if (d_state_in && (rc = gemm_nn(dZh, 4 * H, p->rnn_obs.w_hh, H, d_state_in, 2 * H, R, 4 * H, H, 0, s))) return rc;
        if ((rc = gemm_nn(dZx, 4 * H, p->rnn_obs.w_ih, H, dM, H, R, 4 * H, H, 0, s))) return rc;  // de
    }
    // ---- encoder backward ---------------------------------------------------------------------------------------------
    gm_mlp_grads eg{};
    for (int l = 0; l < m.n_layers; l++) { eg.w[l] = grads->enc_w[l]; eg.b[l] = grads->enc_b[l]; }
    return mlp_backward(&m, R, node_obs, p->in_features, tape + T.enc, dM, H, nullptr, 0, &eg, mlp_scratch, s);
}

}  // extern "C"
