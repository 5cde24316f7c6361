// gemm_sm100.cuh -- interface of the tcgen05 fused linear / LSTM-cell kernel (gemm_sm100.cu).
#pragma once
#include "common.cuh"

namespace gm {

enum { EPI_LINEAR = 0, EPI_LSTM = 1, EPI_QHEAD = 2, EPI_LNLSTM = 3 };
constexpr int TC_MAX_ACT = 8;

// "pk" = tile-packed split activations: an fp32 matrix [R, Kact] (Kact % 32 == 0) stored as bf16
// hi/lo core matrices exactly as the tensor core reads them from shared memory, one 16 KiB block
// per (128-row tile mt, 32-column k-block kb) at ((mt * Kact/32) + kb) * 16 KiB:
//   hi part at +0, lo part at +8 KiB; element (r, k) at (r>>3)*512 + ((k&31)>>3)*128 + (r&7)*16 + (k&7)*2
// Producing layers write it from their epilogue, consuming layers pull it with one bulk copy per
// k-block, so no thread touches the activations between layers.
constexpr int TC_BM = 128, TC_BK = 32;
constexpr int64_t TC_PK_BLOCK = 2 * TC_BM * TC_BK * 2;  // 16 KiB
inline int64_t tc_pk_bytes(int64_t rows, int kact) { return ((rows + TC_BM - 1) / TC_BM) * (int64_t)(kact / TC_BK) * TC_PK_BLOCK; }

struct TcArgs {
    // activations: logical row = [seg0 | seg1]; each segment is either fp32 row-major (A*, lda*) read by
    // the producer warps, or tile-packed (A*pk) pulled by bulk copies.  seg1 optional (K1 = 0).
    const float* A0; int64_t lda0; const uint8_t* A0pk; int K0;
    const float* A1; int64_t lda1; const uint8_t* A1pk; int K1;
    int K0p, Kp;              // filled by tc_launch: start of segment 1 / total K in the packed K space
    const uint8_t* Wp;        // weights (+ tile-ordered bias behind them) packed by tc_pack_weights
    const float* bias_tile;   // filled by tc_launch
    // EPI_LINEAR: C fp32 row-major (may be NULL) and/or Cpk tile-packed (may be NULL)
    float* C; int64_t ldc; uint8_t* Cpk; int act; int accumulate;
    int64_t M; int N;
    // EPI_LSTM: c' = sig(f)*c_in + sig(i)*tanh(g), h' = sig(o)*tanh(c'); h also tile-packed if Hpk
    const float* c_in; int64_t ldc_in;
    float* h_out; int64_t ldh; float* c_out; int64_t ldco; uint8_t* Hpk;
    int H;
    // cell state handed from one cell launch to the next may live in a BLOCKED layout (c_in_blocked / c_out_blocked):
    // [32-row group][8-unit chunk][32 rows][8 floats], offset tc_blocked_off(row, unit, H).  The epilogue thread of
    // row r reads / writes 32 bytes per chunk, so a warp instruction covers 1 KiB of contiguous memory (8 full
    // lines) instead of 32 bytes in each of 32 lines -- L2 throughput here is bound by requests, not bytes.
    int c_in_blocked, c_out_blocked;
    // EPI_LNLSTM (H == 128, both segments 128 wide; layernormlstm.py:24-42): the two gate GEMMs keep SEPARATE
    // accumulators (LN_4H is applied to x W_ih^T and h W_hh^T on their own).  A CTA owns whole M tiles and walks
    // 1 + H/32 N tiles per M tile: tile 0 multiplies by the centred Gram matrices of the weights, from which the
    // epilogue gets each row's LayerNorm mean / variance; tiles 1.. carry [i|f|g|o] of 32 hidden units each.
    // Uses c_in / h_out / c_out / Hpk like EPI_LSTM (h_out, c_out double as scratch for the LN_H pass).
    const float* ln_params;   // filled by tc_launch: column sums, per-tile LN affine, ln_cell affine
    // per-CTA scratch [gridDim][128 units x 128 rows] in the blocked layout of tc_blocked_off (row = tile row): sig(o) of the
    // four gate tiles waits here for the LN_H pass (96 registers per thread leave no room for it); a warp instruction
    // covers 1 KiB of contiguous memory.  NULL: parked in the h' slots of h_out instead (32 lines per warp instruction)
    float* ln_scratch;
    // EPI_QHEAD (N <= 256): the layer's activated output never leaves the SM; the epilogue applies the
    // Q head q = y Wq^T + bq, the action mask, argmax and the epsilon mix (model.py:199-203, policy.py:42-51)
    const float* q_w; const float* q_b; int n_act;
    const uint8_t* action_mask; double epsilon; const int* rand_action; const double* rand_u;
    uint64_t philox_seed, philox_step; const uint64_t* philox_step_dev;
    float* q_out; int* act_out;
    void* trace;  // GM_TC_PROBES builds only: per-tile timeline buffer (see gemm_sm100.cu)
    int m_tiles, n_tiles, has_prod, a_stages;  // filled by tc_launch
};

__host__ __device__ inline int64_t tc_blocked_off(int64_t row, int unit, int H) {
    return ((row >> 5) * (H >> 3) + (unit >> 3)) * 256 + (row & 31) * 8 + (unit & 7);
}
inline int64_t tc_blocked_floats(int64_t rows, int H) { return ((rows + 31) / 32) * 32 * (int64_t)H; }

struct TcShape {
    int BN, K0p, Kp, n_tiles;
    int64_t w_bytes, packed_bytes;  // weight tiles; weights + bias, rounded to 256
};

TcShape tc_shape(int N, int K0, int K1, int epi, int H);
// W fp32 [N, K0+K1] (row stride ldw), or W [N,K0] next to W1 [N,K1] -> packed bf16 hi/lo tiles
// (tc_shape(...).packed_bytes, 256-byte aligned destination)
// bias (+ bias2) are summed and stored tile-ordered behind the weights (either may be NULL)
int tc_pack_weights(const float* W, int64_t ldw, const float* W1, int64_t ldw1, const float* bias, const float* bias2, int N,
                    int K0, int K1, int epi, int H, void* out, cudaStream_t s);
int tc_launch(TcArgs a, int math, int epi, cudaStream_t s);

// Encoder layers 1 + 2 as one kernel for caller-supplied sparse input rows of at most 6 terms (gemm_sm100_encfused.inc):
// layer 1 on the CUDA cores inside the producer warps, layer 2 on tcgen05.  W2 is packed by tc_pack_weights(N = U2,
// K0 = U1, EPI_LINEAR) and must come out as ONE 256-column tile; W1 by enc_fused_pack_w1t.
bool enc_fused_ok(int D, int U1, int U2, int math);
int64_t enc_fused_w1t_bytes(int U1, int D);
int enc_fused_pack_w1t(const float* W1, const float* b1, int U1, int D, const float* static_rows, int S, int static_only, void* out,
                       cudaStream_t s);
int enc_fused_launch(const int32_t* sp_rows, int64_t R, int D, const void* w1t, const void* W2p, int U1, int U2, int act, uint8_t* Cpk,
                     cudaStream_t s);

// LayerNormLSTM cell (H == 128) -> packed weights for EPI_LNLSTM: tc_shape(4H, H, H, EPI_LNLSTM, H).packed_bytes
// (Gram + gate tiles, LN parameters, and the staging area the packing kernels use), 256-byte aligned destination.
int tc_pack_lnlstm(const float* w_ih, const float* w_hh, const float* b_ih, const float* ln_in_w, const float* ln_in_b,
                   const float* ln_hid_w, const float* ln_hid_b, const float* ln_cell_w, const float* ln_cell_b, int H, void* out,
                   cudaStream_t s);

}  // namespace gm
