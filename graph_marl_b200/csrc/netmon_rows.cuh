// netmon_rows.cuh -- NetMon's fp32 row kernels (netmon.cu), launched by the inference forward and by the training
// forward (train.cu) through these host launchers.
#pragma once
#include "common.cuh"

namespace gm {

__device__ inline float warp_sum(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
    return x;
}

// M[r] = sum (or mean) of h over the node's neighbour list, in list order (model.py:213-229); M has row stride H
int aggregate_rows(const float* h, int64_t ldh, float* M, int B, int N, int H, const int* nbr, const int* deg, int DM,
                   const int* list_index, int mean, cudaStream_t s);

// out row = [h_v | gmean_b | last[n_1] .. last[n_maxdeg]] for the B * rows_per_graph rows: every node (agent_node NULL,
// rows_per_graph N) or the node under each agent (model.py:458-469, 582-631)
int readout_rows(const float* h, int64_t ldh, const float* last, int64_t ldl, const float* gmean, const int* nbr,
                 const int* deg, int DM, const int* list_index, const int* agent_node, int rows_per_graph, int B, int N,
                 int H, int use_nbr, int use_glob, int max_degree, float* out, int64_t ldo, cudaStream_t s);

// dst[r, 0:W] = src[r, 0:W] for R rows
int copy_rows(const float* src, int64_t lds, float* dst, int64_t ldd, int64_t R, int W, cudaStream_t s);

}  // namespace gm
