// eval_metrics.cu -- per-env accumulation of the episode metrics of a batched evaluation (graph_marl_b200/evaluation.py):
// after each env step, gm_eval_accumulate adds the step's reward, packet delays, shortest-path ratios and info counters
// into acc f64[B, GM_EVAL_FIELDS] (field order in include/graphmarl_b200.h).
//
// One warp per env: lane l sums agents l, l + 32, ... in that order, the warp reduces with shuffles in a fixed tree, and
// lane 0 adds the totals into the env's row.  Nothing is atomic, so two runs (and a captured launch and an eager one) give
// the same bits.
#include "common.cuh"

namespace gm {

constexpr int kEvalWarps = 8;

__device__ inline double warp_tree_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(FULL, v, o);
    return v;  // valid in lane 0
}

__global__ void __launch_bounds__(kEvalWarps * 32) eval_accumulate_kernel(
    const float* __restrict__ reward, const uint8_t* __restrict__ done, const uint8_t* __restrict__ arrived,
    const int32_t* __restrict__ delays, const double* __restrict__ spr, const int32_t* __restrict__ info, int B, int A,
    double* __restrict__ acc) {
    const int b = blockIdx.x * kEvalWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;  // warp-uniform: the shuffles below see full warps only
    const int64_t row = (int64_t)b * A;
    double r = 0.0, d_sum = 0.0, d_cnt = 0.0, a_sum = 0.0, a_cnt = 0.0, s_sum = 0.0;
    for (int a = lane; a < A; a += 32) {
        const int64_t i = row + a;
        r += (double)reward[i];
        const double d = (double)delays[i];
        if (done[i]) d_sum += d, d_cnt += 1.0;
        if (arrived[i]) a_sum += d, a_cnt += 1.0, s_sum += spr[i];  // spr of a packet that did not arrive is never read
    }
    r = warp_tree_sum(r);
    d_sum = warp_tree_sum(d_sum);
    d_cnt = warp_tree_sum(d_cnt);
    a_sum = warp_tree_sum(a_sum);
    a_cnt = warp_tree_sum(a_cnt);
    s_sum = warp_tree_sum(s_sum);
    if (lane == 0) {
        double* q = acc + (int64_t)b * GM_EVAL_FIELDS;
        const int32_t* in = info + (int64_t)b * 4;
        q[GM_EVAL_REWARD_SUM] += r;
        q[GM_EVAL_AGENT_STEPS] += (double)A;
        q[GM_EVAL_DELAY_SUM] += d_sum;
        q[GM_EVAL_DELAY_COUNT] += d_cnt;
        q[GM_EVAL_ARRIVED_DELAY_SUM] += a_sum;
        q[GM_EVAL_ARRIVED_COUNT] += a_cnt;
        q[GM_EVAL_SPR_SUM] += s_sum;
        q[GM_EVAL_LOOPED] += (double)in[0];
        q[GM_EVAL_THROUGHPUT] += (double)in[1];
        q[GM_EVAL_DROPPED] += (double)in[2];
        q[GM_EVAL_BLOCKED] += (double)in[3];
        q[GM_EVAL_STEPS] += 1.0;
    }
}

}  // namespace gm

using namespace gm;

extern "C" {

int gm_eval_accumulate(const float* reward, const uint8_t* done, const uint8_t* arrived, const int32_t* delays,
                       const double* spr, const int32_t* info, int32_t B, int32_t A, double* acc, void* stream) {
    GM_CHECK_ARG(reward && done && arrived && delays && spr && info && acc, "gm_eval_accumulate: null pointer");
    GM_CHECK_ARG(B >= 1 && A >= 1, "gm_eval_accumulate: %d envs x %d agents", B, A);
    eval_accumulate_kernel<<<ceil_div(B, kEvalWarps), kEvalWarps * 32, 0, (cudaStream_t)stream>>>(reward, done, arrived,
                                                                                                 delays, spr, info, B, A, acc);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

}  // extern "C"
