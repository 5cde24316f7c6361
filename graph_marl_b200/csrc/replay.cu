// replay.cu -- device-resident replay ring: batched insert and index gather.
//
// Reference: src/replaybuffer.py:243-287 (add: 17 per-field copies into ring slot `index`,
// then index = (index+1) % size), :132-187 (_get_transition_batch: fancy-index gather plus
// dtype conversion to float32 / int64 / bool).  Here B transitions (one per env) are
// inserted per call into consecutive slots and the ring never leaves HBM.
#include <cuda_fp16.h>

#include <algorithm>

#include "common.cuh"

namespace gm {

struct ReplayFields {
    gm_replay_field f[GM_REPLAY_MAX_FIELDS];
    int n;
};

// grid.y = field, grid.x strides over (transition, 16 / 8 / 4 / 1-byte unit)
__global__ void replay_insert_kernel(ReplayFields F, int64_t capacity, int64_t index0, const int64_t* __restrict__ index_dev,
                                     int64_t n) {
    const int64_t index = index0 + (index_dev ? *index_dev : 0);
    const gm_replay_field fd = F.f[blockIdx.y];
    const int64_t eb = fd.elem_bytes;
    const int64_t tid0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (int64_t)gridDim.x * blockDim.x;
    if (fd.convert == 4) {  // int32 source elements -> int8 ring elements (actions)
        const int64_t total = n * eb;
        for (int64_t t = tid0; t < total; t += nthreads) {
            int64_t i = t / eb, e = t - i * eb;
            int64_t slot = (index + i) % capacity;
            ((int8_t*)fd.ring)[slot * eb + e] = (int8_t)((const int32_t*)fd.src)[(fd.broadcast ? 0 : i) * eb + e];
        }
        return;
    }
    // One warp per contiguous run (a transition, or one row of a transition's 2-D block): the three 64-bit divisions
    // that locate a run are paid once per warp and run, the lanes then stride over its 16 / 8 / 4 / 1-byte units with
    // up to four independent loads in flight.
    const bool two_d = fd.rows > 0;
    const int64_t rb = two_d ? fd.row_bytes : eb;           // contiguous run
    const int64_t runs = two_d ? fd.rows : 1;               // runs per transition
    const uintptr_t src_bits = (uintptr_t)fd.src | (uintptr_t)rb;
    const uintptr_t dst_bits = (uintptr_t)fd.ring | (uintptr_t)eb | (two_d ? ((uintptr_t)fd.ring_pitch | (uintptr_t)fd.ring_offset) : 0);
    const uintptr_t align_bits = src_bits | dst_bits;
    // 16-byte aligned source with a destination that is only 8-byte aligned (the graph part of a joint observation
    // row starts 520 bytes into the ring row): 16-byte loads, two 8-byte stores each
    const bool split_store = align_bits % 16 != 0 && src_bits % 16 == 0 && dst_bits % 8 == 0;
    const int unit = split_store ? 16 : (align_bits % 16 == 0) ? 16 : (align_bits % 8 == 0) ? 8 : (align_bits % 4 == 0) ? 4 : 1;
    const int upr = (int)(rb / unit);  // units per run
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = tid0 >> 5, nwarps = nthreads >> 5;
    for (int64_t q = warp0; q < n * runs; q += nwarps) {
        const int64_t i = q / runs, row = q - i * runs;
        const int64_t slot = (index + i) % capacity;
        const char* s = (const char*)fd.src + ((fd.broadcast ? 0 : i) * runs + row) * rb;
        char* d = (char*)fd.ring + slot * eb + (two_d ? fd.ring_offset + row * fd.ring_pitch : 0);
        if (unit == 16) {
            int u = lane;
            for (; u + 96 < upr; u += 128) {
                uint4 v[4];
#pragma unroll
                for (int k = 0; k < 4; k++) v[k] = __ldcs((const uint4*)s + u + 32 * k);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    if (split_store) {
                        uint2* d2 = (uint2*)(d + (size_t)(u + 32 * k) * 16);
                        __stcs(d2, make_uint2(v[k].x, v[k].y));
                        __stcs(d2 + 1, make_uint2(v[k].z, v[k].w));
                    } else {
                        __stcs((uint4*)d + u + 32 * k, v[k]);
                    }
                }
            }
            for (; u < upr; u += 32) {
                const uint4 v = __ldcs((const uint4*)s + u);
                if (split_store) {
                    uint2* d2 = (uint2*)(d + (size_t)u * 16);
                    __stcs(d2, make_uint2(v.x, v.y));
                    __stcs(d2 + 1, make_uint2(v.z, v.w));
                } else {
                    __stcs((uint4*)d + u, v);
                }
            }
        } else if (unit == 8) {
            int u = lane;
            for (; u + 32 < upr; u += 64) {
                const uint2 v0 = __ldcs((const uint2*)s + u), v1 = __ldcs((const uint2*)s + u + 32);
                __stcs((uint2*)d + u, v0);
                __stcs((uint2*)d + u + 32, v1);
            }
            for (; u < upr; u += 32) __stcs((uint2*)d + u, __ldcs((const uint2*)s + u));
        } else if (unit == 4) {
            for (int u = lane; u < upr; u += 32) ((uint32_t*)d)[u] = ((const uint32_t*)s)[u];
        } else {
            for (int u = lane; u < upr; u += 32) d[u] = s[u];
        }
    }
}

// gather with conversion: one thread per output element
__global__ void replay_sample_kernel(ReplayFields F, const int64_t* __restrict__ indices, int64_t n) {
    const gm_replay_field fd = F.f[blockIdx.y];
    const int in_size = (fd.convert == 0) ? 1 : (fd.convert == 3 ? 2 : 1);
    const int64_t elems = fd.elem_bytes / in_size;  // for convert==0 this is bytes
    const int64_t total = n * elems;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        int64_t i = t / elems, e = t - i * elems;
        int64_t slot = indices[i];
        const char* s = (const char*)fd.ring + slot * fd.elem_bytes;
        switch (fd.convert) {
            case 0: ((char*)fd.dst)[t] = s[e]; break;
            case 1: ((float*)fd.dst)[t] = (float)(((const uint8_t*)s)[e] != 0); break;
            case 2: ((int64_t*)fd.dst)[t] = (int64_t)((const int8_t*)s)[e]; break;
            case 3: ((float*)fd.dst)[t] = __half2float(((const __half*)s)[e]); break;
        }
    }
}

}  // namespace gm

using namespace gm;

extern "C" {

int gm_replay_insert(const gm_replay_field* fields, int32_t n_fields, int64_t capacity, int64_t index, const int64_t* index_dev,
                     int64_t n, void* stream) {
    GM_CHECK_ARG(fields && n_fields > 0 && n_fields <= GM_REPLAY_MAX_FIELDS, "bad field count %d", n_fields);
    GM_CHECK_ARG(capacity > 0 && n >= 0 && n <= capacity && index >= 0 && (index_dev != nullptr || index < capacity), "bad ring arguments");
    if (n == 0) return GM_OK;
    ReplayFields F;
    F.n = n_fields;
    int64_t maxb = 0;
    for (int i = 0; i < n_fields; i++) {
        GM_CHECK_ARG(fields[i].ring && fields[i].src && fields[i].elem_bytes > 0, "field %d: null ring/src", i);
        GM_CHECK_ARG(fields[i].convert == 0 || fields[i].convert == 4, "field %d: insert convert %d", i, fields[i].convert);
        GM_CHECK_ARG(fields[i].rows == 0 ||
                         (fields[i].row_bytes > 0 && fields[i].ring_offset >= 0 &&
                          fields[i].ring_offset + (fields[i].rows - 1) * fields[i].ring_pitch + fields[i].row_bytes <= fields[i].elem_bytes),
                     "field %d: 2-D block does not fit the ring element", i);
        F.f[i] = fields[i];
        maxb = max(maxb, fields[i].elem_bytes * n);
    }
    int64_t blocks = std::min<int64_t>((maxb / 64 + 255) / 256 + 1, 148 * 4);
    dim3 grid((unsigned)blocks, n_fields);
    {
        ProfileScope prof(PROF_REPLAY, (cudaStream_t)stream);
        replay_insert_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(F, capacity, index, index_dev, n);
    }
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int gm_replay_sample(const gm_replay_field* fields, int32_t n_fields, const int64_t* indices, int64_t n, void* stream) {
    GM_CHECK_ARG(fields && n_fields > 0 && n_fields <= GM_REPLAY_MAX_FIELDS && indices, "bad sample arguments");
    if (n == 0) return GM_OK;
    ReplayFields F;
    F.n = n_fields;
    int64_t maxe = 0;
    for (int i = 0; i < n_fields; i++) {
        GM_CHECK_ARG(fields[i].ring && fields[i].dst && fields[i].elem_bytes > 0, "field %d: null ring/dst", i);
        GM_CHECK_ARG(fields[i].convert >= 0 && fields[i].convert <= 3, "field %d: convert %d", i, fields[i].convert);
        F.f[i] = fields[i];
        maxe = max(maxe, fields[i].elem_bytes * n);
    }
    int64_t blocks = std::min<int64_t>((maxe + 255) / 256, 148 * 8);
    dim3 grid((unsigned)blocks, n_fields);
    replay_sample_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(F, indices, n);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

}  // extern "C"
