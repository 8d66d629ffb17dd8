// Camera-gradient reductions shared by the preprocess backward (32 floats: dL/dviewmatrix, dL/dprojmatrix) and the
// decode backward (3 floats: dL/dcamera_center).  Two stages, both in a fixed order, so that the same inputs give
// bitwise the same camera gradient on every run (pose optimisation stays reproducible; no float atomics):
//   1. every CTA of CAM_ROWS threads sums its threads' 32-vectors into one row of a caller-owned workspace;
//   2. camera_sum_kernel (one CTA) sums the rows and writes the result.
#pragma once
#include "common.cuh"

namespace splatco {

constexpr int CAM_ROWS = 256;      // rows (Gaussians / anchors) per partial
constexpr int CAM_COLS = 32;       // floats per partial

inline size_t camera_grad_ws_bytes(int n) {
    return align_up((size_t)(n > 0 ? ceil_div(n, CAM_ROWS) : 1) * CAM_COLS * sizeof(float));
}

// Column sums of a 32-vector per lane over the warp (transposing butterfly, 31 shuffles): lane l returns column l.
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[CAM_COLS]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool hi = lane & s;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float keep = hi ? v[i + s] : v[i], send = hi ? v[i] : v[i + s];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0];
}

// Stage 1, called by all CAM_ROWS threads of the CTA: part[blockIdx.x][c] = sum over the CTA's threads of v[c].
__device__ __forceinline__ void camera_block_partial(float (&v)[CAM_COLS], float *__restrict__ part) {
    __shared__ float s_w[CAM_ROWS / 32][CAM_COLS];
    const float w = warp_transpose_sum32(v);
    s_w[threadIdx.x >> 5][threadIdx.x & 31] = w;
    __syncthreads();
    if (threadIdx.x < CAM_COLS) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < CAM_ROWS / 32; ++k) t += s_w[k][threadIdx.x];
        part[(size_t)blockIdx.x * CAM_COLS + threadIdx.x] = t;
    }
}

// Stage 2, one CTA of 1024 threads: t[c] = sign * sum_b part[b][c]; out0[c] = t[c] for c < split and
// out1[c - split] = t[c] for split <= c < ncols.  Warp w takes the rows b = w mod 32 (coalesced: lane = column), four
// independent accumulators each; the 32 warp sums are added in warp order.
static __global__ void __launch_bounds__(1024)
camera_sum_kernel(int nb, int ncols, int split, float sign, const float *__restrict__ part, float *__restrict__ out0,
                  float *__restrict__ out1) {
    __shared__ float s_w[32][CAM_COLS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int b = warp; b < nb; b += 4 * 32) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = b + 32 * k;
            if (r < nb) acc[k] += __ldg(part + (size_t)r * CAM_COLS + lane);
        }
    }
    s_w[warp][lane] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
    __syncthreads();
    if (threadIdx.x < CAM_COLS) {
        float t = 0.f;
        for (int w = 0; w < 32; ++w) t += s_w[w][threadIdx.x];
        const int c = threadIdx.x;
        if (c < split) out0[c] = sign * t;
        else if (c < ncols) out1[c - split] = sign * t;
    }
}

}  // namespace splatco
