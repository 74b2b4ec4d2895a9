// Classifier head (reference roko/rnn_model.py:59 fc4) fused with the caller's argmax
// (reference roko/inference.py:116):  logits[m][c] = b4[c] + sum_q W4[c][q] * h[m][q],
// label[m] = first index of the maximum.  One warp per (window, position) row: the 1 KB row of
// the last GRU layer is read once with 32-byte lane chunks, W4 lives in 40 registers per lane.
#include "common.cuh"

namespace roko {

constexpr int HD_THREADS = 256;

__global__ void __launch_bounds__(HD_THREADS)
head_kernel(const float* __restrict__ h, const float* __restrict__ w4, const float* __restrict__ b4,
            float* __restrict__ logits, uint8_t* __restrict__ labels, int rows) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * HD_THREADS + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * HD_THREADS) >> 5;
    float w[CLASSES][8];
#pragma unroll
    for (int c = 0; c < CLASSES; ++c) {
        const float4 a = *reinterpret_cast<const float4*>(w4 + c * OUT_W + lane * 8);
        const float4 b = *reinterpret_cast<const float4*>(w4 + c * OUT_W + lane * 8 + 4);
        w[c][0] = a.x; w[c][1] = a.y; w[c][2] = a.z; w[c][3] = a.w;
        w[c][4] = b.x; w[c][5] = b.y; w[c][6] = b.z; w[c][7] = b.w;
    }
    float bias[CLASSES];
#pragma unroll
    for (int c = 0; c < CLASSES; ++c) bias[c] = b4[c];

    // two rows per warp and iteration: both rows' loads are in flight together (one row at a time left the kernel at half the
    // HBM rate: a warp waited out the latency of 1 KB before asking for the next)
    for (int m0 = 2 * warp; m0 < rows; m0 += 2 * nwarps) {
        const bool two = m0 + 1 < rows;
        const float4* p0 = reinterpret_cast<const float4*>(h + (size_t)m0 * OUT_W + lane * 8);
        const float4* p1 = reinterpret_cast<const float4*>(h + (size_t)(two ? m0 + 1 : m0) * OUT_W + lane * 8);
        const float4 a0 = p0[0], b0 = p0[1], a1 = p1[0], b1 = p1[1];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            if (r == 1 && !two) break;
            const float4 a = r ? a1 : a0, b = r ? b1 : b0;
            const int m = m0 + r;
            const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
            float s[CLASSES];
#pragma unroll
            for (int c = 0; c < CLASSES; ++c) {
                float t = 0.f;
#pragma unroll
                for (int q = 0; q < 8; ++q) t = fmaf(w[c][q], v[q], t);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
                s[c] = t + bias[c];
            }
            if (lane == 0) {
                int best = 0;
                float bv = s[0];
#pragma unroll
                for (int c = 1; c < CLASSES; ++c)
                    if (s[c] > bv) { bv = s[c]; best = c; }      // strict '>' keeps the first maximum
                if (labels) labels[m] = (uint8_t)best;
                if (logits) {
#pragma unroll
                    for (int c = 0; c < CLASSES; ++c) logits[(size_t)m * CLASSES + c] = s[c];
                }
            }
        }
    }
}

cudaError_t launch_head(const float* h, const float* w4, const float* b4, float* logits, uint8_t* labels,
                        int rows, int max_blocks, cudaStream_t s) {
    if (rows <= 0) return cudaSuccess;
    if (max_blocks < 1) return cudaErrorInvalidValue;
    int blocks = ((rows + 1) / 2 + (HD_THREADS / 32) - 1) / (HD_THREADS / 32);
    if (blocks > max_blocks) blocks = max_blocks;
    head_kernel<<<blocks, HD_THREADS, 0, s>>>(h, w4, b4, logits, labels, rows);
    return cudaGetLastError();
}

}  // namespace roko
