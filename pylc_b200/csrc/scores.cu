// Proper scores of the mean-mode probabilities against the full-resolution ground truth (temperature fitting).
//
// Each full-resolution pixel (y, x) reads P at the fitted pixel (y_ofs[y], x_ofs[x]) -- the label map's OpenCV
// INTER_NEAREST index maps -- and, with g its encoded true class, scores in f32
//     nll   = -logf(fmaxf(P[g], 1e-12f))
//     brier = sum over c in class order of (P[c] - [c == g])^2
// A block owns whole destination rows (rows b, b + grid, ...), so the per-row y_ofs and row pointers are loaded
// once per row and there is no integer division in the loop.  A thread owns units of four consecutive pixels of
// a row; x_ofs is monotone, so a warp's gathers from one class plane fall on a short run of the fitted row.
// The NLL-only form reads one plane per pixel, the Brier form all C.
//
// Determinism: every thread accumulates its pixels in f64 in a fixed order, a block reduces its threads with a
// fixed shuffle tree and a fixed warp order, and a second single-block launch adds the block partials in block
// order.  The grid depends only on h_full, so the same inputs give the same bits on every call.
#include <math.h>

#include "common.cuh"

namespace pylc {

struct ScoreArgs {
    const float *probs;
    const int32_t *x_ofs, *y_ofs;
    const uint8_t *truth;
    int C, h, w, h_full, w_full;
    double *partials;                 // [gridDim.x][2]
};

__device__ __forceinline__ void block_sum2(double &a, double &b, double *s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
        b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
    }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        s_red[2 * warp] = a;
        s_red[2 * warp + 1] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        a = s_red[0];
        b = s_red[1];
        for (int i = 1; i < kWarps; ++i) {
            a += s_red[2 * i];
            b += s_red[2 * i + 1];
        }
    }
}

template <bool BRIER>
__global__ void __launch_bounds__(kThreads) prob_scores_kernel(ScoreArgs a) {
    __shared__ double s_red[2 * kWarps];
    const size_t plane = (size_t)a.h * a.w;
    double acc_n = 0.0, acc_b = 0.0;
    for (int y = blockIdx.x; y < a.h_full; y += gridDim.x) {
        const float *row = a.probs + (size_t)__ldg(a.y_ofs + y) * a.w;
        const uint8_t *truth = a.truth + (size_t)y * a.w_full;
        for (int x = threadIdx.x * 4; x < a.w_full; x += kThreads * 4) {
            const int valid = min(4, a.w_full - x);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (j < valid) {
                    const int sx = __ldg(a.x_ofs + x + j);
                    const int g = __ldg(truth + x + j);
                    float q = 0.f;                         // a class >= C has no plane: scored as probability 0
                    if (BRIER) {
                        float s = 0.f;
                        for (int c = 0; c < a.C; ++c) {
                            const float p = __ldg(row + c * plane + sx);
                            const float d = c == g ? p - 1.f : p;
                            if (c == g) q = p;
                            s = fmaf(d, d, s);
                        }
                        acc_b += (double)s;
                    } else if (g < a.C) {
                        q = __ldg(row + g * plane + sx);
                    }
                    acc_n += (double)(-logf(fmaxf(q, 1e-12f)));
                }
            }
        }
    }
    block_sum2(acc_n, acc_b, s_red);
    if (threadIdx.x == 0) {
        a.partials[2 * blockIdx.x] = acc_n;
        a.partials[2 * blockIdx.x + 1] = acc_b;
    }
}

// sums[0..1] = the block partials added in block order (strided per thread, then the fixed tree of block_sum2)
__global__ void __launch_bounds__(kThreads) prob_scores_finish_kernel(const double *partials, int n, double *sums) {
    __shared__ double s_red[2 * kWarps];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < n; i += kThreads) {
        a += partials[2 * i];
        b += partials[2 * i + 1];
    }
    block_sum2(a, b, s_red);
    if (threadIdx.x == 0) {
        sums[0] = a;
        sums[1] = b;
    }
}

}  // namespace pylc

using namespace pylc;

extern "C" int pylc_prob_scores(const float *probs, int C, int h, int w, const int32_t *x_ofs, const int32_t *y_ofs, int h_full,
                                int w_full, const uint8_t *y_true_full, int want_brier, double *workspace, double *sums,
                                pylc_stream_t stream) {
    if (!probs || !x_ofs || !y_ofs || !y_true_full || !workspace || !sums) return PYLC_ERR_ARG;
    if (h < 1 || w < 1 || h_full < 1 || w_full < 1) return PYLC_ERR_ARG;
    if (C < 1 || C > PYLC_MAX_CLASSES) return PYLC_ERR_CLASSES;
    ScoreArgs a;
    a.probs = probs; a.x_ofs = x_ofs; a.y_ofs = y_ofs; a.truth = y_true_full;
    a.C = C; a.h = h; a.w = w; a.h_full = h_full; a.w_full = w_full;
    a.partials = workspace;
    const int grid = h_full < PYLC_SCORES_BLOCKS ? h_full : PYLC_SCORES_BLOCKS;
    cudaStream_t st = (cudaStream_t)stream;
    if (want_brier) prob_scores_kernel<true><<<grid, kThreads, 0, st>>>(a);
    else prob_scores_kernel<false><<<grid, kThreads, 0, st>>>(a);
    int rc = finish_launch();
    if (rc) return rc;
    prob_scores_finish_kernel<<<1, kThreads, 0, st>>>(workspace, grid, sums);
    return finish_launch();
}
