// Multi-scale combine: per-pixel class probabilities of K image scales averaged on one output grid.
//
// Each member k is a [C, h_k, w_k] f32 probability map (the mean-mode P of pylc_stitch_probs for the image resized
// by s_k and fitted to the tile grid).  Output pixel (y, x) reads P_k at (y_ofs_k[y], x_ofs_k[x]), OpenCV's
// INTER_NEAREST index maps from (w_k, h_k) to (w_full, h_full), and forms, per class, in f32 and in this order
//     sum = P_1[c] + P_2[c] + ... + P_K[c]      Pbar[c] = sum * f32(1/K)
// label = first argmax of Pbar, confidence = min(255, rn(Pbar[label] * 255)) (the expression of the stitch).
// __fadd_rn / __fmul_rn keep the compiler from contracting or reordering, so a NumPy restatement matches bit
// for bit, and with K = 1 the result is the mean-mode label and confidence of the member, resampled.
//
// A thread owns a unit of four consecutive output pixels of a row; consecutive lanes own consecutive units.
// The class loop is outside and keeps a running first maximum, so no C-sized register array is needed; the
// scale loop is inside, unrolled (K is a template parameter) with each member's four source columns and row
// pointer held in registers.  For the common s <= 1 members neighbouring lanes read the same or adjacent
// source columns, so the gathers coalesce.  Loads go through the read-only path.
#include "common.cuh"

namespace pylc {

struct MultiscaleArgs {
    const float *probs[PYLC_MAX_SCALES];
    const int32_t *x_ofs[PYLC_MAX_SCALES], *y_ofs[PYLC_MAX_SCALES];
    int h[PYLC_MAX_SCALES], w[PYLC_MAX_SCALES];
    int C, h_full, w_full, upr;   // upr: 4-pixel units per output row
    long long units;
    float inv_k;
    uint8_t *labels, *rgb, *confidence;
    bool vec;                     // w_full % 4 == 0 and labels / confidence / rgb 4-byte aligned
    bool ofs_vec;                 // every x_ofs 16-byte aligned
    ColourLut lut;
};

template <int K>
__global__ void __launch_bounds__(kThreads) multiscale_combine_kernel(const MultiscaleArgs a) {
    const long long stride = (long long)gridDim.x * kThreads;
    for (long long u = (long long)blockIdx.x * kThreads + threadIdx.x; u < a.units; u += stride) {
        const int y = (int)(u / a.upr);
        const int x = (int)(u - (long long)y * a.upr) * 4;
        const int valid = min(4, a.w_full - x);
        const float *row[K];
        size_t plane[K];
        int sx[K][4];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            plane[k] = (size_t)a.h[k] * a.w[k];
            row[k] = a.probs[k] + (size_t)__ldg(a.y_ofs[k] + y) * a.w[k];
            if (a.ofs_vec && valid == 4) {
                const int4 v = __ldg(reinterpret_cast<const int4 *>(a.x_ofs[k] + x));
                sx[k][0] = v.x, sx[k][1] = v.y, sx[k][2] = v.z, sx[k][3] = v.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) sx[k][j] = __ldg(a.x_ofs[k] + x + min(j, valid - 1));
            }
        }
        float best[4];
        uint32_t lab[4] = {0u, 0u, 0u, 0u};
#pragma unroll 2
        for (int c = 0; c < a.C; ++c) {
            float s[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) s[j] = __ldg(row[0] + sx[0][j]);
#pragma unroll
            for (int k = 1; k < K; ++k)
#pragma unroll
                for (int j = 0; j < 4; ++j) s[j] = __fadd_rn(s[j], __ldg(row[k] + sx[k][j]));
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float p = __fmul_rn(s[j], a.inv_k);
                if (c == 0 || p > best[j]) {   // strict: first maximum wins (np.argmax)
                    best[j] = p;
                    lab[j] = (uint32_t)c;
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k) row[k] += plane[k];
        }
        const size_t o = (size_t)y * a.w_full + x;
        if (a.labels) {
            if (a.vec) *reinterpret_cast<unsigned int *>(a.labels + o) = lab[0] | (lab[1] << 8) | (lab[2] << 16) | (lab[3] << 24);
            else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < valid) a.labels[o + j] = (uint8_t)lab[j];
            }
        }
        if (a.confidence) {
            uint32_t q[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) q[j] = min(255u, __float2uint_rn(__fmul_rn(best[j], 255.f)));
            if (a.vec) *reinterpret_cast<unsigned int *>(a.confidence + o) = q[0] | (q[1] << 8) | (q[2] << 16) | (q[3] << 24);
            else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < valid) a.confidence[o + j] = (uint8_t)q[j];
            }
        }
        if (a.rgb) {
            uint32_t p[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) p[j] = a.lut.rgb[lab[j]];
            uint8_t *d = a.rgb + o * 3;
            if (a.vec) {   // 12 bytes at a 4-byte aligned address: three words
                unsigned int *d4 = reinterpret_cast<unsigned int *>(d);
                d4[0] = (p[0] & 0xFFFFFFu) | (p[1] << 24);
                d4[1] = ((p[1] >> 8) & 0xFFFFu) | (p[2] << 16);
                d4[2] = ((p[2] >> 16) & 0xFFu) | (p[3] << 8);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < valid) {
                        d[3 * j] = (uint8_t)p[j];
                        d[3 * j + 1] = (uint8_t)(p[j] >> 8);
                        d[3 * j + 2] = (uint8_t)(p[j] >> 16);
                    }
            }
        }
    }
}

}  // namespace pylc

using namespace pylc;

extern "C" int pylc_multiscale_combine(const float *const *probs, const int32_t *const *x_ofs, const int32_t *const *y_ofs,
                                       const int *h, const int *w, int K, int C, int h_full, int w_full, const uint8_t *lut_rgb,
                                       uint8_t *labels, uint8_t *rgb, uint8_t *confidence, pylc_stream_t stream) {
    if (K < 1 || K > PYLC_MAX_SCALES || !probs || !x_ofs || !y_ofs || !h || !w || h_full < 1 || w_full < 1) return PYLC_ERR_ARG;
    if (!labels && !rgb && !confidence) return PYLC_ERR_ARG;
    if (rgb && !lut_rgb) return PYLC_ERR_ARG;
    if (C < 1 || C > PYLC_MAX_CLASSES) return PYLC_ERR_CLASSES;
    MultiscaleArgs a;
    bool ofs_vec = true;
    for (int k = 0; k < PYLC_MAX_SCALES; ++k) {
        a.probs[k] = nullptr; a.x_ofs[k] = a.y_ofs[k] = nullptr; a.h[k] = a.w[k] = 0;
        if (k >= K) continue;
        if (!probs[k] || !x_ofs[k] || !y_ofs[k] || h[k] < 1 || w[k] < 1) return PYLC_ERR_ARG;
        a.probs[k] = probs[k]; a.x_ofs[k] = x_ofs[k]; a.y_ofs[k] = y_ofs[k]; a.h[k] = h[k]; a.w[k] = w[k];
        ofs_vec = ofs_vec && (uintptr_t)x_ofs[k] % 16 == 0;
    }
    a.C = C; a.h_full = h_full; a.w_full = w_full;
    a.upr = (w_full + 3) / 4;
    a.units = (long long)h_full * a.upr;
    a.inv_k = (float)(1.0 / K);
    a.labels = labels; a.rgb = rgb; a.confidence = confidence;
    a.vec = w_full % 4 == 0 && (uintptr_t)labels % 4 == 0 && (uintptr_t)rgb % 4 == 0 && (uintptr_t)confidence % 4 == 0;
    a.ofs_vec = ofs_vec;
    if (rgb) build_colour_lut(lut_rgb, C, &a.lut);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long want = (a.units + kThreads - 1) / kThreads;
    const unsigned grid = (unsigned)(want < 8LL * sms ? want : 8LL * sms);
    cudaStream_t st = (cudaStream_t)stream;
    switch (K) {
        case 1: multiscale_combine_kernel<1><<<grid, kThreads, 0, st>>>(a); break;
        case 2: multiscale_combine_kernel<2><<<grid, kThreads, 0, st>>>(a); break;
        case 3: multiscale_combine_kernel<3><<<grid, kThreads, 0, st>>>(a); break;
        case 4: multiscale_combine_kernel<4><<<grid, kThreads, 0, st>>>(a); break;
        case 5: multiscale_combine_kernel<5><<<grid, kThreads, 0, st>>>(a); break;
        case 6: multiscale_combine_kernel<6><<<grid, kThreads, 0, st>>>(a); break;
        case 7: multiscale_combine_kernel<7><<<grid, kThreads, 0, st>>>(a); break;
        default: multiscale_combine_kernel<8><<<grid, kThreads, 0, st>>>(a); break;
    }
    return finish_launch();
}
