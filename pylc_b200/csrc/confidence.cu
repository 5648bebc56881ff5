// Confidence plane to full resolution + reliability table (calibration counts).
//
// The fitted u8 confidence of pylc_stitch_probs is resampled with the label map's OpenCV INTER_NEAREST
// index maps (x_ofs / y_ofs, as pylc_resample_encode_confusion uses them), so the full-resolution
// confidence of a pixel belongs to the same fitted pixel as its predicted label.  With the full-resolution
// predicted and true classes the kernel also counts every pixel into rel[pred][q][pred == true].
//
// A thread owns units of four consecutive destination pixels of a row; consecutive lanes own consecutive
// units, so the label planes and the output stream through in 128-byte warp rows.  The table is privatised
// per CTA in shared memory as u32 (C * 256 * 2 words: 18 KB at C = 9) and flushed to the i64 table once per
// CTA.  Before each shared-memory atomic the warp aggregates equal keys with __match_any_sync: a uniform
// region (one class, one confidence level, all right or all wrong) costs one atomic per warp instead of 32,
// which is what keeps a saturated or constant confidence map from serialising on one counter.
#include "common.cuh"

namespace pylc {

struct ConfResampleArgs {
    const uint8_t *conf;
    const int32_t *x_ofs, *y_ofs;
    const uint8_t *pred, *truth;
    int h, w, h_full, w_full, C, upr;   // upr: 4-pixel units per destination row
    long long units;
    uint8_t *out;
    long long *rel;
    bool vec;                           // w_full % 4 == 0 and every full-resolution plane 4-byte aligned
    bool ofs_vec;                       // x_ofs 16-byte aligned
};

__device__ __forceinline__ void load4(const uint8_t *p, bool vec, int valid, uint32_t (&v)[4]) {
    if (vec) {
        const uint32_t w = __ldg(reinterpret_cast<const unsigned int *>(p));
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (w >> (8 * j)) & 0xFFu;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = j < valid ? __ldg(p + j) : 0u;
    }
}

template <bool REL>
__global__ void __launch_bounds__(kThreads) confidence_resample_kernel(ConfResampleArgs a) {
    extern __shared__ unsigned s_rel[];
    const int n_keys = a.C * 512;
    if (REL) {
        for (int i = threadIdx.x; i < n_keys; i += kThreads) s_rel[i] = 0;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * kThreads;
    // the loop bound depends on the warp's first unit only, so every lane of a warp runs the same iterations
    // and __match_any_sync sees a converged warp
    for (long long base = (long long)blockIdx.x * kThreads + (threadIdx.x & ~31); base < a.units; base += stride) {
        const long long u = base + lane;
        int valid = 0;
        uint32_t q[4] = {0u, 0u, 0u, 0u}, p[4] = {0u, 0u, 0u, 0u}, t[4] = {0u, 0u, 0u, 0u};
        if (u < a.units) {
            const int y = (int)(u / a.upr);
            const int x = (int)(u - (long long)y * a.upr) * 4;
            valid = min(4, a.w_full - x);
            const uint8_t *src = a.conf + (size_t)__ldg(a.y_ofs + y) * a.w;
            int sx[4];
            if (a.ofs_vec && valid == 4) {
                const int4 v = __ldg(reinterpret_cast<const int4 *>(a.x_ofs + x));
                sx[0] = v.x, sx[1] = v.y, sx[2] = v.z, sx[3] = v.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) sx[j] = j < valid ? __ldg(a.x_ofs + x + j) : 0;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) q[j] = j < valid ? (uint32_t)src[sx[j]] : 0u;
            const size_t o = (size_t)y * a.w_full + x;
            if (a.out) {
                if (a.vec) *reinterpret_cast<unsigned int *>(a.out + o) = q[0] | (q[1] << 8) | (q[2] << 16) | (q[3] << 24);
                else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (j < valid) a.out[o + j] = (uint8_t)q[j];
                }
            }
            if (REL) {
                load4(a.pred + o, a.vec, valid, p);
                load4(a.truth + o, a.vec, valid, t);
            }
        }
        if (REL) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t key = 0xFFFFFFFFu;
                if (j < valid && p[j] < (uint32_t)a.C && t[j] < (uint32_t)a.C) key = ((p[j] << 8 | q[j]) << 1) | (p[j] == t[j] ? 1u : 0u);
                const unsigned peers = __match_any_sync(0xFFFFFFFFu, key);
                if (key != 0xFFFFFFFFu && lane == __ffs(peers) - 1) atomicAdd(&s_rel[key], (unsigned)__popc(peers));
            }
        }
    }
    if (REL) {
        __syncthreads();
        for (int i = threadIdx.x; i < n_keys; i += kThreads)
            if (s_rel[i]) atomicAdd(reinterpret_cast<unsigned long long *>(&a.rel[i]), (unsigned long long)s_rel[i]);
    }
}

}  // namespace pylc

using namespace pylc;

extern "C" int pylc_confidence_resample(const uint8_t *confidence, int h, int w, const int32_t *x_ofs, const int32_t *y_ofs,
                                        int h_full, int w_full, const uint8_t *y_pred_full, const uint8_t *y_true_full, int C,
                                        uint8_t *confidence_full, int64_t *reliability, pylc_stream_t stream) {
    if (!confidence || !x_ofs || !y_ofs || h < 1 || w < 1 || h_full < 1 || w_full < 1) return PYLC_ERR_ARG;
    if (!confidence_full && !reliability) return PYLC_ERR_ARG;
    if (reliability && (!y_pred_full || !y_true_full)) return PYLC_ERR_ARG;
    if (reliability && (C < 1 || C > PYLC_MAX_CLASSES)) return PYLC_ERR_CLASSES;
    ConfResampleArgs a;
    a.conf = confidence; a.x_ofs = x_ofs; a.y_ofs = y_ofs;
    a.pred = y_pred_full; a.truth = y_true_full;
    a.h = h; a.w = w; a.h_full = h_full; a.w_full = w_full; a.C = reliability ? C : 0;
    a.upr = (w_full + 3) / 4;
    a.units = (long long)h_full * a.upr;
    a.out = confidence_full;
    a.rel = reinterpret_cast<long long *>(reliability);
    a.vec = w_full % 4 == 0 && (uintptr_t)confidence_full % 4 == 0 && (uintptr_t)y_pred_full % 4 == 0 &&
            (uintptr_t)y_true_full % 4 == 0;
    a.ofs_vec = (uintptr_t)x_ofs % 16 == 0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long want = (a.units + kThreads - 1) / kThreads;
    cudaStream_t st = (cudaStream_t)stream;
    if (reliability) {
        // two CTAs per SM: each flushes up to C * 512 counters, so fewer, longer-lived CTAs
        const unsigned grid = (unsigned)(want < 2LL * sms ? want : 2LL * sms);
        const size_t smem = (size_t)C * 512 * sizeof(unsigned);
        const cudaError_t e = cudaFuncSetAttribute(confidence_resample_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        confidence_resample_kernel<true><<<grid, kThreads, smem, st>>>(a);
    } else {
        const unsigned grid = (unsigned)(want < 8LL * sms ? want : 8LL * sms);
        confidence_resample_kernel<false><<<grid, kThreads, 0, st>>>(a);
    }
    return finish_launch();
}
