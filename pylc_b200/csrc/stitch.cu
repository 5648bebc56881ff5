// Fused stitch + softmax + argmax + colourise (tools.reconstruct, utils/tools.py:239-313).
//
// Closed form of the reference's in-place band merging (SURVEY.md A.3), S = T/2:
//   output block (ky,kx) of S x S pixels draws on one quadrant of up to four tiles
//     Hrow(i, ty, x) = raw L[i,0] / L[i,nc-1] at the left / right border,
//                      else (softmax(L[i,kx-1]) + softmax(L[i,kx])) / 2
//     M(y, x)        = Hrow(0) / Hrow(nr-1) at the top / bottom border,
//                      else (softmax(Hrow(ky-1)) + softmax(Hrow(ky))) / 2
//   so corners are raw logits, edges one softmax-average, the interior a double softmax.
// Every logit is read exactly once; a CTA owns a slab of rows of one block, so the block kind
// (how many tiles feed it) is uniform per CTA and there is no divergence.
//
// Probabilities (pylc_stitch_probs): P(y, x) = the mean over the covering tiles of their softmaxes.  In the
// terms above it is softmax(L) on corners (and everywhere when S == T), exactly M on edges, and the sum of
// the two strip sums x 1/4 in the interior, taken before the second softmax.  MODE selects the labels:
// PYLC_STITCH_REFERENCE (0) takes the first argmax of M (the reference's labels), PYLC_STITCH_MEAN (1) that
// of P, and then `stitched` holds P instead of M.  CONF adds the u8 plane q = min(255, rn(P[label] * 255)).
// MODE = 0 without CONF is the reference's stitch: labels, rgb and M.
//
// Temperature: in mean mode every softmax the kernels evaluate is a softmax of raw tile logits, so
// softmax(L / T) is exp_cls with k = fl32(log2(e) / T) in place of log2(e).  The mean-mode instantiations
// take k from the kernel argument `k`; the reference-mode instantiations ignore it and keep the
// compile-time constant.
#include <type_traits>

#include "common.cuh"

namespace pylc {

struct StitchArgs {
    const float *logits;            // contiguous [nr*nc, C, T, T] or NULL
    const float *const *batches;    // device array of batch pointers or NULL
    int tiles_per_batch;
    int nr, nc, C, T, S;
    int overlap;                    // 1: S == T/2, 0: S == T
    int h, w, nbx, nby;
    int rows_per_cta, slabs, upr;   // units (PX pixels) per block row
    uint8_t *labels;
    uint8_t *rgb;
    float *stitched;
};

// What emit_unit writes, the same for both kernel forms; every pointer is nullable.
struct StitchOut {
    int h, w;                       // output map size
    uint8_t *labels;                // [h, w]
    uint8_t *rgb;                   // [h, w, 3]
    float *stitched;                // [C, h, w]: M, or P in mean mode
    uint8_t *confidence;            // [h, w], written by the CONF instantiations
};

// The output fields are kept in the argument structs rather than in a StitchOut member: moving them changes the
// kernels' parameter layout, and with it the code ptxas generates for every stitch_kernel instantiation.
template <class Args>
__device__ __forceinline__ StitchOut stitch_out(const Args &a, uint8_t *conf) {
    return {a.h, a.w, a.labels, a.rgb, a.stitched, conf};
}

__device__ __forceinline__ const float *tile_base(const StitchArgs &a, int i, int j) {
    const int k = i * a.nc + j;
    const size_t tile_elems = (size_t)a.C * a.T * a.T;
    if (a.logits) return a.logits + (size_t)k * tile_elems;
    const int b = k / a.tiles_per_batch;
    return a.batches[b] + (size_t)(k - b * a.tiles_per_batch) * tile_elems;
}

template <int PX>
struct Vec;
template <>
struct Vec<2> {
    static __device__ __forceinline__ void load(const float *p, float (&o)[2]) {
        const float2 t = ld_stream_f2(p);
        o[0] = t.x;
        o[1] = t.y;
    }
    static __device__ __forceinline__ void store(float *p, const float (&v)[2]) {
        *reinterpret_cast<float2 *>(p) = make_float2(v[0], v[1]);
    }
};
template <>
struct Vec<1> {
    static __device__ __forceinline__ void load(const float *p, float (&o)[1]) { o[0] = __ldg(p); }
    static __device__ __forceinline__ void store(float *p, const float (&v)[1]) { *p = v[0]; }
};

// softmax over the class axis, fp32, split in two steps so that the scale by 1/sum can be folded into
// whatever consumes the probabilities:
//   exp_cls     : v[c] <- 2^(v[c]*k - max*k), returns r = 1/sum.  k = log2(e) for logits; for the SUM of
//                 two probability vectors (an average that was never scaled by 1/2) k = log2(e)/2, which
//                 is bit-identical to halving first because scaling by a power of two is exact.
//                 SUBMAX = false skips the max subtraction: inputs that are probabilities (or sums of
//                 two) lie in [0, 2], so 2^(x*k) cannot overflow and softmax is shift-invariant.
//   combine_cls : a[c] <- (a[c]*ra + b[c]*rb) * w as one FMUL + one FFMA per class.
// All classes of a pixel share the same rounded max*k and the same reciprocals, so neither
// approximation can reorder classes; values stay within ~1e-6 relative of torch's CPU softmax.
template <int CMAX, int PX, bool SUBMAX>
__device__ __forceinline__ void exp_cls(float (&v)[CMAX][PX], int C, float k, float (&r)[PX]) {
#pragma unroll
    for (int j = 0; j < PX; ++j) {
        float ms = 0.f;
        if (SUBMAX) {
            float m = v[0][j];
#pragma unroll
            for (int c = 1; c < CMAX; ++c)
                if (c < C) m = fmaxf(m, v[c][j]);
            ms = -m * k;
        }
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < C) {
                const float e = ex2_approx(SUBMAX ? fmaf(v[c][j], k, ms) : v[c][j] * k);
                v[c][j] = e;
                s += e;
            }
        r[j] = rcp_approx(s);
    }
}

template <int CMAX, int PX>
__device__ __forceinline__ void combine_cls(float (&a)[CMAX][PX], const float (&ra)[PX], const float (&b)[CMAX][PX],
                                            const float (&rb)[PX], int C, float w) {
#pragma unroll
    for (int j = 0; j < PX; ++j) {
        const float wa = ra[j] * w, wb = rb[j] * w;
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < C) a[c][j] = fmaf(a[c][j], wa, b[c][j] * wb);
    }
}

template <int CMAX, int PX>
__device__ __forceinline__ void load_cls(const float *p, size_t cstride, int C, float (&v)[CMAX][PX]) {
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
        if (c < C) Vec<PX>::load(p + c * cstride, v[c]);
}

// Writes one unit: optional f32 map, first-maximum argmax (np.argmax), label bytes, optional RGB and, with
// CONF, the confidence byte of P at the label.
template <int CMAX, int PX, bool CONF = false>
__device__ __forceinline__ void emit_unit(const StitchOut &a, const uint32_t *s_lut, int C, const float (&m)[CMAX][PX],
                                          const float (&p)[CMAX][PX], size_t o) {
    if (a.stitched) {
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < C) Vec<PX>::store(a.stitched + (size_t)c * a.h * a.w + o, m[c]);
    }
    uint32_t lab[PX];
    float pl[PX];
#pragma unroll
    for (int j = 0; j < PX; ++j) {
        float best = m[0][j];
        uint32_t bi = 0;
        if constexpr (CONF) pl[j] = p[0][j];
#pragma unroll
        for (int c = 1; c < CMAX; ++c)
            if (c < C && m[c][j] > best) {  // strict: first maximum wins (np.argmax)
                best = m[c][j];
                bi = c;
                if constexpr (CONF) pl[j] = p[c][j];
            }
        lab[j] = bi;
    }
    if (a.labels) {
        if (PX == 2) *reinterpret_cast<uint16_t *>(a.labels + o) = (uint16_t)(lab[0] | (lab[PX - 1] << 8));
        else a.labels[o] = (uint8_t)lab[0];
    }
    if constexpr (CONF) {
        if (a.confidence) {
            uint32_t q[PX];
#pragma unroll
            for (int j = 0; j < PX; ++j) q[j] = min(255u, __float2uint_rn(pl[j] * 255.f));
            if (PX == 2) *reinterpret_cast<uint16_t *>(a.confidence + o) = (uint16_t)(q[0] | (q[PX - 1] << 8));
            else a.confidence[o] = (uint8_t)q[0];
        }
    }
    if (a.rgb) {
        uint8_t *d = a.rgb + o * 3;
        if (PX == 2) {
            const uint32_t p0 = s_lut[lab[0]], p1 = s_lut[lab[PX - 1]];
            uint16_t *d2 = reinterpret_cast<uint16_t *>(d);
            d2[0] = (uint16_t)p0;
            d2[1] = (uint16_t)((p0 >> 16) | (p1 << 8));
            d2[2] = (uint16_t)(p1 >> 8);
        } else {
            const uint32_t p0 = s_lut[lab[0]];
            d[0] = (uint8_t)p0;
            d[1] = (uint8_t)(p0 >> 8);
            d[2] = (uint8_t)(p0 >> 16);
        }
    }
}

// P of a corner block (or of any block when S == T): softmax of the raw logits, e[c] * (1 / sum).
template <int CMAX, int PX>
__device__ __forceinline__ void softmax_copy(const float (&v)[CMAX][PX], int C, float k, float (&p)[CMAX][PX]) {
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
#pragma unroll
        for (int j = 0; j < PX; ++j) p[c][j] = v[c][j];
    float r[PX];
    exp_cls<CMAX, PX, true>(p, C, k, r);
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
#pragma unroll
        for (int j = 0; j < PX; ++j)
            if (c < C) p[c][j] *= r[j];
}

// P of an interior block: the two strip SUMS (each the sum of two softmaxes) added and scaled by 1/4.
template <int CMAX, int PX>
__device__ __forceinline__ void quarter_sum(const float (&s0)[CMAX][PX], const float (&s1)[CMAX][PX], int C, float (&p)[CMAX][PX]) {
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
#pragma unroll
        for (int j = 0; j < PX; ++j)
            if (c < C) p[c][j] = (s0[c][j] + s1[c][j]) * 0.25f;
}

// Source tiles of output block (ky, kx): strip s in {0,1} reads tile row ti[s] from tile row ty0[s] on, column
// q in {0,1} tile column tj[q] from tile column tx0[q] on.  NH: tiles per strip (1 border / 2 interior
// columns); NV: strips (1 border / 2 interior rows).
template <int NH, int NV, class Args>
__device__ __forceinline__ void select_tiles(const Args &a, int ky, int kx, int (&ti)[2], int (&ty0)[2], int (&tj)[2],
                                             int (&tx0)[2]) {
    const int S = a.S;
    if (!a.overlap) {
        ti[0] = ky; ty0[0] = 0; tj[0] = kx; tx0[0] = 0;
    } else {
        if (NV == 1) {
            ti[0] = ky == 0 ? 0 : a.nr - 1;
            ty0[0] = ky == 0 ? 0 : S;
        } else {
            ti[0] = ky - 1; ty0[0] = S;
            ti[1] = ky;     ty0[1] = 0;
        }
        if (NH == 1) {
            tj[0] = kx == 0 ? 0 : a.nc - 1;
            tx0[0] = kx == 0 ? 0 : S;
        } else {
            tj[0] = kx - 1; tx0[0] = S;
            tj[1] = kx;     tx0[1] = 0;
        }
    }
}

// Column merge of one strip at interior columns: the two tiles' softmaxes averaged into v0.  When a second
// softmax follows (NV == 2) the strip keeps the SUM of the two and the 1/2 moves into that softmax's scale.
template <int CMAX, int PX, int NV>
__device__ __forceinline__ void merge_columns(float (&v0)[CMAX][PX], float (&v1)[CMAX][PX], int C, float kl) {
    float r0[PX], r1[PX];
    exp_cls<CMAX, PX, true>(v0, C, kl, r0);
    exp_cls<CMAX, PX, true>(v1, C, kl, r1);
    combine_cls<CMAX, PX>(v0, r0, v1, r1, C, NV == 2 ? 1.f : 0.5f);
}

// Everything after the column merge, given the merged strips s0 and s1 (the same array when NV == 1): P where it
// is not M itself, the row merge into s0 (mean mode needs no second softmax in the interior) and the write of
// output pixel (y0 + yl, x0 + xl): block origin and the unit's place in the block.  The offset is formed after the
// merge, as the kernels have always done; computing it before changes the generated code.
template <int CMAX, int PX, int NH, int NV, int MODE, bool CONF>
__device__ __forceinline__ void merge_rows_emit(const StitchOut &out, const uint32_t *s_lut, int C, float kl,
                                                float (&s0)[CMAX][PX], float (&s1)[CMAX][PX], int y0, int yl, int x0, int xl) {
    constexpr bool NEED_P = MODE == 1 || CONF;
    float p[CMAX][PX];          // P where it is not M itself (interior and corner blocks)
    if constexpr (NEED_P && NV == 2 && NH == 2) quarter_sum<CMAX, PX>(s0, s1, C, p);
    if constexpr (NEED_P && NV == 1 && NH == 1) softmax_copy<CMAX, PX>(s0, C, kl, p);
    if (NV == 2 && !(MODE == 1 && NH == 2)) {
        float r0[PX], r1[PX];
        if (NH == 2) {   // inputs: sums of two probability vectors, in [0, 2]
            exp_cls<CMAX, PX, false>(s0, C, 0.5f * kLog2e, r0);
            exp_cls<CMAX, PX, false>(s1, C, 0.5f * kLog2e, r1);
        } else {         // left / right border: raw logits
            exp_cls<CMAX, PX, true>(s0, C, kl, r0);
            exp_cls<CMAX, PX, true>(s1, C, kl, r1);
        }
        combine_cls<CMAX, PX>(s0, r0, s1, r1, C, 0.5f);
    }
    const size_t o = (size_t)(y0 + yl) * out.w + (size_t)(x0 + xl);
    constexpr bool P_IS_M = NH + NV == 3;         // edge blocks: P is the reference's M
    if constexpr (!NEED_P) emit_unit<CMAX, PX>(out, s_lut, C, s0, s0, o);
    else if constexpr (P_IS_M) emit_unit<CMAX, PX, CONF>(out, s_lut, C, s0, s0, o);
    else if constexpr (MODE == 1) emit_unit<CMAX, PX, CONF>(out, s_lut, C, p, p, o);
    else emit_unit<CMAX, PX, CONF>(out, s_lut, C, s0, p, o);
}

template <int C_T, int CMAX, int PX, int NH, int NV, int MODE, bool CONF>
__device__ __forceinline__ void stitch_units(const StitchArgs &a, const uint32_t *s_lut, uint8_t *conf, float k, int ky, int kx, int row0,
                                             int nrows) {
    const int C = C_T > 0 ? C_T : a.C;
    const float kl = MODE == 1 ? k : kLog2e;     // scale of every raw-logit softmax: log2(e) / temperature
    const int T = a.T, S = a.S;
    const size_t cstride = (size_t)T * T;
    int ti[2], ty0[2], tj[2], tx0[2];
    select_tiles<NH, NV>(a, ky, kx, ti, ty0, tj, tx0);
    const StitchOut out = stitch_out(a, conf);
    const float *base[NV][NH];
#pragma unroll
    for (int s = 0; s < NV; ++s)
#pragma unroll
        for (int q = 0; q < NH; ++q) base[s][q] = tile_base(a, ti[s], tj[q]) + (size_t)ty0[s] * T + tx0[q];

    // a thread's units are kThreads apart: (row, column) advance by constants with a carry
    int row = threadIdx.x / a.upr, col = threadIdx.x - row * a.upr;
    const int d_row = kThreads / a.upr, d_col = kThreads - d_row * a.upr;
    for (; row < nrows; row += d_row, col += d_col) {
        if (col >= a.upr) {
            col -= a.upr;
            if (++row >= nrows) break;
        }
        const int yl = row0 + row;
        const int xl = col * PX;
        const size_t off = (size_t)yl * T + xl;

        float v[NV][NH][CMAX][PX];
#pragma unroll
        for (int s = 0; s < NV; ++s)
#pragma unroll
            for (int q = 0; q < NH; ++q) load_cls<CMAX, PX>(base[s][q] + off, cstride, C, v[s][q]);
        if constexpr (NH == 2) {
#pragma unroll
            for (int s = 0; s < NV; ++s) merge_columns<CMAX, PX, NV>(v[s][0], v[s][1], C, kl);
        }
        merge_rows_emit<CMAX, PX, NH, NV, MODE, CONF>(out, s_lut, C, kl, v[0][0], v[NV - 1][0], ky * S, yl, kx * S, xl);
    }
}

template <int C_T, int CMAX, int PX, int MODE = 0, bool CONF = false>
__global__ void __launch_bounds__(kThreads, 2) stitch_kernel(StitchArgs a, const __grid_constant__ ColourLut lut, uint8_t *conf,
                                                             float k) {
    __shared__ uint32_t s_lut[PYLC_MAX_CLASSES];
    if (threadIdx.x < PYLC_MAX_CLASSES) s_lut[threadIdx.x] = lut.rgb[threadIdx.x];
    __syncthreads();
    int bid = blockIdx.x;
    const int slab = bid % a.slabs;
    bid /= a.slabs;
    // Blocks are walked from the LAST tile row to the first.  In the tiled pipeline the logits were
    // written tile by tile just before this launch and are several times the L2: what is still cached
    // are the most recently written tiles, so reading those first turns the tail of the producer's
    // stores into L2 hits instead of evicting them unread.  (Ordering the blocks by weight -- interior
    // blocks read four quadrants per pixel, corners one -- was measured and makes no difference.)
    bid = a.nbx * a.nby - 1 - bid;
    const int kx = bid % a.nbx, ky = bid / a.nbx;
    const bool two_h = a.overlap && kx > 0 && kx < a.nc;
    const bool two_v = a.overlap && ky > 0 && ky < a.nr;
    if (two_h) {
        if (two_v) stitch_units<C_T, CMAX, PX, 2, 2, MODE, CONF>(a, s_lut, conf, k, ky, kx, slab * a.rows_per_cta, a.rows_per_cta);
        else stitch_units<C_T, CMAX, PX, 2, 1, MODE, CONF>(a, s_lut, conf, k, ky, kx, slab * a.rows_per_cta, a.rows_per_cta);
    } else {
        if (two_v) stitch_units<C_T, CMAX, PX, 1, 2, MODE, CONF>(a, s_lut, conf, k, ky, kx, slab * a.rows_per_cta, a.rows_per_cta);
        else stitch_units<C_T, CMAX, PX, 1, 1, MODE, CONF>(a, s_lut, conf, k, ky, kx, slab * a.rows_per_cta, a.rows_per_cta);
    }
}


// ------------------------------------------------------------------------------------------------
// Fused form (SURVEY.md 8f-1): stitch straight from the decoder's [b, T/4, T/4, C] channels-last output.
// The network's last step, F.interpolate(x, size=T, mode='bilinear', align_corners=True)
// (models/architectures/deeplab.py:38), is evaluated here per output pixel instead of being written out
// as [b, C, T, T] logits and read back: 16x less input (26.5 MB instead of 424.7 MB per 3000x2000 image)
// and one kernel instead of two.  The bilinear arithmetic is the same, in the same order, as
// upsample_to_nchw_staged_kernel (netglue.cu) -- rows blended first: v = fma(hl0, r0, hl1 * r1), then
// res = fma(l, v_left, r * v_right) -- so the logits, and with them the stitched map and the labels, are
// bit-identical to the two-kernel route.
//
// A CTA owns kUpR output rows of one S x S block.  For each of the (up to four) source tiles it copies the
// few decoder rows / columns those output rows touch into shared memory, one 48-byte padded record per
// decoder pixel (4-byte cp.async; a record is three 16-byte shared loads later); a thread then produces
// 2-pixel units exactly as stitch_units does, with "load the logits" replaced by "blend them".
constexpr int kUpR = 8;            // output rows per CTA
constexpr int kUpSrcRows = 4;      // decoder rows staged per tile: kUpR * (hs-1)/(T-1) < 2, + the row below, + float rounding
constexpr int kUpCpad = 12;        // floats per staged decoder pixel (C <= 12)

struct StitchUpArgs {
    const float *const *batches;   // device array of channels-last decoder outputs [b, hs, ws, C]
    int tiles_per_batch;
    int nr, nc, C, T, S, hs, ws;
    int overlap, h, w, nbx, nby, slabs;
    int cols_max;                  // staged decoder columns per tile (S * (ws-1)/(T-1) + 3)
    uint8_t *labels;
    uint8_t *rgb;
    float *stitched;
};

template <int C_T, int CMAX, int NH, int NV, int MODE, bool CONF>
__device__ __forceinline__ void stitch_up_units(const StitchUpArgs &a, const uint32_t *s_lut, uint8_t *conf, float k, float *s_src, int ky, int kx,
                                                int row0) {
    constexpr int PX = 2;
    const int C = C_T > 0 ? C_T : a.C;
    const float kl = MODE == 1 ? k : kLog2e;     // as in stitch_units
    const int T = a.T, S = a.S, hs = a.hs, ws = a.ws;
    const float rh = (float)(hs - 1) / (float)(T - 1), rw = (float)(ws - 1) / (float)(T - 1);
    int ti[2], ty0[2], tj[2], tx0[2];
    select_tiles<NH, NV>(a, ky, kx, ti, ty0, tj, tx0);
    const StitchOut out = stitch_out(a, conf);
    // ---- stage ---------------------------------------------------------------------------------------
    int ys0[NV], xs0[NH], ncol[NH];
#pragma unroll
    for (int s = 0; s < NV; ++s) ys0[s] = (int)(rh * (float)(ty0[s] + row0));
#pragma unroll
    for (int q = 0; q < NH; ++q) {
        xs0[q] = (int)(rw * (float)tx0[q]);
        ncol[q] = min(ws - 1, (int)(rw * (float)(tx0[q] + S - 1)) + 1) - xs0[q] + 1;
    }
    const int tile_f = kUpSrcRows * a.cols_max * kUpCpad;          // floats per staged tile
    const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(s_src);
#pragma unroll
    for (int s = 0; s < NV; ++s) {
        const int nrow = min(hs - 1, (int)(rh * (float)(ty0[s] + row0 + kUpR - 1)) + 1) - ys0[s] + 1;
#pragma unroll
        for (int q = 0; q < NH; ++q) {
            const int k = ti[s] * a.nc + tj[q], b = k / a.tiles_per_batch;
            const float *tile = a.batches[b] + (size_t)(k - b * a.tiles_per_batch) * hs * ws * C;
            const int run = ncol[q] * C;                            // contiguous floats per staged row
            const uint32_t dst0 = s0 + (uint32_t)((s * NH + q) * tile_f) * 4u;
            for (int i = threadIdx.x; i < nrow * run; i += kThreads) {
                const int r = i / run, e = i - r * run;
                const int col = e / C, c = e - col * C;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst0 + (uint32_t)((r * a.cols_max + col) * kUpCpad + c) * 4u),
                             "l"(tile + ((size_t)(ys0[s] + r) * ws + xs0[q]) * C + e)
                             : "memory");
            }
        }
    }
    cp_async_commit();

    // ---- per-thread column set-up (row-invariant): the pair (X, X+1) touches at most three decoder columns
    const int u = threadIdx.x & (S / PX - 1), rsel = threadIdx.x / (S / PX);     // S/2 units per row (a power of two)
    const int rstep = kThreads / (S / PX);
    const int X = u * PX;
    uint32_t coff[NH][3];
    float cw[NH][PX][3];
#pragma unroll
    for (int q = 0; q < NH; ++q) {
        int x1[PX], xr[PX];
        float l0[PX], l1[PX];
#pragma unroll
        for (int j = 0; j < PX; ++j) {
            const float w1r = rw * (float)(tx0[q] + X + j);
            x1[j] = (int)w1r;
            xr[j] = min(x1[j] + 1, ws - 1);
            l1[j] = w1r - (float)x1[j];
            l0[j] = 1.f - l1[j];
        }
        const int xa = x1[0] - xs0[q];
        coff[q][0] = (uint32_t)(xa * kUpCpad) * 4u;
        coff[q][1] = (uint32_t)(min(xa + 1, ncol[q] - 1) * kUpCpad) * 4u;
        coff[q][2] = (uint32_t)(min(xa + 2, ncol[q] - 1) * kUpCpad) * 4u;
#pragma unroll
        for (int j = 0; j < PX; ++j) {
            const bool first = x1[j] == x1[0], right_same = xr[j] == x1[j];
            float c0 = 0.f, c1 = 0.f, c2 = 0.f;
            if (first) { c0 = l0[j]; if (right_same) c0 += l1[j]; else c1 = l1[j]; }
            else { c1 = l0[j]; if (right_same) c1 += l1[j]; else c2 = l1[j]; }
            cw[q][j][0] = c0; cw[q][j][1] = c1; cw[q][j][2] = c2;
        }
    }
    cp_async_wait<0>();
    __syncthreads();

    const uint32_t row_b = (uint32_t)(a.cols_max * kUpCpad) * 4u;
    for (int r = rsel; r < kUpR; r += rstep) {
        const int yl = row0 + r;
        float strip[NV][CMAX][PX];
#pragma unroll
        for (int s = 0; s < NV; ++s) {
            const float h1r = rh * (float)(ty0[s] + yl);
            const int y1 = (int)h1r, y1p = y1 < hs - 1 ? 1 : 0;
            const float hl1 = h1r - (float)y1, hl0 = 1.f - hl1;
            float v[NH][CMAX][PX];
#pragma unroll
            for (int q = 0; q < NH; ++q) {
                const uint32_t p0 = s0 + (uint32_t)((s * NH + q) * tile_f) * 4u + (uint32_t)(y1 - ys0[s]) * row_b;
                const uint32_t p1 = p0 + (uint32_t)y1p * row_b;
                float col[3][CMAX];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
#pragma unroll
                    for (int c4 = 0; c4 < (CMAX + 3) / 4; ++c4) {
                        const uint4 t0 = lds128(p0 + coff[q][k] + 16u * c4), t1 = lds128(p1 + coff[q][k] + 16u * c4);
                        const float a0[4] = {__uint_as_float(t0.x), __uint_as_float(t0.y), __uint_as_float(t0.z), __uint_as_float(t0.w)};
                        const float a1[4] = {__uint_as_float(t1.x), __uint_as_float(t1.y), __uint_as_float(t1.z), __uint_as_float(t1.w)};
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (c4 * 4 + i < CMAX) col[k][c4 * 4 + i] = fmaf(hl0, a0[i], hl1 * a1[i]);
                    }
                }
#pragma unroll
                for (int c = 0; c < CMAX; ++c)
#pragma unroll
                    for (int j = 0; j < PX; ++j)
                        v[q][c][j] = fmaf(cw[q][j][0], col[0][c], fmaf(cw[q][j][1], col[1][c], cw[q][j][2] * col[2][c]));
            }
            if constexpr (NH == 2) merge_columns<CMAX, PX, NV>(v[0], v[1], C, kl);
#pragma unroll
            for (int c = 0; c < CMAX; ++c)
#pragma unroll
                for (int j = 0; j < PX; ++j) strip[s][c][j] = v[0][c][j];
        }
        merge_rows_emit<CMAX, PX, NH, NV, MODE, CONF>(out, s_lut, C, kl, strip[0], strip[NV - 1], ky * S, yl, kx * S, X);
    }
}

template <int C_T, int CMAX, int MODE = 0, bool CONF = false>
__global__ void __launch_bounds__(kThreads, 2) stitch_up_kernel(StitchUpArgs a, const __grid_constant__ ColourLut lut, uint8_t *conf,
                                                                float k) {
    extern __shared__ __align__(16) float s_up[];
    __shared__ uint32_t s_lut[PYLC_MAX_CLASSES];
    if (threadIdx.x < PYLC_MAX_CLASSES) s_lut[threadIdx.x] = lut.rgb[threadIdx.x];
    // (the barrier inside stitch_up_units, after the staging copies, also covers s_lut)
    int bid = blockIdx.x;
    const int slab = bid % a.slabs;
    bid /= a.slabs;
    bid = a.nbx * a.nby - 1 - bid;       // last tile row first, as stitch_kernel does
    const int kx = bid % a.nbx, ky = bid / a.nbx;
    const bool two_h = a.overlap && kx > 0 && kx < a.nc;
    const bool two_v = a.overlap && ky > 0 && ky < a.nr;
    if (two_h) {
        if (two_v) stitch_up_units<C_T, CMAX, 2, 2, MODE, CONF>(a, s_lut, conf, k, s_up, ky, kx, slab * kUpR);
        else stitch_up_units<C_T, CMAX, 2, 1, MODE, CONF>(a, s_lut, conf, k, s_up, ky, kx, slab * kUpR);
    } else {
        if (two_v) stitch_up_units<C_T, CMAX, 1, 2, MODE, CONF>(a, s_lut, conf, k, s_up, ky, kx, slab * kUpR);
        else stitch_up_units<C_T, CMAX, 1, 1, MODE, CONF>(a, s_lut, conf, k, s_up, ky, kx, slab * kUpR);
    }
}

}  // namespace pylc

using namespace pylc;

// Checks both forms make, after their own checks of the tile source (PYLC_ERR_ARG too).  A temperature is finite and
// > 0, and other than 1 only for the mean stitch: reference mode mixes raw-logit corners, a second softmax of
// probability sums and labels from M, so a temperature has no single meaning there.
static int check_stitch(int nr, int nc, int C, int T, int S, int mode, float temperature, const uint8_t *lut_rgb,
                        const uint8_t *rgb) {
    if (nr < 1 || nc < 1 || T < 1 || S < 1) return PYLC_ERR_ARG;
    if (!(temperature > 0.f) || !isfinite(temperature)) return PYLC_ERR_ARG;
    if (mode != PYLC_STITCH_MEAN && temperature != 1.f) return PYLC_ERR_ARG;
    if (rgb && !lut_rgb) return PYLC_ERR_ARG;
    if (mode != PYLC_STITCH_REFERENCE && mode != PYLC_STITCH_MEAN) return PYLC_ERR_ARG;
    if (C < 1 || C > PYLC_MAX_CLASSES) return PYLC_ERR_CLASSES;
    if (!(S == T || 2 * S == T)) return PYLC_ERR_GEOMETRY;  // the reference is only correct for these (tools.py:235-236)
    return PYLC_OK;
}

// The block grid and the outputs, the fields both argument structs share.
template <class Args>
static void set_blocks(Args &a, int nr, int nc, int C, int T, int S, uint8_t *labels, uint8_t *rgb, float *stitched) {
    a.nr = nr; a.nc = nc; a.C = C; a.T = T; a.S = S;
    a.overlap = S < T;
    a.nbx = a.overlap ? nc + 1 : nc;
    a.nby = a.overlap ? nr + 1 : nr;
    a.h = a.nby * S;
    a.w = a.nbx * S;
    a.labels = labels; a.rgb = rgb; a.stitched = stitched;
}

static ColourLut stitch_lut(const uint8_t *lut_rgb, int C) {
    ColourLut lut;
    if (lut_rgb) build_colour_lut(lut_rgb, C, &lut);
    else for (int i = 0; i < PYLC_MAX_CLASSES; ++i) lut.rgb[i] = 0;
    return lut;
}

// Calls launch(std::integral_constant<int, MODE>, std::bool_constant<CONF>, k) for the instantiation (mode, confidence)
// selects; k = log2(e) / temperature is the softmax scale of the mean-mode kernels, exactly log2(e) at T = 1.
template <class Launch>
static int launch_mode(int mode, bool confidence, float temperature, Launch launch) {
    using Ref = std::integral_constant<int, 0>;
    using Mean = std::integral_constant<int, 1>;
    int rc;
    if (mode == PYLC_STITCH_MEAN) {
        const float k = kLog2e / temperature;
        rc = confidence ? launch(Mean{}, std::true_type{}, k) : launch(Mean{}, std::false_type{}, k);
    } else {
        rc = confidence ? launch(Ref{}, std::true_type{}, kLog2e) : launch(Ref{}, std::false_type{}, kLog2e);
    }
    if (rc) return rc;
    return finish_launch();
}

template <int MODE, bool CONF>
static int launch_stitch(bool px2, int C, unsigned grid, cudaStream_t st, const StitchArgs &a, const ColourLut &lut,
                         uint8_t *conf, float k) {
    if (px2) {
        if (C == 9) stitch_kernel<9, 9, 2, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
        else if (C == 11) stitch_kernel<11, 11, 2, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
        else if (C <= 4) stitch_kernel<0, 4, 2, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
        else if (C <= 8) stitch_kernel<0, 8, 2, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
        else stitch_kernel<0, 12, 2, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
    } else {
        if (C <= 12) stitch_kernel<0, 12, 1, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
        else if (C <= 16) stitch_kernel<0, 16, 1, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
        else stitch_kernel<0, 32, 1, MODE, CONF><<<grid, kThreads, 0, st>>>(a, lut, conf, k);
    }
    return 0;
}

extern "C" int pylc_stitch_probs(const float *logits, const float *const *tile_batches, int tiles_per_batch, int nr, int nc,
                                 int C, int T, int S, int mode, const uint8_t *lut_rgb, uint8_t *labels, uint8_t *rgb,
                                 uint8_t *confidence, float *stitched, float temperature, pylc_stream_t stream) {
    if (!logits && (!tile_batches || tiles_per_batch < 1)) return PYLC_ERR_ARG;
    if (int rc = check_stitch(nr, nc, C, T, S, mode, temperature, lut_rgb, rgb)) return rc;
    StitchArgs a;
    a.logits = logits;
    a.batches = tile_batches;
    a.tiles_per_batch = logits ? nr * nc : tiles_per_batch;
    set_blocks(a, nr, nc, C, T, S, labels, rgb, stitched);
    const bool px2 = (S % 2 == 0) && C <= 12 && ((uintptr_t)logits % 8 == 0) &&
                     (!stitched || (uintptr_t)stitched % 8 == 0) && (!labels || (uintptr_t)labels % 2 == 0) &&
                     (!rgb || (uintptr_t)rgb % 2 == 0) && (!confidence || (uintptr_t)confidence % 2 == 0);
    const int PX = px2 ? 2 : 1;
    a.upr = S / PX;
    // One CTA per slab of up to eight units per thread.  Measured on B200 (273 / 45 tiles, C = 9): 8 units
    // 0.395 / 0.078 ms, 4 units 0.416 / 0.080, 2 units 0.449 / 0.084, 16 units 0.428 / 0.082.  Persistent
    // variants (round-robin groups with register double-buffering; weight-balanced contiguous runs per
    // CTA) were slower, 0.43-0.67 / 0.085-0.125 ms: neighbouring CTAs walking neighbouring slabs of the
    // same class planes is what keeps the DRAM pages open, and 16 resident warps hide the softmax.
    int rows = S;
    while (rows > 1 && rows * a.upr > kThreads * 8 && rows % 2 == 0) rows /= 2;
    a.rows_per_cta = rows;
    a.slabs = S / rows;
    const ColourLut lut = stitch_lut(lut_rgb, C);
    const unsigned grid = (unsigned)((long long)a.nbx * a.nby * a.slabs);
    cudaStream_t st = (cudaStream_t)stream;
    return launch_mode(mode, confidence, temperature, [&](auto m, auto conf, float k) {
        return launch_stitch<decltype(m)::value, decltype(conf)::value>(px2, C, grid, st, a, lut, confidence, k);
    });
}

template <int MODE, bool CONF>
static int launch_stitch_up(int C, unsigned grid, size_t smem, cudaStream_t st, const StitchUpArgs &a, const ColourLut &lut,
                            uint8_t *conf, float k) {
#define LAUNCH_UP(CT, CM)                                                                                                  \
    do {                                                                                                                   \
        cudaError_t e = cudaFuncSetAttribute(stitch_up_kernel<CT, CM, MODE, CONF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return (int)e;                                                                               \
        stitch_up_kernel<CT, CM, MODE, CONF><<<grid, kThreads, smem, st>>>(a, lut, conf, k);                                     \
    } while (0)
    if (C == 9) LAUNCH_UP(9, 9);
    else if (C == 11) LAUNCH_UP(11, 11);
    else if (C <= 4) LAUNCH_UP(0, 4);
    else if (C <= 8) LAUNCH_UP(0, 8);
    else LAUNCH_UP(0, 12);
#undef LAUNCH_UP
    return 0;
}

extern "C" int pylc_stitch_upsample_probs(const float *const *decoder_batches, int tiles_per_batch, int nr, int nc, int C,
                                          int T, int S, int hs, int ws, int mode, const uint8_t *lut_rgb, uint8_t *labels,
                                          uint8_t *rgb, uint8_t *confidence, float *stitched, float temperature,
                                          pylc_stream_t stream) {
    if (!decoder_batches || tiles_per_batch < 1 || hs < 2 || ws < 2) return PYLC_ERR_ARG;
    if (int rc = check_stitch(nr, nc, C, T, S, mode, temperature, lut_rgb, rgb)) return rc;
    // this form covers the network's geometry: a x4 up-sample, rows of 2-pixel units that fill a CTA evenly
    if (C > kUpCpad || hs * 4 != T || ws * 4 != T || S % kUpR || (S / 2) > kThreads || kThreads % (S / 2) || (S & (S - 1))) return PYLC_ERR_GEOMETRY;
    if ((stitched && (uintptr_t)stitched % 8) || (labels && (uintptr_t)labels % 2) || (rgb && (uintptr_t)rgb % 2) ||
        (confidence && (uintptr_t)confidence % 2))
        return PYLC_ERR_ALIGN;
    StitchUpArgs a;
    a.batches = decoder_batches;
    a.tiles_per_batch = tiles_per_batch;
    a.hs = hs; a.ws = ws;
    set_blocks(a, nr, nc, C, T, S, labels, rgb, stitched);
    a.slabs = S / kUpR;
    a.cols_max = (int)((double)S * (ws - 1) / (T - 1)) + 4;
    const ColourLut lut = stitch_lut(lut_rgb, C);
    const size_t smem = (size_t)4 * kUpSrcRows * a.cols_max * kUpCpad * sizeof(float);
    const unsigned grid = (unsigned)((long long)a.nbx * a.nby * a.slabs);
    cudaStream_t st = (cudaStream_t)stream;
    return launch_mode(mode, confidence, temperature, [&](auto m, auto conf, float k) {
        return launch_stitch_up<decltype(m)::value, decltype(conf)::value>(C, grid, smem, st, a, lut, confidence, k);
    });
}
