/*
 * pylc_b200 -- C ABI of the sm_100a kernel library for PyLC's tiled-segmentation hot path.
 *
 * This is the drop-in boundary.  The PyLC reference has no FFI layer (it is pure Python); each
 * entry point below replaces the NumPy / Torch-CPU / scikit-learn body of one reference function
 * (cited per function, paths relative to the PyLC source root).  The Python host layer
 * (the modules under pylc_b200/utils and pylc_b200/models/modules/loss.py) binds these with ctypes and keeps the
 * reference's own signatures; INTEGRATION.md shows the stub a PyLC maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - Every pointer is a DEVICE pointer owned by the caller unless marked HOST.
 *   - `stream` is a cudaStream_t passed as void*; NULL = legacy default stream.
 *   - Nothing allocates, synchronises or calls back; a call returns once the launch is enqueued.
 *   - Return value: 0 = ok, > 0 = cudaError_t of the failed launch, < 0 = PYLC_ERR_* below.
 *   - Accumulator outputs (stat, px_dist, conf, partials) are ADDED INTO; the caller zeroes them.
 *     Integer accumulators make every result independent of launch geometry and GPU count.
 *   - Pitches are in bytes.  Sources whose base and pitch are 16-byte aligned take the vectorised
 *     path; anything else takes a slower byte-wise path with identical results.
 */
#ifndef PYLC_B200_H
#define PYLC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PYLC_ABI_VERSION 5
#define PYLC_MAX_CLASSES 32

#define PYLC_OK 0
#define PYLC_ERR_ARG (-1)         /* null pointer / non-positive size                        */
#define PYLC_ERR_CLASSES (-2)     /* n_classes outside [1, PYLC_MAX_CLASSES]                 */
#define PYLC_ERR_GEOMETRY (-3)    /* tile/stride combination the kernels do not implement    */
#define PYLC_ERR_ALIGN (-4)       /* destination pointer not 16-byte aligned                 */
#define PYLC_ERR_PALETTE (-5)     /* no collision-free hash found for the palette            */

#if defined(__GNUC__)
#define PYLC_API __attribute__((visibility("default")))
#else
#define PYLC_API
#endif

typedef void *pylc_stream_t;

/* ---- library ------------------------------------------------------------------------------ */

PYLC_API int pylc_abi_version(void);
/* Human-readable text for any return code of this library (never NULL). */
PYLC_API const char *pylc_error_string(int code);
/* Device the calling thread is bound to: SM count and compute capability (major*10+minor). */
PYLC_API int pylc_device_info(int *sm_count, int *compute_capability);
/* Counts kernel launches issued through this library since load (bench.py's gpu_launches). */
PYLC_API int64_t pylc_launch_count(void);

/* ---- tile extraction ---------------------------------------------------------------------- */

/* Number of tiles Tensor.unfold(0,T,S).unfold(1,T,S) yields (utils/extract.py:302-305). */
PYLC_API int pylc_tile_grid(int H, int W, int T, int S, int *nH, int *nW);

/*
 * Overlapping tile gather, replaces Extractor.__split + np.copyto (utils/extract.py:279-310,182).
 *   src   [H, W] (ch=1) or [H, W, 3] interleaved (ch=3) u8, row pitch `src_pitch` bytes
 *   dst   [nH*nW, ch, T, T] u8, tile k = r*nW + c covers rows [rS, rS+T), cols [cS, cS+T)
 *   stat  nullable [nH*nW, ch, 2] u64: per tile/channel sum(x), sum(x*x) (exact integers; the
 *         host derives torch.mean / torch.std of utils/profile.py:101-106 from them)
 * Requires T % 16 == 0, S % 16 == 0, T % S == 0 (vector path) -- otherwise PYLC_ERR_GEOMETRY.
 */
PYLC_API int pylc_tile_gather_u8(const uint8_t *src, int H, int W, int ch, size_t src_pitch, int T, int S,
                        uint8_t *dst, uint64_t *stat, pylc_stream_t stream);

/*
 * Fused mask tile gather + palette encode + per-tile class histogram; replaces
 * Extractor.__split + tools.class_encode + the one_hot/np.sum histogram
 * (utils/extract.py:195-214, utils/tools.py:412-449, utils/profile.py:109-111).
 *   src      [H, W, 3] RGB u8, pitch bytes
 *   palette  HOST [C, 3] u8.  Unmatched colours encode to class 1, later duplicates win.
 *   dst      [nH*nW, T, T] u8 class indices
 *   px_dist  nullable [nH*nW, C] i64
 */
PYLC_API int pylc_mask_gather_encode_hist(const uint8_t *src, int H, int W, size_t src_pitch, int T, int S,
                                 const uint8_t *palette, int C, uint8_t *dst, int64_t *px_dist,
                                 pylc_stream_t stream);

/*
 * Extraction sweep over a STACK of n_img equally sized sources in one call (one launch on the staged / TMA
 * forms): what the file loop of Extractor.extract (utils/extract.py:136-222) does image by image.
 *   src        image i starts at src + i * img_stride (img_stride >= H * src_pitch; a multiple of 16 keeps
 *              the vector / TMA forms), each [H, W(,3)] with row pitch `src_pitch`
 *   dst        [n_img * nH*nW, ...]: the tiles of image i follow those of image i-1, as the reference's
 *              tile buffers are filled (utils/extract.py:182,214)
 *   stat / px_dist  nullable, [n_img * nH*nW, ...], same order; px_dist is added into
 * Results are identical to n_img single-image calls.
 */
PYLC_API int pylc_tile_gather_u8_stack(const uint8_t *src, int n_img, size_t img_stride, int H, int W, int ch,
                              size_t src_pitch, int T, int S, uint8_t *dst, uint64_t *stat, pylc_stream_t stream);
PYLC_API int pylc_mask_gather_encode_hist_stack(const uint8_t *src, int n_img, size_t img_stride, int H, int W,
                                       size_t src_pitch, int T, int S, const uint8_t *palette, int C, uint8_t *dst,
                                       int64_t *px_dist, pylc_stream_t stream);

/*
 * Standalone tools.class_encode (utils/tools.py:412-449).
 *   layout 0: rgb is [n_img, rows, cols, 3] interleaved with row pitch `pitch` (n_img images
 *             stored back to back, rows*pitch bytes each)          -> out [n_img, rows, cols]
 *   layout 1: rgb is [n_img, 3, rows*cols] planar (the reference's NCHW argument); pitch ignored
 *   hist     nullable [C] i64, histogram of the encoded output
 */
PYLC_API int pylc_class_encode(const uint8_t *rgb, int n_img, int rows, int cols, size_t pitch, int layout,
                      const uint8_t *palette, int C, uint8_t *out, int64_t *hist,
                      pylc_stream_t stream);

/*
 * Profiling sweep over already extracted tiles (utils/profile.py:98-111): per-tile class
 * histograms and per-tile/channel sum(x), sum(x*x).  Either input may be NULL.
 *   imgs [n, ch, tile_px] u8 -> stat [n, ch, 2] u64 ;  masks [n, tile_px] u8 -> px_dist [n, C] i64
 */
PYLC_API int pylc_profile_tiles(const uint8_t *imgs, int ch, const uint8_t *masks, int n, int64_t tile_px,
                       int C, uint64_t *stat, int64_t *px_dist, pylc_stream_t stream);

/*
 * Tile gather fused with Model.normalize_image (models/model.py:416-445) and the grayscale
 * x3 channel replicate (models/model.py:376-377): writes network-ready f32 tiles.
 *   dst [nH*nW, out_ch, T, T] f32, value = ((x - mean[c]) / std[c]) / post_div in IEEE f32, the
 *       reference's operation order (post_div 255, or 1 for the grayscale `default` branch)
 *   mean / std: HOST [3] f32 (index 0 used for ch=1).  out_ch is 3 (ch=1 replicates) or ch.
 */
PYLC_API int pylc_tile_gather_norm_f32(const uint8_t *src, int H, int W, int ch, size_t src_pitch, int T,
                              int S, const float *mean, const float *std, float post_div,
                              int out_ch, float *dst, pylc_stream_t stream);

/*
 * Augmentor.optimize grid search (utils/augment.py:92-187) over rate coefficients x thresholds: for
 * grid point g = i*n_thresholds + j,
 *     rates[n]        = clip(int((scores[n] > thresholds[j]) * rate_coefs[i] * scores[n]), rate_lo, rate_hi)
 *     sum_rates[g]    = sum_n rates[n]
 *     full_px_dist[g] = sum_n (1 + rates[n]) * px_dist[n, :]            (exact int64)
 * scores [N] f64 (the host computes them with NumPy exactly as the reference, augment.py:108-116),
 * px_dist [N, C] i64, rate_coefs / thresholds f64 -- all DEVICE.  The O(grid x C) tail (probabilities,
 * M2, JSD, argmin) stays on the host in float64.
 */
PYLC_API int pylc_sample_rate_grid(const double *scores, const int64_t *px_dist, int N, int C,
                          const double *rate_coefs, int n_coefs, const double *thresholds,
                          int n_thresholds, int rate_lo, int rate_hi, int64_t *sum_rates,
                          int64_t *full_px_dist, pylc_stream_t stream);

/*
 * Over-sampled copies of tiles, replaces tools.augment_transform = perspective_shift + channel_shift
 * (utils/tools.py:452-594) for every copy Augmentor.oversample appends (utils/augment.py:205-222): cv2.warpPerspective
 * (bilinear image / nearest mask, BORDER_REFLECT_101), the 30-pixel crop, cv2.resize back to T (INTER_AREA image /
 * INTER_NEAREST mask) and the brightness shift, bit-identical to that OpenCV call chain (arithmetic: csrc/augment_math.cuh).
 *   src_img   [n_src, ch, T, T] u8, src_mask [n_src, T, T] u8 (class indices)
 *   job_src   [n_jobs] i32   source tile of copy j
 *   job_minv  [n_jobs, 9] f64  row-major INVERSE of cv2.getPerspectiveTransform(pts1, pts2) (cv2.invert; the host draws
 *             pts2 from RandomState(j) exactly as the reference, tools.py:577-580)
 *   job_shift [n_jobs] i32   brightness shift int(uniform(10, 20)) (tools.py:550)          -- all DEVICE
 *   dst_img   [n_jobs, ch, T, T] u8, dst_mask [n_jobs, T, T] u8
 * ch is 1 or 3, T > 61.  Copies with a source index outside [0, n_src) are left unwritten.
 */
PYLC_API int pylc_augment_tiles_u8(const uint8_t *src_img, const uint8_t *src_mask, int n_src, int ch, int T,
                          const int32_t *job_src, const double *job_minv, const int32_t *job_shift, int n_jobs,
                          uint8_t *dst_img, uint8_t *dst_mask, pylc_stream_t stream);

/* ---- test-time fit resize ----------------------------------------------------------------- */

#define PYLC_AREA_TAPS 6 /* source cells per destination cell and axis: scale factors below 5 */

/*
 * cv2.resize(img, (w, h), interpolation=INTER_AREA) of tools.adjust_to_tile
 * (utils/tools.py:189-206) on the device, bit-exact with OpenCV's general area filter for u8
 * (imgproc/resize.cpp: computeResizeAreaTab + resizeArea_<uchar,float>; OpenCV is a third-party
 * dependency of the reference, requirements.txt:8).
 *
 *   pylc_area_supported   HOST: 1 if OpenCV resizes (W,H)->(w,h) with that filter (a down-scale by
 *                         non-integer factors below 5, or the identity); 0 otherwise -- the caller
 *                         then keeps the host cv2 call
 *   pylc_area_table       HOST: one axis of the area table.  For destination index d the source
 *                         cells are start[d] .. start[d]+count[d]-1 with float weights
 *                         weights[d*PYLC_AREA_TAPS + k]; all three arrays are HOST, length dsize
 *                         (weights: dsize*PYLC_AREA_TAPS).  The caller uploads them once per geometry.
 *   pylc_fit_resize_area_u8  src [H,W,ch] u8 (pitch bytes, any alignment) -> dst [h,w,ch] u8
 *                         (dst_pitch bytes); x_* / y_* are DEVICE copies of the two tables.
 */
PYLC_API int pylc_area_supported(int W, int H, int w, int h);
PYLC_API int pylc_area_table(int ssize, int dsize, int32_t *start, int32_t *count, float *weights);
PYLC_API int pylc_fit_resize_area_u8(const uint8_t *src, int H, int W, int ch, size_t src_pitch, uint8_t *dst,
                            int h, int w, size_t dst_pitch, const int32_t *x_start,
                            const int32_t *x_count, const float *x_weights, const int32_t *y_start,
                            const int32_t *y_count, const float *y_weights, pylc_stream_t stream);

/*
 * Pitched host -> device upload on the copy engine (cudaMemcpy2DAsync): a tightly packed decoded
 * image (tools.get_image's array, utils/tools.py:127-131) lands in the 16-byte-pitched device
 * layout the vectorised kernels want, without a host-side repack.  src_host: HOST, pinned for an
 * asynchronous copy.
 */
PYLC_API int pylc_upload_pitched(void *dst, size_t dst_pitch, const void *src_host, size_t src_pitch,
                        size_t width_bytes, size_t rows, pylc_stream_t stream);

/* ---- network glue (non-convolution steps of the DeepLabv3+ inference plan) ---------------- */

/*
 * The convolutions stay library tensor-core kernels; these are the HBM-bound data-movement steps
 * between them, for channels-last (NHWC) f32 activations.  Bilinear = PyTorch's
 * upsample_bilinear2d with align_corners=True (same index and weight arithmetic).
 *
 *   pylc_upsample_concat_nhwc_f32   F.interpolate(x, size=low.shape[2:]) + torch.cat((x, low), 1) of the
 *                                   decoder (models/decoder.py:46-48):
 *                                   x [B,h,w,Cx], low [B,H,W,Cl] -> out [B,H,W,Cx+Cl]   (Cx, Cl % 4 == 0)
 *   pylc_maxpool3x3s2_nhwc_f32      nn.MaxPool2d(3, stride=2, padding=1) of the ResNet stem
 *                                   (models/backbone/resnet.py): in [B,H,W,C] -> out [B,(H-1)/2+1,(W-1)/2+1,C]
 *   pylc_upsample_nhwc_to_nchw_f32  the final F.interpolate(x, size=input.shape[2:]) (models/architectures/
 *                                   deeplab.py:38), emitting planar logits for the stitch kernel:
 *                                   in [B,h,w,C] NHWC -> out [B,C,H,W]                   (W % 4 == 0)
 */
PYLC_API int pylc_upsample_concat_nhwc_f32(const float *x, int B, int h, int w, int Cx, const float *low, int H,
                                  int W, int Cl, float *out, pylc_stream_t stream);
PYLC_API int pylc_maxpool3x3s2_nhwc_f32(const float *in, int B, int H, int W, int C, float *out, pylc_stream_t stream);
PYLC_API int pylc_upsample_nhwc_to_nchw_f32(const float *in, int B, int h, int w, int C, float *out, int H, int W,
                                   pylc_stream_t stream);

/*
 * Reduction step of the inference plan's tap-split route for a dilated 3x3 convolution the library has no
 * sm_100 kernel for (models/modules/aspp.py: the dilation-18 branch on a 32x32 map, reference aspp.py:40-60).
 * The plan computes every tap's product as a cuBLAS GEMM over a contiguous run of flat pixels of the
 * channels-last activation, shifted by dy*W + dx pixels; this kernel adds them where the tap's source pixel
 * lies inside the map and applies the ReLU:
 *     out[b,y,x,:] = relu(out[b,y,x,:] + sum_t [0 <= y+dy_t < H and 0 <= x+dx_t < W] z_t[b, y*W + x - p0_t, :])
 *   out  [B,H,W,O] f32 in/out (holds the centre tap's product + bias on entry), O % 4 == 0
 *   z    HOST array [ntaps] of DEVICE pointers, z_t = [B, m_t, O] f32; p0 / m / dy / dx: HOST arrays [ntaps]
 *        (flat range [p0_t, p0_t + m_t) of output pixels tap t was computed for; must cover every pixel the mask
 *        lets through, else PYLC_ERR_GEOMETRY); ntaps <= 8.
 */
PYLC_API int pylc_tap_combine_relu_f32(float *out, int B, int H, int W, int O, const float *const *z,
                              const int32_t *p0, const int32_t *m, const int32_t *dy, const int32_t *dx,
                              int ntaps, pylc_stream_t stream);

/*
 * pylc_tile_gather_norm_f32 in the layout the space-to-depth form of the ResNet stem wants (the 7x7
 * stride-2 convolution over 3 channels == a 4x4 stride-1 convolution over the 2x2 space-to-depth
 * image with the kernel zero-extended to 8x8; models/fused.py rearranges the weights):
 *   dst [nH*nW, T/2+3, T/2+3, 16] f32 channels-last,
 *   dst[n, Y, X, (py*2+px)*3 + c] = ((x - mean[c]) / std[c]) / post_div of tile pixel (c, 2(Y-2)+py, 2(X-2)+px),
 *   zero outside the tile (two border rows/columns before, one after) and in channels 12..15.
 * ch = 1 replicates the grey value into the three channels (models/model.py:376-377).
 */
PYLC_API int pylc_tile_gather_norm_s2d_f32(const uint8_t *src, int H, int W, int ch, size_t src_pitch, int T,
                                  int S, const float *mean, const float *std, float post_div,
                                  float *dst, pylc_stream_t stream);

/* ---- stitching ---------------------------------------------------------------------------- */

/*
 * Fused stitch + softmax + argmax + colourise, replaces tools.reconstruct up to and including
 * colourize (utils/tools.py:239-313, 322-358) with the reference's exact band semantics
 * (raw logits at the borders, one softmax-average on edges, double softmax in the interior).
 *   logits        one contiguous [nr*nc, C, T, T] f32 buffer, row-major tile order, or NULL
 *   tile_batches  (used when logits == NULL) device array of pointers, batch b =
 *                 [tiles_per_batch, C, T, T] f32 holding tiles b*tiles_per_batch ... -- the list of
 *                 per-batch network outputs the reference concatenates (utils/tools.py:221-222)
 *   S             T/2 (output (nr+1)S x (nc+1)S) or T (pure scatter, output nr*T x nc*T)
 *   lut_rgb       HOST [C, 3] u8 colour per label (colourize's final mapping); needed iff rgb
 *   labels        [h, w] u8 first-maximum argmax     (nullable)
 *   rgb           [h, w, 3] u8                       (nullable)
 *   stitched      [C, h, w] f32 merged map           (nullable; parity tests / save_logits)
 */
PYLC_API int pylc_stitch_argmax_colour(const float *logits, const float *const *tile_batches,
                              int tiles_per_batch, int nr, int nc, int C, int T, int S,
                              const uint8_t *lut_rgb, uint8_t *labels, uint8_t *rgb,
                              float *stitched, pylc_stream_t stream);

/* tools.colourize (utils/tools.py:322-358) on a flat u8 label array: rgb[i] = lut_rgb[labels[i]]. */
/*
 * Fused form of the network's last step + the stitch (SURVEY.md 8f-1): takes the decoder's output
 * BEFORE the final x4 bilinear up-sample -- `decoder_batches`: device array of device pointers to
 * channels-last [b, hs, ws, C] f32 batches, hs = ws = T/4 -- evaluates
 * F.interpolate(..., size=T, mode='bilinear', align_corners=True) (models/architectures/deeplab.py:38) per
 * output pixel with the arithmetic of pylc_upsample_nhwc_to_nchw_f32, and stitches as
 * pylc_stitch_argmax_colour does.  Outputs are bit-identical to that two-call route.
 * PYLC_ERR_GEOMETRY for C > 12 or a geometry other than the x4 up-sample of 512-class tile sizes: the
 * caller keeps the two-call route.
 */
PYLC_API int pylc_stitch_upsample_argmax_colour(const float *const *decoder_batches, int tiles_per_batch, int nr, int nc,
                                       int C, int T, int S, int hs, int ws, const uint8_t *lut_rgb, uint8_t *labels,
                                       uint8_t *rgb, float *stitched, pylc_stream_t stream);
PYLC_API int pylc_colourise_u8(const uint8_t *labels, int64_t n_px, const uint8_t *lut_rgb, int C,
                      uint8_t *rgb, pylc_stream_t stream);

/*
 * Per-pixel class probabilities and confidence from the same stitch (an extension: the reference never forms a
 * clean probability map).  P(y, x) is the mean, over the 1, 2 or 4 tiles covering the pixel, of softmax_c of
 * that tile's logits.  On edge blocks it is exactly the reference's merged map M; on corners (and everywhere
 * when S == T) the softmax of the raw logits; in the interior the mean of the four softmaxes.
 *   mode          PYLC_STITCH_REFERENCE: labels / rgb / stitched are those of pylc_stitch_argmax_colour (first
 *                 argmax of M, stitched = M), bit for bit.
 *                 PYLC_STITCH_MEAN: labels = first argmax of P, stitched = P.
 *   confidence    nullable [h, w] u8, q = min(255, round-to-nearest(P[label] * 255)); the same P in both modes
 * Other arguments as pylc_stitch_argmax_colour / pylc_stitch_upsample_argmax_colour (the fused form also
 * returns PYLC_ERR_ALIGN for an odd `confidence` address).  An unknown mode is PYLC_ERR_ARG.
 */
#define PYLC_STITCH_REFERENCE 0
#define PYLC_STITCH_MEAN 1
PYLC_API int pylc_stitch_probs(const float *logits, const float *const *tile_batches, int tiles_per_batch,
                      int nr, int nc, int C, int T, int S, int mode, const uint8_t *lut_rgb,
                      uint8_t *labels, uint8_t *rgb, uint8_t *confidence, float *stitched, pylc_stream_t stream);
PYLC_API int pylc_stitch_upsample_probs(const float *const *decoder_batches, int tiles_per_batch, int nr, int nc,
                               int C, int T, int S, int hs, int ws, int mode, const uint8_t *lut_rgb,
                               uint8_t *labels, uint8_t *rgb, uint8_t *confidence, float *stitched, pylc_stream_t stream);

/*
 * Temperature-scaled probabilities (post-hoc calibration): pylc_stitch_probs / pylc_stitch_upsample_probs with every
 * tile softmax taken of L / temperature.  In PYLC_STITCH_MEAN mode every softmax of the stitch is a softmax of raw
 * tile logits, so the kernels evaluate it with k_T = f32(log2(e) / f32(temperature)) in place of log2(e):
 *     P_T(y, x) = the mean over the covering tiles of softmax(L / T),  labels = first argmax of P_T,
 *     confidence = min(255, round-to-nearest(P_T[label] * 255)),  stitched = P_T.
 * At temperature 1 every output equals the untempered call bit for bit.  Labels in overlap zones may change with T:
 * the argmax of a mean of softmaxes depends on the temperature.
 * PYLC_ERR_ARG for a temperature that is not finite and > 0, or other than 1 in PYLC_STITCH_REFERENCE mode (that
 * mode mixes raw-logit corners, a second softmax of probability sums and labels from M: a temperature has no single
 * meaning there).  Other arguments and return codes as the untempered calls.
 */
PYLC_API int pylc_stitch_probs_t(const float *logits, const float *const *tile_batches, int tiles_per_batch,
                        int nr, int nc, int C, int T, int S, int mode, const uint8_t *lut_rgb,
                        uint8_t *labels, uint8_t *rgb, uint8_t *confidence, float *stitched, float temperature,
                        pylc_stream_t stream);
PYLC_API int pylc_stitch_upsample_probs_t(const float *const *decoder_batches, int tiles_per_batch, int nr, int nc,
                                 int C, int T, int S, int hs, int ws, int mode, const uint8_t *lut_rgb,
                                 uint8_t *labels, uint8_t *rgb, uint8_t *confidence, float *stitched, float temperature,
                                 pylc_stream_t stream);

/* ---- evaluation --------------------------------------------------------------------------- */

/*
 * Nearest-neighbour resample of the fitted label map to full resolution + ground-truth palette
 * encode + confusion matrix; replaces cv2.resize(INTER_NEAREST) of the colourised map,
 * Evaluator.load's two class_encode passes, Evaluator.validate's coverage injection and every
 * scikit-learn confusion matrix (utils/tools.py:316-317, utils/evaluate.py:87-119,150-176,
 * utils/metrics.py:45-87).
 *   labels    [h, w] u8 fitted-resolution labels, every value < C (what pylc_stitch_*_argmax_colour and
 *             pylc_class_encode emit).  PRECONDITION, not checked: a per-pixel test costs 10-15 % of the kernel
 *             (measured); a label >= C indexes the shared-memory counters out of range
 *   x_ofs     [w_full] i32, y_ofs [h_full] i32: OpenCV nearest source index per destination index
 *   gt_rgb    nullable [h_full, w_full, 3] u8 ground truth, pitch bytes (NULL: no confusion)
 *   palette   HOST [C, 3] u8 (class_encode rules as above) ; lut_rgb HOST [C,3] (for pred_rgb)
 *   n_inject  flat pixels i < n_inject count as (i, i)  (utils/evaluate.py:172-174)
 *   conf      nullable [C, C] i64, conf[t*C + p] += 1
 *   pred_full nullable [h_full, w_full] u8 ; pred_rgb nullable [h_full, w_full, 3] u8
 *   gt_full   nullable [h_full, w_full] u8 encoded ground truth
 */
PYLC_API int pylc_resample_encode_confusion(const uint8_t *labels, int h, int w, const int32_t *x_ofs,
                                   const int32_t *y_ofs, int h_full, int w_full,
                                   const uint8_t *gt_rgb, size_t gt_pitch, const uint8_t *palette,
                                   const uint8_t *lut_rgb, int C, int n_inject, int64_t *conf,
                                   uint8_t *pred_full, uint8_t *pred_rgb, uint8_t *gt_full,
                                   pylc_stream_t stream);

/* Confusion matrix of two flat u8 label vectors (aggregate mode, utils/evaluate.py:158-174). */
PYLC_API int pylc_confusion_u8(const uint8_t *y_true, const uint8_t *y_pred, int64_t n, int C, int n_inject,
                      int64_t *conf, pylc_stream_t stream);

/*
 * Nearest-neighbour resample of the fitted confidence plane (pylc_stitch_probs) with the label map's OpenCV
 * index maps, and the reliability table of a calibration figure.
 *   confidence       [h, w] u8 fitted-resolution confidence
 *   x_ofs / y_ofs    as pylc_resample_encode_confusion
 *   y_pred_full / y_true_full  nullable [h_full, w_full] u8 predicted / true classes (pred_full / gt_full of
 *                    pylc_resample_encode_confusion); pixels whose class is >= C are not counted
 *   confidence_full  nullable [h_full, w_full] u8
 *   reliability      nullable [C, 256, 2] i64, ADDED INTO: [pred][q][pred == true] += 1 per full-resolution pixel
 *                    (no coverage injection).  Needs both label planes, else PYLC_ERR_ARG.
 * Any width and any alignment; rows are dense (pitch = w_full).
 */
PYLC_API int pylc_confidence_resample(const uint8_t *confidence, int h, int w, const int32_t *x_ofs,
                             const int32_t *y_ofs, int h_full, int w_full, const uint8_t *y_pred_full,
                             const uint8_t *y_true_full, int C, uint8_t *confidence_full, int64_t *reliability,
                             pylc_stream_t stream);

/*
 * Proper scores of mean-mode probabilities against the ground truth at full resolution (temperature fitting).
 *   probs         [C, h, w] f32, the `stitched` output of a PYLC_STITCH_MEAN stitch
 *   x_ofs / y_ofs [w_full] / [h_full] i32, the label map's INTER_NEAREST index maps (as pylc_resample_encode_confusion
 *                 takes them).  PRECONDITION, not checked on the device: every value lies in [0, w) / [0, h)
 *   y_true_full   [h_full, w_full] u8 encoded true classes (gt_full of pylc_resample_encode_confusion: unmatched
 *                 colours are class 1), any alignment.  A class >= C is scored as probability 0 for it.
 *   want_brier    0: NLL only (one plane read per pixel); 1: also the Brier score (all C planes)
 *   workspace     [PYLC_SCORES_WS_DOUBLES] f64 scratch
 *   sums          [2] f64, OVERWRITTEN: {sum of nll, sum of brier (0 without want_brier)} over all h_full * w_full
 *                 pixels, where per pixel, in f32, with g its class and q = P[g][y_ofs[y]][x_ofs[x]]:
 *                     nll = -logf(fmaxf(q, 1e-12f)),  brier = sum over c in class order of (P[c] - [c == g])^2
 * Each pixel is added in f64 and the sums are reduced in a fixed order: the same inputs give the same bits on every
 * call.  Two launches.  PYLC_ERR_ARG for a null pointer or a non-positive size; PYLC_ERR_CLASSES for C outside [1, 32].
 */
#define PYLC_SCORES_BLOCKS 1024
#define PYLC_SCORES_WS_DOUBLES (2 * PYLC_SCORES_BLOCKS)
PYLC_API int pylc_prob_scores(const float *probs, int C, int h, int w, const int32_t *x_ofs, const int32_t *y_ofs,
                     int h_full, int w_full, const uint8_t *y_true_full, int want_brier, double *workspace,
                     double *sums, pylc_stream_t stream);

/*
 * Multi-scale combine (an extension): the mean-mode probability maps of K image scales averaged on one output grid.
 *   probs         HOST [K] array of DEVICE pointers, member k = [C, h[k], w[k]] f32 (pylc_stitch_probs' `stitched`
 *                 in PYLC_STITCH_MEAN mode for the image resized by s_k and fitted to the tiles)
 *   x_ofs / y_ofs HOST [K] arrays of DEVICE pointers, x_ofs[k] = [w_full] i32, y_ofs[k] = [h_full] i32: OpenCV's
 *                 INTER_NEAREST source index per output index from (w[k], h[k]) to (w_full, h_full), as
 *                 pylc_resample_encode_confusion takes them.  PRECONDITION, not checked on the device: every value
 *                 lies in [0, w[k]) / [0, h[k]); the host layer checks its maps once per geometry
 *   h / w         HOST [K] member plane sizes
 * Per output pixel and class, in f32 and in this order: sum = P_1[c] + ... + P_K[c] (scale order),
 * Pbar[c] = sum * f32(1/K); label = first argmax of Pbar; confidence = min(255, round-to-nearest(Pbar[label] * 255)).
 * With K = 1 these are the member's mean-mode labels and confidence, resampled with the maps.
 *   labels        nullable [h_full, w_full] u8 ; rgb nullable [h_full, w_full, 3] u8 (lut_rgb HOST [C, 3], needed iff
 *                 rgb) ; confidence nullable [h_full, w_full] u8.  At least one output.
 * Any width and any output alignment; rows are dense.  PYLC_ERR_ARG for K outside [1, PYLC_MAX_SCALES], a null
 * plane or map, a non-positive size or no output; PYLC_ERR_CLASSES for C outside [1, 32].
 */
#define PYLC_MAX_SCALES 8
PYLC_API int pylc_multiscale_combine(const float *const *probs, const int32_t *const *x_ofs, const int32_t *const *y_ofs,
                            const int *h, const int *w, int K, int C, int h_full, int w_full, const uint8_t *lut_rgb,
                            uint8_t *labels, uint8_t *rgb, uint8_t *confidence, pylc_stream_t stream);

/* ---- multi-loss --------------------------------------------------------------------------- */

/*
 * MultiLoss = ce_w*CE + dice_w*Dice + focal_w*Focal (models/modules/loss.py:71-194), computed in
 * two passes because Dice needs batch-global sums before any gradient exists:
 *
 *   pylc_multiloss_reduce    logits + target -> partials[2C+3] f64 (ADDED INTO):
 *                            [0,C) I_c = sum p_c [t=c]; [C,2C) K_c = sum (p_c + [t=c]);
 *                            2C: sum w_t (-ln p_t); 2C+1: sum w_t; 2C+2: sum focal_px
 *                            (data-parallel ranks all-reduce `partials` here)
 *   pylc_multiloss_finalize  partials -> out[4] f32 = {loss, ce, dice, focal}
 *   pylc_multiloss_grad      logits + target + partials -> grad[B,C,HW] f32 = grad_scale * dL/dz
 *                            (times *grad_scale_dev when that device pointer is non-NULL: the
 *                            upstream autograd gradient, read on the device, no host sync)
 *
 *   logits  [B, C, HW] f32 ; target [B, HW], target_is_i64 ? int64 (the reference dtype) : u8
 *   class_w nullable [C] f32 device (CrossEntropyLoss weights; NULL = unweighted)
 *   n_px_total: pixels over ALL ranks (= B*HW on one GPU)
 *   target_u8_out (reduce) / target_u8_ws (fwd_bwd): nullable [B*HW] u8 device workspace.  With int64
 *     targets the reduce pass leaves a one-byte copy of them there, which the gradient pass reads
 *     instead (1 B/px instead of 8): pass it to pylc_multiloss_grad as `target` with target_is_i64 = 0;
 *     the single-launch form does so itself.  Ignored for u8 targets.
 *   A target outside [0, C) makes every loss value and gradient of the batch NaN (the reference's
 *     CrossEntropyLoss / one_hot raise, models/modules/loss.py:66-69,137); the host mirror raises.
 */
typedef struct pylc_loss_cfg {
    float ce_weight, dice_weight, focal_weight; /* config.py:201-203, defaults 0.5 each */
    float dice_smooth;                          /* config.py:204, 1.0                   */
    float fl_gamma, fl_alpha;                   /* config.py:206-207, 2 and 0.25        */
    float eps;                                  /* models/modules/loss.py:51, 1e-8      */
} pylc_loss_cfg;

PYLC_API int pylc_multiloss_reduce(const float *logits, const void *target, int target_is_i64, int B, int C,
                          int64_t HW, const float *class_w, const pylc_loss_cfg *cfg,
                          double *partials, uint8_t *target_u8_out, pylc_stream_t stream);
PYLC_API int pylc_multiloss_finalize(const double *partials, int C, int64_t n_px_total,
                            const pylc_loss_cfg *cfg, float *out4, pylc_stream_t stream);
PYLC_API int pylc_multiloss_grad(const float *logits, const void *target, int target_is_i64, int B, int C,
                        int64_t HW, const float *class_w, const pylc_loss_cfg *cfg,
                        const double *partials, int64_t n_px_total, float grad_scale,
                        const float *grad_scale_dev, float *grad, pylc_stream_t stream);

/*
 * Forward AND backward in one cooperative launch, for the single-GPU training step (no all-reduce
 * between the passes): reduce pass -> grid-wide barrier -> out4 = {loss, ce, dice, focal} ->
 * gradient pass, which walks the logits back to front so that it starts on what the reduce pass
 * left in L2.  Same arguments as the two calls above; `partials` must be zeroed by the caller and
 * holds the 2C+3 sums afterwards; out4 is nullable; n_px_total is B*HW.
 *
 * pylc_scale_unless_one_f32: data[i] *= *scale_dev unless *scale_dev == 1 -- applies autograd's
 * upstream gradient to the stashed dL/dz without a host sync (a no-op for loss.backward()).
 */
PYLC_API int pylc_multiloss_fwd_bwd(const float *logits, const void *target, int target_is_i64, int B, int C,
                           int64_t HW, const float *class_w, const pylc_loss_cfg *cfg,
                           double *partials, float grad_scale, const float *grad_scale_dev,
                           float *grad, float *out4, uint8_t *target_u8_ws, pylc_stream_t stream);
PYLC_API int pylc_scale_unless_one_f32(float *data, int64_t n, const float *scale_dev, pylc_stream_t stream);

/*
 * The same single launch for a DATA-PARALLEL training step (one process per GPU): reduce pass -> grid barrier ->
 * all-reduce of the 2C+3 partials INSIDE the kernel, over peer-addressable memory (NVLink / NVSwitch loads and
 * stores; no NCCL call, no second launch) -> grid barrier -> loss values -> gradient pass.  The result is the loss
 * of the single large batch of all ranks and d(that loss)/d(local logits); `partials` returns the global sums,
 * identical to the last bit on every rank (added in rank order); n_px_total is B*HW*world.
 * Replaces the reference's loss of one training step (models/model.py:317-325, models/modules/loss.py:71-194)
 * under data parallelism, which the reference does not have (models/model.py:185-188).
 *
 *   peer_ws  DEVICE array [world]: pointer to every rank's exchange workspace as addressable from THIS process, in
 *            rank order (torch.distributed._symmetric_memory: rendezvous(...).buffer_ptrs_dev).  A workspace is
 *            PYLC_DP_WS_BYTES bytes, zero-initialised once; only these calls write it.
 *   epoch    call counter, the same on every rank, 1, 2, 3, ... per workspace.
 * Every rank of the group must make the call; a rank that does not arrive within ~1 s turns the results into NaN.
 */
#define PYLC_DP_MAX_RANKS 16
#define PYLC_DP_MAX_PARTIALS 80 /* >= 2 * PYLC_MAX_CLASSES + 3 */
#define PYLC_DP_WS_BYTES 2048
PYLC_API int pylc_multiloss_fwd_bwd_dp(const float *logits, const void *target, int target_is_i64, int B, int C,
                              int64_t HW, const float *class_w, const pylc_loss_cfg *cfg,
                              double *partials, float grad_scale, const float *grad_scale_dev,
                              float *grad, float *out4, uint8_t *target_u8_ws,
                              double *const *peer_ws, int rank, int world, uint64_t epoch, pylc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PYLC_B200_H */
