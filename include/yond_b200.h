/*
 * yond_b200.h — C-ABI of libyond_b200.so: B200 (sm_100a) kernels for YOND's per-image blind raw
 * denoising path (fenghansen/YOND_public).  This is the drop-in boundary: plain pointers and sizes,
 * no torch / C++ types.  Every entry point names the reference interface it replaces (file:line in
 * the reference tree).  The reference is pure Python; a maintainer binds this library with ctypes
 * (see INTEGRATION.md — the stub is yond_public_b200/_lib.py).
 *
 * Conventions
 *   - All data pointers are DEVICE pointers unless the name says `host`.  The caller (PyTorch) owns
 *     every buffer; the library never frees caller memory.  Opaque handles own packed weights.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  All functions are
 *     asynchronous with respect to the host unless stated otherwise.
 *   - Return value: 0 = ok, non-zero = error; yond_last_error() gives the message (thread-local).
 *   - Layouts: Bayer frames (B,H,W) f32; packed frames NHWC (B,h,w,4) f32 with channel = 2*(row&1)+(col&1)
 *     (the reference's `bayer2rggb` order, CFA-agnostic); activations NHWC bf16.
 */
#ifndef YOND_B200_H
#define YOND_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YOND_OK 0
#define YOND_ERR_INVALID 1
#define YOND_ERR_CUDA 2
#define YOND_ERR_UNSUPPORTED 3

const char* yond_last_error(void);
int yond_version(void);
/* Number of kernels launched by this library since process start (bench.py's `gpu_launches`). */
uint64_t yond_launch_count(void);

/* Live stage profiler (bench.py's per-kernel roofline): while enabled, every library stage is bracketed by CUDA events on
 * its launching stream and booked with its algorithmic bytes / FLOPs (SURVEY 8(d)).  yond_prof_read writes a JSON object
 * {"stage": {"scopes": n, "ms": t, "bytes": b, "flops": f}, ...} (it waits for the recorded events). */
int yond_prof_enable(int on);
int yond_prof_read(char* buf, size_t cap, int reset);

/* ---- A1/A2: Bayer pack / unpack — utils/isp_ops.py:57-63 (bayer2rggb, rggb2bayer), batched :65-71 ---- */
int yond_pack(const float* bayer, float* rggb, int B, int H, int W, void* stream);
int yond_unpack(const float* rggb, float* bayer, int B, int h, int w, void* stream);

/* ---- SURVEY 8(f)-1: RAW ingest — data_process/process.py:40-64 (pack_raw_bayer) ----
 * uint16 sensor mosaic -> four float32 planes in the order R, G1, B, G2 given by the 2x2 `raw_pattern`
 * (pos4[c] = 2*row + col of colour c inside the CFA cell), out = (v - black[c]) / (white - black[c]) in float32 with
 * IEEE subtraction / division like NumPy, optionally clipped to [0,1].  `pos4` and `black4` are HOST arrays.
 * layout 0: (B,4,H/2,W/2) planes like the reference; layout 1: (B,H/2,W/2,4) interleaved (what yond_vst_fwd-style
 * kernels and the estimator consume).  Reads 2 B/px instead of the 4 B/px of a float32 mosaic. */
int yond_pack_raw(const uint16_t* raw, float* out, int B, int H, int W, const int* pos4, const float* black4, float white,
                  int clip, int layout, void* stream);

/* How a uint16 sensor mosaic becomes the float32 frame the path works on (the *_raw16 entry points apply it on load). */
typedef struct yond_raw_norm {
  float black, white, ratio; /* out = (float32(raw) - black) * ratio / (white - black), float32 arithmetic in that order */
  int clip;                  /* clip to [0,1] afterwards */
} yond_raw_norm;

/* Dataset normalisation of the 14-bit drivers — data_process/yond_datasets.py:955-961, :1053-1056:
 * out = (float32(raw) - black) * ratio / (white - black) on the mosaic itself, float32 arithmetic in that order, unclipped unless
 * `clip`.  `n` pixels (any shape), 2 B/px read + 4 B/px written.  The result is the `data['lr']` the drivers hand to IterDenoise
 * with p = {wp: white, bl: black, ratio, scale: (white - black) / ratio}. */
int yond_ingest_mosaic(const uint16_t* raw, float* out, size_t n, float black, float white, float ratio, int clip, void* stream);

/* CFA canonicalisation — utils/sidd_utils.py:198-213 (rot_bayer = np.rot90 by k quarter turns, counter-clockwise, over the
 * last two axes; the driver rotates every SIDD frame to the RGGB phase before denoising and back afterwards,
 * YOND_SIDD.py:403,463).  in: (B,H,W) float32, out: (B,W,H) for odd k, (B,H,W) for even k.  Pure data movement. */
int yond_rot90(const float* in, float* out, int B, int H, int W, int k, void* stream);

/* ---- SURVEY 8(f)-3: image-quality metrics of the SIDD driver — YOND_SIDD.py:651-652 (per-block raw PSNR / SSIM),
 * :679-697 (ssim), :700-721 (calculate_ssim); compare_psnr = skimage.metrics.peak_signal_noise_ratio (third-party) ----
 * a, b: (nimg, H, Wm) float32 mosaics of nblk blocks side by side (Wm = nblk * block width); every block is measured alone.
 * psnr[nimg*nblk] = 10 log10(data_range^2 / mean((a-b)^2)) with the float32 difference / square and float64 mean skimage
 * uses for float32 inputs.  ssim[nimg*nblk] = mean over the valid region of the SSIM map of (a*ssim_scale, b*ssim_scale)
 * (float32 products like `dn*255`, then float64), 11x11 window = outer(window11, window11) (HOST array: cv2.getGaussianKernel(11,
 * 1.5)), C1 = (0.01*255)^2, C2 = (0.03*255)^2.  Either output may be null.  Results stay on the device. */
int yond_block_metrics(const float* a, const float* b, int nimg, int H, int Wm, int nblk, double data_range, float ssim_scale,
                       const double* window11, double* psnr, double* ssim, void* stream);

/* The sRGB pictures' numbers — YOND_SIDD.py:661-665: a, b (nimg, H, Wm, 3) uint8 (BGR or RGB), nblk blocks along W
 * (np.split(..., axis=-2)).  psnr = 10 log10(255^2 / mean((a-b)^2)) over the block's three channels (scikit-image promotes
 * integer inputs to float64: exact), ssim = mean of the three per-channel SSIMs, window as above. */
int yond_block_metrics_rgb8(const uint8_t* a, const uint8_t* b, int nimg, int H, int Wm, int nblk, const double* window11,
                            double* psnr, double* ssim, void* stream);

/* ---- SURVEY 8(f)-3: sRGB render of a mosaic — utils/sidd_utils.py:156-180 (process_sidd_image) with :182-196 (flip_bayer),
 * :241-247 (demosaic_CV2), :249-252 (apply_gains), :260-266 (apply_ccm, gamma_compression), :270-277 (process), :226-232
 * (swap_channels) ----
 * bayer: (B,H,W) float32 in the sensor's CFA phase; flip_lr / flip_ud: the flips that bring that phase to RGGB (flip_bayer; the
 * picture stays flipped like the reference's).  gains3 = (1/wb_r, 1/wb_g, 1/wb_b), cam2rgb9 = row-normalised inv(cst x rgb2xyz),
 * both float64 HOST arrays (3x3 host algebra stays with the caller: NumPy on both sides).  One kernel: clip, gains and clip in
 * float64, truncation to a 14-bit mosaic, OpenCV's edge-aware demosaic (integer), float32 / 16383, CCM and 1/2.2 gamma in float64,
 * x255, truncation.  bgr: (B,H,W,3) uint8, channel order B, G, R.  H, W even and >= 4. */
int yond_render_srgb(const float* bayer, uint8_t* bgr, int B, int H, int W, int flip_lr, int flip_ud, const double* gains3,
                     const double* cam2rgb9, void* stream);
/* cv2.cvtColor(bayer, cv2.COLOR_BayerBG2RGB_EA) for uint16 mosaics (third party: OpenCV imgproc/demosaicing.cpp, edge-aware
 * variant), the integer stage of the render on its own: (B,H,W) uint16 -> (B,H,W,3) uint16, site (0,0) of the cell in channel 0.
 * Bit-exact against opencv-python 4.13.0. */
int yond_demosaic_ea(const uint16_t* bayer, uint16_t* rgb, int B, int H, int W, void* stream);

/* ---- the pictures and numbers of a whole SIDD evaluation — YOND_SIDD.py:635-668 (multiprocess_plot) over every image and round at
 * once, each image rendered with its own metadata (:601-607: bayer_2by2, wb and cst2 of the image) ----
 * yond_render_cam: one image's camera, the numbers process_sidd_image derives from its metadata (utils/sidd_utils.py:156-180):
 *   gain = (1/wb_r, 1/wb_g, 1/wb_g, 1/wb_b) per 2x2 site of the flipped frame, row-major (:249-252, :272); cam2rgb = row-normalised
 *   inv(cst2 x rgb2xyz), row-major (:161-170); flip_lr / flip_ud: the flips of flip_bayer (:182-196).
 * yond_render_pic: one picture: `src` the (H,W) float32 mosaic (NULL: not rendered), `cam` the index of its camera record, `src_max`
 *   (optional) a DEVICE float holding max(src, 0) (yond_seg_max): 0 means not rendered — the reference renders and scores nothing for
 *   an output without a positive value (:644-647).  `reserved` is not read.
 * yond_render_srgb_cams: yond_render_srgb of B pictures of one size (H, W) in one launch, picture b from pics_dev[b] with camera
 *   cams_dev[pics_dev[b].cam] (both DEVICE arrays; `cam` is not range-checked), into bgr (B,H,W,3).  Same arithmetic and bytes as
 *   yond_render_srgb with that camera; a picture that is not rendered leaves its bytes of bgr as they were.
 * yond_sidd_scores: the per-image table from per-block numbers.  psnr / ssim: (nround, nimg, nblk) float64, yond_block_metrics of
 *   every round's output against the clean mosaics; psnr_rgb / ssim_rgb (both or neither may be NULL): the same layout,
 *   yond_block_metrics_rgb8 of the rendered pictures; out_max: (nround, nimg) float32 max(output, 0) per round (yond_seg_max);
 *   rounds_dev: (nimg) int32, the rounds each image completed.  table: (nround, nimg, 4) float64 = (psnr, ssim, psnr_rgb, ssim_rgb),
 *   each the sum over the nblk blocks in block order / nblk (:651-665).  Where out_max is 0: psnr = ssim = -1 and the sRGB entries
 *   NaN; rounds at or beyond rounds_dev[i]: all four NaN; without sRGB inputs the sRGB entries are NaN. */
typedef struct yond_render_cam {
  double gain[4];
  double cam2rgb[9];
  int32_t flip_lr, flip_ud;
} yond_render_cam;
typedef struct yond_render_pic {
  const float* src;
  const float* src_max;
  int32_t cam;
  int32_t reserved;
} yond_render_pic;
int yond_render_srgb_cams(const yond_render_pic* pics_dev, const yond_render_cam* cams_dev, uint8_t* bgr, int B, int H, int W,
                          void* stream);
int yond_sidd_scores(const double* psnr, const double* ssim, const double* psnr_rgb, const double* ssim_rgb, const float* out_max,
                     const int32_t* rounds_dev, int nround, int nimg, int nblk, double* table, void* stream);

/* ---- A3/A4 elementwise, for the function-level surface — utils/isp_algos.py:5-14, :17-33 ---- */
int yond_vst(const float* x, float* z, size_t n, double sigma, double gain, void* stream);
int yond_inverse_vst(const float* z, float* x, size_t n, double sigma, double gain, int exact, void* stream);

/* ---- A5: BiasLUT — utils/isp_algos.py:162-231.
 * yond_lut_row: sigma-lerp of the (nx=1921, nsg=1101) [x,sigma] table into one nx-entry row (data_merge over
 *   sigma, :225); `sg_pos` is the fractional sigma index computed on the host (pos_interp, :199).
 * yond_lut_apply: per-element lookup bias(max(x,0)/K) with the reference's piecewise-linear node inversion
 *   (pos_interp :179-186 + data_merge :188-194); x in DN units.  `xnodes` = the nx node positions (electrons). */
int yond_lut_row(const float* lut2d, int nx, int nsg, double sg_pos, float* row, void* stream);
int yond_lut_apply(const float* x, float* bias, size_t n, const float* row, const float* xnodes, int nx,
                   double gain, double sigma, void* stream);

/* interp1d(nodes, vals)(clip(max(x,0), <= nodes[-1])): how the reference applies a get_bias table (YOND_SIDD.py:257). */
int yond_table_apply(const float* x, float* bias, size_t n, const float* vals, const float* nodes, int n_nodes, void* stream);

/* Per-frame parameters of the fused VST stages (one entry per frame of a batch). */
typedef struct {
  float gain;      /* K   (DN)                                   YOND_SIDD.py:356 */
  float sigma;     /* sigma_read (DN)                                               */
  float scale;     /* wp - bl (/ratio)                            YOND_SIDD.py:251,504 */
  float lower;     /* VST(0)                                      YOND_SIDD.py:264 */
  float upper;     /* VST(scale)                                  YOND_SIDD.py:265 */
  int32_t lut_row; /* row index into `rows` (−1: no bias correction, bias_corr=None) */
  int32_t table_n; /* 0: `rows[lut_row]` is a sigma-interpolated BiasLUT row (1921 nodes, electrons);
                      >0: a fallback get_bias table (isp_algos.py:98-140) with `table_n` nodes in DN */
  int32_t exact_inverse; /* 1: closed-form exact unbiased inverse (isp_algos.py:20-27) */
} yond_vst_params;

/* ---- A18 front half (YOND_SIDD.py:251-269,275,281-282,286): pack*scale -> bias -> VST-bias -> normalise ->
 * clamp(0,1) -> reflect-pad to (hp,wp) -> z (B,hp,wp,4) f32; also ub[b] = max(z[b]) (A14, modules.py:15-21).
 * `rows`: (nrows, row_stride) f32 bias tables; `xnodes`: (nrows, row_stride) node positions of each row (the BiasLUT
 * x-grid in electrons for LUT rows, the get_bias nodes in DN for fallback tables).  p2d = (left, right, top, bottom) in packed pixels (utils/utils.py:246-252). */
int yond_vst_fwd(const float* bayer, float* z, float* ub, int B, int H, int W, int pad_l, int pad_r, int pad_t,
                 int pad_b, const yond_vst_params* params_dev, const float* rows, const float* xnodes,
                 int row_stride, void* stream);
/* The same front end reading the uint16 sensor mosaic (B,H,W) and normalising it on load (SURVEY 8(f)-1: 2 B/px reads; the
 * float32 frame of data_process/yond_datasets.py:955-961 / :1053-1056 never exists in memory).  `nrm` (HOST) applies to every frame.
 * nrm_dev (optional, DEVICE, one entry per image of frames_per_img consecutive frames; may be NULL): frame b is normalised with
 * nrm_dev[b / frames_per_img] instead (per-image white / black level / ratio of a mixed batch, same float32 arithmetic; `nrm`
 * may then be NULL).  The call must start at an image boundary: pass the entry of its first image. */
int yond_vst_fwd_raw16(const uint16_t* raw, const yond_raw_norm* nrm, float* z, float* ub, int B, int H, int W, int pad_l, int pad_r,
                       int pad_t, int pad_b, const yond_vst_params* params_dev, const float* rows, const float* xnodes, int row_stride,
                       void* stream, const yond_raw_norm* nrm_dev, int frames_per_img);
/* ---- A18 back half (YOND_SIDD.py:286,289-298, caller's clip :389/:406): y (B,hp,wp,4) f32 -> clamp(0,1) -> crop ->
 * de-normalise -> inverse VST -> unpack -> /scale -> [clip 0..1] -> Bayer (B,H,W) f32. */
int yond_vst_inv(const float* y, float* bayer, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                 const yond_vst_params* params_dev, int clip01, void* stream);
/* Back half with output placement and round selection: frames frame0 .. frame0+B-1 of a batch whose whole output is
 * `out`.  frames_per_row = 1: (N,H,W); n > 1: frame f is block f % n of mosaic f / n, (N/n, H, n*W) — the reference's
 * np.concatenate(blocks, axis=-1) (YOND_SIDD.py:408).  seg_ok_dev (optional, per image of frames_per_seg frames): where 0
 * (round-2 beta1 < 0, :445-447) the frame is copied from `fallback` (round-1 output, same layout) instead. */
int yond_vst_inv_place(const float* y, float* out, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                       const yond_vst_params* params_dev, int clip01, int frames_per_row, int frame0,
                       const int32_t* seg_ok_dev, int frames_per_seg, const float* fallback, void* stream);
/* Simple_Denoiser's front/back (YOND_SIDD.py:238-248): pack -> reflect pad -> clamp, and clamp -> crop -> unpack. */
int yond_pack_pad(const float* bayer, float* z, float* ub, int B, int H, int W, int pad_l, int pad_r, int pad_t,
                  int pad_b, void* stream);
int yond_crop_unpack(const float* y, float* bayer, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                     void* stream);

/* ---- A7/A8/A11: box statistics — utils/isp_algos.py:234-242 (stdfilt = cv2.blur pair), YOND_SIDD.py:62-71, :89-98.
 * Input: packed frames (B,h,w,C) f32 interleaved (C = 4, or 128 for the SIDD_256 channel stack).
 * yond_box_blur: normalised k x k box, BORDER_REFLECT_101, float64 sums -> f32 (what cv2.blur computes).
 * yond_nlf_maps: mode 0 (self)  : var = std_k(x)^2, mean = blur_k(x), lap = std_k(blur_k2(x)), k2 = k/3*2+1
 *                mode 1 (collab): var = std_k(x)^2 - std_k(y)^2, mean = blur_k(y), lap = std_k(y)
 * `work`: scratch of yond_nlf_work_bytes(). */
int yond_box_blur(const float* x, float* out, int B, int h, int w, int C, int k, int square_input, void* work,
                  void* stream);
size_t yond_nlf_work_bytes(int B, int h, int w, int C);
int yond_nlf_maps(const float* x, const float* y, float* var, float* mean, float* lap, int B, int h, int w, int C,
                  int k, int mode, void* work, void* stream);

/* ---- the estimator on the device — A9 get_threshold('score3') YOND_SIDD.py:22-49, A10 masked line fit :77-86 and
 * utils/isp_algos.py:345-365, in float64 ----
 * yond_nlf_maps_bayer: the maps straight from the Bayer frames (no pack pass).  Inputs are `nimg` images of `nblk`
 *   blocks of (H,W) each, in the blocks layout (nimg,nblk,H,W) (`*_mosaic` = 0, the SIDD dataset layout) or the mosaic
 *   layout (nimg,H,nblk*W) (`*_mosaic` = 1, np.concatenate(blocks, -1) of YOND_SIDD.py:315/:408).  split_blocks = 0: an
 *   image's blocks form one mosaic for the box filters (SelfNLF on the mosaic, :315,:341; plain frames are nblk = 1);
 *   split_blocks = 1: every block is its own image (SIDD_256, :65,:91-93).  Maps come out packed, (B,h,w,4) with
 *   B = nimg*nblk / w = W/2 (split) or B = nimg / w = nblk*W/2.  `seg_max` (optional, nimg floats): max(x, 0) per image
 *   of the first input — the bound of the fallback bias table (:393, isp_algos.py:101).  `work`: yond_nlf_work_bytes(B,h,w,4).
 *   mode 0: self maps (y unused); 1: collab maps; 3: var = stdfilt(x, k)**2 alone (y, mean, lap untouched): the noisy-frame
 *   statistics every collab round of IterDenoise shares.  Any other mode is rejected with YOND_ERR_INVALID.
 * yond_nlf_maps_collab_cached: the collab maps of a round from a cached `lr_var` = stdfilt(lr, k)**2 in the same geometry (the
 *   var map of mode 0 or mode 3; read only, may be `var` itself): var = lr_var - stdfilt(y, k)**2, mean = blur_k(y),
 *   lap = stdfilt(y, k), one box pass over the float32 frame y (layout / geometry arguments as above).  The noisy frame is not
 *   an argument, so the call is the same for float32 and uint16 sensor inputs.
 * yond_nlf_fit: percentiles -> score3 threshold -> masked sums (with the empty-mask fallbacks of :77-84) -> line fit,
 *   per segment, all on the device: regs_dev (nseg,2) float64 = (beta1, beta2).
 *   The order statistics behind the percentiles are exact, computed by radix select.  `quants_host`: the nq <= 24 ascending
 *   percentiles of get_threshold (np.linspace(step,100,100//step)).  detail_dev (optional, (nseg, 52) float64):
 *   th, index, percent, redo flag, ths[24], npeaks[24].  `work`: yond_nlf_fit_work_bytes(nseg), 256-byte aligned. */
int yond_nlf_maps_bayer(const float* x, int x_mosaic, const float* y, int y_mosaic, float* var, float* mean, float* lap,
                        int nimg, int nblk, int H, int W, int split_blocks, int k, int mode, float* seg_max, void* work,
                        void* stream);
/* The same maps with the FIRST input given as the uint16 sensor mosaic, normalised on load (the second input of the collab mode is
 * the float32 output of round 1).  `nrm` (HOST) applies to every image.
 * yond_nlf_maps_raw16_per_image: the same with `nrm_dev`, a DEVICE array of nimg entries: image i (with split_blocks, every block
 *   of image i) is normalised with nrm_dev[i] — the per-image white / black level / ratio of a mixed batch, same float32
 *   arithmetic.  A separate entry point, so that bindings of yond_nlf_maps_raw16 keep their argument list. */
int yond_nlf_maps_raw16(const uint16_t* x, const yond_raw_norm* nrm, int x_mosaic, const float* y, int y_mosaic, float* var, float* mean,
                        float* lap, int nimg, int nblk, int H, int W, int split_blocks, int k, int mode, float* seg_max, void* work,
                        void* stream);
int yond_nlf_maps_raw16_per_image(const uint16_t* x, const yond_raw_norm* nrm_dev, int x_mosaic, const float* y, int y_mosaic,
                                  float* var, float* mean, float* lap, int nimg, int nblk, int H, int W, int split_blocks, int k,
                                  int mode, float* seg_max, void* work, void* stream);
int yond_nlf_maps_collab_cached(const float* y, int y_mosaic, const float* lr_var, float* var, float* mean, float* lap, int nimg,
                                int nblk, int H, int W, int split_blocks, int k, void* stream);
size_t yond_nlf_fit_work_bytes(int nseg);
int yond_nlf_fit(const float* var, const float* mean, const float* lap, size_t seg_len, int nseg, const double* quants_host,
                 int nq, double* regs_dev, double* detail_dev, void* work, void* stream);

/* ---- the self estimate of frames of different sizes in one pass — YOND_SIDD.py:338-341 (round 1 of IterDenoise on the
 * full-resolution frame `lr_path_full` when it exists), :62-71 (SelfNLF), :22-49 (score3), :77-86 + utils/isp_algos.py:345-365 (fit).
 * yond_frame_geom: one record per frame, in DEVICE memory.  Frame i's packed maps (H/2, W/2, 4) sit at float offset `off` of the
 *   concatenated var / mean / lap buffers (off = sum of H*W over the frames before it).
 * yond_nlf_maps_frames: the self maps (mode 0 of yond_nlf_maps_bayer) of `nframes` float32 Bayer frames given by `frames_dev`, in
 *   one launch per box pass whatever the sizes.  max_H / max_W: the largest H and W of the records (they size the grid; CTAs past a
 *   smaller frame's extent return at once).  Every frame needs even H, W with H/2 and W/2 larger than k/2; frames narrower than the
 *   box filter's block take the same wide layout as large frames.  `work`: 16 bytes per packed pixel of all frames (sum of H*W*4
 *   bytes), 16-byte aligned.
 * yond_nlf_fit_ragged: yond_nlf_fit over segments of different lengths: segment s is [seg_off_dev[s], seg_off_dev[s + 1]) of the
 *   maps (a DEVICE array of nseg + 1 float offsets, multiples of 4).  max_seg_len (host) is the longest segment; it sizes the grids.
 *   The percentile ranks and weights are computed per segment on the device.  `work`: yond_nlf_fit_ragged_work_bytes(nseg), 256-byte
 *   aligned.  Same outputs and arithmetic as yond_nlf_fit.
 * yond_seg_max: seg_max[s] = max(x, 0) over the nseg contiguous segments of seg_len floats of x (the blocks of image s) — the bound
 *   of the fallback bias table when round 1 estimated on the full frame (:393-395: the maximum of the blocks, not of lr_full).
 *   seg_len a multiple of 4, x 16-byte aligned. */
typedef struct yond_frame_geom {
  const float* base; /* the (H, W) float32 Bayer frame */
  int H, W;
  long long off;
} yond_frame_geom;
int yond_nlf_maps_frames(const yond_frame_geom* frames_dev, int nframes, int max_H, int max_W, float* var, float* mean, float* lap,
                         int k, void* work, void* stream);
size_t yond_nlf_fit_ragged_work_bytes(int nseg);
int yond_nlf_fit_ragged(const float* var, const float* mean, const float* lap, const unsigned long long* seg_off_dev,
                        size_t max_seg_len, int nseg, const double* quants_host, int nq, double* regs_dev, double* detail_dev,
                        void* work, void* stream);
int yond_seg_max(const float* x, size_t seg_len, int nseg, float* seg_max, void* stream);

/* ---- IterDenoise over full frames of different sizes in one batch — YOND_SIDD.py:301-483 with the frame as the image (round 1
 * :315/:338-341 self estimate, :356 + :252-269 VST constants, :419-472 collab rounds on (lr, previous output), :445-447 selection).
 * Every record table below is in DEVICE memory, and the caller keeps every frame it points to alive and unchanged until the work
 * is done.  A float32 frame must be 8-byte aligned (64-bit Bayer loads), a uint16 mosaic 4-byte aligned; these are not checked here.
 * yond_nlf_maps_frames_max: yond_nlf_maps_frames plus `seg_max` (optional, nframes floats): max(x, 0) per frame from the first box
 *   pass — the bound of the fallback bias table (:256, isp_algos.py:101).
 * yond_nlf_maps_frames_raw16: the same self maps (and seg_max) with every record's `base` holding the address of a uint16 (H, W)
 *   sensor mosaic, not a float32 frame: frame i is normalised on load with nrm_dev[i] (a DEVICE array of nframes entries), the same
 *   float32 arithmetic as yond_nlf_maps_raw16_per_image (data_process/yond_datasets.py:955-961, :1053-1056).
 * yond_nlf_maps_frames_collab_cached: the collab maps (yond_nlf_maps_collab_cached, :89-98 with stdfilt(lr, k)**2 cached) of every
 *   frame in one launch: frame i of the round's output is the float32 Bayer frame at y + off_i (the flat layout of the maps, so a
 *   round's outputs concatenated in record order), lr_var the var maps of the self estimate of the same records.  The records'
 *   `base` is not read.  y and lr_var 16-byte aligned.
 * yond_vst_fwd_frames: yond_vst_fwd (nrm_dev NULL, float32 frames) or yond_vst_fwd_raw16 (nrm_dev set: uint16 mosaics, frame b
 *   normalised with nrm_dev[b]) over B records that all hold (H, W) frames: frame b is read from frames_dev[b].base, wherever it
 *   lies.  z, ub, params_dev and the padding as in yond_vst_fwd. */
int yond_nlf_maps_frames_max(const yond_frame_geom* frames_dev, int nframes, int max_H, int max_W, float* var, float* mean, float* lap,
                             int k, void* work, void* stream, float* seg_max);
int yond_nlf_maps_frames_raw16(const yond_frame_geom* frames_dev, const yond_raw_norm* nrm_dev, int nframes, int max_H, int max_W,
                               float* var, float* mean, float* lap, int k, float* seg_max, void* work, void* stream);
int yond_nlf_maps_frames_collab_cached(const float* y, const yond_frame_geom* frames_dev, int nframes, int max_H, int max_W,
                                       const float* lr_var, float* var, float* mean, float* lap, int k, void* stream);
int yond_vst_fwd_frames(const yond_frame_geom* frames_dev, const yond_raw_norm* nrm_dev, float* z, float* ub, int B, int H, int W,
                        int pad_l, int pad_r, int pad_t, int pad_b, const yond_vst_params* params_dev, const float* rows,
                        const float* xnodes, int row_stride, void* stream);

/* ---- the VST parameter chain on the device — YOND_SIDD.py:356 (round 1) / :438-447 (round 2 guards), :252-269,
 * :284-285 (bias source, VST(0), VST(scale), t = nsr*1.03), utils/isp_algos.py:179-231 (sigma row of the BiasLUT),
 * :49-140 (get_bias: the numeric Poisson (*) Gaussian fallback table — SURVEY 8(f)-2, generated on the device).
 * yond_vst_params_fill: regs_dev (nseg,2) -> per-frame yond_vst_params (nseg*frames_per_seg), t_dev (same count), and per
 *   image one bias row + its node positions in rows / xnodes (nseg, row_stride).  round 1: sigma = sqrt(max(beta2,0));
 *   round >= 2: beta2 < 0 -> beta1^2 and ok_dev[s] = (beta1 >= 0) && prev_ok[s] (images with ok = 0 get `prev_params`, their
 *   output is discarded by yond_vst_inv_place).  prev_ok (optional, the previous round's ok_dev; NULL = every image live):
 *   chains the live mask over the rounds of IterDenoise, an image that stopped never comes back whatever its later beta1.  bias_mode: 0 = None, 1 = 'pre' (bias applied, t*1.03), 2 = 'post' (no bias is
 *   applied, like the reference).  lut2d (nx,nsg) f32 + sg_lut_dev (nsg) f64 + x_lut_dev (nx) f32: the BiasLUT, or NULL:
 *   then — and for sigma/K beyond the table — the numeric table up to bound = seg_max[s]*bound_scale (float32 product).
 *   regs_out (optional, (nseg,4) f64): beta1, beta2 (after the guard), gain, sigma.  `work`: yond_chain_work_bytes(nseg).
 *   seg_scales_dev (optional, DEVICE, (nseg,3) f64; may be NULL): per image (scale_est, scale, bound_scale), replacing the scalar
 *   arguments of the same names: a batch of images with their own white / black levels and ratios.  gain = beta1*scale_est,
 *   sigma = sqrt(beta2)*scale_est, VST(scale), q.scale = scale, the fallback table bound seg_max[s]*bound_scale.  An array of equal
 *   entries gives the same bits as the scalar call.
 * yond_bias_table: get_bias(bound, sigma, gain) nodes / values (float32, `cap` entries available) for one parameter
 *   set; n_nodes_dev receives the node count (= yond_bias_table_nodes(bound), a host-side helper). */
size_t yond_chain_work_bytes(int nseg);
int yond_bias_table_nodes(float bound);
int yond_vst_params_fill(const double* regs_dev, const float* seg_max_dev, int nseg, int frames_per_seg, double scale_est,
                         double scale, double bound_scale, int round, int bias_mode, int exact_inverse, const float* lut2d,
                         const double* sg_lut_dev, const float* x_lut_dev, int nx, int nsg,
                         const yond_vst_params* prev_params, yond_vst_params* params_dev, float* t_dev, float* rows,
                         float* xnodes, int row_stride, double* regs_out, int32_t* ok_dev, void* work, void* stream,
                         const int32_t* prev_ok, const double* seg_scales_dev);
int yond_bias_table(double gain, double sigma, float bound, float* nodes_dev, float* vals_dev, int cap,
                    int32_t* n_nodes_dev, void* work, void* stream);
/* get_bias_points(lams, K, sigGs, pho_min, close_form=True) (isp_algos.py:142-160): the bias at explicit float64 points
 * (BiasLUT.get_lut's small-input fallback, :204-212, and — with K = 1, pho_min = 100 on the x-grid — one column of the
 * offline bias_lut_2d.npy builder).  float64 in / out. */
int yond_bias_points(const double* lams_dev, int n, double gain, double sigma, int pho_min, double* bias_dev, void* work,
                     void* stream);

/* ---- A14-A17, A20: denoiser networks — archs/Unet.py:4-104 (UNetSeeInDark), :380-470 (GuidedResUnet),
 * :288-378 (SNRnet); blocks archs/modules.py:117-125,163-233.  Plugin descriptor = the yml `arch:` block. */
typedef struct yond_net yond_net_t;
#define YOND_ARCH_UNET 0     /* UNetSeeInDark  */
#define YOND_ARCH_GUIDED 1   /* GuidedResUnet  */
#define YOND_ARCH_SNR 2      /* SNRnet         */
#define YOND_ARCH_RES2 3     /* ResUnet2 (archs/Unet.py:197-286): GuidedResUnet's graph and state_dict keys, blocks without the
                                conditioning (ResBlock.forward never uses gamma / beta, archs/modules.py:258-265), LeakyReLU(0.2)
                                after conv_in, called as net(x) */
#define YOND_ARCH_SELFRES 4  /* SelfResUNet (archs/comp.py:745-802): constant-width residual U-Net (nf down, 2 nf up), max-pool down,
                                nearest-neighbour up, network input concatenated at the last up level; called as net(x); H, W
                                multiples of 32 */
#define YOND_ARCH_GSELF 5    /* GuidedSelfUnet (archs/comp.py:852-910): the same graph with noise-level conditioning — the second conv
                                of every block and the single conv of every down level are GLRs (conv, z*tk + tb, LeakyReLU);
                                called as net(x, t); res must be 0 (the reference's res branch cannot run) */
/* Creates a network; weights are set tensor-by-tensor with the reference's state_dict keys. */
int yond_net_create(int arch, int in_nc, int out_nc, int nf, int res, int norm, yond_net_t** out);
void yond_net_destroy(yond_net_t* net);
/* `host_data`: f32 tensor in the reference's (PyTorch) layout — Conv2d (Cout,Cin,kh,kw), ConvTranspose2d
 * (Cin,Cout,2,2), bias (C).  Repacked once to the kernels' layouts (per-tap K-major bf16).  utils/utils.py:160-209. */
int yond_net_set_tensor(yond_net_t* net, const char* key, const float* host_data, const int64_t* shape, int ndim);
/* The state_dict this network expects, in the reference's registration order (keys, shapes). */
int yond_net_num_keys(yond_net_t* net);
const char* yond_net_key(yond_net_t* net, int i);
int yond_net_key_shape(yond_net_t* net, int i, int64_t* shape4); /* returns ndim */
/* Returns the number of state-dict tensors still unset (0 = ready); `missing` receives a ';'-joined key list. */
int yond_net_missing(yond_net_t* net, char* missing, size_t cap);
size_t yond_net_workspace_bytes(yond_net_t* net, int B, int H, int W);
/* net(x[, t]) on NHWC input: z (B,H,W,4) f32 in [0,1] (H,W multiples of 16), ub (B) = per-sample max (used when
 * norm=1; pass the buffer yond_vst_fwd / yond_pack_pad filled), t (B) f32 per-sample guidance value BEFORE the
 * division by ub (archs/Unet.py:427-429; NULL for UNetSeeInDark).  y (B,H,W,4) f32 = network output (not clamped). */
int yond_net_forward(yond_net_t* net, const float* z, const float* ub, const float* t, float* y, int B, int H,
                     int W, void* workspace, size_t workspace_bytes, void* stream);
/* Module-level drop-in: NCHW f32 in / out like nn.Module.forward; computes ub itself (data_normalize). */
int yond_net_forward_nchw(yond_net_t* net, const float* x, const float* t, float* y, int B, int H, int W,
                          void* workspace, size_t workspace_bytes, void* stream);
/* FLOPs of the tensor-core conv stack for one forward of this shape (2*MAC, algorithmic, no halo / padding). */
double yond_net_flops(yond_net_t* net, int B, int H, int W);
/* 0: tcgen05 implicit-GEMM kernels (product path).  1: CUDA-core direct convolution (debug cross-check only).
 * 2: the tcgen05 kernels with the layer fusions off (up-sampling + shortcut, output conv in the last epilogue): A/B checks. */
int yond_net_set_conv_impl(yond_net_t* net, int impl);
/* Device time (ms) accumulated by the conv-stack kernels since the last reset, measured with CUDA events on
 * `stream` when profiling is enabled (bench.py's live roofline). */
int yond_net_profile(yond_net_t* net, int enable);
int yond_net_profile_read(yond_net_t* net, double* conv_ms, double* conv_flops, int* launches, int reset);

/* ---- single conv layer on NHWC bf16 activations (the building block of the networks above; torch.nn.Conv2d /
 * ConvTranspose2d in archs/Unet.py).  mode: 0 = 3x3 s1 p1, 1 = 1x1, 2 = 3x3 s2 p1, 3 = ConvTranspose 2x2 s2.
 * The input is the channel concatenation of src0 (Cin0) and src1 (Cin1, may be 0/NULL).  `weight_host`: f32 in the
 * PyTorch layout; bias/scale/shift/res/out are device pointers.  Epilogue: v = acc + bias; v = v*scale[b] + shift[b];
 * act (0 none, 1 LeakyReLU(slope), 2 SiLU); v += res; out0 = bf16(v); out1 = bf16(SiLU(v)) if given.
 * impl: 0 = tcgen05 kernel, 1 = CUDA-core cross-check.  Synchronous (packs and uploads the weights per call). */
int yond_conv2d(int mode, int impl, int B, int Hin, int Win, int Cin0, int Cin1, const void* src0, const void* src1,
                int Cout, const float* weight_host, const float* bias, const float* scale, const float* shift, int act,
                float slope, const void* res, void* out0, void* out1, void* stream);

/* ---- tiling helpers (new design; reference semantics utils/utils.py:254-268 + whole-frame forward) ----
 * Copies a halo-extended tile out of / back into a padded NHWC4 frame; out-of-frame halo pixels are zero
 * (what the network's own zero padding would have seen). */
int yond_tile_extract(const float* frame, float* tile, int H, int W, int y0, int x0, int th, int tw, void* stream);
int yond_tile_insert(const float* tile, float* frame, int H, int W, int y0, int x0, int th, int tw, int halo_t,
                     int halo_l, int core_h, int core_w, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* YOND_B200_H */
