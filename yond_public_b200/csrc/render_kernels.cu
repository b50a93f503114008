// sRGB render of the SIDD driver on the device (SURVEY 8(f)-3): the reference turns every noisy / denoised / clean mosaic into an
// 8-bit BGR picture on the CPU before it saves it and before the sRGB PSNR / SSIM (YOND_SIDD.py:601-607, :637-665).
//   reference: utils/sidd_utils.py:156-180 (process_sidd_image), :182-196 (flip_bayer), :215-224 (stack_rggb_channels),
//              :241-247 (demosaic_CV2: 14-bit truncation, cv2.COLOR_BayerBG2RGB_EA, float32 / 16383), :249-252 (apply_gains),
//              :260-266 (apply_ccm, gamma_compression), :270-277 (process), :226-232 (swap_channels)
//   third party: OpenCV's edge-aware demosaic (imgproc/demosaicing.cpp; opencv-python 4.13.0 in this image) — integer, bit-exact
//              here: green at a colour site from the pair across the SMALLER gradient (|l-r| > |d-u| strict -> vertical pair),
//              opposite colour from the four diagonals, the colours at a green site from the horizontal / vertical pair, all
//              with round-half-up shifts; the outermost ring repeats its inner neighbours.
// One kernel: clip -> flip -> white-balance gains (float64) -> clip -> 14-bit mosaic in shared memory -> demosaic -> CCM -> clip ->
// gamma -> BGR uint8.  4 B/px read, 3 B/px written; nothing intermediate touches HBM.
// Gamma without a float64 pow per sample: uint8(255 * x^(1/2.2)) is a monotone step function of the float64 x, so it is fully
// described by its 255 step positions T[k] = the smallest double with uint8(255 * pow(T, 1/2.2)) >= k.  The table is found once on
// the host by bisection over the double's bit pattern with libm's pow (the function NumPy calls), and the kernel only locates x
// among the steps: a float32 estimate of the level, corrected by exact float64 comparisons.  Same bytes as evaluating pow in
// float64 for every sample, at a fraction of the float64 work.
#include <math.h>
#include <string.h>

#include <mutex>

#include "common.cuh"

namespace {

constexpr int kTW = 128, kTH = 8;          // output pixels per block: 32 lanes x 4 pixels, 8 rows
constexpr int kSW = kTW + 2, kSH = kTH + 2;

__device__ double g_gamma_steps[256];  // [0] = 0; [k] = first double that reaches level k

struct RenderParams {
  double gain[4];   // per 2x2 site, row-major (R, G, G, B)
  double ccm[9];    // cam2rgb, row-major
  double inv_gamma;
  int flip_lr, flip_ud;
};

// 14-bit mosaic value of flipped-frame pixel (y, x): sidd_utils.py:158 (clip), :250-252 + :272 (gains, clip), :244 (x16383, clip,
// truncation to uint16)
__device__ __forceinline__ uint16_t quantise(const float* __restrict__ img, int H, int W, int y, int x, const RenderParams& p) {
  const int sy = p.flip_ud ? H - 1 - y : y, sx = p.flip_lr ? W - 1 - x : x;
  const float v = fminf(fmaxf(__ldg(img + (size_t)sy * W + sx), 0.f), 1.f);
  const double gain = (y & 1) ? ((x & 1) ? p.gain[3] : p.gain[2]) : ((x & 1) ? p.gain[1] : p.gain[0]);
  double g = __dmul_rn((double)v, gain);
  g = fmin(fmax(g, 0.0), 1.0);
  g = fmin(fmax(__dmul_rn(g, 16383.0), 0.0), 16383.0);
  return (uint16_t)(int)g;
}

// Edge-aware demosaic of the pixel whose (border-clamped) position in the tile is (ty, tx) and whose frame parity is (py, px).
__device__ __forceinline__ void demosaic_px(const uint16_t (*q)[kSW], int ty, int tx, int py, int px, int& r, int& g, int& b) {
  const int c = q[ty][tx], l = q[ty][tx - 1], rr = q[ty][tx + 1], u = q[ty - 1][tx], d = q[ty + 1][tx];
  const int hh = (l + rr + 1) >> 1, vv = (u + d + 1) >> 1;
  if (py != px) {  // green site: row 0 has R left/right and B above/below, row 1 the other way round
    g = c;
    r = py == 0 ? hh : vv;
    b = py == 0 ? vv : hh;
  } else {
    const int diag = (q[ty - 1][tx - 1] + q[ty - 1][tx + 1] + q[ty + 1][tx - 1] + q[ty + 1][tx + 1] + 2) >> 2;
    g = abs(l - rr) > abs(d - u) ? vv : hh;
    r = py == 0 ? c : diag;
    b = py == 0 ? diag : c;
  }
}

// kTable (render only): picture bz is the (H, W) mosaic of record pics[bz] with the camera cams[pics[bz].cam] (yond_render_pic,
// yond_render_cam), read once per CTA, instead of picture bz of one (B, H, W) tensor under the by-value `p` — every image of a SIDD
// evaluation with its own metadata, the clean mosaics and each round's output where their owners keep them.  A record without a
// source, or whose src_max holds no positive value (YOND_SIDD.py:644-647: such an output is neither rendered nor scored), returns
// before its first load.  p.inv_gamma still comes from the argument.  The arithmetic is the uniform form's.
template <bool kRender, bool kTable = false>
__global__ void __launch_bounds__(256) render_kernel(const float* __restrict__ img, const uint16_t* __restrict__ mosaic,
                                                     uint8_t* __restrict__ bgr, uint16_t* __restrict__ rgb16, int H, int W,
                                                     RenderParams p, const yond_render_pic* __restrict__ pics,
                                                     const yond_render_cam* __restrict__ cams) {
  __shared__ uint16_t q[kSH][kSW];
  __shared__ double steps[256];
  const yond_render_cam* cam = nullptr;
  if constexpr (kTable) {
    const yond_render_pic pic = pics[blockIdx.z];
    if (pic.src == nullptr || (pic.src_max != nullptr && !(*pic.src_max > 0.f))) return;
    cam = cams + pic.cam;
#pragma unroll
    for (int i = 0; i < 4; ++i) p.gain[i] = cam->gain[i];
    p.flip_lr = cam->flip_lr, p.flip_ud = cam->flip_ud;
    img = pic.src;
  }
  if (kRender) steps[threadIdx.x] = g_gamma_steps[threadIdx.x];
  const int x0 = blockIdx.x * kTW, y0 = blockIdx.y * kTH;
  const size_t plane = (size_t)H * W;
  const int bz = blockIdx.z;
  for (int i = threadIdx.x; i < kSH * kSW; i += blockDim.x) {
    const int ty = i / kSW, tx = i - ty * kSW;
    const int y = min(max(y0 + ty - 1, 0), H - 1), x = min(max(x0 + tx - 1, 0), W - 1);
    q[ty][tx] = kRender ? quantise(kTable ? img : img + bz * plane, H, W, y, x, p) : __ldg(mosaic + bz * plane + (size_t)y * W + x);
  }
  __syncthreads();
  if constexpr (kTable) {  // read after the tile is built, so that the gains and the matrix are not live at the same time
#pragma unroll
    for (int i = 0; i < 9; ++i) p.ccm[i] = cam->cam2rgb[i];
  }
  const int ly = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int y = y0 + ly;
  if (y >= H) return;
  const int cy = min(max(y, 1), H - 2);
  uint32_t packed[3] = {0u, 0u, 0u};
  uint8_t* orow = kRender ? bgr + (bz * plane + (size_t)y * W) * 3 : nullptr;
  const bool vec = kRender && (W % 4 == 0);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int x = x0 + lane * 4 + k;
    if (x >= W) break;
    const int cx = min(max(x, 1), W - 2);
    int r, g, b;
    demosaic_px(q, cy - y0 + 1, cx - x0 + 1, cy & 1, cx & 1, r, g, b);
    if (!kRender) {
      uint16_t* o = rgb16 + (bz * plane + (size_t)y * W + x) * 3;
      o[0] = (uint16_t)r, o[1] = (uint16_t)g, o[2] = (uint16_t)b;
      continue;
    }
    // :246 float32 / 16383, :260-263 float64 products summed in index order, :275 clip, :265-266 gamma, :176-177 x255 -> uint8
    const double d0 = (double)__fdiv_rn((float)r, 16383.f), d1 = (double)__fdiv_rn((float)g, 16383.f),
                 d2 = (double)__fdiv_rn((float)b, 16383.f);
    uint32_t out3[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double v = __dadd_rn(__dadd_rn(__dmul_rn(d0, p.ccm[i * 3]), __dmul_rn(d1, p.ccm[i * 3 + 1])), __dmul_rn(d2, p.ccm[i * 3 + 2]));
      v = fmax(fmin(fmax(v, 0.0), 1.0), 1e-8);
      int level = min(max((int)(255.f * __powf((float)v, (float)p.inv_gamma)), 0), 255);
      while (level < 255 && v >= steps[level + 1]) ++level;
      while (level > 0 && v < steps[level]) --level;
      out3[2 - i] = (uint32_t)level;  // swap_channels: RGB -> BGR
    }
    if (vec) {
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const int byte = k * 3 + i;
        packed[byte >> 2] |= out3[i] << ((byte & 3) * 8);
      }
    } else {
      orow[(size_t)x * 3] = (uint8_t)out3[0], orow[(size_t)x * 3 + 1] = (uint8_t)out3[1], orow[(size_t)x * 3 + 2] = (uint8_t)out3[2];
    }
  }
  if (vec && x0 + lane * 4 < W) {
    uint32_t* o = reinterpret_cast<uint32_t*>(orow + (size_t)(x0 + lane * 4) * 3);
    o[0] = packed[0], o[1] = packed[1], o[2] = packed[2];
  }
}

// uint8(255 * max(x, 1e-8)^(1/2.2)) as the reference evaluates it (sidd_utils.py:265-266, :176-177)
int gamma_level(double x, double inv_gamma) { return (int)(pow(x, inv_gamma) * 255.0); }

int upload_gamma_steps(double inv_gamma) {
  static std::mutex mu;
  static bool done[64] = {};
  int dev = 0;
  YOND_CUDA_CHECK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  if (dev >= 0 && dev < 64 && done[dev]) return YOND_OK;
  double steps[256];
  steps[0] = 0.0;
  for (int k = 1; k < 256; ++k) {
    uint64_t lo, hi;  // positive doubles order like their bit patterns; level(lo) < k <= level(hi) throughout
    const double a = 1e-8, b = 1.0;
    memcpy(&lo, &a, 8);
    memcpy(&hi, &b, 8);
    while (hi - lo > 1) {
      const uint64_t mid = lo + (hi - lo) / 2;
      double x;
      memcpy(&x, &mid, 8);
      if (gamma_level(x, inv_gamma) >= k) hi = mid; else lo = mid;
    }
    memcpy(&steps[k], &hi, 8);
  }
  YOND_CUDA_CHECK(cudaMemcpyToSymbol(g_gamma_steps, steps, sizeof(steps)));
  if (dev >= 0 && dev < 64) done[dev] = true;
  return YOND_OK;
}

int check_shape(const char* who, int B, int H, int W) {
  YOND_REQUIRE(B > 0 && H >= 4 && W >= 4 && H % 2 == 0 && W % 2 == 0, "%s: need B > 0 and even H, W >= 4 (got %d x %d x %d)", who, B, H, W);
  YOND_REQUIRE(B <= 65535, "%s: at most 65535 images per call", who);
  return YOND_OK;
}

}  // namespace

extern "C" int yond_render_srgb(const float* bayer, uint8_t* bgr, int B, int H, int W, int flip_lr, int flip_ud, const double* gains3,
                                const double* cam2rgb9, void* stream) {
  YOND_REQUIRE(bayer && bgr && gains3 && cam2rgb9, "yond_render_srgb: null pointer");
  if (int e = check_shape("yond_render_srgb", B, H, W)) return e;
  RenderParams p;
  p.gain[0] = gains3[0], p.gain[1] = gains3[1], p.gain[2] = gains3[1], p.gain[3] = gains3[2];
  for (int i = 0; i < 9; ++i) p.ccm[i] = cam2rgb9[i];
  p.inv_gamma = 1.0 / 2.2;
  p.flip_lr = flip_lr != 0, p.flip_ud = flip_ud != 0;
  if (int e = upload_gamma_steps(p.inv_gamma)) return e;
  cudaStream_t s = (cudaStream_t)stream;
  YondProfScope prof("render_srgb", s, 7.0 * (double)B * H * W);
  dim3 grid(ceil_div(W, kTW), ceil_div(H, kTH), B);
  render_kernel<true><<<grid, 256, 0, s>>>(bayer, nullptr, bgr, nullptr, H, W, p, nullptr, nullptr);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

extern "C" int yond_render_srgb_cams(const yond_render_pic* pics_dev, const yond_render_cam* cams_dev, uint8_t* bgr, int B, int H,
                                     int W, void* stream) {
  YOND_REQUIRE(pics_dev && cams_dev && bgr, "yond_render_srgb_cams: null pointer");
  if (int e = check_shape("yond_render_srgb_cams", B, H, W)) return e;
  RenderParams p = {};
  p.inv_gamma = 1.0 / 2.2;
  if (int e = upload_gamma_steps(p.inv_gamma)) return e;
  cudaStream_t s = (cudaStream_t)stream;
  YondProfScope prof("render_srgb", s, 7.0 * (double)B * H * W);
  dim3 grid(ceil_div(W, kTW), ceil_div(H, kTH), B);
  render_kernel<true, true><<<grid, 256, 0, s>>>(nullptr, nullptr, bgr, nullptr, H, W, p, pics_dev, cams_dev);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

extern "C" int yond_demosaic_ea(const uint16_t* bayer, uint16_t* rgb, int B, int H, int W, void* stream) {
  YOND_REQUIRE(bayer && rgb, "yond_demosaic_ea: null pointer");
  if (int e = check_shape("yond_demosaic_ea", B, H, W)) return e;
  RenderParams p = {};
  cudaStream_t s = (cudaStream_t)stream;
  YondProfScope prof("demosaic_ea", s, 8.0 * (double)B * H * W);
  dim3 grid(ceil_div(W, kTW), ceil_div(H, kTH), B);
  render_kernel<false><<<grid, 256, 0, s>>>(nullptr, bayer, nullptr, rgb, H, W, p, nullptr, nullptr);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}
