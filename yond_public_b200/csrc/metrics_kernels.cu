// Image-quality metrics of the SIDD driver on the device (SURVEY 8(f)-3): raw PSNR and the MATLAB-style SSIM that
// YOND_SIDD.py:652-653 evaluates per 256x256 block of the mosaic in a CPU worker thread.
//   reference: YOND_SIDD.py:679-697 (ssim: 11x11 Gaussian window sigma 1.5 from cv2.getGaussianKernel, float64
//              cv2.filter2D, valid region, C1 = (0.01*255)^2, C2 = (0.03*255)^2), :700-721 (calculate_ssim),
//              :651-652 (32 blocks split along W, data_range 1 / images scaled by 255);
//              skimage.metrics.peak_signal_noise_ratio (third-party, not vendored): float32 difference and square for
//              float32 inputs, float64 mean, 10 log10(range^2 / mse).
// A mosaic (H, nblk*Wb) holds nblk blocks side by side; every block is measured on its own.
#include "common.cuh"

namespace {

constexpr int kWin = 11, kR = 5;
constexpr int kTile = 16;               // output pixels per block edge
constexpr int kIn = kTile + 2 * kR;     // 26 x 26 input tile

struct SsimWin {
  double w[kWin];
};

// One thread per valid output pixel; the 26x26 input tiles of both images sit in shared memory as float64
// (= double(fl32(x * 255)) like `dn*255` -> np.float64).  The window is outer(kernel, kernel) (YOND_SIDD.py:684-685), so the five
// filtered quantities (x1, x2, x1^2, x2^2, x1 x2) are formed in two passes — 11 taps along the rows into shared memory, 11 taps down
// the columns — 144 float64 FMAs per pixel instead of 605.  (cv2.filter2D itself evaluates an 11x11 float64 window through a DFT;
// all three orders of summation agree to ~1e-9 in the SSIM value.)
__device__ __forceinline__ double metric_value(float v, float scale) { return (double)__fmul_rn(v, scale); }
__device__ __forceinline__ double metric_value(uint8_t v, float) { return (double)v; }  // 8-bit sRGB pictures are already in [0, 255]

// T = float: mosaics (nch = 1).  T = uint8_t: interleaved pictures (H, Wm, nch); every channel is filtered on its own and the
// block's sum runs over all of them (calculate_ssim's mean over the three channel means, YOND_SIDD.py:711-716).
template <typename T>
__global__ void __launch_bounds__(kTile * kTile) ssim_kernel(const T* __restrict__ a, const T* __restrict__ b, int H, int Wb, int nblk,
                                                             int nch, float scale, SsimWin win, double* __restrict__ sums) {
  __shared__ double ta[kIn][kIn + 1], tb[kIn][kIn + 1];
  __shared__ double rows[5][kIn][kTile + 1];  // row-filtered x1, x2, x1^2, x2^2, x1 x2
  __shared__ double red[kTile * kTile / 32];
  const int ch = blockIdx.z % nch, unit = blockIdx.z / nch;
  const int blk = unit % nblk, img = unit / nblk;
  const size_t Wm = (size_t)nblk * Wb;
  const T* pa = a + ((size_t)img * H * Wm + (size_t)blk * Wb) * nch + ch;
  const T* pb = b + ((size_t)img * H * Wm + (size_t)blk * Wb) * nch + ch;
  const int oy0 = blockIdx.y * kTile, ox0 = blockIdx.x * kTile;  // valid-region coordinates
  const int vh = H - 2 * kR, vw = Wb - 2 * kR;
  for (int i = threadIdx.x; i < kIn * kIn; i += blockDim.x) {
    const int ty = i / kIn, tx = i - ty * kIn;
    const int y = oy0 + ty, x = ox0 + tx;  // input coordinates = valid coordinates + window offset (0..10)
    double va = 0.0, vb = 0.0;
    if (y < H && x < Wb) {
      va = metric_value(pa[((size_t)y * Wm + x) * nch], scale);
      vb = metric_value(pb[((size_t)y * Wm + x) * nch], scale);
    }
    ta[ty][tx] = va;
    tb[ty][tx] = vb;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kIn * kTile; i += blockDim.x) {
    const int ty = i / kTile, lx = i - ty * kTile;
    double m1 = 0, m2 = 0, s11 = 0, s22 = 0, s12 = 0;
#pragma unroll
    for (int j = 0; j < kWin; ++j) {
      const double w = win.w[j], x1 = ta[ty][lx + j], x2 = tb[ty][lx + j];
      m1 += w * x1;
      m2 += w * x2;
      s11 += w * (x1 * x1);
      s22 += w * (x2 * x2);
      s12 += w * (x1 * x2);
    }
    rows[0][ty][lx] = m1, rows[1][ty][lx] = m2, rows[2][ty][lx] = s11, rows[3][ty][lx] = s22, rows[4][ty][lx] = s12;
  }
  __syncthreads();
  const int ly = threadIdx.x / kTile, lx = threadIdx.x % kTile;
  double v = 0.0;
  if (oy0 + ly < vh && ox0 + lx < vw) {
    double m1 = 0, m2 = 0, s11 = 0, s22 = 0, s12 = 0;
#pragma unroll
    for (int i = 0; i < kWin; ++i) {
      const double w = win.w[i];
      m1 += w * rows[0][ly + i][lx];
      m2 += w * rows[1][ly + i][lx];
      s11 += w * rows[2][ly + i][lx];
      s22 += w * rows[3][ly + i][lx];
      s12 += w * rows[4][ly + i][lx];
    }
    const double C1 = (0.01 * 255) * (0.01 * 255), C2 = (0.03 * 255) * (0.03 * 255);
    const double m11 = m1 * m1, m22 = m2 * m2, m12 = m1 * m2;
    v = ((2 * m12 + C1) * (2 * (s12 - m12) + C2)) / ((m11 + m22 + C1) * ((s11 - m11) + (s22 - m22) + C2));
  }
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < kTile * kTile / 32; ++i) s += red[i];
    atomicAdd(&sums[unit], s);
  }
}

__device__ __forceinline__ double sq_diff(float a, float b) {  // float32 inputs stay float32 in skimage (`_as_floats`)
  const float d = __fsub_rn(a, b);
  return (double)__fmul_rn(d, d);
}
__device__ __forceinline__ double sq_diff(uint8_t a, uint8_t b) {  // integer inputs are promoted to float64: exact
  const double d = (double)((int)a - (int)b);
  return d * d;
}

// Sum of squared differences per block (all nch interleaved channels together), accumulated in float64.
template <typename T>
__global__ void __launch_bounds__(256) sqdiff_kernel(const T* __restrict__ a, const T* __restrict__ b, int H, int Wb, int nblk, int nch,
                                                     double* __restrict__ sums) {
  const int blk = blockIdx.z % nblk, img = blockIdx.z / nblk;
  const size_t Wm = (size_t)nblk * Wb;
  const T* pa = a + ((size_t)img * H * Wm + (size_t)blk * Wb) * nch;
  const T* pb = b + ((size_t)img * H * Wm + (size_t)blk * Wb) * nch;
  double acc = 0.0;
  for (int y = blockIdx.y; y < H; y += gridDim.y)
    for (int x = threadIdx.x; x < Wb * nch; x += blockDim.x) acc += sq_diff(pa[(size_t)y * Wm * nch + x], pb[(size_t)y * Wm * nch + x]);
  __shared__ double red[8];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < 8; ++i) s += red[i];
    atomicAdd(&sums[blockIdx.z], s);
  }
}

__global__ void metrics_finish_kernel(double* psnr, double* ssim, int n, double npix, double nvalid, double range2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (psnr) psnr[i] = 10.0 * log10(range2 / (psnr[i] / npix));
  if (ssim) ssim[i] = ssim[i] / nvalid;
}

// One thread per (round, image) of a SIDD evaluation: the per-image numbers of multiprocess_plot (YOND_SIDD.py:643-665) from the
// per-block ones — the sum over the blocks in block order / nblk; (-1, -1) and no sRGB numbers where the output has no positive value
// (:644-647); nothing for rounds the image did not complete.
__global__ void sidd_scores_kernel(const double* __restrict__ psnr, const double* __restrict__ ssim, const double* __restrict__ psnr_rgb,
                                   const double* __restrict__ ssim_rgb, const float* __restrict__ out_max,
                                   const int32_t* __restrict__ rounds, int nround, int nimg, int nblk, double* __restrict__ table) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // round * nimg + image
  if (i >= nround * nimg) return;
  const int r = i / nimg, img = i - r * nimg;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  double* o = table + (size_t)i * 4;
  if (r >= rounds[img]) {
    o[0] = o[1] = o[2] = o[3] = nan;
    return;
  }
  if (!(out_max[i] > 0.f)) {
    o[0] = o[1] = -1.0;
    o[2] = o[3] = nan;
    return;
  }
  const double* src[4] = {psnr, ssim, psnr_rgb, ssim_rgb};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (!src[k]) {
      o[k] = nan;
      continue;
    }
    const double* v = src[k] + (size_t)i * nblk;
    double sum = 0.0;
    for (int b = 0; b < nblk; ++b) sum += v[b];
    o[k] = sum / nblk;
  }
}

template <typename T>
int block_metrics_impl(const char* who, const T* a, const T* b, int nimg, int H, int Wm, int nblk, int nch, double data_range,
                       float ssim_scale, const double* window11, double* psnr, double* ssim, void* stream) {
  YOND_REQUIRE(a && b && nimg > 0 && H > 0 && Wm > 0 && nblk > 0 && Wm % nblk == 0, "%s: bad shape", who);
  YOND_REQUIRE(psnr || ssim, "%s: no output requested", who);
  YOND_REQUIRE((size_t)nimg * nblk * nch <= 65535, "%s: at most 65535 block-channels per call", who);
  cudaStream_t s = (cudaStream_t)stream;
  const int Wb = Wm / nblk, n = nimg * nblk;
  if (psnr) {
    YOND_CUDA_CHECK(cudaMemsetAsync(psnr, 0, sizeof(double) * n, s));
    const int rows_wanted = n >= 1184 ? 1 : 1184 / n;  // ~8 blocks per SM in flight also when one large image is measured
    dim3 g(1, H < rows_wanted ? H : rows_wanted, n);
    sqdiff_kernel<T><<<g, 256, 0, s>>>(a, b, H, Wb, nblk, nch, psnr);
    YOND_LAUNCH_CHECK();
  }
  if (ssim) {
    YOND_REQUIRE(window11 != nullptr, "%s: SSIM needs the 11-tap window (host array)", who);
    YOND_REQUIRE(H > 2 * kR && Wb > 2 * kR, "%s: blocks smaller than the SSIM window", who);
    SsimWin win;
    for (int i = 0; i < kWin; ++i) win.w[i] = window11[i];
    YOND_CUDA_CHECK(cudaMemsetAsync(ssim, 0, sizeof(double) * n, s));
    dim3 g(ceil_div(Wb - 2 * kR, kTile), ceil_div(H - 2 * kR, kTile), n * nch);
    ssim_kernel<T><<<g, kTile * kTile, 0, s>>>(a, b, H, Wb, nblk, nch, ssim_scale, win, ssim);
    YOND_LAUNCH_CHECK();
  }
  metrics_finish_kernel<<<ceil_div(n, 128), 128, 0, s>>>(psnr, ssim, n, (double)H * Wb * nch,
                                                        (double)(H - 2 * kR) * (Wb - 2 * kR) * nch, data_range * data_range);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

}  // namespace

extern "C" int yond_block_metrics(const float* a, const float* b, int nimg, int H, int Wm, int nblk, double data_range, float ssim_scale,
                                  const double* window11, double* psnr, double* ssim, void* stream) {
  return block_metrics_impl<float>("yond_block_metrics", a, b, nimg, H, Wm, nblk, 1, data_range, ssim_scale, window11, psnr, ssim,
                                   stream);
}

extern "C" int yond_block_metrics_rgb8(const uint8_t* a, const uint8_t* b, int nimg, int H, int Wm, int nblk, const double* window11,
                                       double* psnr, double* ssim, void* stream) {
  return block_metrics_impl<uint8_t>("yond_block_metrics_rgb8", a, b, nimg, H, Wm, nblk, 3, 255.0, 1.0f, window11, psnr, ssim, stream);
}

extern "C" int yond_sidd_scores(const double* psnr, const double* ssim, const double* psnr_rgb, const double* ssim_rgb, const float* out_max,
                                const int32_t* rounds_dev, int nround, int nimg, int nblk, double* table, void* stream) {
  YOND_REQUIRE(psnr && ssim && out_max && rounds_dev && table, "yond_sidd_scores: null pointer");
  YOND_REQUIRE(!psnr_rgb == !ssim_rgb, "yond_sidd_scores: give both sRGB inputs or neither");
  YOND_REQUIRE(nround > 0 && nimg > 0 && nblk > 0 && (long long)nround * nimg <= (1ll << 30), "yond_sidd_scores: bad shape");
  const int n = nround * nimg;
  sidd_scores_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(psnr, ssim, psnr_rgb, ssim_rgb, out_max, rounds_dev, nround, nimg,
                                                                         nblk, table);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}
