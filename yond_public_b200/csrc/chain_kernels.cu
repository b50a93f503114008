// Device-resident VST parameter chain: from the estimator's (beta1, beta2) to everything the fused VST kernels need,
// without a host read-back.
//   reference: YOND_SIDD.py:356 / :419-472 (gain, sigma and the guards of the collab rounds), :252-269,284-285 (bias source, VST(0),
//              VST(scale), nsr, t), utils/isp_algos.py:179-231 (BiasLUT.pos_interp / data_merge over sigma),
//              :49-82,84-96,98-140 (getGsP / close_form_bias / get_bias: the fallback bias table).
// All scalar arithmetic is float64 with explicit round-to-nearest operations in NumPy's evaluation order.
#include <cmath>
#include <mutex>

#include "common.cuh"

namespace {

struct SegChain {     // per image; written by params_fill_kernel, consumed by the table generator and the LUT-row kernel
  double gain, sigma; // DN
  double sg_pos;      // fractional sigma index into the BiasLUT (valid when use_lut)
  float bound;        // upper bound of the fallback table in DN (float32 product, like lr_raw.max()*(wp-bl))
  int use_lut;        // 1: sigma-interpolated BiasLUT row
  int need_table;     // 1: numeric get_bias table
  int n_nodes;        // nodes of that table
  int ok;             // rounds >= 2: still live (beta1 >= 0 in this round and every earlier one)
};

__device__ __forceinline__ double vst_d(double v, double K, double sig) {
  // utils/isp_algos.py:5-14 with mu = 0
  const double fz = __dadd_rn(__dadd_rn(__dmul_rn(K, v), __dmul_rn(0.375, __dmul_rn(K, K))), __dmul_rn(sig, sig));
  return __dmul_rn(__ddiv_rn(2.0, K), sqrt(fz > 0.0 ? fz : 0.0));
}

// ---- node positions of get_bias (isp_algos.py:101-108).  `ub` = ceil(img.max()) + 1 is a float32 scalar in the reference
// (NumPy keeps float32 for float32-scalar <op> Python-scalar), so the pieces that end in `ub` are float32 linspaces and the
// fixed pieces float64 ones; the concatenation upcasts exactly.
__device__ __forceinline__ double linspace64(double a, double b, int n, int j) {
  if (j == n - 1 && n > 1) return b;
  const double step = __ddiv_rn(__dsub_rn(b, a), (double)(n - 1));
  return __dadd_rn(__dmul_rn((double)j, step), a);
}
__device__ __forceinline__ double linspace32(float a, float b, int n, int j) {
  if (j == n - 1 && n > 1) return (double)b;
  const float step = __fdiv_rn(__fsub_rn(b, a), (float)(n - 1));
  return (double)__fadd_rn(__fmul_rn((float)j, step), a);
}
__host__ __device__ inline int table_nodes(float bound) {
  const float ub = ceilf(bound) + 1.f;
  if (ub < 50.f) return (int)(ub / 0.1f) + 2;
  if (ub < 500.f) return 501 + (int)(ub - 50.f) + 2;
  return 501 + 451 + (int)(ub - 500.f) / 10 + 2;
}
__device__ __forceinline__ double table_node(float bound, int j) {
  const float ub = ceilf(bound) + 1.f;
  if (ub < 50.f) return linspace32(0.f, ub, (int)__fdiv_rn(ub, 0.1f) + 2, j);
  if (j < 501) return linspace64(0.0, 50.0, 501, j);
  if (ub < 500.f) return linspace32(50.f, ub, (int)(ub - 50.f) + 2, j - 501);
  if (j < 952) return linspace64(50.0, 500.0, 451, j - 501);
  return linspace32(500.f, ub, (int)(ub - 500.f) / 10 + 2, j - 952);
}

// Foi's closed form (isp_algos.py:84-96), float64
__device__ __forceinline__ double close_form_bias_d(double x, double sig, double K) {
  const double y = x / K, s = sig / K;
  const double yh = y + 0.375 + s * s;
  const double m1 = (y + s * s) / (yh * yh);
  const double m2 = y / (yh * yh * yh);
  const double m3 = (y + 3.0 * (y + s * s) * (y + s * s)) / (yh * yh * yh * yh);
  return 2.0 * sqrt(yh) * (-0.125 * m1 + 0.0625 * m2 - 0.0390625 * m3);
}

// ---- the fallback table on the device (SURVEY 8(f)-2).  One block = kNodesPerBlock consecutive nodes of one image.
// Per node (getGsP, isp_algos.py:49-82): the grid x = linspace(-r, r, 2*pho*r+1) has step 1/pho; poisson.pmf is non-zero
// only on its integer points, so convolve(pmf, norm.pdf, 'same')[j] = sum_k P(k; lam/K) * phi((j - c)/pho - k) over the
// integers k whose distance to x_j is inside the 'same' window (|j - i_k| <= c = pho*r).  The Poisson weights of a node and
// the Gaussian samples of an image are tabulated once in shared memory; the double sum is plain FMAs.
// bias = sum(pdf * VST(K x)) / sum(pdf) - VST(lam)  (the reference's two /pho normalisations cancel).
constexpr int kNodesPerBlock = 8;
constexpr int kTableThreads = 256;
constexpr int kGaussTab = 4096;   // tabulated Gaussian samples in the pipeline (32 KB); farther ones are evaluated directly
constexpr int kGaussTabMax = 24576;  // get_bias_points with pho_min = 100 (the offline LUT builder): 192 KB
constexpr int kPoisTab = 1024;
// `lam_list` (optional): explicit float64 evaluation points instead of get_bias's node layout (get_bias_points,
// isp_algos.py:142-160); the values then go to `vals64` in float64.
__global__ void __launch_bounds__(kTableThreads) bias_table_kernel(const SegChain* __restrict__ chain, float* __restrict__ rows,
                                                                   float* __restrict__ xnodes, int row_stride, int gauss_tab,
                                                                   int pho_min, const double* __restrict__ lam_list,
                                                                   double* __restrict__ vals64) {
  const int s = blockIdx.y;
  const SegChain ch = chain[s];
  if (!ch.need_table) return;
  const int j0 = blockIdx.x * kNodesPerBlock;
  if (j0 >= ch.n_nodes) return;
  extern __shared__ double G[];  // gauss_tab entries
  __shared__ double P[kPoisTab];
  __shared__ double red[2][kTableThreads / 32];
  const double K = ch.gain, sig = ch.sigma;
  const double sg = sig / K;
  const double rootK = sqrt(K);  // K**0.5
  int pho = (int)rootK;
  if (pho < pho_min) pho = pho_min;
  const double th = K < 1.0 ? 50.0 * K : 50.0 * rootK;
  const bool gauss = sig > 0.0;
  // Gaussian samples phi(d / pho): exactly zero (float64 underflow) beyond ~38.6 sigma
  const double inv_sg = gauss ? 1.0 / sg : 0.0;
  const double gnorm = gauss ? 1.0 / (sg * 2.5066282746310002) : 1.0;  // sqrt(2 pi)
  long long dcut = gauss ? (long long)(39.0 * sg * pho) + 1 : 0;
  auto gval = [&](long long d) -> double {
    if (!gauss) return d == 0 ? 1.0 : 0.0;
    const double t = ((double)d / (double)pho) * inv_sg;
    return exp(-0.5 * t * t) * gnorm;
  };
  const int gtab = (int)(dcut < (long long)gauss_tab - 1 ? dcut + 1 : gauss_tab);
  for (int d = threadIdx.x; d < gtab; d += kTableThreads) G[d] = gval(d);
  __syncthreads();
  for (int jn = j0; jn < j0 + kNodesPerBlock && jn < ch.n_nodes; ++jn) {
    const double lam = lam_list ? lam_list[jn] : table_node(ch.bound, jn);
    double bias;
    if (lam > th) {
      bias = close_form_bias_d(lam, sig, K);
    } else {
      const double mu = lam / K;
      const long long r = (long long)(lam * (1.0 / K) * 2.0 + sig * 2.0 + lam + 10.0);
      const long long c = (long long)pho * r;
      // Poisson weights worth keeping: |k - mu| <= 14 sqrt(mu) + 40 (tail < 1e-30), inside [0, r]
      const double spread = 14.0 * sqrt(mu) + 40.0;
      long long kmin = (long long)floor(mu - spread), kmax = (long long)ceil(mu + spread);
      if (kmin < 0) kmin = 0;
      if (kmax > r) kmax = r;
      if (kmax - kmin + 1 > kPoisTab) kmax = kmin + kPoisTab - 1;
      const int nk = (int)(kmax - kmin + 1);
      const double logmu = mu > 0.0 ? log(mu) : 0.0;
      __syncthreads();  // P is reused across the nodes of this block
      for (int i = threadIdx.x; i < nk; i += kTableThreads) {
        const double k = (double)(kmin + i);
        // scipy: exp(xlogy(k, mu) - gammaln(k + 1) - mu)
        P[i] = mu > 0.0 ? exp(k * logmu - lgamma(k + 1.0) - mu) : (k == 0.0 ? 1.0 : 0.0);
      }
      __syncthreads();
      const long long dwin = dcut < c ? dcut : c;  // Gaussian support, cut by the 'same' window
      long long jlo = c + kmin * pho - dwin, jhi = c + kmax * pho + dwin;
      if (jlo < 0) jlo = 0;
      if (jhi > 2 * c) jhi = 2 * c;
      double s0 = 0.0, s1 = 0.0;
      for (long long j = jlo + threadIdx.x; j <= jhi; j += kTableThreads) {
        // integers k with |j - c - k*pho| <= dwin
        const long long rel = j - c;
        long long ka = (rel - dwin + pho - 1 >= 0) ? (rel - dwin + pho - 1) / pho : -((dwin - rel) / pho);
        long long kb = (rel + dwin >= 0) ? (rel + dwin) / pho : -1;
        if (ka < kmin) ka = kmin;
        if (kb > kmax) kb = kmax;
        double acc = 0.0;
        for (long long k = ka; k <= kb; ++k) {
          long long d = rel - k * pho;
          if (d < 0) d = -d;
          const double g = d < gtab ? G[d] : gval(d);
          acc = fma(P[k - kmin], g, acc);
        }
        if (acc > 0.0) {
          s0 += acc;
          s1 = fma(acc, vst_d(K * ((double)rel / (double)pho), K, sig), s1);
        }
      }
      for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      }
      if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = s0;
        red[1][threadIdx.x >> 5] = s1;
      }
      __syncthreads();
      s0 = s1 = 0.0;
      for (int w = 0; w < kTableThreads / 32; ++w) {
        s0 += red[0][w];
        s1 += red[1][w];
      }
      bias = s1 / s0 - vst_d(lam, K, sig);
    }
    if (threadIdx.x == 0) {
      if (vals64) {
        vals64[jn] = bias;
      } else {
        rows[(size_t)s * row_stride + jn] = (float)bias;
        xnodes[(size_t)s * row_stride + jn] = (float)lam;
      }
    }
  }
}

// ---- BiasLUT.pos_interp over sigma (isp_algos.py:179-186): data = [-inf, sg_lut...], idx = searchsorted (left), clipped
__device__ __forceinline__ double sigma_pos_d(const double* __restrict__ sg_lut, int nsg, double sg) {
  // first index i in [0, nsg] of the extended array with data[i] >= sg; data[0] = -inf
  int lo = 0, hi = nsg + 1;  // searchsorted over nsg + 1 entries
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const double v = mid == 0 ? -__longlong_as_double(0x7ff0000000000000LL) : sg_lut[mid - 1];
    if (v < sg) lo = mid + 1; else hi = mid;
  }
  int idx = lo;
  if (idx > nsg) idx = nsg;
  const double hi_v = idx == 0 ? -__longlong_as_double(0x7ff0000000000000LL) : sg_lut[idx - 1];
  const double lo_v = idx <= 1 ? -__longlong_as_double(0x7ff0000000000000LL) : sg_lut[idx - 2];
  const double w = __dsub_rn(hi_v, sg), diff = __dsub_rn(hi_v, lo_v);
  return __dsub_rn(__dsub_rn((double)idx, __ddiv_rn(w, diff)), 1.0);
}

struct FillArgs {
  double scale_est, scale, bound_scale;
  int round, bias_mode, exact_inverse, frames_per_seg, nseg, nsg, has_lut, max_nodes;
};
// One thread per image.
__global__ void params_fill_kernel(FillArgs a, const double* __restrict__ regs, const float* __restrict__ seg_max,
                                   const double* __restrict__ sg_lut, const yond_vst_params* __restrict__ prev,
                                   const int32_t* __restrict__ prev_ok, yond_vst_params* __restrict__ params, float* __restrict__ t_out,
                                   SegChain* __restrict__ chain, double* __restrict__ regs_out, int32_t* __restrict__ ok_out,
                                   const double* __restrict__ seg_scales) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= a.nseg) return;
  double scale_est = a.scale_est, scale = a.scale, bound_scale = a.bound_scale;
  if (seg_scales) {  // this image's (scale_est, scale, bound_scale)
    scale_est = seg_scales[3 * s];
    scale = seg_scales[3 * s + 1];
    bound_scale = seg_scales[3 * s + 2];
  }
  double b1 = regs[2 * s], b2 = regs[2 * s + 1];
  int ok = 1;
  double sig;
  if (a.round >= 2) {  // YOND_SIDD.py:438-447
    if (b2 < 0.0) b2 = __dmul_rn(b1, b1);
    sig = __dmul_rn(sqrt(b2), scale_est);
    // the reference leaves its loop at the first beta1 < 0: an image that stopped in an earlier round stays stopped
    ok = !(b1 < 0.0) && (!prev_ok || prev_ok[s]);
  } else {             // :356  sqrt(max(beta2, 0))
    sig = __dmul_rn(sqrt(0.0 > b2 ? 0.0 : b2), scale_est);
  }
  const double gain = __dmul_rn(b1, scale_est);
  if (regs_out) {
    regs_out[4 * s] = b1;
    regs_out[4 * s + 1] = b2;
    regs_out[4 * s + 2] = gain;
    regs_out[4 * s + 3] = sig;
  }
  if (ok_out) ok_out[s] = ok;
  SegChain ch{};
  ch.ok = ok;
  ch.gain = gain;
  ch.sigma = sig;
  yond_vst_params q{};
  float t = 0.f;
  if (!ok && prev) {
    // stopped: the reference keeps the previous round's result; this image's output of this round is discarded by the back half,
    // the parameters of its last live round (carried from round to round in `prev`) keep the wasted pass well-defined
    q = prev[(size_t)s * a.frames_per_seg];
    q.lut_row = -1;
    q.table_n = 0;
  } else {
    const double c0 = __dadd_rn(__dmul_rn(0.375, __dmul_rn(gain, gain)), __dmul_rn(sig, sig));
    const double two_g = __ddiv_rn(2.0, gain);
    const double lower = __dmul_rn(two_g, sqrt(c0 > 0.0 ? c0 : 0.0));
    const double up_arg = __dadd_rn(__dmul_rn(gain, scale), c0);
    const double upper = __dmul_rn(two_g, sqrt(up_arg > 0.0 ? up_arg : 0.0));
    q.gain = (float)gain;
    q.sigma = (float)sig;
    q.scale = (float)scale;
    q.lower = (float)lower;
    q.upper = (float)upper;
    q.exact_inverse = a.exact_inverse;
    q.lut_row = -1;
    q.table_n = 0;
    t = (float)__dmul_rn(__ddiv_rn(1.0, __dsub_rn(upper, lower)), a.bias_mode == 1 ? 1.03 : 1.0);  // :268, :284-285
    if (a.bias_mode == 1) {  // only 'pre' applies a bias (:261-262)
      q.lut_row = s;
      bool in_range = false;
      if (a.has_lut) {
        const double pos = sigma_pos_d(sg_lut, a.nsg, __ddiv_rn(sig, gain));
        in_range = pos <= (double)(a.nsg - 1);
        ch.sg_pos = pos;
      }
      if (in_range) {
        ch.use_lut = 1;
      } else {  // no LUT, or sigma/K beyond it: the numeric table up to this image's maximum (:254-257, isp_algos.py:204-212)
        const float mx = seg_max ? seg_max[s] : 1.0f;
        ch.bound = __fmul_rn(mx > 0.f ? mx : 0.f, (float)bound_scale);
        int n = table_nodes(ch.bound);
        if (n > a.max_nodes) n = a.max_nodes;  // the caller sized the rows for its data range
        ch.n_nodes = n;
        ch.need_table = 1;
        q.table_n = n;
      }
    }
  }
  chain[s] = ch;
  for (int f = 0; f < a.frames_per_seg; ++f) {
    params[(size_t)s * a.frames_per_seg + f] = q;
    t_out[(size_t)s * a.frames_per_seg + f] = t;
  }
}

// sigma-lerp of the 2-D table into one row per image (data_merge over sigma, isp_algos.py:225) + the row's node positions
__global__ void lut_rows_kernel(const float* __restrict__ lut, const float* __restrict__ xlut, int nx, int nsg,
                                const SegChain* __restrict__ chain, float* __restrict__ rows, float* __restrict__ xnodes,
                                int row_stride) {
  const int s = blockIdx.y;
  if (!chain[s].use_lut) return;
  double pos = chain[s].sg_pos;
  if (pos < 0) pos = 0;
  if (pos > nsg - 1) pos = nsg - 1;
  const int l = (int)floor(pos), r = (int)ceil(pos);
  const float wr = (float)(pos - l);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nx) {
    rows[(size_t)s * row_stride + i] = lut[(size_t)i * nsg + l] * (1.f - wr) + lut[(size_t)i * nsg + r] * wr;
    xnodes[(size_t)s * row_stride + i] = xlut[i];
  }
}

__global__ void single_chain_kernel(SegChain* chain, double gain, double sigma, float bound, int max_nodes, int* n_out, int n_list) {
  SegChain ch{};
  ch.gain = gain;
  ch.sigma = sigma;
  ch.bound = bound;
  ch.need_table = 1;
  int n = n_list > 0 ? n_list : table_nodes(bound);
  if (n > max_nodes) n = max_nodes;
  ch.n_nodes = n;
  chain[0] = ch;
  if (n_out) *n_out = n;
}

}  // namespace

extern "C" {

size_t yond_chain_work_bytes(int nseg) { return (size_t)(nseg < 1 ? 1 : nseg) * sizeof(SegChain) + 256; }

int yond_bias_table_nodes(float bound) { return table_nodes(bound); }

int yond_vst_params_fill(const double* regs_dev, const float* seg_max_dev, int nseg, int frames_per_seg, double scale_est,
                         double scale, double bound_scale, int round, int bias_mode, int exact_inverse, const float* lut2d,
                         const double* sg_lut_dev, const float* x_lut_dev, int nx, int nsg, const yond_vst_params* prev_params,
                         yond_vst_params* params_dev, float* t_dev, float* rows, float* xnodes, int row_stride, double* regs_out,
                         int32_t* ok_dev, void* work, void* stream, const int32_t* prev_ok, const double* seg_scales_dev) {
  YOND_REQUIRE(regs_dev && params_dev && t_dev && work, "yond_vst_params_fill: null argument");
  YOND_REQUIRE(nseg > 0 && nseg <= 65535 && frames_per_seg > 0, "yond_vst_params_fill: bad batch geometry");
  YOND_REQUIRE(bias_mode >= 0 && bias_mode <= 2, "yond_vst_params_fill: bias_mode 0 (None), 1 ('pre'), 2 ('post')");
  YOND_REQUIRE(bias_mode != 1 || (rows && xnodes && row_stride >= 2), "yond_vst_params_fill: bias rows required for 'pre'");
  YOND_REQUIRE(!lut2d || (sg_lut_dev && x_lut_dev && nx > 1 && nsg > 1 && row_stride >= nx), "yond_vst_params_fill: incomplete LUT description");
  cudaStream_t s = (cudaStream_t)stream;
  SegChain* chain = reinterpret_cast<SegChain*>(work);
  FillArgs a{};
  a.scale_est = scale_est;
  a.scale = scale;
  a.bound_scale = bound_scale;
  a.round = round;
  a.bias_mode = bias_mode;
  a.exact_inverse = exact_inverse;
  a.frames_per_seg = frames_per_seg;
  a.nseg = nseg;
  a.nsg = nsg;
  a.has_lut = lut2d != nullptr;
  a.max_nodes = row_stride;
  params_fill_kernel<<<ceil_div(nseg, 64), 64, 0, s>>>(a, regs_dev, seg_max_dev, sg_lut_dev, prev_params, prev_ok, params_dev, t_dev,
                                                      chain, regs_out, ok_dev, seg_scales_dev);
  YOND_LAUNCH_CHECK();
  if (bias_mode == 1) {
    if (lut2d) {
      lut_rows_kernel<<<dim3(ceil_div(nx, 256), nseg), 256, 0, s>>>(lut2d, x_lut_dev, nx, nsg, chain, rows, xnodes, row_stride);
      YOND_LAUNCH_CHECK();
    }
    bias_table_kernel<<<dim3(ceil_div(row_stride, kNodesPerBlock), nseg), kTableThreads, kGaussTab * sizeof(double), s>>>(
        chain, rows, xnodes, row_stride, kGaussTab, 1, nullptr, nullptr);
    YOND_LAUNCH_CHECK();
  }
  return YOND_OK;
}

int yond_bias_table(double gain, double sigma, float bound, float* nodes_dev, float* vals_dev, int cap, int32_t* n_nodes_dev,
                    void* work, void* stream) {
  YOND_REQUIRE(nodes_dev && vals_dev && work && cap >= 2, "yond_bias_table: null argument");
  YOND_REQUIRE(gain > 0, "yond_bias_table: gain must be positive");
  cudaStream_t s = (cudaStream_t)stream;
  SegChain* chain = reinterpret_cast<SegChain*>(work);
  single_chain_kernel<<<1, 1, 0, s>>>(chain, gain, sigma, bound, cap, n_nodes_dev, 0);
  YOND_LAUNCH_CHECK();
  int n = table_nodes(bound);
  if (n > cap) n = cap;
  bias_table_kernel<<<dim3(ceil_div(n, kNodesPerBlock), 1), kTableThreads, kGaussTab * sizeof(double), s>>>(chain, vals_dev, nodes_dev, cap,
                                                                                                     kGaussTab, 1, nullptr, nullptr);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_bias_points(const double* lams_dev, int n, double gain, double sigma, int pho_min, double* bias_dev, void* work,
                     void* stream) {
  YOND_REQUIRE(lams_dev && bias_dev && work && n > 0, "yond_bias_points: null argument");
  YOND_REQUIRE(gain > 0 && pho_min >= 1, "yond_bias_points: gain must be positive, pho_min >= 1");
  cudaStream_t s = (cudaStream_t)stream;
  SegChain* chain = reinterpret_cast<SegChain*>(work);
  single_chain_kernel<<<1, 1, 0, s>>>(chain, gain, sigma, 0.f, n, nullptr, n);
  YOND_LAUNCH_CHECK();
  const int gtab = pho_min > 8 ? kGaussTabMax : kGaussTab;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(bias_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGaussTabMax * (int)sizeof(double));
  });
  if (attr_err != cudaSuccess) return yond_set_error(YOND_ERR_CUDA, "cudaFuncSetAttribute(bias_table_kernel) failed: %s", cudaGetErrorString(attr_err));
  bias_table_kernel<<<dim3(ceil_div(n, kNodesPerBlock), 1), kTableThreads, gtab * sizeof(double), s>>>(chain, nullptr, nullptr, 0, gtab,
                                                                                                  pho_min, lams_dev, bias_dev);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

}  // extern "C"
