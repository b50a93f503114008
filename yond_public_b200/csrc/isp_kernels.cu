// Elementwise / LUT kernels of the YOND path: Bayer pack/unpack, generalized-Anscombe VST with LUT bias
// correction, normalisation, reflect padding, inverse VST.  All HBM-bound: one pass, 64/128-bit accesses.
//   reference: utils/isp_ops.py:57-63, utils/isp_algos.py:5-33,162-231, YOND_SIDD.py:238-299.
#include <mutex>

#include "common.cuh"

namespace {

constexpr int kBlock = 256;

// ------------------------------------------------------------------ A1 / A2
// One thread packs two adjacent quads: two 128-bit loads (rows 2i, 2i+1), two 128-bit stores.
__global__ void pack_kernel(const float* __restrict__ bayer, float* __restrict__ rggb, int B, int H, int W) {
  const int h = H >> 1, w2 = W >> 2;  // w2 = pairs of quads per row
  const size_t total = (size_t)B * h * w2;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int jp = (int)(idx % w2);
    const int i = (int)((idx / w2) % h);
    const int b = (int)(idx / ((size_t)w2 * h));
    const float* r0 = bayer + ((size_t)b * H + 2 * i) * W + 4 * jp;
    const float4 a = ldg_stream_f4(reinterpret_cast<const float4*>(r0));
    const float4 c = ldg_stream_f4(reinterpret_cast<const float4*>(r0 + W));
    float4* o = reinterpret_cast<float4*>(rggb + (((size_t)b * h + i) * (W >> 1) + 2 * jp) * 4);
    o[0] = make_float4(a.x, a.y, c.x, c.y);
    o[1] = make_float4(a.z, a.w, c.z, c.w);
  }
}
__global__ void pack_kernel_scalar(const float* __restrict__ bayer, float* __restrict__ rggb, int B, int H, int W) {
  const int h = H >> 1, w = W >> 1;
  const size_t total = (size_t)B * h * w;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(idx % w);
    const int i = (int)((idx / w) % h);
    const int b = (int)(idx / ((size_t)w * h));
    const float* r0 = bayer + ((size_t)b * H + 2 * i) * W + 2 * j;
    float* o = rggb + idx * 4;
    o[0] = r0[0]; o[1] = r0[1]; o[2] = r0[W]; o[3] = r0[W + 1];
  }
}
__global__ void unpack_kernel(const float* __restrict__ rggb, float* __restrict__ bayer, int B, int h, int w) {
  const int W = 2 * w, H = 2 * h;
  const size_t total = (size_t)B * h * w;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(idx % w);
    const int i = (int)((idx / w) % h);
    const int b = (int)(idx / ((size_t)w * h));
    const float4 v = ldg_stream_f4(reinterpret_cast<const float4*>(rggb) + idx);
    float* r0 = bayer + ((size_t)b * H + 2 * i) * W + 2 * j;
    *reinterpret_cast<float2*>(r0) = make_float2(v.x, v.y);
    *reinterpret_cast<float2*>(r0 + W) = make_float2(v.z, v.w);
  }
}

// ------------------------------------------------------------------ 8(f)-1 RAW ingest (process.py:40-64)
// One thread = one CFA cell: two 32-bit loads (2 x uint16 each), four IEEE float32 (v - black) / (white - black), one
// 128-bit store (interleaved layout) or four plane stores.  2 B/px in, 4 B/px out.
struct RawParams {
  int pos[4];       // position (2*row + col) of R, G1, B, G2 inside the cell
  float black[4];
  float denom[4];   // fl32(white) - black[c], rounded like NumPy's float32 subtraction
};
__device__ __forceinline__ void raw_cell(uint32_t a, uint32_t d, const RawParams& q, int clip, float (&v)[4]) {
  const float c0 = (float)(a & 0xffffu), c1 = (float)(a >> 16), c2 = (float)(d & 0xffffu), c3 = (float)(d >> 16);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int p = q.pos[c];
    const float cell = p == 0 ? c0 : (p == 1 ? c1 : (p == 2 ? c2 : c3));  // selects: no dynamically indexed local array
    float t = __fdiv_rn(__fsub_rn(cell, q.black[c]), q.denom[c]);
    if (clip) t = fminf(fmaxf(t, 0.f), 1.f);
    v[c] = t;
  }
}
// kCells = CFA cells per thread along the row: 2 (64-bit loads; W % 4 == 0 and 8-byte aligned rows) or 1.
template <int kCells>
__global__ void pack_raw_kernel(const uint16_t* __restrict__ raw, float* __restrict__ out, int B, int H, int W, RawParams q,
                                int clip, int layout) {
  const int h = H >> 1, w = W >> 1, wq = w / kCells;
  const size_t total = (size_t)B * h * wq;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(idx % wq) * kCells;
    const int i = (int)((idx / wq) % h);
    const int b = (int)(idx / ((size_t)wq * h));
    const uint16_t* r0 = raw + ((size_t)b * H + 2 * i) * W + 2 * j;
    uint32_t a[kCells], d[kCells];
    if (kCells == 2) {
      const uint2 ua = ldg_stream_u2(reinterpret_cast<const uint2*>(r0)), ud = ldg_stream_u2(reinterpret_cast<const uint2*>(r0 + W));
      a[0] = ua.x; a[kCells - 1] = ua.y; d[0] = ud.x; d[kCells - 1] = ud.y;
    } else {
      a[0] = __ldg(reinterpret_cast<const uint32_t*>(r0));
      d[0] = __ldg(reinterpret_cast<const uint32_t*>(r0 + W));
    }
    const size_t plane = (size_t)h * w, cellidx = ((size_t)b * h + i) * w + j, pbase = (size_t)b * 4 * plane + (size_t)i * w + j;
    float v[kCells][4];
#pragma unroll
    for (int k = 0; k < kCells; ++k) raw_cell(a[k], d[k], q, clip, v[k]);
    if (layout == 1) {
#pragma unroll
      for (int k = 0; k < kCells; ++k) reinterpret_cast<float4*>(out)[cellidx + k] = make_float4(v[k][0], v[k][1], v[k][2], v[k][3]);
    } else if (kCells == 2) {
#pragma unroll
      for (int c = 0; c < 4; ++c) *reinterpret_cast<float2*>(out + pbase + c * plane) = make_float2(v[0][c], v[kCells - 1][c]);
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) out[pbase + c * plane] = v[0][c];
    }
  }
}

// ------------------------------------------------------------------ dataset normalisation of the 14-bit drivers
// data_process/yond_datasets.py:955-961, :1053-1056: lr = (raw.astype(float32) - bl) * ratio / (wp - bl) on the MOSAIC, float32
// arithmetic in that order (array op scalar keeps float32 under the NumPy the reference was written for), no clipping unless asked.
// Reads 2 B/px; eight pixels (one 128-bit load, two 128-bit stores) per thread.
__global__ void ingest_mosaic_kernel(const uint16_t* __restrict__ raw, float* __restrict__ out, size_t n8, float bl, float ratio, float denom,
                                     int clip) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(raw) + i);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    float v[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      v[2 * k] = (float)(w[k] & 0xffffu);
      v[2 * k + 1] = (float)(w[k] >> 16);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float t = __fdiv_rn(__fmul_rn(__fsub_rn(v[k], bl), ratio), denom);
      if (clip) t = fminf(fmaxf(t, 0.f), 1.f);
      v[k] = t;
    }
    float4* o = reinterpret_cast<float4*>(out) + 2 * i;
    o[0] = make_float4(v[0], v[1], v[2], v[3]);
    o[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
}
__global__ void ingest_mosaic_tail_kernel(const uint16_t* __restrict__ raw, float* __restrict__ out, size_t i0, size_t n, float bl, float ratio,
                                          float denom, int clip) {
  const size_t i = i0 + blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float t = __fdiv_rn(__fmul_rn(__fsub_rn((float)raw[i], bl), ratio), denom);
  if (clip) t = fminf(fmaxf(t, 0.f), 1.f);
  out[i] = t;
}

// ------------------------------------------------------------------ rot_bayer (sidd_utils.py:198-213): np.rot90
// Quarter turns go through a 32x32 shared-memory tile so that both the global read and the global write are row-contiguous:
//   k = 1: out[i][j] = in[j][W-1-i]      tile[r][c] = in[j0 + r][W-1-i0-31 + c],   out(i0+a, j0+b) = tile[b][31-a]
//   k = 3: out[i][j] = in[H-1-j][i]      tile[r][c] = in[H-1-j0-31 + r][i0 + c],   out(i0+a, j0+b) = tile[31-b][a]
// block (32, 8); out is (W, H) per image.
__global__ void rot90_odd_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W, int k) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const float* src = in + (size_t)b * H * W;
  float* dst = out + (size_t)b * H * W;
  const int Ho = W, Wo = H;
  const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
  const int rb = k == 1 ? j0 : H - 1 - j0 - 31;
  const int cb = k == 1 ? W - 1 - i0 - 31 : i0;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int rr = rb + r, cc = cb + (int)threadIdx.x;
    tile[r][threadIdx.x] = (rr >= 0 && rr < H && cc >= 0 && cc < W) ? src[(size_t)rr * W + cc] : 0.f;
  }
  __syncthreads();
  for (int a = threadIdx.y; a < 32; a += 8) {
    const int i = i0 + a, j = j0 + (int)threadIdx.x;
    if (i < Ho && j < Wo) dst[(size_t)i * Wo + j] = k == 1 ? tile[threadIdx.x][31 - a] : tile[31 - threadIdx.x][a];
  }
}
// k = 2: out[i][j] = in[H-1-i][W-1-j]; k = 0: copy
__global__ void rot90_even_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int H, int W, int k) {
  const size_t per = (size_t)H * W, total = (size_t)B * per;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t b = idx / per, e = idx - b * per;
    out[idx] = k == 2 ? in[b * per + (per - 1 - e)] : in[idx];  // reversing both axes = reversing the flattened image
  }
}

// ------------------------------------------------------------------ A3 / A4 / A5 device functions
struct VstConst {
  float K, c0, two_over_K, lower, inv_range, range, scale, inv_scale, sig2e, sigma;
  int lut_row, table_n, exact;
};
__device__ __forceinline__ VstConst load_const(const yond_vst_params& q) {
  VstConst c;
  c.K = q.gain;
  c.sigma = q.sigma;
  c.c0 = 0.375f * q.gain * q.gain + q.sigma * q.sigma;
  c.two_over_K = 2.0f / q.gain;
  c.lower = q.lower;
  c.range = q.upper - q.lower;
  c.inv_range = 1.0f / c.range;
  c.scale = q.scale;
  c.inv_scale = 1.0f / q.scale;
  const float se = q.sigma / q.gain;
  c.sig2e = se * se;
  c.lut_row = q.lut_row;
  c.table_n = q.table_n;
  c.exact = q.exact_inverse;
  return c;
}
__device__ __forceinline__ float vst_f(float x, const VstConst& c) {
  // sqrt.approx: 1 ulp (2^-23 relative) instead of correctly rounded — far below the 2e-3 output budget, a third of the
  // instructions of the IEEE sequence; the function-level VST (vst_elem_kernel) keeps sqrtf
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaxf(fmaf(c.K, x, c.c0), 0.f)));
  return c.two_over_K * r;
}
// Foi's closed-form bias (utils/isp_algos.py:84-96), used beyond the table like the reference does (:228-230).
__device__ __forceinline__ float close_form_bias_f(float x, const VstConst& c) {
  const float y = x / c.K, s2 = c.sig2e;
  const float yh = y + 0.375f + s2;
  const float m1 = (y + s2) / (yh * yh);
  const float m2 = y / (yh * yh * yh);
  const float m3 = (y + 3.f * (y + s2) * (y + s2)) / (yh * yh * yh * yh);
  return 2.f * sqrtf(yh) * (-0.125f * m1 + 0.0625f * m2 - 0.0390625f * m3);
}
// Piecewise-linear table lookup with the reference's node inversion (pos_interp + data_merge).
//   `nodes` ascending, n entries; LUT mode (analytic first guess on the lin+log grid) or generic (binary search).
__device__ __forceinline__ float table_eval(float xq, const float* __restrict__ row, const float* __restrict__ nodes, int n,
                                            bool lut_grid) {
  if (xq <= __ldg(nodes)) return __ldg(row);
  int l;
  if (lut_grid) {
    int g = xq < 0.0625f ? (int)(xq * 2048.f) : 128 + (int)floorf(128.f * (log2f(xq) + 4.f));
    g = max(0, min(g, n - 2));
    while (g + 1 < n - 1 && __ldg(nodes + g + 1) < xq) ++g;
    while (g > 0 && __ldg(nodes + g) >= xq) --g;
    l = g;
  } else {
    int lo = 0, hi = n - 1;  // invariant: nodes[lo] < xq, find last such lo with lo <= n-2
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(nodes + mid) < xq) lo = mid; else hi = mid;
    }
    l = lo;
  }
  const float xl = __ldg(nodes + l), xr = __ldg(nodes + l + 1);
  float wr = (xq - xl) / (xr - xl);
  wr = fminf(wr, 1.0f);  // beyond the last node the reference clips the position (data_merge)
  const float yl = __ldg(row + l), yr = __ldg(row + l + 1);
  return yl * (1.f - wr) + yr * wr;
}
__device__ __forceinline__ float bias_eval(float x_dn, const VstConst& c, const float* __restrict__ rows,
                                           const float* __restrict__ xnodes, int row_stride) {
  if (c.lut_row < 0) return 0.f;
  const float xb = fmaxf(x_dn, 0.f);
  const float* row = rows + (size_t)c.lut_row * row_stride;
  const float* nodes = xnodes + (size_t)c.lut_row * row_stride;  // every row carries its own node positions
  if (c.table_n > 0) {  // fallback get_bias table (isp_algos.py:98-140): nodes in DN
    const float xc = fminf(xb, __ldg(nodes + c.table_n - 1));
    return table_eval(xc, row, nodes, c.table_n, false);
  }
  const float xe = xb / c.K;  // BiasLUT row: nodes in electrons on the 1921-node lin+log grid
  const int nx = 1921;
  const float last = __ldg(nodes + nx - 1), prev = __ldg(nodes + nx - 2);
  if (xe >= last + (last - prev)) return close_form_bias_f(xb, c);  // x_pos >= len(x_lut): isp_algos.py:228-230
  return table_eval(xe, row, nodes, nx, true);
}
__device__ __forceinline__ float inverse_vst_f(float z, const VstConst& c) {
  float f;
  if (c.exact) {
    if (z > 0.f) {
      const float iz = 1.f / z;
      f = 0.25f * z * z + 0.30618621784789724f * iz - 1.375f * iz * iz + 0.7654655446197431f * iz * iz * iz - 0.125f - c.sig2e;
    } else {
      f = 0.f;
    }
  } else {
    f = 0.25f * z * z - 0.375f - c.sig2e;
  }
  return fmaxf(f, 0.f) * c.K;
}

__device__ __forceinline__ void block_max_to(float v, float* dst) {
  // v >= 0: integer order == float order
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __shared__ float wmax[kBlock / 32];
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    float m = threadIdx.x < kBlock / 32 ? wmax[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) atomicMax(reinterpret_cast<int*>(dst), __float_as_int(m));
  }
}

// ------------------------------------------------------------------ A18 front: fused pack+bias+VST+normalise+clamp+pad
// grid = (blocks per frame, B); every block stays inside one frame so the per-frame constants are uniform.
// The frame's bias row is staged in shared memory as one 16-byte record per interval {x_l, y_l, slope, x_r}: a lookup is
// an index guess (analytic on the BiasLUT's lin+log grid and on get_bias's three uniform pieces, binary search for
// anything else), one LDS.128, a fix-up that almost never iterates, and one FMA.  The float32 slope form differs from the
// reference's y_l (1 - w) + y_r w by one rounding of a value that is itself ~0.1 (BiasLUT goldens: <= 2e-6 allowed, ~1e-8 seen).
constexpr int kFwdPix = 16;  // packed pixels per thread: amortises the table staging (1921 records per block)
struct TabInfo {
  int n;            // nodes
  int kind;         // 0: none, 1: BiasLUT grid (electrons), 2: get_bias pieces (DN), 3: generic ascending nodes
  float last;       // last node
  float ext;        // LUT: last + (last - prev): beyond it the closed form applies (isp_algos.py:228-230)
  int n1, n2;       // get_bias pieces: first index of piece 2 / piece 3
  float v1, v2;     // their first node values
  float is0, is1, is2;  // inverse steps of the pieces
};
// tab / ti: 32-bit shared addresses (smem_addr) of the interval records and of the TabInfo; kind and n are held in registers
__device__ __forceinline__ float tab_lookup(float xq, uint32_t tab, int kind, int n, uint32_t ti) {
  int g;
  if (kind == 1) {
    g = xq < 0.0625f ? (int)(xq * 2048.f) : 128 + (int)(128.f * (__log2f(xq) + 4.f));
  } else if (kind == 2) {
    const float v1 = lds_f32(ti + offsetof(TabInfo, v1)), v2 = lds_f32(ti + offsetof(TabInfo, v2));
    g = xq < v1 ? (int)(xq * lds_f32(ti + offsetof(TabInfo, is0)))
                : (xq < v2 ? (int)lds_u32(ti + offsetof(TabInfo, n1)) + (int)((xq - v1) * lds_f32(ti + offsetof(TabInfo, is1)))
                           : (int)lds_u32(ti + offsetof(TabInfo, n2)) + (int)((xq - v2) * lds_f32(ti + offsetof(TabInfo, is2))));
  } else {
    int lo = 0, hi = n - 1;  // last interval whose left node is < xq
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (lds_f32(tab + 16u * (uint32_t)mid) < xq) lo = mid; else hi = mid;
    }
    g = lo;
  }
  g = max(0, min(g, n - 2));
  float4 e = lds_v4f(tab + 16u * (uint32_t)g);
  while (xq > e.w && g < n - 2) e = lds_v4f(tab + 16u * (uint32_t)(++g));
  while (xq < e.x && g > 0) e = lds_v4f(tab + 16u * (uint32_t)(--g));
  return fmaf(fmaxf(xq - e.x, 0.f), e.z, e.y);
}
// kTable: frame b is the (H, W) frame of record frames[b] (yond_frame_geom), read once per CTA, instead of frame b of one (B, H, W)
// tensor — the frames of one size of a batch stay where their owners keep them.  With raw_in.per_img set the record's `base` is a uint16
// sensor mosaic, normalised with raw_in.per_img[b].  The arithmetic and the z / ub outputs are the uniform form's.
template <bool kVst, bool kTable = false>
__global__ void __launch_bounds__(kBlock, 5) vst_fwd_kernel(const float* __restrict__ bayer, float* __restrict__ z,
                                                         float* __restrict__ ub, int H, int W, int pl, int pt, int hp, int wp,
                                                         const yond_vst_params* __restrict__ params,
                                                         const float* __restrict__ rows, const float* __restrict__ xnodes,
                                                         int row_stride, RawNorm raw_in, const yond_frame_geom* frames) {
  extern __shared__ float4 tab[];
  __shared__ TabInfo ti;
  const int b = blockIdx.y;
  if constexpr (kTable) {
    bayer = frames[b].base;
    if (raw_in.per_img) raw_in.base = reinterpret_cast<const uint16_t*>(bayer);
  }
  const RawNorm raw = raw_norm_at(raw_in, b);  // every pixel of a CTA belongs to frame b
  const int h = H >> 1, w = W >> 1;
  VstConst c{};
  if (kVst) {
    c = load_const(params[b]);
    if (c.lut_row >= 0) {
      const float* row = rows + (size_t)c.lut_row * row_stride;
      const float* nodes = xnodes + (size_t)c.lut_row * row_stride;
      const int n = c.table_n > 0 ? c.table_n : 1921;
      for (int i = threadIdx.x; i < n - 1; i += kBlock) {
        const float xl = __ldg(nodes + i), xr = __ldg(nodes + i + 1), yl = __ldg(row + i), yr = __ldg(row + i + 1);
        tab[i] = make_float4(xl, yl, xr > xl ? (yr - yl) / (xr - xl) : 0.f, xr);
      }
      if (threadIdx.x == 0) {
        TabInfo t{};
        t.n = n;
        t.last = __ldg(nodes + n - 1);
        t.ext = t.last + (t.last - __ldg(nodes + n - 2));
        if (c.table_n == 0) {
          t.kind = 1;
        } else {
          // get_bias node layout (isp_algos.py:101-108): [0,50] step 0.1 | [50,500] step 1 | [500,ub] step ~10, or a single
          // piece below 50 — recognised from the node values, anything else takes the binary search
          t.kind = 3;
          const float n0 = __ldg(nodes);
          if (n0 == 0.f && t.last < 50.f && n >= 3) {
            t.kind = 2; t.n1 = t.n2 = n; t.v1 = t.v2 = 3.0e38f; t.is0 = (float)(n - 1) / t.last;
          } else if (n0 == 0.f && n >= 504 && __ldg(nodes + 500) == 50.f && __ldg(nodes + 501) == 50.f) {
            t.kind = 2; t.n1 = 501; t.v1 = 50.f; t.is0 = 10.f;
            if (t.last < 500.f || n < 955) {
              t.n2 = n; t.v2 = 3.0e38f; t.is1 = (float)(n - 502) / (t.last - 50.f);
            } else if (__ldg(nodes + 951) == 500.f && __ldg(nodes + 952) == 500.f) {
              t.n2 = 952; t.v2 = 500.f; t.is1 = 1.f; t.is2 = (float)(n - 953) / (t.last - 500.f);
            } else {
              t.kind = 3;
            }
          }
        }
        ti = t;
      }
    }
  }
  __syncthreads();
  const uint32_t a_tab = smem_addr(tab), a_ti = smem_addr(&ti);
  const int t_kind = ti.kind, t_n = ti.n;
  const float t_last = ti.last, t_ext = ti.ext;
  const float invK = kVst ? 1.0f / c.K : 0.f;
  const float* frame = bayer + (kTable ? 0 : (size_t)b * H * W);
  float4* zo = reinterpret_cast<float4*>(z) + (size_t)b * hp * wp;
  const int npix = hp * wp;
  float vmax = 0.f;
  int idx = blockIdx.x * (kBlock * kFwdPix) + threadIdx.x;
  int i = idx / wp, j = idx - i * wp;
  // the padding is smaller than the frame (checked by the launcher): one reflection per side
  auto refl = [](int t, int n) { t = t < 0 ? -t : t; return t >= n ? 2 * (n - 1) - t : t; };
#pragma unroll 1
  for (int it = 0; it < kFwdPix && idx < npix; ++it) {
    const size_t poff = (size_t)(2 * refl(i - pt, h)) * W + 2 * refl(j - pl, w);
    float v[4];
    if (raw.base) {  // uint16 sensor mosaic, normalised on load (SURVEY 8(f)-1)
      const uint16_t* r16 = raw.base + (kTable ? 0 : (size_t)b * H * W) + poff;
      const uint32_t a = __ldg(reinterpret_cast<const uint32_t*>(r16)), d = __ldg(reinterpret_cast<const uint32_t*>(r16 + W));
      v[0] = raw_norm(a & 0xffffu, raw); v[1] = raw_norm(a >> 16, raw); v[2] = raw_norm(d & 0xffffu, raw); v[3] = raw_norm(d >> 16, raw);
    } else {
      const float* r0 = frame + poff;
      const float2 a = ldg_stream_f2(reinterpret_cast<const float2*>(r0));
      const float2 d = ldg_stream_f2(reinterpret_cast<const float2*>(r0 + W));
      v[0] = a.x; v[1] = a.y; v[2] = d.x; v[3] = d.y;
    }
    if (kVst) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float x = v[k] * c.scale;
        float bias = 0.f;
        if (c.lut_row >= 0) {
          const float xb = fmaxf(x, 0.f);
          if (c.table_n > 0) {
            bias = tab_lookup(fminf(xb, t_last), a_tab, t_kind, t_n, a_ti);
          } else {
            const float xe = xb * invK;
            bias = xe >= t_ext ? close_form_bias_f(xb, c) : tab_lookup(xe, a_tab, t_kind, t_n, a_ti);
          }
        }
        const float zz = vst_f(x, c) - bias;
        v[k] = (zz - c.lower) * c.inv_range;
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      v[k] = fminf(fmaxf(v[k], 0.f), 1.f);
      vmax = fmaxf(vmax, v[k]);
    }
    zo[idx] = make_float4(v[0], v[1], v[2], v[3]);
    idx += kBlock;
    j += kBlock;
    while (j >= wp) {
      j -= wp;
      ++i;
    }
  }
  block_max_to(vmax, ub + b);
}

// ------------------------------------------------------------------ A18 back: clamp+crop+denorm+inverse+unpack(+clip)
// Output placement: frames_per_row = 1 writes (B,H,W); n > 1 writes frame b as block b % n of the mosaic b / n — the
// reference's np.concatenate(blocks, axis=-1) layout (YOND_SIDD.py:408) — so no permute pass follows.
// Round selection: with `seg_ok`, frames of an image whose round-2 estimate failed the beta1 >= 0 guard (:445-447) copy
// `fallback` (the round-1 result, same layout as the output) instead of the network output.
struct InvPlace {
  int frames_per_row;
  const int32_t* seg_ok;
  int frames_per_seg;
  const float* fallback;
};
template <bool kVst>
__global__ void __launch_bounds__(kBlock) vst_inv_kernel(const float* __restrict__ y, float* __restrict__ bayer, int H, int W,
                                                         int pl, int pt, int hp, int wp,
                                                         const yond_vst_params* __restrict__ params, int clip01, InvPlace place) {
  const int b = blockIdx.y;
  const int h = H >> 1, w = W >> 1;
  VstConst c{};
  if (kVst) c = load_const(params[b]);
  const float4* yi = reinterpret_cast<const float4*>(y) + (size_t)b * hp * wp;
  const int fpr = place.frames_per_row;
  const size_t pitch = (size_t)fpr * W;
  const size_t origin = (size_t)(b / fpr) * H * pitch + (size_t)(b % fpr) * W;
  float* frame = bayer + origin;
  const bool keep = place.seg_ok == nullptr || place.seg_ok[b / place.frames_per_seg] != 0;
  const float* fb = place.fallback ? place.fallback + origin : nullptr;
  const int npix = h * w;
  for (int idx = blockIdx.x * kBlock + threadIdx.x; idx < npix; idx += gridDim.x * kBlock) {
    const int j = idx % w, i = idx / w;
    float* r0 = frame + (size_t)(2 * i) * pitch + 2 * j;
    if (!keep) {
      if (fb) {
        const float* f0 = fb + (size_t)(2 * i) * pitch + 2 * j;
        *reinterpret_cast<float2*>(r0) = ldg_stream_f2(reinterpret_cast<const float2*>(f0));
        *reinterpret_cast<float2*>(r0 + pitch) = ldg_stream_f2(reinterpret_cast<const float2*>(f0 + pitch));
      }
      continue;
    }
    const float4 q = ldg_stream_f4(yi + (size_t)(i + pt) * wp + (j + pl));
    float v[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float t = fminf(fmaxf(v[k], 0.f), 1.f);
      if (kVst) {
        t = inverse_vst_f(fmaf(t, c.range, c.lower), c) * c.inv_scale;
        if (clip01) t = fminf(fmaxf(t, 0.f), 1.f);
      }
      v[k] = t;
    }
    *reinterpret_cast<float2*>(r0) = make_float2(v[0], v[1]);
    *reinterpret_cast<float2*>(r0 + pitch) = make_float2(v[2], v[3]);
  }
}

// ------------------------------------------------------------------ function-level surface
__global__ void vst_elem_kernel(const float* __restrict__ x, float* __restrict__ z, size_t n, float K, float c0) {
  const float tk = 2.f / K;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    z[i] = tk * sqrtf(fmaxf(fmaf(K, x[i], c0), 0.f));
}
__global__ void ivst_elem_kernel(const float* __restrict__ z, float* __restrict__ x, size_t n, VstConst c) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    x[i] = inverse_vst_f(z[i], c);
}
__global__ void lut_row_kernel(const float* __restrict__ lut, int nx, int nsg, int l, int r, float wr, float* __restrict__ row) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nx) row[i] = lut[(size_t)i * nsg + l] * (1.f - wr) + lut[(size_t)i * nsg + r] * wr;
}
__global__ void lut_apply_kernel(const float* __restrict__ x, float* __restrict__ bias, size_t n, const float* __restrict__ row,
                                 const float* __restrict__ xnodes, int nx, VstConst c) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    bias[i] = bias_eval(x[i], c, row, xnodes, nx);
}

inline int grid_for(size_t n, int per_thread = 1) {
  size_t g = (n + (size_t)kBlock * per_thread - 1) / ((size_t)kBlock * per_thread);
  const size_t cap = (size_t)yond_num_sms() * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

extern "C" {

int yond_pack(const float* bayer, float* rggb, int B, int H, int W, void* stream) {
  YOND_REQUIRE(B > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "yond_pack: H,W must be even (got %d,%d)", H, W);
  cudaStream_t s = (cudaStream_t)stream;
  const bool vec = (W % 4 == 0) && ((uintptr_t)bayer % 16 == 0) && ((uintptr_t)rggb % 16 == 0);
  YondProfScope prof("pack", s, 8.0 * (double)B * H * W);
  if (vec) pack_kernel<<<grid_for((size_t)B * (H / 2) * (W / 4)), kBlock, 0, s>>>(bayer, rggb, B, H, W);
  else pack_kernel_scalar<<<grid_for((size_t)B * (H / 2) * (W / 2)), kBlock, 0, s>>>(bayer, rggb, B, H, W);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_rot90(const float* in, float* out, int B, int H, int W, int k, void* stream) {
  YOND_REQUIRE(in && out && in != out && B > 0 && H > 0 && W > 0, "yond_rot90: bad arguments (out of place only)");
  YOND_REQUIRE(B <= 65535, "yond_rot90: at most 65535 images per call");
  k = ((k % 4) + 4) % 4;
  cudaStream_t s = (cudaStream_t)stream;
  if (k & 1) rot90_odd_kernel<<<dim3((H + 31) / 32, (W + 31) / 32, B), dim3(32, 8), 0, s>>>(in, out, H, W, k);
  else rot90_even_kernel<<<grid_for((size_t)B * H * W), kBlock, 0, s>>>(in, out, B, H, W, k);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_pack_raw(const uint16_t* raw, float* out, int B, int H, int W, const int* pos4, const float* black4, float white,
                  int clip, int layout, void* stream) {
  YOND_REQUIRE(raw && out && pos4 && black4, "yond_pack_raw: null argument");
  YOND_REQUIRE(B > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "yond_pack_raw: H,W must be even (got %d,%d)", H, W);
  YOND_REQUIRE((uintptr_t)raw % 4 == 0 && (uintptr_t)out % 16 == 0, "yond_pack_raw: raw must be 4-byte and out 16-byte aligned");
  YOND_REQUIRE(layout == 0 || layout == 1, "yond_pack_raw: layout 0 (planes) or 1 (interleaved)");
  RawParams q;
  int seen = 0;
  for (int c = 0; c < 4; ++c) {
    YOND_REQUIRE(pos4[c] >= 0 && pos4[c] < 4, "yond_pack_raw: CFA position out of range");
    seen |= 1 << pos4[c];
    q.pos[c] = pos4[c];
    q.black[c] = black4[c];
    q.denom[c] = white - black4[c];  // float32 subtraction, like `white_point - black_level` on a float32 array
  }
  YOND_REQUIRE(seen == 15, "yond_pack_raw: raw_pattern must place R, G1, B, G2 on four distinct cell positions");
  YondProfScope prof("pack_raw", (cudaStream_t)stream, 6.0 * (double)B * H * W);
  if (W % 4 == 0 && (uintptr_t)raw % 8 == 0)
    pack_raw_kernel<2><<<grid_for((size_t)B * (H / 2) * (W / 4)), kBlock, 0, (cudaStream_t)stream>>>(raw, out, B, H, W, q, clip, layout);
  else
    pack_raw_kernel<1><<<grid_for((size_t)B * (H / 2) * (W / 2)), kBlock, 0, (cudaStream_t)stream>>>(raw, out, B, H, W, q, clip, layout);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_ingest_mosaic(const uint16_t* raw, float* out, size_t n, float black, float white, float ratio, int clip, void* stream) {
  YOND_REQUIRE(raw && out && n > 0, "yond_ingest_mosaic: null argument");
  YOND_REQUIRE((uintptr_t)raw % 16 == 0 && (uintptr_t)out % 16 == 0, "yond_ingest_mosaic: 16-byte aligned buffers required");
  YOND_REQUIRE(white > black, "yond_ingest_mosaic: white level must exceed the black level");
  const float denom = white - black;  // the reference subtracts the integer levels: exact in float32 for sensor ranges
  YondProfScope prof("ingest_mosaic", (cudaStream_t)stream, 6.0 * (double)n);
  const size_t n8 = n / 8;
  if (n8) {
    ingest_mosaic_kernel<<<grid_for(n8), kBlock, 0, (cudaStream_t)stream>>>(raw, out, n8, black, ratio, denom, clip);
    YOND_LAUNCH_CHECK();
  }
  if (n % 8) {
    ingest_mosaic_tail_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(raw, out, n8 * 8, n, black, ratio, denom, clip);
    YOND_LAUNCH_CHECK();
  }
  return YOND_OK;
}

int yond_unpack(const float* rggb, float* bayer, int B, int h, int w, void* stream) {
  YOND_REQUIRE(B > 0 && h > 0 && w > 0, "yond_unpack: bad shape");
  unpack_kernel<<<grid_for((size_t)B * h * w), kBlock, 0, (cudaStream_t)stream>>>(rggb, bayer, B, h, w);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_vst(const float* x, float* z, size_t n, double sigma, double gain, void* stream) {
  YOND_REQUIRE(gain > 0, "yond_vst: gain must be positive");
  vst_elem_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(x, z, n, (float)gain,
                                                                    (float)(0.375 * gain * gain + sigma * sigma));
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_inverse_vst(const float* z, float* x, size_t n, double sigma, double gain, int exact, void* stream) {
  YOND_REQUIRE(gain > 0, "yond_inverse_vst: gain must be positive");
  VstConst c{};
  c.K = (float)gain;
  c.sig2e = (float)((sigma / gain) * (sigma / gain));
  c.exact = exact;
  ivst_elem_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(z, x, n, c);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_lut_row(const float* lut2d, int nx, int nsg, double sg_pos, float* row, void* stream) {
  YOND_REQUIRE(nx > 1 && nsg > 1, "yond_lut_row: bad table shape");
  if (sg_pos < 0) sg_pos = 0;
  if (sg_pos > nsg - 1) sg_pos = nsg - 1;  // the reference clips with len(x_lut)-1 (isp_algos.py:189): guarded here
  const int l = (int)floor(sg_pos), r = (int)ceil(sg_pos);
  lut_row_kernel<<<ceil_div(nx, kBlock), kBlock, 0, (cudaStream_t)stream>>>(lut2d, nx, nsg, l, r, (float)(sg_pos - l), row);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_lut_apply(const float* x, float* bias, size_t n, const float* row, const float* xnodes, int nx, double gain,
                   double sigma, void* stream) {
  YOND_REQUIRE(nx == 1921, "yond_lut_apply: expects the 1921-node BiasLUT grid");
  VstConst c{};
  c.K = (float)gain;
  c.lut_row = 0;
  c.table_n = 0;
  c.sig2e = (float)((sigma / gain) * (sigma / gain));
  lut_apply_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(x, bias, n, row, xnodes, nx, c);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_table_apply(const float* x, float* bias, size_t n, const float* vals, const float* nodes, int n_nodes, void* stream) {
  YOND_REQUIRE(x && bias && vals && nodes && n_nodes >= 2, "yond_table_apply: bad arguments");
  VstConst c{};
  c.K = 1.f;
  c.lut_row = 0;
  c.table_n = n_nodes;
  lut_apply_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(x, bias, n, vals, nodes, n_nodes, c);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

static int launch_fwd(bool vst, const float* bayer, float* z, float* ub, int B, int H, int W, int pl, int pr, int pt, int pb,
                      const yond_vst_params* params, const float* rows, const float* xnodes, int row_stride, void* stream,
                      RawNorm raw = RawNorm{}, const yond_frame_geom* frames = nullptr) {
  YOND_REQUIRE(B > 0 && H % 2 == 0 && W % 2 == 0 && H > 0 && W > 0, "vst_fwd: H,W must be even");
  const int h = H / 2, w = W / 2;
  YOND_REQUIRE(pl >= 0 && pr >= 0 && pt >= 0 && pb >= 0 && pl < w && pr < w && pt < h && pb < h,
               "vst_fwd: reflect padding must be smaller than the frame");
  const int hp = h + pt + pb, wp = w + pl + pr;
  cudaStream_t s = (cudaStream_t)stream;
  YOND_CUDA_CHECK(cudaMemsetAsync(ub, 0, sizeof(float) * B, s));
  YOND_REQUIRE(B <= 65535, "vst_fwd: at most 65535 frames per call");
  const int gx = ceil_div(hp * wp, kBlock * kFwdPix);
  dim3 grid(gx, B);
  if (vst) {
    const int tab_n = rows ? (row_stride > 1921 ? row_stride : 1921) : 0;
    const size_t smem = (size_t)tab_n * sizeof(float4);
    YOND_REQUIRE(smem <= 200 * 1024, "vst_fwd: bias tables of more than %d nodes are not supported (row_stride %d)", 200 * 1024 / 16, row_stride);
    static std::once_flag once, once_tab;
    static cudaError_t attr_err = cudaSuccess, attr_err_tab = cudaSuccess;
    cudaError_t err;
    if (frames) {
      std::call_once(once_tab, [] { attr_err_tab = cudaFuncSetAttribute(vst_fwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
      err = attr_err_tab;
    } else {
      std::call_once(once, [] { attr_err = cudaFuncSetAttribute(vst_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
      err = attr_err;
    }
    if (err != cudaSuccess) return yond_set_error(YOND_ERR_CUDA, "cudaFuncSetAttribute(vst_fwd_kernel) failed: %s", cudaGetErrorString(err));
    YondProfScope prof("vst_fwd", s, 8.0 * (double)B * H * W);  // 4 R (Bayer f32) + 4 W (z f32) per Bayer pixel
    if (frames)
      vst_fwd_kernel<true, true><<<grid, kBlock, smem, s>>>(nullptr, z, ub, H, W, pl, pt, hp, wp, params, rows, xnodes, row_stride, raw, frames);
    else
      vst_fwd_kernel<true><<<grid, kBlock, smem, s>>>(bayer, z, ub, H, W, pl, pt, hp, wp, params, rows, xnodes, row_stride, raw, nullptr);
  } else {
    vst_fwd_kernel<false><<<grid, kBlock, 0, s>>>(bayer, z, ub, H, W, pl, pt, hp, wp, nullptr, nullptr, nullptr, 0, raw, nullptr);
  }
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

int yond_vst_fwd(const float* bayer, float* z, float* ub, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                 const yond_vst_params* params_dev, const float* rows, const float* xnodes, int row_stride, void* stream) {
  YOND_REQUIRE(params_dev != nullptr, "yond_vst_fwd: params required");
  return launch_fwd(true, bayer, z, ub, B, H, W, pad_l, pad_r, pad_t, pad_b, params_dev, rows, xnodes, row_stride, stream);
}
int yond_vst_fwd_raw16(const uint16_t* raw, const yond_raw_norm* nrm, float* z, float* ub, int B, int H, int W, int pad_l, int pad_r,
                       int pad_t, int pad_b, const yond_vst_params* params_dev, const float* rows, const float* xnodes, int row_stride,
                       void* stream, const yond_raw_norm* nrm_dev, int frames_per_img) {
  YOND_REQUIRE(params_dev != nullptr && raw != nullptr && (nrm != nullptr || nrm_dev != nullptr), "yond_vst_fwd_raw16: null argument");
  YOND_REQUIRE((nrm_dev ? frames_per_img >= 1 : nrm->white > nrm->black) && (uintptr_t)raw % 4 == 0 && W % 2 == 0,
               "yond_vst_fwd_raw16: bad normalisation / alignment");
  return launch_fwd(true, nullptr, z, ub, B, H, W, pad_l, pad_r, pad_t, pad_b, params_dev, rows, xnodes, row_stride, stream,
                    make_raw_norm(raw, nrm, nrm_dev, frames_per_img));
}
int yond_vst_fwd_frames(const yond_frame_geom* frames_dev, const yond_raw_norm* nrm_dev, float* z, float* ub, int B, int H, int W,
                        int pad_l, int pad_r, int pad_t, int pad_b, const yond_vst_params* params_dev, const float* rows,
                        const float* xnodes, int row_stride, void* stream) {
  YOND_REQUIRE(frames_dev != nullptr && params_dev != nullptr, "yond_vst_fwd_frames: null argument");
  RawNorm raw{};
  raw.per_img = nrm_dev;  // uint16 records: the kernel takes each mosaic's address from its record
  raw.units_per_img = 1;
  return launch_fwd(true, nullptr, z, ub, B, H, W, pad_l, pad_r, pad_t, pad_b, params_dev, rows, xnodes, row_stride, stream, raw, frames_dev);
}
int yond_pack_pad(const float* bayer, float* z, float* ub, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                  void* stream) {
  return launch_fwd(false, bayer, z, ub, B, H, W, pad_l, pad_r, pad_t, pad_b, nullptr, nullptr, nullptr, 0, stream);
}

static int launch_inv(bool vst, const float* y, float* bayer, int B, int H, int W, int pl, int pr, int pt, int pb,
                      const yond_vst_params* params, int clip01, const InvPlace& place, void* stream) {
  YOND_REQUIRE(B > 0 && H % 2 == 0 && W % 2 == 0 && H > 0 && W > 0, "vst_inv: H,W must be even");
  YOND_REQUIRE(B <= 65535, "vst_inv: at most 65535 frames per call");
  const int h = H / 2, w = W / 2, hp = h + pt + pb, wp = w + pl + pr;
  int gx = ceil_div(h * w, kBlock * 4);
  if (gx < 1) gx = 1;
  if (gx > 65535) gx = 65535;
  dim3 grid(gx, B);
  cudaStream_t s = (cudaStream_t)stream;
  YondProfScope prof(vst ? "vst_inv" : "crop_unpack", s, 8.0 * (double)B * H * W);
  if (vst) vst_inv_kernel<true><<<grid, kBlock, 0, s>>>(y, bayer, H, W, pl, pt, hp, wp, params, clip01, place);
  else vst_inv_kernel<false><<<grid, kBlock, 0, s>>>(y, bayer, H, W, pl, pt, hp, wp, nullptr, 0, place);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}
int yond_vst_inv(const float* y, float* bayer, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                 const yond_vst_params* params_dev, int clip01, void* stream) {
  YOND_REQUIRE(params_dev != nullptr, "yond_vst_inv: params required");
  return launch_inv(true, y, bayer, B, H, W, pad_l, pad_r, pad_t, pad_b, params_dev, clip01, InvPlace{1, nullptr, 1, nullptr}, stream);
}
int yond_vst_inv_place(const float* y, float* out, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                       const yond_vst_params* params_dev, int clip01, int frames_per_row, int frame0, const int32_t* seg_ok_dev,
                       int frames_per_seg, const float* fallback, void* stream) {
  YOND_REQUIRE(params_dev != nullptr, "yond_vst_inv_place: params required");
  YOND_REQUIRE(frames_per_row >= 1 && frame0 >= 0 && frame0 % frames_per_row == 0 && B % frames_per_row == 0,
               "yond_vst_inv_place: a call covers whole mosaics (B and frame0 multiples of frames_per_row)");
  YOND_REQUIRE(!seg_ok_dev || (frames_per_seg >= 1 && frame0 % frames_per_seg == 0), "yond_vst_inv_place: frame0 must start an image");
  // `out` / `fallback` / `seg_ok_dev` are the buffers of the WHOLE batch; this call covers frames frame0 .. frame0 + B - 1
  const size_t off = (size_t)frame0 * H * W;
  InvPlace place{frames_per_row, seg_ok_dev ? seg_ok_dev + frame0 / frames_per_seg : nullptr, frames_per_seg < 1 ? 1 : frames_per_seg,
                 fallback ? fallback + off : nullptr};
  return launch_inv(true, y, out + off, B, H, W, pad_l, pad_r, pad_t, pad_b, params_dev, clip01, place, stream);
}
int yond_crop_unpack(const float* y, float* bayer, int B, int H, int W, int pad_l, int pad_r, int pad_t, int pad_b,
                     void* stream) {
  return launch_inv(false, y, bayer, B, H, W, pad_l, pad_r, pad_t, pad_b, nullptr, 0, InvPlace{1, nullptr, 1, nullptr}, stream);
}

}  // extern "C"
