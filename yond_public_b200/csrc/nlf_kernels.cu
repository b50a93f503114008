// Noise-level-function estimation kernels (SimpleNLF): box statistics, exact order statistics, the
// 'score3' bin-occupancy count and the masked regression sums.
//   reference: utils/isp_algos.py:234-242 (stdfilt via cv2.blur), :345-365 (polyfit);
//              YOND_SIDD.py:22-49 (get_threshold 'score3'), :62-115 (SelfNLF / CollabNLF).
// cv2.blur on float32 = normalised box, BORDER_REFLECT_101, float64 running sums, result rounded to float32;
// the box kernel below keeps float64 sums (vertical sliding window in registers, horizontal prefix in shared memory).
#include <mutex>

#include "common.cuh"

namespace {

constexpr int kMaxK = 31;

__device__ __forceinline__ float4 sq4(const float4& v) {
  return make_float4(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y), __fmul_rn(v.z, v.z), __fmul_rn(v.w, v.w));
}

// Fused box statistics: one kernel, no float64 scratch in HBM.
// A block owns kCols consecutive columns (output columns + a halo of k/2 on each side) of a strip of rows.  Thread c
// slides a k-tall window down column c (float64 sums of x and of fl32(x*x), 4 channels = NQ running sums).  For each
// row the k-wide horizontal sums come from an inclusive prefix over the block's columns, window(c) = P[c+r] - P[c-r-1],
// computed in shared memory as a chunked scan: warp q owns quantity q, lane j scans the CH = kCols/32 consecutive
// columns of chunk j sequentially, one warp shuffle-scan of the 32 chunk totals gives the offsets.  That is one
// 5-step shuffle scan per quantity and row instead of one per quantity and WARP OF COLUMNS (8x fewer shuffles, ~3x
// fewer instructions than scanning the column sums where they live).  All sums are float64 sums of float32 values,
// so the result equals cv2.blur's float64 accumulation rounded to float32 up to the (far below float32) float64
// rounding of the summation order.  S is double-buffered by row parity: two __syncthreads per row.
// OP_MEAN_VAR: out0 = mean, out1 = std^2 (SelfNLF's var).  OP_VAR: out0 = std^2.  OP_COLLAB: out0 = mean, out1 = std (lap),
// out2 = aux - std^2 with aux = std_k(other frame)^2 (CollabNLF's var), a read-only map that may be out2 itself (in place).
// Squares / difference in float32 with explicit rounding, like the reference's elementwise float32 expressions.
enum { OP_MEAN = 0, OP_MEAN_STD = 1, OP_STD = 2, OP_MEAN_VAR = 3, OP_VAR = 4, OP_COLLAB = 5 };
constexpr int kBoxThreads = 256;
// Where the k x k window reads its pixels from.  kBayer = false: packed frames (B,h,w,4) float32.  kBayer = true: the Bayer
// mosaic itself (two 64-bit loads per packed pixel, rows 2i and 2i+1) — the estimator then needs no pack pass at all — with
// optional SIDD geometry: packed column c of image b lives in block c / blk_w of that image (blocks laid side by side,
// YOND_SIDD.py:315), `blk_stride` floats apart.
struct BoxSrc {
  const float* base;
  long long img_stride;  // floats between images
  long long blk_stride;  // floats between the blocks of an image (Bayer mode)
  int blk_w;             // packed pixels per block row (Bayer mode; = w for plain frames)
  int row_len;           // floats per source row: Bayer W of a block, or 4*w
  float* seg_max;        // optional: per-image maximum of max(x, 0) (atomicMax on the float bits), image = b / imgs_per_seg
  int imgs_per_seg;
  int mosaic_blocks;     // > 0: box-filter image b is block b % n of mosaic b / n (mosaic layout, blocks as separate images)
  RawNorm raw;           // raw.base != nullptr (Bayer mode only): the source is the uint16 sensor mosaic, normalised on load
};
// BORDER_REFLECT_101 for an index at most one image away from the valid range (the filter radius is smaller than the image)
__device__ __forceinline__ int reflect_once(int i, int n) {
  i = i < 0 ? -i : i;
  return i >= n ? 2 * (n - 1) - i : i;
}
// kNarrow: images no wider than half a block (SIDD blocks: 128 packed pixels) — a block then holds 256 / w WHOLE images side
// by side, every thread is a real column (no halo threads), and the reflected border columns are taken from the same
// prefix array: sum over [c-r, c+r] with reflection = P[min(c+r, w-1)] - P[c-r-1] + (P[r-c] - P[0]) on the left edge and
// + (P[w-2] - P[2(w-1)-(c+r)-1]) on the right edge.
// kRows: image rows per barrier round.  Every round a column thread pushes the window down kRows rows (all 2 kRows loads
// of the round are issued up front), stores the kRows sets of column sums, the scan warps prefix kRows x NQ rows of the
// staging array (two at a time, interleaved), the writers emit kRows image rows: three block barriers per kRows rows
// instead of two per row, and kRows-fold more independent work between them.
constexpr int kRows = 4;
template <bool kSq, int kCols, bool kBayer, bool kNarrow>  // kCols = 256, or 160 when a whole row plus both halos fits
__global__ void __launch_bounds__(kBoxThreads) box_fused_kernel(BoxSrc src, float4* __restrict__ out0,
                                                                float4* __restrict__ out1, int B, int h, int w, int k, int op,
                                                                int rows_per_strip, const float4* aux,  // may alias out2
                                                                float4* __restrict__ out2) {
  constexpr int NQ = kSq ? 8 : 4;
  constexpr int CH = kCols / 32;           // columns per scan chunk (8 or 5)
  // Staging rows.  kCols = 256: 16-byte slots (column pairs) XOR-swizzled, slot s -> s ^ ((s >> 3) & 3): 64-bit accesses of 16
  // consecutive aligned columns (the column threads' stores, the writers' upper window end) and the scan's 128-bit accesses of
  // four slots per lane are both bank-conflict free without padding (the padded layout cost every column-indexed access a second
  // wavefront: 4.3 shared-memory wavefronts per pixel, one third of them conflicts).  kCols = 160: padded, column c at c + c / CH.
  constexpr bool kSwz = kCols == 256;
  constexpr int PITCH = kSwz ? kCols : kCols + 32 + 1;
  extern __shared__ __align__(16) double S[];  // [kRows][NQ][PITCH]
  const int r = k / 2;
  const int outc = kCols - 2 * r;
  const int c = threadIdx.x, lane = c & 31, warp = c >> 5;
  int b, col_out, col_src, img0 = 0;
  bool colthread, writer;
  if (kNarrow) {
    const int ipb = kCols / w, il = c / w;  // images per block, this thread's image inside the block
    b = blockIdx.z * ipb + il;
    col_out = col_src = c - il * w;
    img0 = il * w;                           // first column of this image in the block's prefix array
    colthread = writer = il < ipb && b < B;
    if (!colthread) b = B - 1;
  } else {
    b = blockIdx.z;
    col_out = blockIdx.x * outc + (c - r);          // image column this thread's window is centred on
    col_src = reflect101(col_out, w);               // BORDER_REFLECT_101
    colthread = c < kCols;
    writer = (c >= r) && (c < r + outc) && (col_out < w);
  }
  // Wide layout: the thread that WRITES output column oc is thread oc + r, so that its upper window end P[oc + r] sits at its own
  // (aligned) position; only the lower end P[oc - r - 1] is an unaligned access.
  int col_w = col_out;
  if (!kNarrow) {
    col_w = blockIdx.x * outc + (c - 2 * r);
    writer = (c >= 2 * r) && (col_w < w);
  }
  const int i0 = blockIdx.y * rows_per_strip;
  const int i1 = min(h, i0 + rows_per_strip);
  size_t coloff;  // element offset of this thread's column in row 0 of its image
  if (kBayer) {
    const int blk = col_src / src.blk_w;
    coloff = (size_t)b * src.img_stride + (size_t)blk * src.blk_stride + 2 * (col_src - blk * src.blk_w);
    if (src.mosaic_blocks > 0)
      coloff += (size_t)(b / src.mosaic_blocks) * (2 * h) * src.row_len + (size_t)(b % src.mosaic_blocks) * src.blk_stride;
  } else {
    coloff = (size_t)b * src.img_stride + 4 * (size_t)col_src;
  }
  const float* colbase = src.base + coloff;
  const uint16_t* colbase16 = kBayer && src.raw.base ? src.raw.base + coloff : nullptr;
  // per thread: in the narrow layout one block holds images of different dataset images
  const RawNorm rn = kBayer ? raw_norm_at(src.raw, b) : src.raw;
  const uint32_t row_pitch = kBayer ? 2u * (uint32_t)src.row_len : (uint32_t)src.row_len;  // an image stays below 2^32 floats
  float vmax = 0.f;
  double s[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) s[q] = 0.0;
  auto accum = [&](const float4& v, double sign) {
    s[0] += sign * v.x; s[1] += sign * v.y; s[2] += sign * v.z; s[3] += sign * v.w;
    if (kSq) {
      const float4 q2 = sq4(v);
      s[4] += sign * q2.x; s[5] += sign * q2.y; s[6] += sign * q2.z; s[7] += sign * q2.w;
    }
  };
  auto load = [&](int i) {
    const uint32_t roff = (uint32_t)reflect_once(i, h) * row_pitch;
    const float* p = colbase + roff;
    float4 v;
    if (kBayer && colbase16) {  // uint16 mosaic: two 32-bit loads per packed pixel, normalised on load
      const uint32_t a = __ldg(reinterpret_cast<const uint32_t*>(colbase16 + roff));
      const uint32_t d = __ldg(reinterpret_cast<const uint32_t*>(colbase16 + roff + src.row_len));
      v = make_float4(raw_norm(a & 0xffffu, rn), raw_norm(a >> 16, rn), raw_norm(d & 0xffffu, rn), raw_norm(d >> 16, rn));
    } else if (kBayer) {
      const float2 a = __ldg(reinterpret_cast<const float2*>(p)), d = __ldg(reinterpret_cast<const float2*>(p + src.row_len));
      v = make_float4(a.x, a.y, d.x, d.y);
    } else {
      v = __ldg(reinterpret_cast<const float4*>(p));
    }
    return v;
  };
  // every pixel of a column enters the window exactly once: the running maximum rides on the accumulate step (NOT on the
  // load, which would make the load's first use immediate and expose its latency)
  auto enter = [&](const float4& v) {
    accum(v, 1.0);
    if (src.seg_max) vmax = fmaxf(vmax, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
  };
  if (colthread) {  // initial window, loads batched four at a time
    int i = i0 - r;
    for (; i + 3 <= i0 + r; i += 4) {
      const float4 v0 = load(i), v1 = load(i + 1), v2 = load(i + 2), v3 = load(i + 3);
      enter(v0); enter(v1); enter(v2); enter(v3);
    }
    for (; i <= i0 + r; ++i) enter(load(i));
  }
  const double inv = 1.0 / ((double)k * (double)k);
  // stdfilt (isp_algos.py:236-241): float32 square of the blurred image, float32 difference, sqrt; explicit
  // round-to-nearest mul/sub: an FMA contraction would skip the float32 rounding of mean^2 the reference has
  auto sd = [](float e2, float e1) { return sqrtf(fmaxf(__fsub_rn(e2, __fmul_rn(e1, e1)), 0.f)); };
  auto pidx = [](int col) {  // position of block column `col` in a staging row
    return kSwz ? ((((col >> 1) ^ ((col >> 4) & 3)) << 1) | (col & 1)) : col + col / CH;
  };
  const int my_idx = pidx(c);
  // window = P[hi] - P[lo] (+ P[e1] - P[e0] for the reflected part of a border column in the narrow layout); index -1 = "0"
  int hi_idx, lo_idx, e1_idx = -1, e0_idx = -1;
  if (kNarrow) {
    const int hc = min(col_out + r, w - 1), lc = col_out - r - 1;
    hi_idx = pidx(img0 + hc);
    lo_idx = lc >= 0 ? pidx(img0 + lc) : (img0 > 0 ? pidx(img0 - 1) : -1);
    if (col_out - r < 0) {                 // columns -1 .. col-r reflect onto 1 .. r-col
      e1_idx = pidx(img0 + (r - col_out));
      e0_idx = pidx(img0);
    } else if (col_out + r > w - 1) {      // columns w .. col+r reflect onto w-2 .. 2(w-1)-(col+r)
      e1_idx = pidx(img0 + w - 2);
      e0_idx = pidx(img0 + 2 * (w - 1) - (col_out + r) - 1);
    }
  } else {
    hi_idx = pidx(c);
    lo_idx = c - 2 * r - 1 >= 0 ? pidx(c - 2 * r - 1) : -1;
  }
  auto Srow = [&](int j, int q) { return S + (size_t)(j * NQ + q) * PITCH; };
  for (int i = i0; i < i1; i += kRows) {
    const int nr = min(kRows, i1 - i);
    // rows entering / leaving the window for the next kRows positions (the last pair prepares the next round)
    float4 vin[kRows], vout[kRows];
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
      if (colthread && i + j + 1 < i1) {
        vin[j] = load(i + j + 1 + r);
        vout[j] = load(i + j - r);
      }
    }
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
      if (colthread && j < nr) {
#pragma unroll
        for (int q = 0; q < NQ; ++q) Srow(j, q)[my_idx] = s[q];
      }
      if (colthread && i + j + 1 < i1) {
        enter(vin[j]);
        accum(vout[j], -1.0);
      }
    }
    __syncthreads();
    // chunked inclusive scans of the nr x NQ staging rows: task t = (row j, quantity q), two tasks per step per warp
    for (int t0 = warp; t0 < nr * NQ; t0 += 2 * (kBoxThreads / 32)) {
      const int t1 = t0 + kBoxThreads / 32;
      const bool two = t1 < nr * NQ;
      double la[CH], lb[CH];
      double ra = 0.0, rb = 0.0;
      if (kSwz) {  // lane = chunk of 8 columns = 4 swizzled slots, 128-bit accesses
        double2* rowa = reinterpret_cast<double2*>(S + (size_t)t0 * PITCH);
        double2* rowb = reinterpret_cast<double2*>(S + (size_t)(two ? t1 : t0) * PITCH);
        const int x = (lane >> 1) & 3;
#pragma unroll
        for (int j = 0; j < CH / 2; ++j) {
          const double2 va = rowa[(4 * lane + j) ^ x], vb = rowb[(4 * lane + j) ^ x];
          ra += va.x; la[2 * j] = ra; ra += va.y; la[2 * j + 1] = ra;
          rb += vb.x; lb[2 * j] = rb; rb += vb.y; lb[2 * j + 1] = rb;
        }
        double ia = ra, ib = rb;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const double ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
          if (lane >= o) { ia += ta; ib += tb; }
        }
        const double ea = ia - ra, eb = ib - rb;
#pragma unroll
        for (int j = 0; j < CH / 2; ++j) rowa[(4 * lane + j) ^ x] = make_double2(la[2 * j] + ea, la[2 * j + 1] + ea);
        if (two) {
#pragma unroll
          for (int j = 0; j < CH / 2; ++j) rowb[(4 * lane + j) ^ x] = make_double2(lb[2 * j] + eb, lb[2 * j + 1] + eb);
        }
        continue;
      }
      double* rowa = S + (size_t)t0 * PITCH + lane * (CH + 1);  // chunk `lane` starts at column lane*CH, i.e. index lane*CH + lane
      double* rowb = S + (size_t)(two ? t1 : t0) * PITCH + lane * (CH + 1);
#pragma unroll
      for (int j = 0; j < CH; ++j) {
        ra += rowa[j];
        rb += rowb[j];
        la[j] = ra;
        lb[j] = rb;
      }
      double ia = ra, ib = rb;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += ta; ib += tb; }
      }
      const double ea = ia - ra, eb = ib - rb;
#pragma unroll
      for (int j = 0; j < CH; ++j) rowa[j] = la[j] + ea;
      if (two) {
#pragma unroll
        for (int j = 0; j < CH; ++j) rowb[j] = lb[j] + eb;
      }
    }
    __syncthreads();
    if (writer) {
#pragma unroll
      for (int j = 0; j < kRows; ++j) {
        if (j >= nr) break;
        double a[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          const double* Sq = Srow(j, q);
          a[q] = Sq[hi_idx] - (lo_idx >= 0 ? Sq[lo_idx] : 0.0);
          if (kNarrow && e1_idx >= 0) a[q] += Sq[e1_idx] - Sq[e0_idx];
        }
        const size_t o = ((size_t)b * h + (i + j)) * w + col_w;
        const float4 m = make_float4((float)(a[0] * inv), (float)(a[1] * inv), (float)(a[2] * inv), (float)(a[3] * inv));
        if (!kSq || op == OP_MEAN) {
          out0[o] = m;
        } else {
          const float4 m2 = make_float4((float)(a[4] * inv), (float)(a[5] * inv), (float)(a[6] * inv), (float)(a[7] * inv));
          const float4 st = make_float4(sd(m2.x, m.x), sd(m2.y, m.y), sd(m2.z, m.z), sd(m2.w, m.w));
          if (op == OP_MEAN_STD) {
            out0[o] = m;
            out1[o] = st;
          } else if (op == OP_MEAN_VAR) {
            out0[o] = m;
            out1[o] = sq4(st);
          } else if (op == OP_VAR) {
            out0[o] = sq4(st);
          } else if (op == OP_COLLAB) {
            out0[o] = m;
            out1[o] = st;
            const float4 a2 = aux[o], s2 = sq4(st);
            out2[o] = make_float4(__fsub_rn(a2.x, s2.x), __fsub_rn(a2.y, s2.y), __fsub_rn(a2.z, s2.z), __fsub_rn(a2.w, s2.w));
          } else {
            out0[o] = st;
          }
        }
      }
    }
    __syncthreads();  // the staging rows are rewritten by the next round
  }
  if (src.seg_max) {  // values are >= 0: integer order of the bits == float order
    if (!colthread) vmax = 0.f;
    if (kNarrow) {    // a warp may straddle two images
      if (vmax > 0.f) atomicMax(reinterpret_cast<int*>(src.seg_max + b / src.imgs_per_seg), __float_as_int(vmax));
    } else {
      for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
      if (lane == 0 && vmax > 0.f) atomicMax(reinterpret_cast<int*>(src.seg_max + b / src.imgs_per_seg), __float_as_int(vmax));
    }
  }
}

// ------------------------------------------------------------------ exact order statistics (radix select)
// Three counting passes over the data (11 + 11 + 10 key bits), each followed by a one-block-per-segment "select" kernel
// that turns the histogram into the bucket of every queried rank (block prefix sum + binary search).
__device__ __forceinline__ uint32_t f2key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  const uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

constexpr int kMaxRanks = 64;
constexpr int kBins = 1001;  // get_threshold: int(clip(mean,0,1)*1000) -> 1001 bins (YOND_SIDD.py:26,38-41)
struct SelectWork {
  unsigned int hist0[2048];
  unsigned int hist1[kMaxRanks][2048];
  unsigned int hist2[kMaxRanks][1024];
  unsigned int rank_in[kMaxRanks];          // residual rank of each query inside its current bucket
  int slot1_of_prefix[2048];                // top-11-bit prefix -> slot (or -1)
  int q_slot1[kMaxRanks], q_slot2[kMaxRanks];
  uint32_t q_prefix[kMaxRanks];
  int nslot1, nslot2, nq_live;
  unsigned int hist2_hits;                  // elements the third pass will count (sum of the queried 22-bit buckets), set by select1
  int level;  // 1 after select0 (q_prefix = 11 bits), 2 after select1 (22 bits)
};

// Streaming loops keep kUnroll 128-bit loads in flight per thread (one float4 per thread and a dependent shared-memory
// atomic leave ~16 KB in flight per SM against the ~40 KB Little's law asks for).
constexpr int kUnroll = 4;
template <typename F>
__device__ __forceinline__ void stream_f4(const float4* __restrict__ d4, size_t n4, F&& body) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; i + (kUnroll - 1) * stride < n4; i += kUnroll * stride) {
    float4 v[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) v[u] = ldg_stream_f4(d4 + i + u * stride);
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      body(v[u].x); body(v[u].y); body(v[u].z); body(v[u].w);
    }
  }
  for (; i < n4; i += stride) {
    const float4 v = ldg_stream_f4(d4 + i);
    body(v.x); body(v.y); body(v.z); body(v.w);
  }
}

// First level, optionally fused with the score3 bin pass (get_threshold 'score3', YOND_SIDD.py:34-43): npeaks[i] counts
// the `mean` bins that hold a pixel with lap <= ths[i], i.e. the bins whose SMALLEST lap is <= ths[i] — so the pass only
// needs the per-bin minimum of lap and does not depend on the thresholds: it rides along with the first histogram.
template <bool kBinMin>
__global__ void __launch_bounds__(256) hist0_kernel(const float* __restrict__ d, const float* __restrict__ mean, size_t n,
                                                    SelectWork* wk, unsigned int* __restrict__ binmin) {
  d += (size_t)blockIdx.y * n;  // one segment (image) per blockIdx.y
  if (wk) wk += blockIdx.y;
  if (kBinMin) binmin += (size_t)blockIdx.y * 1024;  // smallest lap key per `mean` bin, ~0u = bin empty
  __shared__ unsigned int h[2048];
  __shared__ unsigned int smin[kBinMin ? 1024 : 1];
  for (int i = threadIdx.x; i < 2048; i += blockDim.x) h[i] = 0;
  if (kBinMin)
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) smin[i] = ~0u;
  __syncthreads();
  const float4* d4 = reinterpret_cast<const float4*>(d);  // segments hold 4-channel pixels: n % 4 == 0, 16-byte aligned
  if (!kBinMin) {
    stream_f4(d4, n / 4, [&](float e) { atomicAdd(&h[f2key(e) >> 21], 1u); });
  } else {
    const float4* m4 = reinterpret_cast<const float4*>(mean + (size_t)blockIdx.y * n);
    auto one = [&](float l, float m) {
      const uint32_t k = f2key(l);
      if (wk) atomicAdd(&h[k >> 21], 1u);
      const int bin = (int)__fmul_rn(fminf(fmaxf(m, 0.f), 1.f), 1000.f);
      if (smin[bin] > k) atomicMin(&smin[bin], k);
    };
    const size_t n4 = n / 4, stride = (size_t)gridDim.x * blockDim.x;
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    for (; i + stride < n4; i += 2 * stride) {  // two pixel quads of each map (64 B) in flight per thread
      const float4 l0 = ldg_stream_f4(d4 + i), m0 = ldg_stream_f4(m4 + i);
      const float4 l1 = ldg_stream_f4(d4 + i + stride), m1 = ldg_stream_f4(m4 + i + stride);
      one(l0.x, m0.x); one(l0.y, m0.y); one(l0.z, m0.z); one(l0.w, m0.w);
      one(l1.x, m1.x); one(l1.y, m1.y); one(l1.z, m1.z); one(l1.w, m1.w);
    }
    for (; i < n4; i += stride) {
      const float4 l0 = ldg_stream_f4(d4 + i), m0 = ldg_stream_f4(m4 + i);
      one(l0.x, m0.x); one(l0.y, m0.y); one(l0.z, m0.z); one(l0.w, m0.w);
    }
  }
  __syncthreads();
  if (wk)
    for (int i = threadIdx.x; i < 2048; i += blockDim.x)
      if (h[i]) atomicAdd(&wk->hist0[i], h[i]);
  if (kBinMin)
    for (int i = threadIdx.x; i < kBins; i += blockDim.x)
      if (smin[i] < binmin[i]) atomicMin(&binmin[i], smin[i]);  // plain read first: most blocks have nothing new
}

// Block-wide inclusive prefix sum of a 2048-entry (or shorter) histogram into shared memory; blockDim.x = 1024, each
// thread owns two consecutive entries.
__device__ __forceinline__ void block_prefix(const unsigned int* __restrict__ hist, int nbins, unsigned int* __restrict__ pre,
                                             unsigned int* __restrict__ wsum) {
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const unsigned int a = 2 * t < nbins ? hist[2 * t] : 0u, b = 2 * t + 1 < nbins ? hist[2 * t + 1] : 0u;
  unsigned int incl = a + b;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    unsigned int w = wsum[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int v = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += v;
    }
    wsum[lane] = w;
  }
  __syncthreads();
  const unsigned int off = warp ? wsum[warp - 1] : 0u;
  if (2 * t < nbins) pre[2 * t] = off + incl - b;
  if (2 * t + 1 < nbins) pre[2 * t + 1] = off + incl;
  __syncthreads();
}
// smallest bin with pre[bin] > r (pre inclusive, ascending); *before = elements below that bin
__device__ __forceinline__ int find_bin(const unsigned int* __restrict__ pre, int nbins, unsigned int r, unsigned int* before) {
  int lo = 0, hi = nbins - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (pre[mid] > r) hi = mid; else lo = mid + 1;
  }
  *before = lo ? pre[lo - 1] : 0u;
  return lo;
}

__global__ void __launch_bounds__(1024) select0_kernel(SelectWork* wk, const unsigned long long* __restrict__ ranks, int nranks) {
  wk += blockIdx.x;
  __shared__ unsigned int pre[2048];
  __shared__ unsigned int wsum[32];
  __shared__ int s_bin[kMaxRanks];
  for (int i = threadIdx.x; i < 2048; i += blockDim.x) wk->slot1_of_prefix[i] = -1;
  block_prefix(wk->hist0, 2048, pre, wsum);
  if ((int)threadIdx.x < nranks) {
    const int q = threadIdx.x;
    unsigned int before;
    const int bin = find_bin(pre, 2048, (unsigned int)ranks[q], &before);
    s_bin[q] = bin;
    wk->q_prefix[q] = (uint32_t)bin;
    wk->rank_in[q] = (unsigned int)ranks[q] - before;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int ns = 0;
    for (int q = 0; q < nranks; ++q) {
      const int bin = s_bin[q];
      if (wk->slot1_of_prefix[bin] < 0) wk->slot1_of_prefix[bin] = ns++;
      wk->q_slot1[q] = wk->slot1_of_prefix[bin];
    }
    wk->nslot1 = ns;
    wk->nq_live = nranks;
    wk->level = 1;
  }
}
// Second radix level.  The queried ranks (percentiles 5..95) sit in a handful of top-11-bit buckets that together
// hold most of the data, so nearly every element increments a counter: the counters of the first kHist1Slots buckets
// (slots are handed out in rank order, so these are the dense ones) are privatised in shared memory and flushed once per
// block; later buckets fall back to global atomics.  The pass is bound by the shared-memory atomic rate (one per element).
constexpr int kHist1Slots = 16;
constexpr int kHist1Threads = 1024;
__device__ __forceinline__ void load_slot_table(const SelectWork* wk, signed char* s1tab) {
  // prefix -> slot table from the query list (a handful of entries), not from the 2048-entry global table
  for (int i = threadIdx.x; i < 512; i += blockDim.x) reinterpret_cast<unsigned int*>(s1tab)[i] = 0xffffffffu;
  __syncthreads();
  const int nq = wk->nq_live;
  if ((int)threadIdx.x < nq) s1tab[wk->q_prefix[threadIdx.x] >> ((wk->level - 1) * 11)] = (signed char)wk->q_slot1[threadIdx.x];
}
__global__ void __launch_bounds__(kHist1Threads) hist1_kernel(const float* __restrict__ d, size_t n, SelectWork* wk) {
  extern __shared__ unsigned int hs[];  // [kHist1Slots][2048] counters, then the 2048-entry prefix -> slot table (int8)
  signed char* s1tab = reinterpret_cast<signed char*>(hs + kHist1Slots * 2048);
  d += (size_t)blockIdx.y * n;
  wk += blockIdx.y;
  const int nsh = min(wk->nslot1, kHist1Slots);
  for (int i = threadIdx.x; i < nsh * 2048; i += blockDim.x) hs[i] = 0u;
  load_slot_table(wk, s1tab);
  __syncthreads();
  const uint32_t a_tab = smem_addr(s1tab), a_hs = smem_addr(hs);
  stream_f4(reinterpret_cast<const float4*>(d), n / 4, [=](float e) {
    const uint32_t k = f2key(e);
    const int s = lds_s8(a_tab + (k >> 21));
    if (s >= 0) {
      const uint32_t mid = (k >> 10) & 2047u;
      if (s < kHist1Slots) reds_add(a_hs + 4u * ((uint32_t)s * 2048u + mid));
      else atomicAdd(&wk->hist1[s][mid], 1u);
    }
  });
  __syncthreads();
  for (int i = threadIdx.x; i < nsh * 2048; i += blockDim.x)
    if (hs[i]) atomicAdd(&wk->hist1[i >> 11][i & 2047], hs[i]);
}
// select1 / select2: one WARP per distinct bucket — lane-local sums of the bucket's histogram (64 / 32 entries per lane), a
// warp scan of the lane totals, then the lane that holds a query's rank walks its own entries.
__global__ void __launch_bounds__(1024) select1_kernel(SelectWork* wk, int nranks) {
  wk += blockIdx.x;
  __shared__ int s_bin[kMaxRanks], s_s1[kMaxRanks], s_s2[kMaxRanks];
  __shared__ unsigned int s_rank[kMaxRanks], s_cnt[kMaxRanks];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((int)threadIdx.x < nranks) {
    s_s1[threadIdx.x] = wk->q_slot1[threadIdx.x];
    s_rank[threadIdx.x] = wk->rank_in[threadIdx.x];
  }
  __syncthreads();
  const int ns1 = wk->nslot1;
  extern __shared__ unsigned int stage[];  // [16 warps][2048 + 32]: entry e of a bucket sits at e + e / 64 (conflict-free lane rows)
  for (int s0 = 0; s0 < ns1; s0 += 16) {
    const int s1 = s0 + warp;
    if (warp < 16 && s1 < ns1) {
      const unsigned int* hist = wk->hist1[s1];
      unsigned int* st = stage + warp * (2048 + 32);
#pragma unroll 8
      for (int j = 0; j < 64; ++j) st[j * 32 + lane + ((j * 32 + lane) >> 6)] = hist[j * 32 + lane];  // coalesced
      __syncwarp();
      const unsigned int* mine = st + lane * 65;
      unsigned int tot = 0;
#pragma unroll 8
      for (int j = 0; j < 64; ++j) tot += mine[j];
      unsigned int incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      const unsigned int lane_excl = incl - tot;
      for (int q = 0; q < nranks; ++q) {
        if (s_s1[q] != s1) continue;  // uniform across the warp
        const unsigned int r = s_rank[q];
        const unsigned int m = __ballot_sync(0xffffffffu, lane_excl <= r);
        const int owner = 31 - __clz(m);
        if (lane == owner) {
          unsigned int run = lane_excl;
          int j = 0;
          for (; j < 63; ++j) {
            const unsigned int v = mine[j];
            if (run + v > r) break;
            run += v;
          }
          const int bin = lane * 64 + j;
          s_bin[q] = bin;
          s_cnt[q] = mine[j];
          wk->q_prefix[q] = (wk->q_prefix[q] << 11) | (uint32_t)bin;
          wk->rank_in[q] = r - run;
        }
        __syncwarp();
      }
    }
    __syncthreads();
  }
  __syncthreads();
  if (threadIdx.x == 0) {  // queries sharing (bucket, bin) share a third-level histogram
    int ns = 0;
    unsigned long long hits = 0;
    for (int q = 0; q < nranks; ++q) {
      int found = -1;
      for (int p = 0; p < q && found < 0; ++p)
        if (s_s1[p] == s_s1[q] && s_bin[p] == s_bin[q]) found = s_s2[p];
      s_s2[q] = found >= 0 ? found : ns++;
      wk->q_slot2[q] = s_s2[q];
      if (found < 0) hits += s_cnt[q];
    }
    wk->hist2_hits = hits > 0xffffffffull ? 0xffffffffu : (unsigned int)hits;
    wk->nslot2 = ns;
    wk->level = 2;
  }
}
// Third radix level.  Only elements whose upper 22 bits equal one of the <= 64 queried prefixes count (~0.2 % of the
// data): the membership test runs against shared memory (prefix -> slot table + one 2048-bit map per first-level slot),
// a hit looks its slot up in the query list and takes a global atomic.
// Hits are rare on natural data, but a frame with a saturated / black region has `lap` == 0 over a large area and then millions of
// elements fall into ONE (slot, bin): the hit path therefore aggregates per warp (match.any: one atomic per distinct counter and warp)
// into a per-block copy of the first kHist2Slots slots in shared memory, flushed once — instead of one global atomic per element on a
// single address (measured: see DESIGN.md).
// Both forms are launched; select1 has counted how many elements the pass will hit (`hist2_hits`) and each form returns at once when
// the other one is due: sparse hits (natural data: ~0.2 %) take the lean form with 6 blocks per SM, dense hits the privatised one.
constexpr int kHist2Slots = 16;
__device__ __forceinline__ bool hist2_dense(const SelectWork* wk, size_t n) { return (size_t)wk->hist2_hits > n / 16; }
template <bool privatise>
__global__ void __launch_bounds__(256) hist2_kernel(const float* __restrict__ d, size_t n, SelectWork* wk) {
  extern __shared__ unsigned int hs2[];  // [kHist2Slots][1024] when privatise
  if (hist2_dense(wk + blockIdx.y, n) != privatise) return;
  __shared__ signed char s1tab[2048];
  __shared__ unsigned int bm[kMaxRanks * 64];
  __shared__ uint32_t qpre[kMaxRanks];
  __shared__ int qs2[kMaxRanks];
  __shared__ int nq;
  d += (size_t)blockIdx.y * n;
  wk += blockIdx.y;
  const int ns1 = wk->nslot1;
  const int nsh = privatise ? min(wk->nslot2, kHist2Slots) : 0;
  for (int i = threadIdx.x; i < ns1 * 64; i += blockDim.x) bm[i] = 0u;
  for (int i = threadIdx.x; i < nsh * 1024; i += blockDim.x) hs2[i] = 0u;
  if (threadIdx.x == 0) nq = wk->nq_live;
  load_slot_table(wk, s1tab);
  __syncthreads();
  if ((int)threadIdx.x < nq) {
    const uint32_t pre = wk->q_prefix[threadIdx.x];  // (top 11 bits << 11) | middle 11 bits
    const uint32_t mid = pre & 2047u;
    qpre[threadIdx.x] = pre;
    qs2[threadIdx.x] = wk->q_slot2[threadIdx.x];
    atomicOr(&bm[wk->q_slot1[threadIdx.x] * 64 + (mid >> 5)], 1u << (mid & 31u));
  }
  __syncthreads();
  const uint32_t a_tab = smem_addr(s1tab), a_bm = smem_addr(bm), a_qpre = smem_addr(qpre), a_qs2 = smem_addr(qs2);
  const uint32_t a_hs2 = smem_addr(hs2);
  const int nq_r = nq;
  stream_f4(reinterpret_cast<const float4*>(d), n / 4, [=](float e) {
    const uint32_t k = f2key(e);
    const int s1 = lds_s8(a_tab + (k >> 21));
    if (s1 < 0) return;
    const uint32_t mid = (k >> 10) & 2047u;
    if (!((lds_u32(a_bm + 4u * ((uint32_t)s1 * 64u + (mid >> 5))) >> (mid & 31u)) & 1u)) return;
    const uint32_t p22 = k >> 10;
    int slot = -1;
    for (int q = 0; q < nq_r; ++q)
      if (lds_u32(a_qpre + 4u * q) == p22) {
        slot = (int)lds_u32(a_qs2 + 4u * q);
        break;
      }
    if (slot < 0) return;
    if (!privatise) {
      atomicAdd(&wk->hist2[slot][k & 1023u], 1u);
      return;
    }
    const uint32_t key = ((uint32_t)slot << 10) | (k & 1023u);
    const unsigned m = __match_any_sync(__activemask(), key);  // the lanes that are here together with the same counter
    if ((int)(threadIdx.x & 31) == __ffs(m) - 1) {
      if (slot < nsh) reds_add(a_hs2 + 4u * key, (unsigned)__popc(m));
      else atomicAdd(&wk->hist2[slot][k & 1023u], (unsigned)__popc(m));
    }
  });
  if (nsh) {
    __syncthreads();
    for (int i = threadIdx.x; i < nsh * 1024; i += blockDim.x)
      if (hs2[i]) atomicAdd(&wk->hist2[i >> 10][i & 1023], hs2[i]);
  }
}
__global__ void __launch_bounds__(1024) select2_kernel(SelectWork* wk, int nranks, float* __restrict__ out) {
  wk += blockIdx.x;
  out += (size_t)blockIdx.x * nranks;
  __shared__ int s_s2[kMaxRanks];
  if ((int)threadIdx.x < nranks) s_s2[threadIdx.x] = wk->q_slot2[threadIdx.x];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ns2 = wk->nslot2;
  for (int s2 = warp; s2 < ns2; s2 += 32) {
    const unsigned int* hist = wk->hist2[s2];
    unsigned int tot = 0;
#pragma unroll 8
    for (int j = 0; j < 32; ++j) tot += hist[lane * 32 + j];
    unsigned int incl = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    const unsigned int lane_excl = incl - tot;
    for (int q = 0; q < nranks; ++q) {
      if (s_s2[q] != s2) continue;
      const unsigned int r = wk->rank_in[q];
      const unsigned int m = __ballot_sync(0xffffffffu, lane_excl <= r);
      const int owner = 31 - __clz(m);
      if (lane == owner) {
        unsigned int run = lane_excl;
        int j = 0;
        for (; j < 31; ++j) {
          const unsigned int v = hist[lane * 32 + j];
          if (run + v > r) break;
          run += v;
        }
        out[q] = key2f((wk->q_prefix[q] << 10) | (uint32_t)(lane * 32 + j));
      }
      __syncwarp();
    }
  }
}

// ------------------------------------------------------------------ score3 bin occupancy
// npeaks[s][i] = #bins whose smallest lap is <= ths[s][i]  ((double)lap <= th, like the reference's float32 <= float64)
__global__ void score3_count_kernel(const unsigned int* __restrict__ binmin, const double* __restrict__ ths, int nth,
                                    int* __restrict__ npeaks) {
  binmin += (size_t)blockIdx.x * 1024;
  ths += (size_t)blockIdx.x * nth;
  npeaks += (size_t)blockIdx.x * nth;
  __shared__ int cnt[33];
  if (threadIdx.x < 33) cnt[threadIdx.x] = 0;
  __syncthreads();
  for (int b = threadIdx.x; b < kBins; b += blockDim.x) {
    const unsigned int k = binmin[b];
    if (k == ~0u) continue;
    const double l = (double)key2f(k);
    int j = 0;
    while (j < nth && !(l <= ths[j])) ++j;  // ths ascending: index of the first threshold that admits the bin
    if (j < nth) atomicAdd(&cnt[j], 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int c = 0;
    for (int i = 0; i < nth; ++i) {
      c += cnt[i];
      npeaks[i] = c;
    }
  }
}

// ------------------------------------------------------------------ masked regression sums
__global__ void __launch_bounds__(256) masked_sums_kernel(const float* __restrict__ lap, const float* __restrict__ mean,
                                                          const float* __restrict__ var, size_t n,
                                                          const double* __restrict__ ths, double* __restrict__ sums,
                                                          const int* __restrict__ active) {
  if (active && !active[blockIdx.y]) return;  // second pass of the device-side estimator: only the segments that redo
  lap += (size_t)blockIdx.y * n;
  mean += (size_t)blockIdx.y * n;
  var += (size_t)blockIdx.y * n;
  sums += (size_t)blockIdx.y * 12;
  const double th = ths[blockIdx.y];
  double s[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) s[i] = 0.0;
  const float4* l4 = reinterpret_cast<const float4*>(lap);
  const float4* m4 = reinterpret_cast<const float4*>(mean);
  const float4* v4 = reinterpret_cast<const float4*>(var);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n / 4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 lv = ldg_stream_f4(l4 + i), mv = ldg_stream_f4(m4 + i), vv = ldg_stream_f4(v4 + i);
    const float le[4] = {lv.x, lv.y, lv.z, lv.w}, me[4] = {mv.x, mv.y, mv.z, mv.w}, ve[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if ((double)le[e] < th) {
        const float xf = me[e];
        const double x = xf, y = ve[e];
        s[0] += 1.0; s[1] += x; s[2] += y; s[3] += x * x; s[4] += x * y; s[5] += y * y;
        if (xf > 1e-4f && xf < 0.8f) {
          s[6] += 1.0; s[7] += x; s[8] += y; s[9] += x * x; s[10] += x * y; s[11] += y * y;
        }
      }
    }
  }
  __shared__ double red[8][12];
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    double v = s[i];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    double v = 0;
    for (int wq = 0; wq < 8; ++wq) v += red[wq][threadIdx.x];
    atomicAdd(&sums[threadIdx.x], v);
  }
}

// ------------------------------------------------------------------ device-resident estimator tail
// Everything the reference does on a few dozen scalars per image after the maps (YOND_SIDD.py:22-49 np.percentile lerp,
// score, argmin; :77-84 empty-mask fallback; utils/isp_algos.py:345-365 polyfit) as tiny float64 kernels, so that the
// estimate never leaves the GPU.  Arithmetic follows NumPy operation by operation (explicit round-to-nearest mul / add /
// div: no FMA contraction), so thresholds are the same doubles np.percentile computes (oracle/yond_oracle.py).
constexpr int kMaxQ = 24;
struct QuantList {
  int nq;
  double q[kMaxQ];
};
// np.percentile(method='linear'): virtual index (n-1)*q/100, bracketing order statistics, gamma (numpy _quantile).
// ranks: [lo_0..lo_nq | hi_0..hi_nq] with entry nq = the 25th percentile of the empty-mask fallback (:82).
__global__ void ranks_kernel(QuantList ql, unsigned long long n, unsigned long long* __restrict__ ranks, double* __restrict__ gamma) {
  const int i = threadIdx.x;
  if (i > ql.nq) return;
  const double q = i < ql.nq ? ql.q[i] : 25.0;
  const double vi = __dmul_rn((double)(n - 1), __ddiv_rn(q, 100.0));
  const double lo = floor(vi);
  unsigned long long l = (unsigned long long)lo, h = l + 1;
  if (h > n - 1) h = n - 1;
  ranks[i] = l;
  ranks[ql.nq + 1 + i] = h;
  gamma[i] = __dsub_rn(vi, lo);
}
// numpy _lerp: float32 difference, float64 interpolation, the b - diff*(1-t) form for t >= 0.5
__device__ __forceinline__ double np_lerp(float a, float b, double t) {
  const double diff = (double)__fsub_rn(b, a);
  if (t >= 0.5) return __dsub_rn((double)b, __dmul_rn(diff, __dsub_rn(1.0, t)));
  return __dadd_rn((double)a, __dmul_rn(diff, t));
}
__global__ void pct_kernel(const float* __restrict__ stats, const double* __restrict__ gamma, int nq, double* __restrict__ ths,
                           double* __restrict__ th25) {
  const int s = blockIdx.x, i = threadIdx.x;
  if (i > nq) return;
  const float* st = stats + (size_t)s * (2 * (nq + 1));
  const double v = np_lerp(st[i], st[nq + 1 + i], gamma[i]);
  if (i < nq) ths[(size_t)s * nq + i] = v;
  else th25[s] = v;
}
// score = ths / (quants * npeaks); i = argmin(score[1:]) + 1 (np.argmin: first minimum, a NaN wins)  — YOND_SIDD.py:45-48
__global__ void pick_kernel(QuantList ql, const double* __restrict__ ths, const int* __restrict__ npeaks, double* __restrict__ th,
                            int* __restrict__ idx_out, int nseg) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  int best = 1;
  double bs = 0.0;
  for (int i = 1; i < ql.nq; ++i) {
    const double sc = __ddiv_rn(ths[(size_t)s * ql.nq + i], __dmul_rn(ql.q[i], (double)npeaks[(size_t)s * ql.nq + i]));
    if (i == 1 || sc < bs || (sc != sc && bs == bs)) {
      best = i;
      bs = sc;
    }
    if (bs != bs) break;
  }
  if (ql.nq == 1) best = 0;
  th[s] = ths[(size_t)s * ql.nq + best];
  idx_out[s] = best;
}
// Empty mask (YOND_SIDD.py:77-84): redo with the 25th percentile when it differs from th; when it does not, the
// reference keeps the unmasked maps (fit over every pixel: threshold +inf).
__global__ void backup_kernel(const double* __restrict__ sums, const double* __restrict__ th, const double* __restrict__ th25,
                              double* __restrict__ th2, int* __restrict__ redo, double* __restrict__ sums2, int nseg) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  const bool empty = sums[(size_t)s * 12] == 0.0;
  redo[s] = empty ? 1 : 0;
  th2[s] = !empty ? th[s] : (th[s] != th25[s] ? th25[s] : __longlong_as_double(0x7ff0000000000000LL));
  for (int i = 0; i < 12; ++i) sums2[(size_t)s * 12 + i] = 0.0;
}
// polyfit (isp_algos.py:348-364): the 1e-4 < x < 0.8 subset when it holds more than 1 % of the points, then the least
// squares line through the normal equations in float64.
__global__ void solve_kernel(const double* __restrict__ sums, const double* __restrict__ sums2, const int* __restrict__ redo,
                             const double* __restrict__ th2, const int* __restrict__ idx, const double* __restrict__ ths,
                             const int* __restrict__ npeaks, QuantList ql, double* __restrict__ regs, double* __restrict__ detail,
                             int nseg) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  const double* a = (redo[s] ? sums2 : sums) + (size_t)s * 12;
  const double* u = a[6] > 0.01 * a[0] ? a + 6 : a;
  const double N = u[0], Sx = u[1], Sy = u[2], Sxx = u[3], Sxy = u[4];
  const double det = N * Sxx - Sx * Sx;
  const double b1 = (N * Sxy - Sx * Sy) / det;
  regs[2 * s] = b1;
  regs[2 * s + 1] = (Sy - b1 * Sx) / N;
  if (detail) {
    double* d = detail + (size_t)s * (4 + 2 * kMaxQ);
    d[0] = th2[s];
    d[1] = (double)idx[s];
    d[2] = ql.q[idx[s]];
    d[3] = (double)redo[s];
    for (int i = 0; i < ql.nq; ++i) {
      d[4 + i] = ths[(size_t)s * ql.nq + i];
      d[4 + kMaxQ + i] = (double)npeaks[(size_t)s * ql.nq + i];
    }
  }
}

inline int stream_grid(size_t n) {
  size_t g = (n + 256 * 16 - 1) / (256 * 16);
  const size_t cap = (size_t)yond_num_sms() * 8;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

BoxSrc packed_src(const float* x, int h, int w) {
  BoxSrc s{};
  s.base = x;
  s.img_stride = (long long)h * w * 4;
  s.blk_w = w;
  s.row_len = 4 * w;
  s.imgs_per_seg = 1;
  return s;
}

template <bool SQ, int COLS, bool BAYER, bool NARROW>
int launch_box(dim3 g, cudaStream_t s, const BoxSrc& src, float4* o0, float4* o1, int B, int h, int w, int k, int op, int rows_per_strip,
               const float4* ax, float4* o2) {
  constexpr size_t bytes = (size_t)kRows * (SQ ? 8 : 4) * (COLS == 256 ? COLS : COLS + 33) * sizeof(double);  // = [kRows][NQ][PITCH]
  static std::once_flag once;
  static cudaError_t err = cudaSuccess;
  std::call_once(once, [] {
    err = cudaFuncSetAttribute(box_fused_kernel<SQ, COLS, BAYER, NARROW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  });
  if (err != cudaSuccess) return yond_set_error(YOND_ERR_CUDA, "box filter: cudaFuncSetAttribute failed: %s", cudaGetErrorString(err));
  box_fused_kernel<SQ, COLS, BAYER, NARROW><<<g, kBoxThreads, bytes, s>>>(src, o0, o1, B, h, w, k, op, rows_per_strip, ax, o2);
  return YOND_OK;
}

int box_pass(const BoxSrc& src, bool bayer, float* out0, float* out1, int B, int h, int w, int k, bool with_sq, int op,
             cudaStream_t s, const float* aux = nullptr, float* out2 = nullptr) {
  const int r = k / 2;
  // narrow images (SIDD blocks): 256 / w whole images per block, no halo threads; needs a single reflection (r < w - 1)
  const bool multi = 2 * w <= 256 && w >= 2 * r + 2;
  const bool narrow = !multi && w + 2 * r <= 160;
  const int rows_per_strip = 64;
  const int cols = narrow ? 160 : 256;
  const int outc = cols - 2 * r;
  dim3 g(ceil_div(w, outc), ceil_div(h, rows_per_strip), B);
  if (multi) g = dim3(1, ceil_div(h, rows_per_strip), ceil_div(B, 256 / w));
  YOND_REQUIRE(g.z <= 65535, "box filter: at most 65535 images per call");
  float4* o0 = reinterpret_cast<float4*>(out0);
  float4* o1 = reinterpret_cast<float4*>(out1);
  const float4* ax = reinterpret_cast<const float4*>(aux);
  float4* o2 = reinterpret_cast<float4*>(out2);
  const int opx = with_sq ? op : OP_MEAN;
#define YOND_BOX(SQ, COLS, BAYER, NARROW) \
  rc = launch_box<SQ, COLS, BAYER, NARROW>(g, s, src, o0, o1, B, h, w, k, opx, rows_per_strip, ax, o2)
#define YOND_BOX_B(SQ, COLS, NARROW)                        \
  do {                                                      \
    if (bayer) YOND_BOX(SQ, COLS, true, NARROW);            \
    else YOND_BOX(SQ, COLS, false, NARROW);                 \
  } while (0)
  int rc = YOND_OK;
  if (with_sq) {
    if (multi) YOND_BOX_B(true, 256, true);
    else if (narrow) YOND_BOX_B(true, 160, false);
    else YOND_BOX_B(true, 256, false);
  } else {
    if (multi) YOND_BOX_B(false, 256, true);
    else if (narrow) YOND_BOX_B(false, 160, false);
    else YOND_BOX_B(false, 256, false);
  }
#undef YOND_BOX_B
#undef YOND_BOX
  if (rc) return rc;
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

// CollabNLF's maps from a cached std_k(lr)^2 map `lr_var` in the same geometry (read only; may be `var` itself): the one box pass over
// the denoised frame y.  var = lr_var - std_k(y)^2, mean = blur_k(y), lap = std_k(y).
int collab_from_lr_var(const BoxSrc& y, bool bayer, const float* lr_var, float* var, float* mean, float* lap, int B, int h, int w, int k,
                       cudaStream_t s) {
  return box_pass(y, bayer, mean, lap, B, h, w, k, true, OP_COLLAB, s, lr_var, var);
}

// Maps of SelfNLF / CollabNLF from either source kind
int nlf_maps_impl(const BoxSrc& x, const BoxSrc* y, bool bayer, float* var, float* mean, float* lap, int B, int h, int w, int k, int mode,
                  void* work, cudaStream_t s) {
  const size_t n = (size_t)B * h * w * 4;
  float* tmpA = reinterpret_cast<float*>(work);
  float* tmpB = tmpA + n;
  int rc;
  // algorithmic bytes per Bayer pixel (SURVEY 8d): self 4 R + 12 W (lap, mean, var), collab 8 R + 12 W, lr var 4 R + 4 W
  // Indexed by mode; there is no mode 2, so modes 1 and 3 keep the numbers of the C entry points.
  static const char* names[4] = {"nlf_maps_self (3 box_fused passes)", "nlf_maps_collab (2 box_fused passes)", nullptr,
                                 "nlf_maps_lr_var (1 box_fused pass)"};
  static const double bytes[4] = {16.0, 20.0, 0.0, 8.0};
  YondProfScope prof(names[mode], s, bytes[mode] * (double)n);
  BoxSrc x_nomax = x;
  x_nomax.seg_max = nullptr;
  if (mode == 0) {
    // mean = blur_k(x), var = std_k(x)^2 in one pass
    if ((rc = box_pass(x, bayer, mean, var, B, h, w, k, true, OP_MEAN_VAR, s))) return rc;
    // lap = std_k(blur_k2(x)), k2 = k//3*2+1 (YOND_SIDD.py:70)
    const int k2 = k / 3 * 2 + 1;
    if ((rc = box_pass(x_nomax, bayer, tmpB, nullptr, B, h, w, k2, false, OP_MEAN, s))) return rc;
    if ((rc = box_pass(packed_src(tmpB, h, w), false, lap, nullptr, B, h, w, k, true, OP_STD, s))) return rc;
  } else if (mode == 3) {
    // var = std_k(x)^2 alone: the cached lr statistics of the collab rounds (mean / lap untouched)
    if ((rc = box_pass(x, bayer, var, nullptr, B, h, w, k, true, OP_VAR, s))) return rc;
  } else {
    // std_k(lr)^2 -> tmpA ; mean = blur_k(hr), lap = std_k(hr) ; var = std_lr^2 - std_hr^2
    if ((rc = box_pass(x, bayer, tmpA, nullptr, B, h, w, k, true, OP_VAR, s))) return rc;
    if ((rc = collab_from_lr_var(*y, bayer, tmpA, var, mean, lap, B, h, w, k, s))) return rc;
  }
  return YOND_OK;
}

// Bayer inputs of the box filters: `nimg` images of `nblk` blocks of (H,W), blocks layout (nimg,nblk,H,W) or mosaic layout
// (nimg,H,nblk*W).  split_blocks = 1: every block is its own image for the box filters (SIDD_256, YOND_SIDD.py:65,91-93);
// split_blocks = 0: the nblk blocks of an image form one mosaic (:315), h x (nblk*w) packed pixels.  With split_blocks the
// box-filter image index runs over blocks, and a block's origin in a mosaic is not a multiple of the image stride: it is folded
// into per-image / per-block strides.
BoxSrc bayer_src(const float* base, int mosaic, int nblk, int H, int W, int split_blocks) {
  BoxSrc d{};
  d.base = base;
  d.blk_w = W / 2;
  d.imgs_per_seg = split_blocks ? nblk : 1;
  if (!mosaic) {
    d.row_len = W;
    d.blk_stride = (long long)H * W;
    d.img_stride = split_blocks ? (long long)H * W : (long long)nblk * H * W;
  } else {
    d.row_len = nblk * W;
    d.blk_stride = W;
    d.img_stride = split_blocks ? 0 : (long long)nblk * H * W;  // split_blocks: see box kernel (image b = mosaic b / nblk, block b % nblk)
    d.mosaic_blocks = split_blocks ? nblk : 0;
  }
  return d;
}

}  // namespace

extern "C" {

size_t yond_nlf_work_bytes(int B, int h, int w, int C) {
  (void)C;
  const size_t npix = (size_t)B * h * w;
  // two float32x4 temporaries (blur_k2(x) / std of the first input)
  return 2 * npix * sizeof(float4) + 4096;
}

int yond_box_blur(const float* x, float* out, int B, int h, int w, int C, int k, int square_input, void* work, void* stream) {
  (void)work;
  YOND_REQUIRE(C == 4, "yond_box_blur: packed 4-channel frames only (pass SIDD block stacks as a batch)");
  YOND_REQUIRE(k % 2 == 1 && k >= 1 && k <= kMaxK, "yond_box_blur: odd k <= %d required (got %d)", kMaxK, k);
  YOND_REQUIRE(h > k / 2 && w > k / 2, "yond_box_blur: frame smaller than the filter radius");
  YOND_REQUIRE(square_input == 0, "yond_box_blur: square_input is not supported");
  return box_pass(packed_src(x, h, w), false, out, nullptr, B, h, w, k, false, OP_MEAN, (cudaStream_t)stream);
}

int yond_nlf_maps(const float* x, const float* y, float* var, float* mean, float* lap, int B, int h, int w, int C, int k,
                  int mode, void* work, void* stream) {
  YOND_REQUIRE(C == 4, "yond_nlf_maps: packed 4-channel frames only (pass SIDD block stacks as a batch)");
  YOND_REQUIRE(k % 2 == 1 && k >= 3 && k <= kMaxK, "yond_nlf_maps: odd k <= %d required (got %d)", kMaxK, k);
  YOND_REQUIRE(h > k / 2 && w > k / 2, "yond_nlf_maps: frame smaller than the filter radius");
  YOND_REQUIRE(mode == 0 || (mode == 1 && y != nullptr), "yond_nlf_maps: collab mode needs the second input");
  const BoxSrc xs = packed_src(x, h, w), ys = packed_src(y, h, w);
  return nlf_maps_impl(xs, &ys, false, var, mean, lap, B, h, w, k, mode, work, (cudaStream_t)stream);
}

static int nlf_maps_bayer_impl(const float* x, const uint16_t* x16, const yond_raw_norm* nrm, const yond_raw_norm* nrm_dev, int x_mosaic,
                               const float* y, int y_mosaic, float* var, float* mean, float* lap, int nimg, int nblk, int H, int W,
                               int split_blocks, int k, int mode, float* seg_max, void* work, void* stream) {
  YOND_REQUIRE((x || x16) && var && (mode == 3 || (mean && lap)) && work, "yond_nlf_maps_bayer: null argument");
  YOND_REQUIRE(!x16 || ((nrm_dev || (nrm && nrm->white > nrm->black)) && (uintptr_t)x16 % 4 == 0),
               "yond_nlf_maps_raw16: normalisation / 4-byte aligned mosaic required");
  YOND_REQUIRE(nimg > 0 && nblk > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "yond_nlf_maps_bayer: H,W must be even");
  YOND_REQUIRE(k % 2 == 1 && k >= 3 && k <= kMaxK, "yond_nlf_maps_bayer: odd k <= %d required (got %d)", kMaxK, k);
  YOND_REQUIRE(mode == 0 || mode == 3 || (mode == 1 && y != nullptr), "yond_nlf_maps_bayer: mode 0, 1 or 3, the collab mode needs the second input");
  YOND_REQUIRE((!x || (uintptr_t)x % 8 == 0) && (!y || (uintptr_t)y % 8 == 0), "yond_nlf_maps_bayer: 8-byte aligned frames required");
  cudaStream_t s = (cudaStream_t)stream;
  const int h = H / 2, wb = W / 2;
  const int B = split_blocks ? nimg * nblk : nimg;
  const int w = split_blocks ? wb : nblk * wb;
  YOND_REQUIRE(h > k / 2 && w > k / 2, "yond_nlf_maps_bayer: frame smaller than the filter radius");
  YOND_REQUIRE(B <= 65535, "yond_nlf_maps_bayer: at most 65535 images per call");
  BoxSrc xs = bayer_src(x, x_mosaic, nblk, H, W, split_blocks);
  xs.raw = make_raw_norm(x16, nrm, nrm_dev, xs.imgs_per_seg);  // box-filter image b is dataset image b / imgs_per_seg
  xs.seg_max = seg_max;
  if (seg_max) YOND_CUDA_CHECK(cudaMemsetAsync(seg_max, 0, sizeof(float) * nimg, s));
  BoxSrc ys = bayer_src(y, y_mosaic, nblk, H, W, split_blocks);
  return nlf_maps_impl(xs, &ys, true, var, mean, lap, B, h, w, k, mode, work, s);
}
int yond_nlf_maps_bayer(const float* x, int x_mosaic, const float* y, int y_mosaic, float* var, float* mean, float* lap, int nimg,
                        int nblk, int H, int W, int split_blocks, int k, int mode, float* seg_max, void* work, void* stream) {
  YOND_REQUIRE(x != nullptr, "yond_nlf_maps_bayer: null argument");
  return nlf_maps_bayer_impl(x, nullptr, nullptr, nullptr, x_mosaic, y, y_mosaic, var, mean, lap, nimg, nblk, H, W, split_blocks, k, mode,
                             seg_max, work, stream);
}
int yond_nlf_maps_raw16(const uint16_t* x, const yond_raw_norm* nrm, int x_mosaic, const float* y, int y_mosaic, float* var, float* mean,
                        float* lap, int nimg, int nblk, int H, int W, int split_blocks, int k, int mode, float* seg_max, void* work,
                        void* stream) {
  YOND_REQUIRE(x != nullptr && nrm != nullptr, "yond_nlf_maps_raw16: null argument");
  return nlf_maps_bayer_impl(nullptr, x, nrm, nullptr, x_mosaic, y, y_mosaic, var, mean, lap, nimg, nblk, H, W, split_blocks, k, mode,
                             seg_max, work, stream);
}
int yond_nlf_maps_raw16_per_image(const uint16_t* x, const yond_raw_norm* nrm_dev, int x_mosaic, const float* y, int y_mosaic,
                                  float* var, float* mean, float* lap, int nimg, int nblk, int H, int W, int split_blocks, int k,
                                  int mode, float* seg_max, void* work, void* stream) {
  YOND_REQUIRE(x != nullptr && nrm_dev != nullptr, "yond_nlf_maps_raw16_per_image: null argument");
  return nlf_maps_bayer_impl(nullptr, x, nullptr, nrm_dev, x_mosaic, y, y_mosaic, var, mean, lap, nimg, nblk, H, W, split_blocks, k, mode,
                             seg_max, work, stream);
}

int yond_nlf_maps_collab_cached(const float* y, int y_mosaic, const float* lr_var, float* var, float* mean, float* lap, int nimg, int nblk,
                                int H, int W, int split_blocks, int k, void* stream) {
  YOND_REQUIRE(y && lr_var && var && mean && lap, "yond_nlf_maps_collab_cached: null argument");
  YOND_REQUIRE(nimg > 0 && nblk > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "yond_nlf_maps_collab_cached: H,W must be even");
  YOND_REQUIRE(k % 2 == 1 && k >= 3 && k <= kMaxK, "yond_nlf_maps_collab_cached: odd k <= %d required (got %d)", kMaxK, k);
  YOND_REQUIRE((uintptr_t)y % 8 == 0 && (uintptr_t)lr_var % 16 == 0, "yond_nlf_maps_collab_cached: aligned buffers required");
  const int h = H / 2, wb = W / 2;
  const int B = split_blocks ? nimg * nblk : nimg;
  const int w = split_blocks ? wb : nblk * wb;
  YOND_REQUIRE(h > k / 2 && w > k / 2, "yond_nlf_maps_collab_cached: frame smaller than the filter radius");
  YOND_REQUIRE(B <= 65535, "yond_nlf_maps_collab_cached: at most 65535 images per call");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)B * h * w * 4;
  YondProfScope prof("nlf_maps_collab (1 box_fused pass, lr statistics reused)", s, 20.0 * (double)n);
  return collab_from_lr_var(bayer_src(y, y_mosaic, nblk, H, W, split_blocks), true, lr_var, var, mean, lap, B, h, w, k, s);
}

}  // extern "C"

namespace {
// data = lap; the first counting pass also collects the per-bin minimum of lap over the `mean` bins (score3) into `binmin`
int order_stats_impl(const float* data, const float* mean, unsigned int* binmin, size_t seg_len, int nseg, const uint64_t* ranks_dev,
                     int nranks, float* out_dev, void* work, cudaStream_t s) {
  SelectWork* wk = reinterpret_cast<SelectWork*>(work);
  // one memset for all segments (the slot tables behind the histograms are rewritten by the select kernels anyway)
  YOND_CUDA_CHECK(cudaMemsetAsync(wk, 0, (size_t)nseg * sizeof(SelectWork), s));
  dim3 g(stream_grid(seg_len), nseg);
  if ((size_t)g.x * nseg > (size_t)yond_num_sms() * 16) g.x = (unsigned)((yond_num_sms() * 16 + nseg - 1) / nseg);
  const double nel = (double)seg_len * nseg;
  YOND_CUDA_CHECK(cudaMemsetAsync(binmin, 0xff, (size_t)nseg * 1024 * sizeof(unsigned int), s));
  {
    YondProfScope prof("hist0+score3_binmin", s, 8.0 * nel);
    hist0_kernel<true><<<g, 256, 0, s>>>(data, mean, seg_len, wk, binmin);
  }
  YOND_LAUNCH_CHECK();
  select0_kernel<<<nseg, 1024, 0, s>>>(wk, reinterpret_cast<const unsigned long long*>(ranks_dev), nranks);
  YOND_LAUNCH_CHECK();
  {
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    const size_t smem = (size_t)kHist1Slots * 2048 * sizeof(unsigned int) + 2048;
    std::call_once(once, [&] {
      attr_err = cudaFuncSetAttribute(hist1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (attr_err == cudaSuccess)
        attr_err = cudaFuncSetAttribute(select1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * (2048 + 32) * (int)sizeof(unsigned int));
    });
    if (attr_err != cudaSuccess) return yond_set_error(YOND_ERR_CUDA, "cudaFuncSetAttribute(hist1_kernel) failed: %s", cudaGetErrorString(attr_err));
    int bx = yond_num_sms() / nseg;  // one 130 KB block per SM
    if (bx < 1) bx = 1;
    const size_t need = (seg_len / 4 + kHist1Threads - 1) / kHist1Threads;
    if ((size_t)bx > need) bx = (int)need;
    YondProfScope prof("hist1", s, 4.0 * nel);
    hist1_kernel<<<dim3(bx, nseg), kHist1Threads, smem, s>>>(data, seg_len, wk);
    YOND_LAUNCH_CHECK();
  }
  select1_kernel<<<nseg, 1024, 16 * (2048 + 32) * sizeof(unsigned int), s>>>(wk, nranks);
  YOND_LAUNCH_CHECK();
  {
    YondProfScope prof("hist2", s, 4.0 * nel);
    static std::once_flag h2_once;
    static cudaError_t h2_err = cudaSuccess;
    std::call_once(h2_once, [] { h2_err = cudaFuncSetAttribute(hist2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHist2Slots * 1024 * 4); });
    if (h2_err != cudaSuccess) return yond_set_error(YOND_ERR_CUDA, "cudaFuncSetAttribute(hist2_kernel) failed: %s", cudaGetErrorString(h2_err));
    hist2_kernel<false><<<g, 256, 0, s>>>(data, seg_len, wk);
    YOND_LAUNCH_CHECK();
    hist2_kernel<true><<<g, 256, kHist2Slots * 1024 * sizeof(unsigned int), s>>>(data, seg_len, wk);
  }
  YOND_LAUNCH_CHECK();
  select2_kernel<<<nseg, 1024, 0, s>>>(wk, nranks, out_dev);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

// sums_dev[s][0..5] = {N, Sx, Sy, Sxx, Sxy, Syy} over {lap < ths_dev[s]} (YOND_SIDD.py:77-78, strict), [6..11] the same over
// {lap < th, 1e-4 < mean < 0.8} (polyfit's non-saturated subset, utils/isp_algos.py:348-350), float64
int masked_sums(const float* lap, const float* mean, const float* var, size_t seg_len, int nseg, const double* ths_dev, double* sums_dev,
                cudaStream_t s) {
  YOND_CUDA_CHECK(cudaMemsetAsync(sums_dev, 0, (size_t)nseg * 12 * sizeof(double), s));
  dim3 g(stream_grid(seg_len), nseg);
  if ((size_t)g.x * nseg > (size_t)yond_num_sms() * 16) g.x = (unsigned)((yond_num_sms() * 16 + nseg - 1) / nseg);
  {
    YondProfScope prof("masked_sums", s, 12.0 * (double)seg_len * nseg);
    masked_sums_kernel<<<g, 256, 0, s>>>(lap, mean, var, seg_len, ths_dev, sums_dev, nullptr);
  }
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

// Scratch of yond_nlf_fit: the radix-select tables + a few hundred bytes of scalars per segment.
struct FitWork {
  SelectWork* sel;
  unsigned long long* ranks;
  double *gamma, *ths, *th25, *th, *th2, *sums, *sums2;
  float* stats;
  int *npeaks, *minj, *idx, *redo;
  size_t bytes;
};
FitWork carve_fit(void* base, int nseg) {
  FitWork w{};
  uint8_t* p = reinterpret_cast<uint8_t*>(base);
  size_t off = 0;
  auto take = [&](size_t nbytes) {
    off = align_up(off, 256);
    void* r = p ? p + off : nullptr;
    off += nbytes;
    return r;
  };
  w.sel = (SelectWork*)take((size_t)nseg * sizeof(SelectWork));
  w.ranks = (unsigned long long*)take(kMaxRanks * 8);
  w.gamma = (double*)take(kMaxQ * 2 * 8);
  w.ths = (double*)take((size_t)nseg * kMaxQ * 8);
  w.th25 = (double*)take((size_t)nseg * 8);
  w.th = (double*)take((size_t)nseg * 8);
  w.th2 = (double*)take((size_t)nseg * 8);
  w.sums = (double*)take((size_t)nseg * 12 * 8);
  w.sums2 = (double*)take((size_t)nseg * 12 * 8);
  w.stats = (float*)take((size_t)nseg * kMaxRanks * 4);
  w.npeaks = (int*)take((size_t)nseg * kMaxQ * 4);
  w.minj = (int*)take((size_t)nseg * 1024 * 4);
  w.idx = (int*)take((size_t)nseg * 4);
  w.redo = (int*)take((size_t)nseg * 4);
  w.bytes = align_up(off, 256);
  return w;
}
}  // namespace

extern "C" {

size_t yond_nlf_fit_work_bytes(int nseg) { return carve_fit(nullptr, nseg < 1 ? 1 : nseg).bytes + 256; }

int yond_nlf_fit(const float* var, const float* mean, const float* lap, size_t seg_len, int nseg, const double* quants_host,
                 int nq, double* regs_dev, double* detail_dev, void* work, void* stream) {
  YOND_REQUIRE(var && mean && lap && regs_dev && work && quants_host, "yond_nlf_fit: null argument");
  YOND_REQUIRE(nq >= 1 && nq <= kMaxQ && 2 * (nq + 1) <= kMaxRanks, "yond_nlf_fit: 1..%d quantiles (got %d)", kMaxQ, nq);
  YOND_REQUIRE(seg_len > 0 && nseg > 0 && nseg <= 65535, "yond_nlf_fit: bad segment geometry");
  YOND_REQUIRE((uintptr_t)work % 256 == 0, "yond_nlf_fit: work must be 256-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  const FitWork w = carve_fit(work, nseg);
  QuantList ql{};
  ql.nq = nq;
  for (int i = 0; i < nq; ++i) ql.q[i] = quants_host[i];
  for (int i = 1; i < nq; ++i) YOND_REQUIRE(ql.q[i] > ql.q[i - 1], "yond_nlf_fit: quantiles must ascend");
  const int nranks = 2 * (nq + 1);
  ranks_kernel<<<1, 32, 0, s>>>(ql, (unsigned long long)seg_len, w.ranks, w.gamma);
  YOND_LAUNCH_CHECK();
  YOND_REQUIRE(seg_len < 0xffffffffull && seg_len % 4 == 0 && (uintptr_t)lap % 16 == 0 && (uintptr_t)mean % 16 == 0,
               "yond_nlf_fit: segments must hold whole 4-channel pixels (16-byte aligned), fewer than 2^32 elements");
  unsigned int* binmin = reinterpret_cast<unsigned int*>(w.minj);
  // the first counting pass of the radix select also collects the per-bin minimum of lap (all score3 needs from the maps)
  int rc = order_stats_impl(lap, mean, binmin, seg_len, nseg, reinterpret_cast<const uint64_t*>(w.ranks), nranks, w.stats, w.sel, s);
  if (rc) return rc;
  pct_kernel<<<nseg, 32, 0, s>>>(w.stats, w.gamma, nq, w.ths, w.th25);
  YOND_LAUNCH_CHECK();
  score3_count_kernel<<<nseg, 256, 0, s>>>(binmin, w.ths, nq, w.npeaks);
  YOND_LAUNCH_CHECK();
  pick_kernel<<<ceil_div(nseg, 64), 64, 0, s>>>(ql, w.ths, w.npeaks, w.th, w.idx, nseg);
  YOND_LAUNCH_CHECK();
  if ((rc = masked_sums(lap, mean, var, seg_len, nseg, w.th, w.sums, s))) return rc;
  backup_kernel<<<ceil_div(nseg, 64), 64, 0, s>>>(w.sums, w.th, w.th25, w.th2, w.redo, w.sums2, nseg);
  YOND_LAUNCH_CHECK();
  {  // second pass: only the segments whose mask came out empty do any work
    dim3 g(stream_grid(seg_len), nseg);
    if ((size_t)g.x * nseg > (size_t)yond_num_sms() * 16) g.x = (unsigned)((yond_num_sms() * 16 + nseg - 1) / nseg);
    masked_sums_kernel<<<g, 256, 0, s>>>(lap, mean, var, seg_len, w.th2, w.sums2, w.redo);
    YOND_LAUNCH_CHECK();
  }
  solve_kernel<<<ceil_div(nseg, 64), 64, 0, s>>>(w.sums, w.sums2, w.redo, w.th2, w.idx, w.ths, w.npeaks, ql, regs_dev, detail_dev, nseg);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}

}  // extern "C"
