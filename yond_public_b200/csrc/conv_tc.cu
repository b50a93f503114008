// Implicit-GEMM convolution for the YOND denoisers on Blackwell tensor cores (sm_100a).
//
// Replaces the torch.nn.Conv2d / ConvTranspose2d calls of archs/Unet.py:17-52, :393-421 and
// archs/modules.py:117-125,163-233 (library kernels in the reference) with one persistent,
// warp-specialised kernel:
//
//   warp 0     TMA producer — activations: halo-extended NHWC slabs (cp.async.bulk.tensor.4d; out-of-bounds
//                             zero-fill is the conv's zero padding); weights: per-tap K-major tiles (2d), resident in
//                             shared memory for narrow layers, streamed through a ring otherwise
//   warp 1     MMA issuer   — one elected thread issues tcgen05.mma (M=128 pixels — 256 over a CTA pair —, N<=256
//                             channels, K=16) as straight-line code, accumulating taps x channel blocks into TMEM;
//                             tcgen05.commit frees the stages
//   warps 2-17 epilogue     — tcgen05.ld the accumulators (double-buffered in TMEM so the next tile's MMAs overlap),
//                             bias / FiLM / activation / residual, 256-bit bf16 NHWC stores
//
// GEMM view: M = output pixels, N = Cout, K = taps*Cin.  A 3x3 stride-1 conv loads ONE halo slab per channel
// block — (rows+2) x (8+2) pixels, 128 B (or 64 B) per pixel, hardware-swizzled by TMA — and reaches all nine
// taps by moving the UMMA descriptor's start address by whole pixels (the swizzle XOR is a function of the
// absolute shared-memory address, so any pixel-aligned start reads consistently).  T sub-tiles of 128 pixels
// (stacked rows, or T images) share every weight tile, which cuts weight traffic from L2 by T.  Two builds:
// conv_tc_kernel<false> (one CTA per SM) and conv_tc_kernel<true> (cluster of 2, cta_group::2: each CTA holds its own
// pixels and half of every weight tile; the 3x3 layers that stream their weights with N tiles >= 128).  Modes: 3x3 s1,
// 3x3 s2, 1x1 (on up to two concatenated sources), ConvT 2x2, and the fused ConvT 2x2 + 1x1-on-concat hand-over of the
// decoder (CONV_UPSC).  See DESIGN.md section 4.
#include "conv_tc.cuh"

#include <mutex>

namespace {

constexpr int kEpiWarps = 16;                 // four per TMEM lane quarter, splitting the column chunks
constexpr int kThreads = 64 + 32 * kEpiWarps;  // 2 control warps + the epilogue warps
constexpr int kMaxStagesA = 8;
constexpr int kMaxStagesB = 8;
constexpr int kMaxT = 4;
// The MMA issuer instantiates its loops for T = 1, 2 and 4 only (T is a power of two <= kMaxT).
static_assert(kMaxT == 4, "conv_tc: the issuer dispatches T in {1, 2, 4}");
constexpr int kMaxNT = 256;      // largest UMMA N
constexpr int kCta2MinNT = 128;  // smallest N tile of a streamed layer that runs as a CTA pair
// Resident-weight layers other than 3x3 stride 1 tabulate their stage decode (16 B per stage) in the 1 KB output-conv table.
constexpr int kMaxTabStages = 64;

// Division by a run-time constant as multiply-high + shift (n < 2^31): the epilogue and the tile decode run once per
// tile in every warp, and a 32-bit integer division is ~20 instructions.
struct FastDiv {
  uint32_t mul, shr, d;
};
__host__ FastDiv make_fastdiv(uint32_t d) {
  FastDiv f{0u, 0u, d};
  if (d > 1) {
    uint32_t lg = 0;
    while ((1u << lg) < d) ++lg;
    const uint32_t pw = 31 + lg;
    f.mul = (uint32_t)(((1ull << pw) + d - 1) / d);
    f.shr = pw - 32;
  }
  return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t n, const FastDiv& f) { return f.d == 1 ? n : (__umulhi(n, f.mul) >> f.shr); }

struct TcParams {
  int B, H, W;  // tile-space dims (output dims; input dims for CONVT_2X2)
  int TW, TH, NB, T;  // sub-tile = TH rows x NB images x TW columns = 128 GEMM rows; T sub-tiles per CTA tile
  int t_along_h;      // sub-tiles stacked along H (1) or along the batch (0)
  int tiles_h, tiles_w, tiles_b, tiles_n;
  int NT;     // N tile (UMMA N)
  int N;      // GEMM N total
  int Cout;   // real output channels
  int CB;     // channel block (32 | 64)
  int ncb0, ncb1;
  int mode;
  int wres;   // weights resident in smem
  int SA, SB; // pipeline depths
  uint32_t a_stage_bytes, a_tx_bytes, b_stage_bytes;  // stage pitch (1024-aligned), bytes one slab load writes, weight tile
  uint32_t sub_off, sbo, tap_r_off;  // byte offsets inside an activation stage: next sub-tile, next 8-row group, next image row
  uint32_t smem_b_off, smem_bar_off, smem_epi_off;  // weights, barriers, epilogue parameter rows (128 B per epilogue warp)
  int tmem_cols;
  uint32_t b2_stage_bytes, b2_off;  // CONV_UPSC: skip-part weight tile (Cout rows) and where those tiles start in the weight region
  int cta2;        // CTA pair: cta_group::2 MMAs (M = 256 over two SMs), each CTA loads its own tile and half of every weight tile
  int acc_stages;  // accumulator stages in TMEM: 2 (epilogue of tile i overlaps the MMAs of tile i+1) or 1 (T*NT = 512 columns)
  FastDiv fd_tiles_n, fd_tiles_w, fd_tiles_h, fd_cout;
  int lg_nchunk;       // log2(NT / 16)
  uint32_t t_off;      // output element offset between consecutive sub-tiles
  int epi_split;  // two accumulator stages: the epilogue warps form two groups of kEpiWarps/2 that take alternate tiles (group g owns
                  // accumulator stage g), so one group's TMEM reads / MUFU burst / stores overlap the other group's and a tile's
                  // epilogue may take up to two tile times of MMAs
  int epi_fixed;  // every visit of an epilogue warp covers the same 16 channels of the same image (see epilogue_loop)
  int paired;      // pixel-pair formulation of a 32 -> 32 channel 3x3 conv (conv_tc.cuh): N = CB = 64 over (H, W/2)
  int cvec;        // channels of the bias / scale / shift vectors (= Cout, or 32 in the paired formulation)
  uint32_t cmask;  // paired: 31 (output column n = o*32 + co uses vector entry co), else all ones
  const float* bias;
  const float* scale;
  const float* shift;
  int act;
  float slope;
  const bf16* res;
  bf16* out0;
  bf16* out1;
  // fused last layer (ConvLayer::tail_*): table [32][4] + [4] floats at smem_tail_off
  const float* tail_w;
  const float* tail_b;
  const float* tail_z;
  const float* tail_ub;
  float* tail_y;
  int tail_res;
  uint32_t smem_tail_off;
};

struct TcMaps {
  CUtensorMap a[8];
  CUtensorMap w;
  CUtensorMap w2;  // CONV_UPSC: skip-part weight tiles
};

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a pipeline bug must surface as a trapped kernel (an error on the host), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    if ((it & 0x3ff) == 0x3ff) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 6000000000LL) __trap();  // ~3 s at 1.9 GHz
    }
  }
}
// One lane of a converged warp (elect.sync); returns 1 on the elected lane.
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred px;\n\t"
      "elect.sync _|px, 0xFFFFFFFF;\n\t"
      "selp.u32 %0, 1, 0, px;\n\t}"
      : "=r"(pred));
  return pred;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// ---- CTA pair (cta_group::2): two SMs of one TPC run one M=256 MMA; each holds its own 128 rows of A and of the
// accumulator and HALF of the B tile, so per-SM shared-memory reads and weight traffic halve.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads of a CTA pair: data lands in this CTA's shared memory, the transaction bytes are counted on `bar`, a
// shared::cluster address (the leader CTA's barrier).
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrive on the barrier at this offset in BOTH CTAs of the pair once all previously issued MMAs have completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(h);
}

// SiLU(v) = v * sigmoid(v) = 0.5 v (1 + tanh(v / 2)): one MUFU (tanh.approx, ~2^-11 relative) instead of exp + rcp;
// the result is stored as bf16 (2^-9), so the approximation is below the storage rounding.
__device__ __forceinline__ float fast_silu(float v) {
  float t;
  const float h = 0.5f * v;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// One activation ("A") pipeline stage of the K loop, decoded identically by producer and MMA issuer.
struct AStage {
  int map;       // index into TcMaps::a
  int c;         // channel coordinate
  int dw, dh;    // tile-origin offsets of the load
  int ntaps;     // weight tiles consumed from this stage
  int widx0;     // first weight-tile index
  int sx;        // CONV_UPSC skip part: output parity of this stage, else -1
};
__device__ __forceinline__ AStage decode_astage(const TcParams& p, int ai) {
  AStage s;
  s.sx = -1;
  if (p.mode == CONV_3X3_S1) {  // one halo slab per channel block: all nine taps
    const int src = ai >= p.ncb0;
    s.map = src;
    s.c = (src ? ai - p.ncb0 : ai) * p.CB;
    s.dw = -1;
    s.dh = -1;
    s.ntaps = 9;
    s.widx0 = ai * 9;
  } else if (p.mode == CONV_3X3_S2) {
    int cbg = ai / 9, tap = ai - cbg * 9;
    int r = tap / 3, sx = tap - r * 3;
    int src = cbg >= p.ncb0;
    s.map = src * 4 + (r != 1) * 2 + (sx != 1);
    s.c = (src ? cbg - p.ncb0 : cbg) * p.CB;
    s.dh = (r == 0) ? -1 : 0;
    s.dw = (sx == 0) ? -1 : 0;
    s.ntaps = 1;
    s.widx0 = cbg * 9 + tap;
  } else if (p.mode == CONV_UPSC) {
    s.dw = 0;
    s.dh = 0;
    s.ntaps = 1;
    if (ai < p.ncb0) {  // folded up-sampling part: low-resolution source, all four parities at once (N = 4 Cout)
      s.map = 0;
      s.c = ai * p.CB;
      s.widx0 = ai;
    } else {            // skip part: one stage per (parity, channel block), N = Cout into that parity's columns
      const int j = ai - p.ncb0;
      const int q = j / p.ncb1, cb = j - q * p.ncb1;
      s.map = 4 + q;
      s.c = cb * p.CB;
      s.widx0 = cb;
      s.sx = q;
    }
  } else {
    int src = ai >= p.ncb0;
    s.map = src;
    s.c = (src ? ai - p.ncb0 : ai) * p.CB;
    s.dw = 0;
    s.dh = 0;
    s.ntaps = 1;
    s.widx0 = ai;
  }
  return s;
}
__host__ __device__ __forceinline__ int num_astages(const TcParams& p) {
  int ncb = p.ncb0 + p.ncb1;
  if (p.mode == CONV_3X3_S1) return ncb;
  if (p.mode == CONV_UPSC) return p.ncb0 + 4 * p.ncb1;
  return p.mode == CONV_3X3_S2 ? ncb * 9 : ncb;
}
__device__ __forceinline__ int num_wtiles(const TcParams& p) {
  int ncb = p.ncb0 + p.ncb1;
  return (p.mode == CONV_3X3_S1 || p.mode == CONV_3X3_S2) ? ncb * 9 : ncb;
}

struct TileCoord {
  int n0, w0, h0, b0, n_idx;
};
__device__ __forceinline__ TileCoord decode_tile(const TcParams& p, int tile) {
  TileCoord t;
  uint32_t m = fdiv((uint32_t)tile, p.fd_tiles_n);
  t.n_idx = tile - (int)m * p.tiles_n;
  uint32_t m2 = fdiv(m, p.fd_tiles_w);
  const int tw_i = (int)(m - m2 * p.tiles_w);
  const uint32_t m3 = fdiv(m2, p.fd_tiles_h);
  const int th_i = (int)(m2 - m3 * p.tiles_h);
  const int tb_i = (int)m3;
  t.w0 = tw_i * p.TW;
  t.h0 = th_i * p.TH * (p.t_along_h ? p.T : 1);
  t.b0 = tb_i * p.NB * (p.t_along_h ? 1 : p.T);
  t.n0 = t.n_idx * p.NT;
  return t;
}

// Persistent tile schedule.  Single CTA: tile = blockIdx.x, += gridDim.x.  CTA pair: the pair walks "units" = (pair of
// consecutive M tiles, n tile); rank r of the pair owns M tile 2 m + r (an M tile past the end decodes to images >= B:
// its loads are zero-filled and its stores masked, but it takes part in the pair's MMAs).
struct TileSched {
  int first, step, n_units, rank, cta2;
};
template <bool kPair>
__device__ __forceinline__ TileSched make_sched(const TcParams& p, int total_tiles) {
  TileSched s;
  s.cta2 = kPair ? 1 : 0;
  if (kPair) {
    s.rank = (int)cluster_ctarank();
    s.first = (int)blockIdx.x >> 1;
    s.step = (int)gridDim.x >> 1;
    const int m_tiles = total_tiles / p.tiles_n;
    s.n_units = ((m_tiles + 1) >> 1) * p.tiles_n;
  } else {
    s.rank = 0;
    s.first = (int)blockIdx.x;
    s.step = (int)gridDim.x;
    s.n_units = total_tiles;
  }
  return s;
}
__device__ __forceinline__ int sched_tile(const TcParams& p, const TileSched& s, int u) {
  if (!s.cta2) return u;
  const int m2 = (int)fdiv((uint32_t)u, p.fd_tiles_n);
  return (2 * m2 + s.rank) * p.tiles_n + (u - m2 * p.tiles_n);
}

// All MMAs of one tap (weight tile): TT sub-tile accumulators x KS steps of K=16, fully unrolled so that every
// descriptor is `running low word + immediate` (two uniform adds per MMA; the B200 tensor pipe retires an
// M=128,N=32 SS MMA every 40 cycles, N=64 every 48, N=128 every 64 — tools/mma_rate.cu — so the issue stream must
// stay well below that).
// MMA + in-place advance of both descriptor low words by one K=16 step (32 bytes = 2 units of 16 B).
__device__ __forceinline__ void umma_step(uint32_t tmem_d, uint32_t& a_lo, uint32_t a_hi, uint32_t& b_lo, uint32_t b_hi,
                                          uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%0, %2};\n\t"
      "mov.b64 db, {%1, %3};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%4], da, db, %5, p;\n\t"
      "add.u32 %0, %0, 2;\n\t"
      "add.u32 %1, %1, 2;\n\t}"
      : "+r"(a_lo), "+r"(b_lo)
      : "r"(a_hi), "r"(b_hi), "r"(tmem_d), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_step_pair(uint32_t tmem_d, uint32_t& a_lo, uint32_t a_hi, uint32_t& b_lo, uint32_t b_hi,
                                               uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%0, %2};\n\t"
      "mov.b64 db, {%1, %3};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%4], da, db, %5, p;\n\t"
      "add.u32 %0, %0, 2;\n\t"
      "add.u32 %1, %1, 2;\n\t}"
      : "+r"(a_lo), "+r"(b_lo)
      : "r"(a_hi), "r"(b_hi), "r"(tmem_d), "r"(idesc), "r"(accum)
      : "memory");
}
template <int KS, int TT>
__device__ __forceinline__ void issue_tap_pair(uint32_t d_tmem, uint32_t nt, uint32_t a_lo0, uint32_t sub_step, uint32_t b_lo0,
                                               uint32_t a_hi, uint32_t b_hi, uint32_t idesc, uint32_t accum) {
  uint32_t al = a_lo0, dt = d_tmem;
#pragma unroll
  for (int t = 0; t < TT; ++t) {
    uint32_t bl = b_lo0;
#pragma unroll
    for (int k = 0; k < KS; ++k) umma_step_pair(dt, al, a_hi, bl, b_hi, idesc, k ? 1u : accum);
    al += sub_step - 2u * KS;
    dt += nt;
  }
}
template <int KS, int TT>
__device__ __forceinline__ void issue_tap(uint32_t d_tmem, uint32_t nt, uint32_t a_lo0, uint32_t sub_step, uint32_t b_lo0,
                                          uint32_t a_hi, uint32_t b_hi, uint32_t idesc, uint32_t accum) {
  uint32_t al = a_lo0, dt = d_tmem;
#pragma unroll
  for (int t = 0; t < TT; ++t) {
    uint32_t bl = b_lo0;
#pragma unroll
    for (int k = 0; k < KS; ++k) umma_step(dt, al, a_hi, bl, b_hi, idesc, k ? 1u : accum);
    al += sub_step - 2u * KS;  // next sub-tile, back to K step 0
    dt += nt;
  }
}

// K steps [K0, K1) of one tap (pixel-pair formulation: the other steps multiply all-zero weights)
template <int K0, int K1, int TT>
__device__ __forceinline__ void issue_tap_range(uint32_t d_tmem, uint32_t nt, uint32_t a_lo0, uint32_t sub_step, uint32_t b_lo0,
                                                uint32_t a_hi, uint32_t b_hi, uint32_t idesc, uint32_t accum) {
  uint32_t al = a_lo0 + 2u * K0, dt = d_tmem;
#pragma unroll
  for (int t = 0; t < TT; ++t) {
    uint32_t bl = b_lo0 + 2u * K0;
#pragma unroll
    for (int k = K0; k < K1; ++k) umma_step(dt, al, a_hi, bl, b_hi, idesc, k > K0 ? 1u : accum);
    al += sub_step - 2u * (K1 - K0);
    dt += nt;
  }
}
// Nine taps of a pixel-pair slab (CB = 64: K steps 0,1 = first pixel of the pair, 2,3 = second): the left neighbour pair
// contributes only its second pixel, the right neighbour pair only its first.
template <int TT>
__device__ __forceinline__ void issue_slab_paired(uint32_t d_tmem, uint32_t nt, uint32_t a_stage_lo, uint32_t tap_r16, uint32_t px16,
                                                  uint32_t sub_step, uint32_t b_lo_first, uint32_t b_step16, uint32_t a_hi,
                                                  uint32_t b_hi, uint32_t idesc, uint32_t first_accum) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const uint32_t a0 = a_stage_lo + (uint32_t)r * tap_r16, b0 = b_lo_first + (uint32_t)(r * 3) * b_step16;
    issue_tap_range<2, 4, TT>(d_tmem, nt, a0, sub_step, b0, a_hi, b_hi, idesc, r ? 1u : first_accum);
    issue_tap_range<0, 4, TT>(d_tmem, nt, a0 + px16, sub_step, b0 + b_step16, a_hi, b_hi, idesc, 1u);
    issue_tap_range<0, 2, TT>(d_tmem, nt, a0 + 2u * px16, sub_step, b0 + 2u * b_step16, a_hi, b_hi, idesc, 1u);
  }
}

// All nine taps of one halo slab as straight-line code (resident weights): the only run-time inputs are a handful of
// uniform bases and strides, everything else is an immediate.
template <int KS, int TT>
__device__ __forceinline__ void issue_slab_resident(uint32_t d_tmem, uint32_t nt, uint32_t a_stage_lo, uint32_t tap_r16, uint32_t px16,
                                                    uint32_t sub_step, uint32_t b_lo_first, uint32_t b_step16, uint32_t a_hi,
                                                    uint32_t b_hi, uint32_t idesc, uint32_t first_accum) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int sx = 0; sx < 3; ++sx)
      issue_tap_range<0, KS, TT>(d_tmem, nt, a_stage_lo + (uint32_t)r * tap_r16 + (uint32_t)sx * px16, sub_step,
                                 b_lo_first + (uint32_t)(r * 3 + sx) * b_step16, a_hi, b_hi, idesc, (r | sx) ? 1u : first_accum);
}

// 256-bit global accesses (sm_100): one lane moves a whole 32-byte sector per instruction, so a pixel-per-lane store of
// 16 bf16 channels is one full-sector write instead of two half-sector partial writes.
struct __align__(32) U8 { uint32_t v[8]; };
__device__ __forceinline__ void stg256(void* ptr, const U8& u) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(ptr), "r"(u.v[0]), "r"(u.v[1]), "r"(u.v[2]), "r"(u.v[3]),
               "r"(u.v[4]), "r"(u.v[5]), "r"(u.v[6]), "r"(u.v[7])
               : "memory");
}
__device__ __forceinline__ U8 ldg256(const void* ptr) {
  U8 u;
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(u.v[0]), "=r"(u.v[1]), "=r"(u.v[2]), "=r"(u.v[3]), "=r"(u.v[4]), "=r"(u.v[5]), "=r"(u.v[6]), "=r"(u.v[7])
               : "l"(ptr));
  return u;
}

// Epilogue warps: bias, FiLM scale/shift, activation, residual, bf16 stores of the finished accumulators.
// A warp owns one TMEM lane quarter (32 GEMM rows = 32 pixels) and every fourth 16-column chunk of the tile ("visits":
// 2 to 8 per tile).  16 warps x visits x instructions-per-visit has to fit under the tile's MMA time on 4 issue ports
// (an N=32 tile of 512 pixels is only ~2900 cycles of MMAs), so the loop is written for instruction count:
// no integer divisions (shifts / multiply-high), 32-bit element offsets from one per-tile base, activation and the
// presence of scale / residual resolved at compile time.  Everything with a long latency is issued BEFORE the wait on
// the accumulator barrier, while the tile's MMAs run:
//   - the residual (one 256-bit load per visit, kept in registers),
//   - when the layer is narrow (NT <= 64, one image per tile) a warp's visits all cover the same 16 channels of the
//     same image, so bias / scale / shift collapse to out = act(acc * A + Bc) with A, Bc loaded once per tile
//     (`epi_fixed`); wider layers load them per visit.
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_u4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// kRegP (FiLM layers without a residual input whose visits all use ONE 16-channel parameter set — N = 32, or the pixel-pair form, where
// output columns n and n + 32 are the same channel): the folded scale / shift vectors live in 32 registers and are refreshed when the
// image changes, instead of eight broadcast LDS.128 per visit (512 B into the register file each, on the shared-memory pipe the MMAs
// read their operands through; 77 % LSU data-pipe utilisation in the profile of c1.conv1).
__device__ __forceinline__ bool epilogue_single_set(const TcParams& p) {
  const int nparts = p.epi_split ? 2 : 4, nchunk = 1 << p.lg_nchunk;
  const int nsets = nchunk > nparts ? nchunk / nparts : 1;
  return p.epi_fixed != 0 && nsets <= 2 && (nsets == 1 || (((uint32_t)(nparts << 4) & p.cmask) == 0u));
}
template <bool kScale, bool kRes, bool kSilu, int kV, bool kPair, bool kRegP = false>  // kV: visits per group (residual registers held at once)
__device__ __forceinline__ void epilogue_loop(const TcParams& p, uint32_t tmem_base, uint32_t acc_full, uint32_t acc_empty, uint32_t ptab,
                                              int warp, int lane, int total_tiles) {
  const TileSched sched = make_sched<kPair>(p, total_tiles);
  // the MMA issuer that waits for "accumulator drained" lives in the pair's leader CTA
  const uint32_t acc_empty_remote = kPair ? mapa_shared(acc_empty, 0) : acc_empty;
  const int q = warp & 3;            // TMEM lane quarter this warp may access
  const int part4 = (warp - 2) >> 2; // kEpiWarps/4 warps share a quarter
  const bool split = p.epi_split != 0;
  const int grp = split ? (part4 & 1) : 0;         // tile parity (= accumulator stage) this warp serves
  const int part = split ? (part4 >> 1) : part4;   // the warps of a group that share a quarter split the column chunks
  const int nparts = split ? 2 : 4;
  const int row = q * 32 + lane;     // GEMM row inside a sub-tile
  const int w_i = row & (p.TW - 1);  // TW, NB are powers of two
  const int g_i = row / p.TW;        // (h, b) index inside the sub-tile, h-major
  const int dh = g_i / p.NB, db = g_i & (p.NB - 1);
  const int nchunk = 1 << p.lg_nchunk, nchunk_m1 = nchunk - 1, nvis = p.T << p.lg_nchunk;
  // `fixed`: a warp's visits cover the column chunks part, part + nparts, ... (mod nchunk): nsets = nchunk / nparts distinct
  // 16-channel sets (1 or 2), visit j uses set j mod nsets
  const int nsets = nchunk > nparts ? nchunk / nparts : 1;
  const bool fixed = p.epi_fixed != 0 && nsets <= 2 && !(kScale && kRes);  // both at once would not fit the register budget
  const bool convt = p.mode == CONVT_2X2 || p.mode == CONV_UPSC;  // output pixel (2h+a, 2w+b), n = (a*2+b)*Cout + co
  const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
  const bool lrelu = p.act == ACT_LRELU;
  const float slope = p.slope;
  // `fixed`: A[16] | Bc[16] of each of this warp's channel sets live in a 128-byte shared-memory row (registers are short: 18
  // warps leave 96 per thread, and spilled values miss the ~28 KB of L1 that 227 KB of shared memory leaves); lanes 0-15 fill
  // set 0, lanes 16-31 set 1
  const int lset = lane >> 4;
  const uint32_t cfix_v = (uint32_t)((((part + nparts * lset) & nchunk_m1) << 4) + (lane & 15)) & p.cmask;  // entry of the bias / scale / shift vectors
  const bool pl = fixed && lset < nsets;  // this lane fills a parameter slot
  const uint32_t pslot = ptab + 128 * lset + 4 * (lane & 15);
  const float bias_l = pl ? __ldg(p.bias + cfix_v) : 0.f;
  if (pl) {
    sts_f32(pslot, 1.f);
    sts_f32(pslot + 64, bias_l);
  }
  __syncwarp();
  int as = grp, pacc = 0, b_prev = -1;
  float pa[kRegP && kScale ? 16 : 1], pb[kRegP ? 16 : 1];
  if (kRegP && !kScale) {  // bias only: constant for the whole kernel
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const float4 bc = lds_f4(ptab + 64 + 16 * g);
      pb[g * 4 + 0] = bc.x; pb[g * 4 + 1] = bc.y; pb[g * 4 + 2] = bc.z; pb[g * 4 + 3] = bc.w;
    }
  }
  for (int u = sched.first + grp * sched.step; u < sched.n_units; u += (split ? 2 : 1) * sched.step) {
    const TileCoord tc = decode_tile(p, sched_tile(p, sched, u));
    const int w = tc.w0 + w_i, h0 = tc.h0 + dh;
    const int bb = tc.b0 + (p.t_along_h ? db : db * p.T);  // along the batch: sub-tile t = images t, t+T, ... of the tile
    const bool wv = (w < p.W) && (h0 < p.H) && (bb < p.B);
    // element offset of this thread's pixel in sub-tile 0 (+ first column of the tile unless transposed conv)
    const uint32_t e0 = convt ? (((uint32_t)bb * (2 * p.H) + 2 * h0) * (uint32_t)(2 * p.W) + 2 * w) * (uint32_t)p.Cout
                              : (((uint32_t)bb * p.H + h0) * (uint32_t)p.W + w) * (uint32_t)p.Cout + tc.n0;
    // visits in groups of kV
    for (int k0 = 0; part + nparts * k0 < nvis; k0 += kV) {
      // ---- before the accumulator is ready: addresses, residual loads, per-tile parameters ----
      uint32_t off[kV];
      uint32_t vmask = 0;
      U8 rr[kV];
#pragma unroll
      for (int k = 0; k < kV; ++k) {
        const int ci = part + nparts * (k0 + k);
        off[k] = 0;
        if (ci < nvis) {
          const int t = ci >> p.lg_nchunk, c = (ci & nchunk_m1) << 4;
          const bool ok = wv && (p.t_along_h ? (h0 + t * p.TH < p.H) : (bb + t < p.B));
          uint32_t e = e0 + (uint32_t)t * p.t_off;
          if (convt) {
            const uint32_t n = (uint32_t)(tc.n0 + c), quad = fdiv(n, p.fd_cout);
            e += ((quad >> 1) * (uint32_t)(2 * p.W) + (quad & 1u)) * (uint32_t)p.Cout + (n - quad * p.Cout);
          } else {
            e += (uint32_t)c;
          }
          off[k] = e;
          if (ok) {
            vmask |= 1u << k;
            if (kRes) rr[k] = ldg256(p.res + e);
          }
        }
      }
      if (k0 == 0) {
        if (kScale && fixed) {
          // the folded parameters change with the image only (NB == 1: one image per tile, uniform over the warp); every
          // epilogue warp of every SM re-reading the same two cache lines per tile made this dependent global load the
          // longest step of the epilogue (L2 hot line: ~2000 cycles per tile in the source-level profile)
          const int b = bb < p.B ? bb : p.B - 1;
          if (b != b_prev) {
            b_prev = b;
            if (pl) {
              const float sc = __ldg(p.scale + (size_t)b * p.cvec + cfix_v);
              const float sh = p.shift ? __ldg(p.shift + (size_t)b * p.cvec + cfix_v) : 0.f;
              sts_f32(pslot, sc);
              sts_f32(pslot + 64, fmaf(bias_l, sc, sh));
            }
            __syncwarp();
            if (kRegP) {
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                const float4 a = lds_f4(ptab + 16 * g), bc = lds_f4(ptab + 64 + 16 * g);
                pa[g * 4 + 0] = a.x; pa[g * 4 + 1] = a.y; pa[g * 4 + 2] = a.z; pa[g * 4 + 3] = a.w;
                pb[g * 4 + 0] = bc.x; pb[g * 4 + 1] = bc.y; pb[g * 4 + 2] = bc.z; pb[g * 4 + 3] = bc.w;
              }
            }
          }
        }
        mbar_wait(acc_full + 8 * as, pacc);
        tc_fence_after();
      }
#pragma unroll
      for (int k = 0; k < kV; ++k) {
        const int ci = part + nparts * (k0 + k);
        if (ci >= nvis) break;  // visits are in increasing order: the rest of the group is past the end too
        const int t = ci >> p.lg_nchunk, c = (ci & nchunk_m1) << 4;
        uint32_t v[16];
        tmem_ld16(tmem_row + (uint32_t)((as * p.T + t) * p.NT + c), v);
        tmem_ld_wait();
        if ((vmask >> k) & 1u) {
          float f[16];
          if (kRegP) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = kScale ? fmaf(__uint_as_float(v[j]), pa[j], pb[j]) : __uint_as_float(v[j]) + pb[j];
          } else if (fixed) {
            const uint32_t pt = ptab + 128u * (uint32_t)((k0 + k) & (nsets - 1));
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const float4 bc = lds_f4(pt + 64 + 16 * g);
              if (kScale) {
                const float4 a = lds_f4(pt + 16 * g);
                f[g * 4 + 0] = fmaf(__uint_as_float(v[g * 4 + 0]), a.x, bc.x); f[g * 4 + 1] = fmaf(__uint_as_float(v[g * 4 + 1]), a.y, bc.y);
                f[g * 4 + 2] = fmaf(__uint_as_float(v[g * 4 + 2]), a.z, bc.z); f[g * 4 + 3] = fmaf(__uint_as_float(v[g * 4 + 3]), a.w, bc.w);
              } else {
                f[g * 4 + 0] = __uint_as_float(v[g * 4 + 0]) + bc.x; f[g * 4 + 1] = __uint_as_float(v[g * 4 + 1]) + bc.y;
                f[g * 4 + 2] = __uint_as_float(v[g * 4 + 2]) + bc.z; f[g * 4 + 3] = __uint_as_float(v[g * 4 + 3]) + bc.w;
              }
            }
          } else {
            const uint32_t n = (uint32_t)(tc.n0 + c);
            const uint32_t co = (convt ? n - fdiv(n, p.fd_cout) * p.Cout : n) & p.cmask;
            const float4* b4 = reinterpret_cast<const float4*>(p.bias + co);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const float4 bi = __ldg(b4 + g);
              f[g * 4 + 0] = __uint_as_float(v[g * 4 + 0]) + bi.x; f[g * 4 + 1] = __uint_as_float(v[g * 4 + 1]) + bi.y;
              f[g * 4 + 2] = __uint_as_float(v[g * 4 + 2]) + bi.z; f[g * 4 + 3] = __uint_as_float(v[g * 4 + 3]) + bi.w;
            }
            if (kScale) {
              int b = p.t_along_h ? bb : bb + t;
              if (b > p.B - 1) b = p.B - 1;
              const float4* s4 = reinterpret_cast<const float4*>(p.scale + (size_t)b * p.cvec + co);
              const float4* h4 = p.shift ? reinterpret_cast<const float4*>(p.shift + (size_t)b * p.cvec + co) : nullptr;
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                const float4 sc = __ldg(s4 + g), sh = h4 ? __ldg(h4 + g) : make_float4(0.f, 0.f, 0.f, 0.f);
                f[g * 4 + 0] = fmaf(f[g * 4 + 0], sc.x, sh.x); f[g * 4 + 1] = fmaf(f[g * 4 + 1], sc.y, sh.y);
                f[g * 4 + 2] = fmaf(f[g * 4 + 2], sc.z, sh.z); f[g * 4 + 3] = fmaf(f[g * 4 + 3], sc.w, sh.w);
              }
            }
          }
          if (kSilu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = fast_silu(f[j]);
          } else if (lrelu) {  // slope < 1: LeakyReLU(x) = max(x, slope * x)
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], f[j] * slope);
          }
          if (kRes) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float2 a = unpack_bf16x2(rr[k].v[j]);
              f[2 * j] += a.x;
              f[2 * j + 1] += a.y;
            }
          }
          U8 o;
#pragma unroll
          for (int j = 0; j < 8; ++j) o.v[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
          stg256(p.out0 + off[k], o);
          if (p.out1) {
#pragma unroll
            for (int j = 0; j < 8; ++j) o.v[j] = pack_bf16x2(fast_silu(f[2 * j]), fast_silu(f[2 * j + 1]));
            stg256(p.out1 + off[k], o);
          }
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (kPair) mbar_arrive_cluster(acc_empty_remote + 8 * as);
      else mbar_arrive(acc_empty + 8 * as);
    }
    if (split) pacc ^= 1;  // this group's stage comes round every second tile
    else if (++as == p.acc_stages) { as = 0; pacc ^= 1; }
  }
}

// Epilogue of the network's LAST tensor-core layer with the 1x1 output conv fused in (ConvLayer::tail_*): N = 32, so a pixel's
// channels are two 16-column chunks; warp `part` of a lane quarter takes sub-tile t = part and BOTH chunks, folds
// out[c] = act(acc * A[c] + Bc[c]) + res[c] straight into the four output sums and writes one float4 per pixel.
template <bool kScale, bool kRes>
__device__ __forceinline__ void epilogue_tail(const TcParams& p, uint32_t tmem_base, uint32_t acc_full, uint32_t acc_empty, uint32_t ptab,
                                              uint32_t tailtab, int warp, int lane, int total_tiles) {
  const int q = warp & 3, part = (warp - 2) >> 2;
  const int row = q * 32 + lane;
  const int w_i = row & (p.TW - 1), g_i = row / p.TW;
  const int dh = g_i / p.NB, db = g_i & (p.NB - 1);
  const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
  const bool lrelu = p.act == ACT_LRELU, silu = p.act == ACT_SILU;
  const float slope = p.slope;
  const float bias_l = __ldg(p.bias + lane);  // Cout == 32: lane c holds channel c's parameters
  sts_f32(ptab + 4 * lane, 1.f);
  sts_f32(ptab + 128 + 4 * lane, bias_l);
  __syncwarp();
  const float4 tb = lds_f4(tailtab + 32 * 16);
  int as = 0, pacc = 0, b_prev = -1;
  for (int u = blockIdx.x; u < total_tiles; u += gridDim.x) {
    const TileCoord tc = decode_tile(p, u);
    const int t = part;  // this warp's sub-tile (idle when the tile has fewer)
    const int w = tc.w0 + w_i, h0 = tc.h0 + dh + (p.t_along_h ? t * p.TH : 0);
    const int bb = tc.b0 + (p.t_along_h ? db : db * p.T + t);
    const bool ok = t < p.T && w < p.W && h0 < p.H && bb < p.B;
    const uint32_t pix = ((uint32_t)bb * p.H + h0) * (uint32_t)p.W + w;
    U8 rr[2];
    float4 zi = make_float4(0.f, 0.f, 0.f, 0.f);
    float ub = 1.f;
    if (ok) {
      if (kRes) {
        rr[0] = ldg256(p.res + (size_t)pix * 32);
        rr[1] = ldg256(p.res + (size_t)pix * 32 + 16);
      }
      if (p.tail_res) zi = __ldg(reinterpret_cast<const float4*>(p.tail_z) + pix);
      if (p.tail_ub) ub = __ldg(p.tail_ub + bb);
    }
    if (kScale) {  // per-image A / Bc (NB == 1 is not required here: the table is per warp and reloaded when the image changes)
      const int b = bb < p.B ? bb : p.B - 1;
      const int b0 = __shfl_sync(0xffffffffu, b, 0);
      if (b0 != b_prev) {  // tiles of a CTA share their image for long runs (tile order: n, w, h, b)
        b_prev = b0;
        const float sc = __ldg(p.scale + (size_t)b0 * 32 + lane);
        const float sh = p.shift ? __ldg(p.shift + (size_t)b0 * 32 + lane) : 0.f;
        sts_f32(ptab + 4 * lane, sc);
        sts_f32(ptab + 128 + 4 * lane, fmaf(bias_l, sc, sh));
        __syncwarp();
      }
    }
    mbar_wait(acc_full + 8 * as, pacc);
    tc_fence_after();
    if (t < p.T) {
      float o0 = tb.x, o1 = tb.y, o2 = tb.z, o3 = tb.w;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        uint32_t v[16];
        tmem_ld16(tmem_row + (uint32_t)((as * p.T + t) * 32 + 16 * k), v);
        tmem_ld_wait();
        float f[16];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float4 bc = lds_f4(ptab + 128 + 64 * k + 16 * g);
          if (kScale) {
            const float4 a = lds_f4(ptab + 64 * k + 16 * g);
            f[g * 4 + 0] = fmaf(__uint_as_float(v[g * 4 + 0]), a.x, bc.x); f[g * 4 + 1] = fmaf(__uint_as_float(v[g * 4 + 1]), a.y, bc.y);
            f[g * 4 + 2] = fmaf(__uint_as_float(v[g * 4 + 2]), a.z, bc.z); f[g * 4 + 3] = fmaf(__uint_as_float(v[g * 4 + 3]), a.w, bc.w);
          } else {
            f[g * 4 + 0] = __uint_as_float(v[g * 4 + 0]) + bc.x; f[g * 4 + 1] = __uint_as_float(v[g * 4 + 1]) + bc.y;
            f[g * 4 + 2] = __uint_as_float(v[g * 4 + 2]) + bc.z; f[g * 4 + 3] = __uint_as_float(v[g * 4 + 3]) + bc.w;
          }
        }
        if (silu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = fast_silu(f[j]);
        } else if (lrelu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], f[j] * slope);
        }
        if (kRes) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float2 a = unpack_bf16x2(rr[k].v[j]);
            f[2 * j] += a.x;
            f[2 * j + 1] += a.y;
          }
        }
        // the unfused layer stores bf16 and the output conv reads it back: keep that rounding, so that the fused result is
        // bit-identical to the two-kernel form (same float32 accumulation order below)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float2 a = unpack_bf16x2(pack_bf16x2(f[2 * j], f[2 * j + 1]));
          f[2 * j] = a.x;
          f[2 * j + 1] = a.y;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float4 wj = lds_f4(tailtab + (uint32_t)(16 * k + j) * 16);
          o0 = fmaf(f[j], wj.x, o0); o1 = fmaf(f[j], wj.y, o1); o2 = fmaf(f[j], wj.z, o2); o3 = fmaf(f[j], wj.w, o3);
        }
      }
      if (ok) {
        if (p.tail_res) {
          const float inv = 1.0f / ub;
          o0 += zi.x * inv; o1 += zi.y * inv; o2 += zi.z * inv; o3 += zi.w * inv;
        }
        reinterpret_cast<float4*>(p.tail_y)[pix] = make_float4(o0 * ub, o1 * ub, o2 * ub, o3 * ub);
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(acc_empty + 8 * as);
    if (++as == p.acc_stages) { as = 0; pacc ^= 1; }
  }
}

template <bool kPair>  // kPair: CTA-pair build (cluster of 2, cta_group::2 instructions); launched with a cluster dimension
__global__ void __launch_bounds__(kThreads, 1)
conv_tc_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: swizzle atoms (8 rows x 128 B) are defined on absolute address bits.
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_base + p.smem_b_off;
  const uint32_t bars = smem_base + p.smem_bar_off;
  const uint32_t a_full = bars, a_empty = a_full + 8 * kMaxStagesA;
  const uint32_t b_full = a_empty + 8 * kMaxStagesA, b_empty = b_full + 8 * kMaxStagesB;
  const uint32_t acc_full = b_empty + 8 * kMaxStagesB, acc_empty = acc_full + 16;
  const uint32_t w_full = acc_empty + 16;
  const uint32_t tmem_slot = w_full + 8;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t row_bytes = p.CB * 2;
  const int total_tiles = p.tiles_b * p.tiles_h * p.tiles_w * p.tiles_n;
  const int n_ast = num_astages(p);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.SA; ++i) { mbar_init(a_full + 8 * i, 1); mbar_init(a_empty + 8 * i, 1); }
    for (int i = 0; i < p.SB; ++i) { mbar_init(b_full + 8 * i, 1); mbar_init(b_empty + 8 * i, 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(acc_full + 8 * i, 1);
      // pair: both CTAs' epilogue warps report to the leader; split epilogue: one group of kEpiWarps/2 per stage
      mbar_init(acc_empty + 8 * i, (kPair ? 2 * kEpiWarps : kEpiWarps) >> (p.epi_split ? 1 : 0));
    }
    mbar_init(w_full, 1);
    fence_barrier_init();
  }
  if (p.tail_w) {  // [32][4] weights + [4] bias of the fused output conv
    for (int i = threadIdx.x; i < 132; i += blockDim.x)
      sts_f32(smem_base + p.smem_tail_off + 4 * i, i < 128 ? __ldg(p.tail_w + i) : __ldg(p.tail_b + i - 128));
  }
  if (warp == 1) {
    if (kPair) {
      tmem_alloc_pair(tmem_slot, p.tmem_cols);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_slot, p.tmem_cols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();  // the peer's barriers are initialised before anything is signalled across the pair
  tc_fence_after();
  const TileSched sched = make_sched<kPair>(p, total_tiles);
  const bool pair_leader = sched.rank == 0;
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ===================== TMA producer =====================
    // Converged warp, one elected lane issues (keeps coordinates / addresses in uniform registers).
    const uint32_t is_leader = elect_one();
    if (is_leader) {
      tma_prefetch_desc(&maps.w);
      tma_prefetch_desc(&maps.a[0]);
      if (p.wres && p.mode == CONV_UPSC) {
        mbar_expect_tx(w_full, p.ncb0 * p.b_stage_bytes + p.ncb1 * p.b2_stage_bytes);
        for (int i = 0; i < p.ncb0; ++i) tma_load_2d(smem_b + i * p.b_stage_bytes, &maps.w, w_full, 0, i * p.N);
        for (int i = 0; i < p.ncb1; ++i) tma_load_2d(smem_b + p.b2_off + i * p.b2_stage_bytes, &maps.w2, w_full, 0, i * p.Cout);
      } else if (p.wres) {  // all weight tiles of this layer stay in smem for the kernel's lifetime
        const int nwt = num_wtiles(p);
        mbar_expect_tx(w_full, nwt * p.b_stage_bytes);
        for (int i = 0; i < nwt; ++i) tma_load_2d(smem_b + i * p.b_stage_bytes, &maps.w, w_full, 0, i * p.N);
      }
    }
    __syncwarp();
    int sa = 0, pa = 0, sb = 0, pb = 0;
    // CTA pair: "data landed" is counted on the LEADER's barriers (its MMA consumes both CTAs' stages); the leader
    // expects the bytes of both CTAs, the peer only issues its loads.  "Stage free" arrives on each CTA's own barrier
    // through the multicast commit.
    const uint32_t a_full_sig = kPair ? mapa_shared(a_full, 0) : a_full;
    const uint32_t b_full_sig = kPair ? mapa_shared(b_full, 0) : b_full;
    const uint32_t b_half = kPair ? (uint32_t)(sched.rank * (p.NT / 2)) : 0u;  // this CTA's rows of every weight tile
    for (int u = sched.first; u < sched.n_units; u += sched.step) {
      const TileCoord tc = decode_tile(p, sched_tile(p, sched, u));
      for (int ai = 0; ai < n_ast; ++ai) {
        const AStage s = decode_astage(p, ai);
        mbar_wait(a_empty + 8 * sa, pa ^ 1);
        if (is_leader) {
          if (kPair) {
            if (pair_leader) mbar_expect_tx(a_full + 8 * sa, 2 * p.a_tx_bytes);
            tma_load_4d_pair(smem_a + sa * p.a_stage_bytes, &maps.a[s.map], a_full_sig + 8 * sa, s.c, tc.w0 + s.dw, tc.b0, tc.h0 + s.dh);
          } else {
            mbar_expect_tx(a_full + 8 * sa, p.a_tx_bytes);
            tma_load_4d(smem_a + sa * p.a_stage_bytes, &maps.a[s.map], a_full + 8 * sa, s.c, tc.w0 + s.dw, tc.b0, tc.h0 + s.dh);
          }
        }
        __syncwarp();
        if (++sa == p.SA) { sa = 0; pa ^= 1; }
        if (!p.wres) {
          for (int j = 0; j < s.ntaps; ++j) {
            const int widx = s.widx0 + j;
            mbar_wait(b_empty + 8 * sb, pb ^ 1);
            if (is_leader) {
              if (kPair) {
                if (pair_leader) mbar_expect_tx(b_full + 8 * sb, 2 * p.b_stage_bytes);
                tma_load_2d_pair(smem_b + sb * p.b_stage_bytes, &maps.w, b_full_sig + 8 * sb, 0, widx * p.N + tc.n0 + (int)b_half);
              } else {
                mbar_expect_tx(b_full + 8 * sb, p.b_stage_bytes);
                tma_load_2d(smem_b + sb * p.b_stage_bytes, &maps.w, b_full + 8 * sb, 0, widx * p.N + tc.n0);
              }
            }
            __syncwarp();
            if (++sb == p.SB) { sb = 0; pb ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp stays converged and ONE elected lane issues the tcgen05 instructions.  tcgen05.mma takes its
    // descriptors from UNIFORM registers, so every value on the issue path must be provably warp-uniform for the
    // compiler: values read through inline asm / shared memory (TMEM base, smem base) are laundered through a
    // warp reduction (REDUX writes a uniform register), loop state is only updated in converged code, and the elected
    // region derives everything from that state.  Otherwise each tap pays ~9 R2UR moves (~375 cycles, measured)
    // — far more than its MMAs (40/48/64 cycles each for N = 32/64/128, tools/mma_rate.cu).
    const uint32_t u_tmem = __reduce_max_sync(0xffffffffu, tmem_base);
    const uint32_t u_smem_a = __reduce_max_sync(0xffffffffu, smem_a);
    const uint32_t u_smem_b = __reduce_max_sync(0xffffffffu, smem_b);
    const uint32_t u_bars = __reduce_max_sync(0xffffffffu, bars);
    const uint32_t ua_full = u_bars, ua_empty = ua_full + 8 * kMaxStagesA;
    const uint32_t ub_full = ua_empty + 8 * kMaxStagesA, ub_empty = ub_full + 8 * kMaxStagesB;
    const uint32_t uacc_full = ub_empty + 8 * kMaxStagesB, uacc_empty = uacc_full + 16;
    const uint32_t uw_full = uacc_empty + 16;
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.NT >> 3) << 17) | (((kPair ? 256u : 128u) >> 4) << 24);
    const uint32_t idesc_full = idesc;
    const int ksteps = p.CB / 16;
    const uint32_t layout = (row_bytes == 128) ? 2u : 4u;  // SWIZZLE_128B : SWIZZLE_64B
    // high words: stride byte offset [32,46), version 1 at bit 46, layout type at [61,64)
    const uint32_t a_hi = ((p.sbo >> 4) & 0x3FFFu) | (1u << 14) | (layout << 29);
    const uint32_t b_hi = (((8u * row_bytes) >> 4) & 0x3FFFu) | (1u << 14) | (layout << 29);
    const uint32_t lo_flags = 1u << 16;  // leading byte offset field (ignored for swizzled K-major operands)
    const uint32_t sub_step = p.sub_off >> 4;
    const uint32_t tap_r16 = p.tap_r_off >> 4, px16 = row_bytes >> 4;
    const uint32_t nt = (uint32_t)p.NT;
    const bool leader = elect_one() != 0;
    if (p.wres) mbar_wait(uw_full, 0);
    int sa = 0, pa = 0, sb = 0, pb = 0, as = 0, pacc = 0;
    // The commonest shape — 3x3 stride 1, weights resident, ONE halo slab per tile (32 / 64 input channels: the four layers of
    // each full- and half-resolution block) — gets a loop of its own.  A single warp retires roughly one dependent instruction
    // every 5 cycles, and tcgen05.mma issue blocks once a few MMAs are queued, so whatever this warp executes between the last
    // MMA of a tile and the first of the next is time the tensor pipe drains and idles: the generic loop below spends up to
    // ~1100 cycles per tile there (stage decode, the dispatch on T / K steps / pairing, ring bookkeeping; measured with cycle
    // counters, their own cost included) against 4500-5700 cycles for a tile of these layers.  Here everything tile-invariant is
    // hoisted and the dispatch happens once, outside the loop.
    const bool fast_slab1 = p.wres && p.mode == CONV_3X3_S1 && n_ast == 1 && !kPair;
    if (fast_slab1) {
      const uint32_t b_first = (((u_smem_b) & 0x3FFFFu) >> 4) | lo_flags;  // the slab's channel block is 0: widx0 = 0
      const uint32_t b_step16 = p.b_stage_bytes >> 4;
      const uint32_t a_bytes = p.a_stage_bytes, acc_cols = (uint32_t)p.T * nt;
      const int SA = p.SA, nacc = p.acc_stages;
      auto run = [&](auto issue) {
        for (int u = sched.first; u < sched.n_units; u += sched.step) {
          mbar_wait(uacc_empty + 8 * as, pacc ^ 1);
          mbar_wait(ua_full + 8 * sa, pa);
          tc_fence_after();
          if (leader) {
            issue(u_tmem + (uint32_t)as * acc_cols, (((u_smem_a + (uint32_t)sa * a_bytes) & 0x3FFFFu) >> 4) | lo_flags);
            umma_commit(ua_empty + 8 * sa);
            umma_commit(uacc_full + 8 * as);
          }
          __syncwarp();
          if (++sa == SA) { sa = 0; pa ^= 1; }
          if (++as == nacc) { as = 0; pacc ^= 1; }
        }
      };
#define YOND_SLAB1(FN) run([&](uint32_t d, uint32_t a_lo) { FN(d, nt, a_lo, tap_r16, px16, sub_step, b_first, b_step16, a_hi, b_hi, idesc, 0u); })
      if (p.paired) {
        if (p.T == 1) YOND_SLAB1((issue_slab_paired<1>));
        else if (p.T == 2) YOND_SLAB1((issue_slab_paired<2>));
        else YOND_SLAB1((issue_slab_paired<4>));
      } else if (ksteps == 4) {
        if (p.T == 1) YOND_SLAB1((issue_slab_resident<4, 1>));
        else if (p.T == 2) YOND_SLAB1((issue_slab_resident<4, 2>));
        else YOND_SLAB1((issue_slab_resident<4, 4>));
      } else {
        if (p.T == 1) YOND_SLAB1((issue_slab_resident<2, 1>));
        else if (p.T == 2) YOND_SLAB1((issue_slab_resident<2, 2>));
        else YOND_SLAB1((issue_slab_resident<2, 4>));
      }
#undef YOND_SLAB1
    }
    // The other resident-weight layers (stride-2 3x3, 1x1, ConvT 2x2, the fused up-sampling + shortcut) consume one weight tile per
    // activation stage, 2-36 stages per tile.  Their stage decode (weight-tile address, and for the skip part of CONV_UPSC a
    // narrower N and a column offset into the accumulator) does not depend on the tile: it is tabulated once in shared memory
    // (the unused output-conv table region) and the per-stage work of this warp shrinks to a barrier wait, one 16-byte load and
    // the MMAs.  (conv_tc_launch bounds n_ast by kMaxTabStages; the fused output conv, whose table shares the region, is 3x3 only.)
    const bool fast_tab = p.wres && p.mode != CONV_3X3_S1 && !kPair;
    if (fast_tab) {
      const uint32_t tab = smem_base + p.smem_tail_off;
      for (int ai = lane; ai < n_ast; ai += 32) {
        const AStage s = decode_astage(p, ai);
        uint32_t b_lo0 = (((smem_b + (uint32_t)s.widx0 * p.b_stage_bytes) & 0x3FFFFu) >> 4) | lo_flags;
        uint32_t id = idesc_full, d_off = 0;
        if (p.mode == CONV_UPSC && s.sx >= 0) {  // skip part: N = Cout, accumulate into parity s.sx's columns
          b_lo0 = (((smem_b + p.b2_off + (uint32_t)s.widx0 * p.b2_stage_bytes) & 0x3FFFFu) >> 4) | lo_flags;
          id = (idesc_full & ~(0x3Fu << 17)) | ((uint32_t)(p.Cout >> 3) << 17);
          d_off = (uint32_t)(s.sx * p.Cout);
        }
        sts_u4(tab + 16u * (uint32_t)ai, b_lo0, id, d_off, 0u);
      }
      __syncwarp();
      const uint32_t a_bytes = p.a_stage_bytes, acc_cols = (uint32_t)p.T * nt;
      const int SA = p.SA, nacc = p.acc_stages;
      auto run = [&](auto issue) {
        for (int u = sched.first; u < sched.n_units; u += sched.step) {
          mbar_wait(uacc_empty + 8 * as, pacc ^ 1);
          const uint32_t d_tile = u_tmem + (uint32_t)as * acc_cols;
          for (int ai = 0; ai < n_ast; ++ai) {
            mbar_wait(ua_full + 8 * sa, pa);
            tc_fence_after();
            if (leader) {
              const uint4 e = lds_u4(tab + 16u * (uint32_t)ai);
              issue(d_tile + e.z, (((u_smem_a + (uint32_t)sa * a_bytes) & 0x3FFFFu) >> 4) | lo_flags, e.x, e.y, ai ? 1u : 0u);
              umma_commit(ua_empty + 8 * sa);
            }
            __syncwarp();
            if (++sa == SA) { sa = 0; pa ^= 1; }
          }
          if (leader) umma_commit(uacc_full + 8 * as);
          __syncwarp();
          if (++as == nacc) { as = 0; pacc ^= 1; }
        }
      };
#define YOND_TAB(KS, TT) run([&](uint32_t d, uint32_t a_lo, uint32_t b_lo, uint32_t id, uint32_t acc) { issue_tap<KS, TT>(d, nt, a_lo, sub_step, b_lo, a_hi, b_hi, id, acc); })
      if (ksteps == 4) {
        if (p.T == 1) YOND_TAB(4, 1);
        else if (p.T == 2) YOND_TAB(4, 2);
        else YOND_TAB(4, 4);
      } else {
        if (p.T == 1) YOND_TAB(2, 1);
        else if (p.T == 2) YOND_TAB(2, 2);
        else YOND_TAB(2, 4);
      }
#undef YOND_TAB
    }
    // Streamed weights, one halo slab per 64-channel block (the 128- to 512-channel 3x3 layers, normally as CTA pairs): nine taps
    // per stage, each waiting for its weight tile and handing the ring slot back.  Same hoisting: T is dispatched once, the
    // stage needs no decode at all (the slab is the whole story for this warp; weight tiles arrive in ring order).
    const bool fast_stream = !p.wres && p.mode == CONV_3X3_S1 && ksteps == 4;
    if (fast_stream && (!kPair || pair_leader)) {
      const uint32_t a_bytes = p.a_stage_bytes, b_bytes = p.b_stage_bytes, acc_cols = (uint32_t)p.T * nt;
      const int SA = p.SA, SB = p.SB, nacc = p.acc_stages;
      auto commit = [&](uint32_t bar) {
        if (kPair) umma_commit_pair(bar);
        else umma_commit(bar);
      };
      auto run = [&](auto issue) {
        for (int u = sched.first; u < sched.n_units; u += sched.step) {
          mbar_wait(uacc_empty + 8 * as, pacc ^ 1);
          const uint32_t d_tile = u_tmem + (uint32_t)as * acc_cols;
          for (int ai = 0; ai < n_ast; ++ai) {
            mbar_wait(ua_full + 8 * sa, pa);
            tc_fence_after();
            if (leader) {
              const uint32_t a_stage_lo = (((u_smem_a + (uint32_t)sa * a_bytes) & 0x3FFFFu) >> 4) | lo_flags;
              int lsb = sb, lpb = pb;
#pragma unroll
              for (int j = 0; j < 9; ++j) {
                const uint32_t r = j / 3, sx = j % 3;
                mbar_wait(ub_full + 8 * lsb, lpb);
                tc_fence_after();
                issue(d_tile, a_stage_lo + r * tap_r16 + sx * px16, (((u_smem_b + (uint32_t)lsb * b_bytes) & 0x3FFFFu) >> 4) | lo_flags,
                      (ai | j) ? 1u : 0u);
                commit(ub_empty + 8 * lsb);
                if (++lsb == SB) { lsb = 0; lpb ^= 1; }
              }
              commit(ua_empty + 8 * sa);
            }
            __syncwarp();
            sb += 9;  // advance the weight ring by this stage's taps, in converged code
            while (sb >= SB) { sb -= SB; pb ^= 1; }
            if (++sa == SA) { sa = 0; pa ^= 1; }
          }
          if (leader) commit(uacc_full + 8 * as);
          __syncwarp();
          if (++as == nacc) { as = 0; pacc ^= 1; }
        }
      };
#define YOND_STREAM(TT)                                                                                                   \
  run([&](uint32_t d, uint32_t a_lo, uint32_t b_lo, uint32_t acc) {                                                      \
    if (kPair) issue_tap_pair<4, TT>(d, nt, a_lo, sub_step, b_lo, a_hi, b_hi, idesc, acc);                               \
    else issue_tap<4, TT>(d, nt, a_lo, sub_step, b_lo, a_hi, b_hi, idesc, acc);                                          \
  })
      if (p.T == 1) YOND_STREAM(1);
      else if (p.T == 2) YOND_STREAM(2);
      else YOND_STREAM(4);
#undef YOND_STREAM
    }
    // Everything no loop above takes: resident-weight 3x3 layers with several halo slabs (a concatenation of two 32-channel
    // sources), and streamed layers with one weight tile per stage (stride-2 3x3, 1x1 / ConvT / fused up-sampling too wide to stay
    // resident, and 3x3 with 32-channel blocks).  Every CTA-pair plan takes fast_stream, where the peer CTA's warp 1 idles.
    if (!kPair && !fast_slab1 && !fast_tab && !fast_stream) {
      for (int u = sched.first; u < sched.n_units; u += sched.step) {
        mbar_wait(uacc_empty + 8 * as, pacc ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = u_tmem + (uint32_t)(as * p.T) * nt;
        for (int ai = 0; ai < n_ast; ++ai) {
          const AStage s = decode_astage(p, ai);
          mbar_wait(ua_full + 8 * sa, pa);
          tc_fence_after();
          const uint32_t a_stage_lo = (((u_smem_a + (uint32_t)sa * p.a_stage_bytes) & 0x3FFFFu) >> 4) | lo_flags;
          if (leader && p.wres) {
            // resident weights, 3x3 stride 1: 9 taps x T sub-tiles x K steps of this slab as one straight-line burst
            const uint32_t b_first = (((u_smem_b + (uint32_t)s.widx0 * p.b_stage_bytes) & 0x3FFFFu) >> 4) | lo_flags;
            const uint32_t b_step16 = p.b_stage_bytes >> 4;
            const uint32_t acc0 = ai ? 1u : 0u;
            if (ksteps == 4) {
              if (p.T == 1) issue_slab_resident<4, 1>(d_tmem, nt, a_stage_lo, tap_r16, px16, sub_step, b_first, b_step16, a_hi, b_hi, idesc, acc0);
              else if (p.T == 2) issue_slab_resident<4, 2>(d_tmem, nt, a_stage_lo, tap_r16, px16, sub_step, b_first, b_step16, a_hi, b_hi, idesc, acc0);
              else issue_slab_resident<4, 4>(d_tmem, nt, a_stage_lo, tap_r16, px16, sub_step, b_first, b_step16, a_hi, b_hi, idesc, acc0);
            } else {
              if (p.T == 1) issue_slab_resident<2, 1>(d_tmem, nt, a_stage_lo, tap_r16, px16, sub_step, b_first, b_step16, a_hi, b_hi, idesc, acc0);
              else if (p.T == 2) issue_slab_resident<2, 2>(d_tmem, nt, a_stage_lo, tap_r16, px16, sub_step, b_first, b_step16, a_hi, b_hi, idesc, acc0);
              else issue_slab_resident<2, 4>(d_tmem, nt, a_stage_lo, tap_r16, px16, sub_step, b_first, b_step16, a_hi, b_hi, idesc, acc0);
            }
            umma_commit(ua_empty + 8 * sa);
          } else if (leader) {
            // streamed weights: each tap waits for its weight tile and hands the ring slot back
            int lsb = sb, lpb = pb;  // weight-ring position of this stage's first tap (uniform on entry)
            for (int j = 0; j < s.ntaps; ++j) {
              uint32_t r = 0, sx = 0;
              if (p.mode == CONV_3X3_S1) { r = (j >= 3) + (j >= 6); sx = j - r * 3; }
              mbar_wait(ub_full + 8 * lsb, lpb);
              tc_fence_after();
              const uint32_t a_lo0 = a_stage_lo + r * tap_r16 + sx * px16;
              const uint32_t b_lo0 = (((u_smem_b + (uint32_t)lsb * p.b_stage_bytes) & 0x3FFFFu) >> 4) | lo_flags;
              const uint32_t accum = (ai | j) ? 1u : 0u;
              if (ksteps == 4) {
                if (p.T == 1) issue_tap<4, 1>(d_tmem, nt, a_lo0, sub_step, b_lo0, a_hi, b_hi, idesc, accum);
                else if (p.T == 2) issue_tap<4, 2>(d_tmem, nt, a_lo0, sub_step, b_lo0, a_hi, b_hi, idesc, accum);
                else issue_tap<4, 4>(d_tmem, nt, a_lo0, sub_step, b_lo0, a_hi, b_hi, idesc, accum);
              } else {
                if (p.T == 1) issue_tap<2, 1>(d_tmem, nt, a_lo0, sub_step, b_lo0, a_hi, b_hi, idesc, accum);
                else if (p.T == 2) issue_tap<2, 2>(d_tmem, nt, a_lo0, sub_step, b_lo0, a_hi, b_hi, idesc, accum);
                else issue_tap<2, 4>(d_tmem, nt, a_lo0, sub_step, b_lo0, a_hi, b_hi, idesc, accum);
              }
              umma_commit(ub_empty + 8 * lsb);
              if (++lsb == p.SB) { lsb = 0; lpb ^= 1; }
            }
            umma_commit(ua_empty + 8 * sa);
          }
          __syncwarp();
          if (!p.wres) {  // advance the weight ring by this stage's taps, in converged code
            sb += s.ntaps;
            while (sb >= p.SB) { sb -= p.SB; pb ^= 1; }
          }
          if (++sa == p.SA) { sa = 0; pa ^= 1; }
        }
        if (leader) umma_commit(uacc_full + 8 * as);
        __syncwarp();
        if (++as == p.acc_stages) { as = 0; pacc ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (warps 2..2+kEpiWarps) =====================
    const bool silu = p.act == ACT_SILU;
    const uint32_t ptab = smem_base + p.smem_epi_off + (uint32_t)(warp - 2) * 256u;
#define YOND_EPI(S, R, A, V) epilogue_loop<S, R, A, V, kPair>(p, tmem_base, acc_full, acc_empty, ptab, warp, lane, total_tiles)
    const bool few = p.T * (p.NT / 16) <= 8;  // at most two visits per warp and tile: hold two residual rows, not four
    if (!kPair && p.tail_w) {
      const uint32_t tailtab = smem_base + p.smem_tail_off;
      if (p.scale && p.res) epilogue_tail<true, true>(p, tmem_base, acc_full, acc_empty, ptab, tailtab, warp, lane, total_tiles);
      else if (p.scale) epilogue_tail<true, false>(p, tmem_base, acc_full, acc_empty, ptab, tailtab, warp, lane, total_tiles);
      else if (p.res) epilogue_tail<false, true>(p, tmem_base, acc_full, acc_empty, ptab, tailtab, warp, lane, total_tiles);
      else epilogue_tail<false, false>(p, tmem_base, acc_full, acc_empty, ptab, tailtab, warp, lane, total_tiles);
    }
    else if (p.scale && p.res) { if (silu) YOND_EPI(true, true, true, 2); else YOND_EPI(true, true, false, 2); }
    else if (p.scale && epilogue_single_set(p)) {
      if (silu) epilogue_loop<true, false, true, 4, kPair, true>(p, tmem_base, acc_full, acc_empty, ptab, warp, lane, total_tiles);
      else epilogue_loop<true, false, false, 4, kPair, true>(p, tmem_base, acc_full, acc_empty, ptab, warp, lane, total_tiles);
    }
    else if (p.scale) { if (silu) YOND_EPI(true, false, true, 4); else YOND_EPI(true, false, false, 4); }
    else if (p.res && epilogue_single_set(p)) {
#define YOND_EPI_R(A, V) epilogue_loop<false, true, A, V, kPair, true>(p, tmem_base, acc_full, acc_empty, ptab, warp, lane, total_tiles)
      if (few) { if (silu) YOND_EPI_R(true, 2); else YOND_EPI_R(false, 2); }
      else { if (silu) YOND_EPI_R(true, 4); else YOND_EPI_R(false, 4); }
#undef YOND_EPI_R
    }
    else if (p.res) {
      if (few) { if (silu) YOND_EPI(false, true, true, 2); else YOND_EPI(false, true, false, 2); }
      else { if (silu) YOND_EPI(false, true, true, 4); else YOND_EPI(false, true, false, 4); }
    }
    else if (epilogue_single_set(p)) {
      if (silu) epilogue_loop<false, false, true, 4, kPair, true>(p, tmem_base, acc_full, acc_empty, ptab, warp, lane, total_tiles);
      else epilogue_loop<false, false, false, 4, kPair, true>(p, tmem_base, acc_full, acc_empty, ptab, warp, lane, total_tiles);
    }
    else { if (silu) YOND_EPI(false, false, true, 4); else YOND_EPI(false, false, false, 4); }
#undef YOND_EPI
  }

  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();  // the peer's shared memory / barriers stay valid until both CTAs are done
  if (warp == 1) {
    tc_fence_after();
    if (kPair) tmem_dealloc_pair(tmem_base, p.tmem_cols);
    else tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

// Activation map over an NHWC bf16 tensor viewed as dims (C, W, B, H) so that a box lands in smem as
// [h][b][w][c]: one image row of the tile (all its images, all its columns) is contiguous.
int make_act_map(CUtensorMap* m, const bf16* base, int C, int W, int B, int H, uint64_t strideW, uint64_t strideB,
                 uint64_t strideH, int CB, int box_w, int box_b, int box_h) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return yond_set_error(YOND_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)B, (cuuint64_t)H};
  cuuint64_t strides[3] = {strideW, strideB, strideH};
  cuuint32_t box[4] = {(cuuint32_t)CB, (cuuint32_t)box_w, (cuuint32_t)box_b, (cuuint32_t)box_h};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<bf16*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CB == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return yond_set_error(YOND_ERR_CUDA, "cuTensorMapEncodeTiled(act) failed: %d (C=%d W=%d B=%d H=%d box=%d,%d,%d,%d)",
                          (int)r, C, W, B, H, CB, box_w, box_b, box_h);
  return YOND_OK;
}

int make_weight_map(CUtensorMap* m, const bf16* base, int CB, size_t rows, int NT) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return yond_set_error(YOND_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)CB, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)CB * 2};
  cuuint32_t box[2] = {(cuuint32_t)CB, (cuuint32_t)NT};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CB == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return yond_set_error(YOND_ERR_CUDA, "cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
  return YOND_OK;
}

int pow2_ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

}  // namespace

int conv_tc_channel_block(int Cin0, int Cin1) {
  return (Cin0 % 64 == 0 && Cin1 % 64 == 0) ? 64 : 32;
}

size_t conv_tc_packed_elems(int mode, int Cin_total, int Cout) {
  if (mode == CONV_UPSC) return (size_t)(Cin_total - Cout) * 4 * Cout + (size_t)Cout * Cout;  // folded part + skip part
  int taps = (mode == CONV_3X3_S1 || mode == CONV_3X3_S2) ? 9 : 1;
  int N = (mode == CONVT_2X2) ? 4 * Cout : Cout;
  return (size_t)taps * Cin_total * N;
}

void conv_tc_pack_paired(const float* w, bf16* out) {
  for (int r = 0; r < 3; ++r)
    for (int P = -1; P <= 1; ++P)
      for (int o = 0; o < 2; ++o)
        for (int co = 0; co < 32; ++co)
          for (int i = 0; i < 2; ++i)
            for (int ci = 0; ci < 32; ++ci) {
              const int dx = 2 * P + i - o;
              const float v = (dx >= -1 && dx <= 1) ? w[((size_t)co * 32 + ci) * 9 + r * 3 + (dx + 1)] : 0.f;
              out[((size_t)(r * 3 + P + 1) * 64 + (o * 32 + co)) * 64 + (i * 32 + ci)] = __float2bfloat16_rn(v);
            }
}

int conv_tc_launch(const ConvLayer& Lin, cudaStream_t stream) {
  ConvLayer L = Lin;
  // (layers with a residual input are bound by their 3 x 64 B per pixel of HBM traffic, not by the MMAs: measured 930 us plain
  // vs 990-1030 us paired for 24.8 M pixels, so they keep the N = 32 form)
  const bool paired = L.wpaired && L.mode == CONV_3X3_S1 && L.Cin0 == 32 && L.Cin1 == 0 && L.Cout == 32 && L.Win % 2 == 0 &&
                      L.res == nullptr && L.tail_w == nullptr;
  if (paired) {  // (B,H,W,32) is (B,H,W/2,64): same memory, pixel pairs as 64-channel pixels
    L.Win /= 2;
    L.Cin0 = 64;
    L.Cout = 64;
    L.wpacked = L.wpaired;
  }
  YOND_REQUIRE(L.Cin0 % 32 == 0 && L.Cin1 % 32 == 0 && L.Cin0 > 0, "conv_tc: Cin must be a multiple of 32 (got %d,%d)",
               L.Cin0, L.Cin1);
  YOND_REQUIRE(L.Cout % 32 == 0, "conv_tc: Cout must be a multiple of 32 (got %d)", L.Cout);
  YOND_REQUIRE((double)L.B * L.Hin * L.Win * ((L.mode == CONVT_2X2 || L.mode == CONV_UPSC) ? 4.0 : 1.0) * L.Cout < 4294967296.0,
               "conv_tc: output of %d x %d x %d x %d elements exceeds the 32-bit offset range; split the batch", L.B, L.Hin, L.Win, L.Cout);
  YOND_REQUIRE(L.scale != nullptr || L.shift == nullptr, "conv_tc: a shift vector needs a scale vector");
  TcParams p{};
  p.mode = L.mode;
  p.B = L.B;
  if (L.mode == CONV_3X3_S2) {
    YOND_REQUIRE(L.Hin % 2 == 0 && L.Win % 2 == 0, "conv_tc: stride-2 conv needs even input dims");
    p.H = L.Hin / 2;
    p.W = L.Win / 2;
  } else {
    p.H = L.Hin;
    p.W = L.Win;
  }
  p.Cout = L.Cout;
  p.paired = paired ? 1 : 0;
  p.cvec = paired ? 32 : L.Cout;
  p.cmask = paired ? 31u : 0xffffffffu;
  const bool convt_like = L.mode == CONVT_2X2 || L.mode == CONV_UPSC;
  p.N = convt_like ? 4 * L.Cout : L.Cout;
  p.CB = conv_tc_channel_block(L.Cin0, L.Cin1);
  p.ncb0 = L.Cin0 / p.CB;
  p.ncb1 = L.Cin1 / p.CB;
  p.NT = p.N < kMaxNT ? p.N : kMaxNT;
  YOND_REQUIRE(p.N % p.NT == 0 && (p.NT & (p.NT - 1)) == 0, "conv_tc: unsupported N=%d", p.N);
  p.tiles_n = p.N / p.NT;
  const uint32_t row_bytes = p.CB * 2;
  const bool conv3 = L.mode == CONV_3X3_S1;

  // sub-tile: TH rows x NB images x TW columns = 128 GEMM rows.  3x3 convs use 8-pixel-wide tiles so that every
  // 8-row swizzle group is one image row of the slab (uniform stride between groups whatever the halo width).
  p.TW = conv3 ? 8 : (p.W > 8 ? 16 : 8);
  const int rows = 128 / p.TW;
  p.TH = pow2_ceil(p.H) < rows ? pow2_ceil(p.H) : rows;
  p.NB = rows / p.TH;
  const int ncb = p.ncb0 + p.ncb1;
  const int nwt = ((L.mode == CONV_3X3_S1 || L.mode == CONV_3X3_S2) ? 9 : 1) * ncb;
  const size_t smem_budget = 227 * 1024 - 2048 - kEpiWarps * 256 - 1024;  // ... and the table of a fused output conv  // dynamic smem minus alignment slack, barriers, parameter rows
  p.b_stage_bytes = (uint32_t)p.NT * row_bytes;
  YOND_REQUIRE(p.b_stage_bytes % 1024 == 0, "conv_tc: weight stage not 1024-aligned");
  size_t wres_bytes = (size_t)nwt * p.b_stage_bytes;
  if (L.mode == CONV_UPSC) {
    YOND_REQUIRE(L.Cin1 == L.Cout && L.src1 != nullptr, "conv_tc: fused up-sampling needs a skip source with Cout channels");
    p.b2_stage_bytes = (uint32_t)L.Cout * row_bytes;
    p.b2_off = (uint32_t)p.ncb0 * p.b_stage_bytes;
    wres_bytes = (size_t)p.b2_off + (size_t)p.ncb1 * p.b2_stage_bytes;
    YOND_REQUIRE(p.tiles_n == 1 && wres_bytes <= 80 * 1024 && p.b2_stage_bytes % 1024 == 0,
                 "conv_tc: fused up-sampling is built for resident weights (Cout <= 64); got Cout=%d", L.Cout);
  }
  p.wres = (p.tiles_n == 1 && wres_bytes <= 80 * 1024) ? 1 : 0;
  YOND_REQUIRE(!p.wres || conv3 || num_astages(p) <= kMaxTabStages, "conv_tc: %d resident-weight stages exceed the stage table (%d)",
               num_astages(p), kMaxTabStages);
  // CTA pairs for the layers that stream their weights (>= 128 channels): halves the per-SM weight traffic and the
  // shared-memory reads of the B operand, which is what bounds those layers with single-CTA MMAs.
  // (Resident-weight layers stay single-CTA: at N = 64 the A operand is 4 of the 6 KB an MMA reads, so halving B buys less than
  // the pair's cross-CTA hand-shakes cost; measured 25 % slower, DESIGN.md section 4.)
  p.cta2 = (conv3 && !p.wres && p.CB == 64 && p.NT >= kCta2MinNT && yond_num_sms() >= 2) ? 1 : 0;
  if (p.cta2) p.b_stage_bytes /= 2;  // each CTA of the pair holds NT/2 rows of every weight tile
  // T sub-tiles share each weight tile (and one halo slab): stacked along H when the map is tall enough, else along
  // the batch (sub-tile t = images t, t+T, ... of the tile, so that the 8-row groups keep a uniform stride).  T is
  // bounded by TMEM and by shared memory.  Resident-weight layers keep two accumulator stages (2 T NT <= 512 columns);
  // layers that stream their weights take T NT = 512 with a single stage when they can: the serialised epilogue
  // costs a few percent, re-streaming the whole weight set for half as many pixels costs L2 bandwidth, which is what
  // bounds them (measured: 256/512-channel layers moved ~7.7 TB/s of weights through L2 at T = 1).
  // Stride-2 / 1x1 / transposed layers stack their sub-tiles along H only (a taller box of whole 128-row tiles).
  int T = 1;
  {
    // (a CTA pair already halves the weight traffic per SM: it keeps both accumulator stages)
    int tmax = (p.wres || p.cta2) ? 512 / (2 * p.NT) : 512 / p.NT;
    if (tmax > kMaxT) tmax = kMaxT;
    if (p.NB == 1) {
      while (T * 2 <= tmax && (p.H >= p.TH * T * 2 || (conv3 && p.B >= T * 2))) T *= 2;
    } else if (conv3) {
      while (T * 2 <= tmax && p.B >= p.NB * T * 2) T *= 2;
    }
  }
  int slab_w = 0, slab_h = 0, SBt = 0;
  size_t b_region = 0;
  for (;; T /= 2) {
    p.T = T;
    p.t_along_h = (p.H >= p.TH * T) ? 1 : 0;
    const int SH = p.TH * (p.t_along_h ? T : 1);
    SBt = p.NB * (p.t_along_h ? 1 : T);
    p.tiles_w = ceil_div(p.W, p.TW);
    p.tiles_h = ceil_div(p.H, SH);
    p.tiles_b = ceil_div(p.B, SBt);
    slab_w = conv3 ? p.TW + 2 : p.TW;
    slab_h = conv3 ? SH + 2 : SH;
    const uint32_t line = (uint32_t)slab_w * row_bytes;  // one image row of one image inside a stage
    p.a_tx_bytes = (uint32_t)slab_h * SBt * line;
    p.a_stage_bytes = (uint32_t)align_up((size_t)p.a_tx_bytes, 1024);
    if (conv3) {
      p.tap_r_off = (uint32_t)SBt * line;
      p.sbo = p.t_along_h ? line : (uint32_t)T * line;
      p.sub_off = p.t_along_h ? (uint32_t)p.TH * line : line;
    } else {
      p.tap_r_off = 0;
      p.sbo = 8u * row_bytes;
      p.sub_off = (uint32_t)p.TH * line;  // = 128 rows: sub-tile t is the t-th whole tile of the box
    }
    if (p.wres) {
      p.SB = 1;
      b_region = wres_bytes;
      p.SA = (int)((smem_budget - b_region) / p.a_stage_bytes);
      if (p.SA > kMaxStagesA) p.SA = kMaxStagesA;
      if (p.SA >= 3 || T == 1) break;
    } else {
      // streamed weights: two activation stages (one stage feeds 9 taps x T sub-tiles of MMAs), the rest of the
      // shared memory goes to the weight ring, what is left after that back to the activations
      const size_t rest = smem_budget > 2 * (size_t)p.a_stage_bytes ? smem_budget - 2 * (size_t)p.a_stage_bytes : 0;
      p.SB = (int)(rest / p.b_stage_bytes);
      if (p.SB > kMaxStagesB) p.SB = kMaxStagesB;
      b_region = (size_t)p.SB * p.b_stage_bytes;
      p.SA = p.SB > 0 ? (int)((smem_budget - b_region) / p.a_stage_bytes) : 0;
      if (p.SA > kMaxStagesA) p.SA = kMaxStagesA;
      if ((p.SB >= 3 && p.SA >= 2) || T == 1) break;
    }
  }
  YOND_REQUIRE(p.SB >= 1, "conv_tc: not enough shared memory for the weight ring");
  YOND_REQUIRE(p.SA >= 2, "conv_tc: not enough shared memory for the activation pipeline");
  p.smem_b_off = (uint32_t)p.SA * p.a_stage_bytes;
  p.smem_bar_off = (uint32_t)align_up(p.smem_b_off + b_region, 1024);
  p.smem_epi_off = p.smem_bar_off + 512;
  p.smem_tail_off = p.smem_epi_off + kEpiWarps * 256;
  const size_t smem_bytes = p.smem_tail_off + 1024 + 1024;  // barriers, parameter rows, output-conv table, alignment slack
  p.acc_stages = 2 * p.T * p.NT <= 512 ? 2 : 1;
  // Measured inside a GuidedResUnet forward on 8 x 12 MP frames (ncu, profiles/r02_conv_layers_pairing.txt): the pixel-pair
  // layers 890 -> 767 us; every other layer is within +-2 % or loses 4 % (64-channel FiLM layers, residual layers), and the wide
  // layers (N tile >= 128: many visits per warp) lose up to 10 % in isolation — so only the paired layers split.
  p.epi_split = (p.acc_stages == 2 && p.paired) ? 1 : 0;
  p.tmem_cols = p.acc_stages * p.T * p.NT < 32 ? 32 : p.acc_stages * p.T * p.NT;
  YOND_REQUIRE(p.tmem_cols <= 512, "conv_tc: TMEM budget exceeded");

  p.fd_tiles_n = make_fastdiv((uint32_t)p.tiles_n);
  p.fd_tiles_w = make_fastdiv((uint32_t)p.tiles_w);
  p.fd_tiles_h = make_fastdiv((uint32_t)p.tiles_h);
  p.fd_cout = make_fastdiv((uint32_t)p.Cout);
  p.lg_nchunk = 0;
  while ((16 << p.lg_nchunk) < p.NT) ++p.lg_nchunk;
  if (convt_like) p.t_off = (uint32_t)p.TH * 4u * p.W * p.Cout;  // TH input rows = 2 TH output rows of 2 W pixels
  else p.t_off = (p.t_along_h ? (uint32_t)p.TH * p.W : (uint32_t)p.H * p.W) * (uint32_t)p.Cout;
  YOND_REQUIRE(L.act != ACT_LRELU || (L.slope >= 0.f && L.slope <= 1.f), "conv_tc: LeakyReLU slope must be in [0, 1]");
  {
    const int nchunk = p.NT / 16;
    p.epi_fixed = (p.tiles_n == 1 && nchunk <= 4 && p.NB == 1 && (p.T == 1 || p.t_along_h) && !convt_like) ? 1 : 0;
  }
  p.bias = L.bias;
  p.scale = L.scale;
  p.shift = L.shift;
  p.act = L.act;
  p.slope = L.slope;
  p.res = L.res;
  p.out0 = L.out0;
  p.out1 = L.out1;
  if (L.tail_w) {
    YOND_REQUIRE(L.mode == CONV_3X3_S1 && L.Cout == 32 && !paired && p.tiles_n == 1 && p.NT == 32 && p.T <= 4 && !p.cta2 && L.tail_b &&
                     L.tail_y && (L.tail_z || !L.tail_res),
                 "conv_tc: the fused output conv needs a 3x3 layer with 32 output channels");
    p.tail_w = L.tail_w;
    p.tail_b = L.tail_b;
    p.tail_z = L.tail_z;
    p.tail_ub = L.tail_ub;
    p.tail_y = L.tail_y;
    p.tail_res = L.tail_res;
    p.epi_split = 0;
  }

  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  const bf16* srcs[2] = {L.src0, L.src1};
  const int cins[2] = {L.Cin0, L.Cin1};
  for (int s = 0; s < 2; ++s) {
    if (cins[s] == 0) continue;
    const int C = cins[s];
    if (L.mode == CONV_UPSC && s == 1) {  // skip tensor at twice the tile-space resolution: one map per output parity
      for (int ph = 0; ph < 2; ++ph)
        for (int pw = 0; pw < 2; ++pw) {
          const int Wh = 2 * L.Win, Hh = 2 * L.Hin;
          const bf16* base = srcs[s] + ((size_t)ph * Wh + pw) * C;
          int rc = make_act_map(&maps.a[4 + ph * 2 + pw], base, C, L.Win, L.B, L.Hin, (uint64_t)2 * C * 2,
                                (uint64_t)Hh * Wh * C * 2, (uint64_t)2 * Wh * C * 2, p.CB, slab_w, SBt, slab_h);
          if (rc) return rc;
        }
    } else if (L.mode == CONV_3X3_S2) {
      for (int ph = 0; ph < 2; ++ph)
        for (int pw = 0; pw < 2; ++pw) {
          const bf16* base = srcs[s] + ((size_t)ph * L.Win + pw) * C;
          int rc = make_act_map(&maps.a[s * 4 + ph * 2 + pw], base, C, L.Win / 2, L.B, L.Hin / 2, (uint64_t)2 * C * 2,
                                (uint64_t)L.Hin * L.Win * C * 2, (uint64_t)2 * L.Win * C * 2, p.CB, slab_w, SBt, slab_h);
          if (rc) return rc;
        }
    } else {
      int rc = make_act_map(&maps.a[s], srcs[s], C, L.Win, L.B, L.Hin, (uint64_t)C * 2, (uint64_t)L.Hin * L.Win * C * 2,
                            (uint64_t)L.Win * C * 2, p.CB, slab_w, SBt, slab_h);
      if (rc) return rc;
    }
  }
  {
    const size_t rows_a = L.mode == CONV_UPSC ? (size_t)p.ncb0 * p.N : (size_t)nwt * p.N;
    int rc = make_weight_map(&maps.w, L.wpacked, p.CB, rows_a, p.cta2 ? p.NT / 2 : p.NT);
    if (rc) return rc;
    if (L.mode == CONV_UPSC) {
      rc = make_weight_map(&maps.w2, L.wpacked + rows_a * p.CB, p.CB, (size_t)p.ncb1 * L.Cout, L.Cout);
      if (rc) return rc;
    }
  }
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    attr_err = cudaFuncSetAttribute(conv_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (attr_err == cudaSuccess)
      attr_err = cudaFuncSetAttribute(conv_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  });
  if (attr_err != cudaSuccess)
    return yond_set_error(YOND_ERR_CUDA, "cudaFuncSetAttribute(conv_tc_kernel) failed: %s", cudaGetErrorString(attr_err));

  const int total_tiles = p.tiles_b * p.tiles_h * p.tiles_w * p.tiles_n;
  if (p.cta2) {
    const int m_tiles = total_tiles / p.tiles_n;
    const int units = ((m_tiles + 1) / 2) * p.tiles_n;
    int grid = yond_num_sms() & ~1;
    if (grid > 2 * units) grid = 2 * units;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<true>, maps, p);
    if (e != cudaSuccess) return yond_set_error(YOND_ERR_CUDA, "conv_tc: cluster launch failed: %s", cudaGetErrorString(e));
    yond_count_launch(1);
    return YOND_OK;
  }
  int grid = yond_num_sms();
  if (grid > total_tiles) grid = total_tiles;
  conv_tc_kernel<false><<<grid, kThreads, smem_bytes, stream>>>(maps, p);
  YOND_LAUNCH_CHECK();
  return YOND_OK;
}
