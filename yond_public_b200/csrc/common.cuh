// Shared helpers for libyond_b200 (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/yond_b200.h"

typedef __nv_bfloat16 bf16;

int yond_set_error(int code, const char* fmt, ...);
void yond_count_launch(int n = 1);

#define YOND_CUDA_CHECK(expr)                                                                        \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return yond_set_error(YOND_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),   \
                            __FILE__, __LINE__);                                                     \
  } while (0)

#define YOND_LAUNCH_CHECK()                                                                          \
  do {                                                                                               \
    cudaError_t _e = cudaGetLastError();                                                             \
    if (_e != cudaSuccess)                                                                           \
      return yond_set_error(YOND_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), \
                            __FILE__, __LINE__);                                                     \
    yond_count_launch();                                                                             \
  } while (0)

#define YOND_REQUIRE(cond, ...)                                                                      \
  do {                                                                                               \
    if (!(cond)) return yond_set_error(YOND_ERR_INVALID, __VA_ARGS__);                               \
  } while (0)

// Library-wide stage profiler (bench.py's live per-kernel roofline): while enabled (yond_prof_enable), a scope brackets
// the launches issued during its lifetime with CUDA events on the launching stream and books them under `name` together
// with the ALGORITHMIC bytes / FLOPs the caller states for them (SURVEY 8(d)).  Disabled: one relaxed atomic load.
struct YondProfScope {
  int slot;
  cudaStream_t stream;
  void* end_event;
  YondProfScope(const char* name, cudaStream_t s, double bytes, double flops = 0.0);
  ~YondProfScope();
};

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

// Number of SMs of the current device (148 on B200); cached.
int yond_num_sms();

__device__ __forceinline__ float silu_f(float v) { return v / (1.0f + __expf(-v)); }

// cv2.blur's border rule (BORDER_REFLECT_101) and torch's F.pad(mode='reflect') are the same map.
__host__ __device__ __forceinline__ int reflect101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) {
    if (i < 0) i = -i;
    if (i >= n) i = 2 * (n - 1) - i;
  }
  return i;
}

// 32-bit shared-window address of a __shared__ object, opaque to the compiler.  Indexing shared arrays inside hot per-element code
// otherwise makes nvcc REMATERIALISE the window base (S2R SR_CgaCtaId + shift + add) in front of every access on sm_100 — several
// extra instructions per element, one of them on the slow S2R path.  Take the address once, then ld.shared with register + immediate.
__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("" : "+r"(a));
  return a;
}
__device__ __forceinline__ int lds_s8(uint32_t a) {
  int v;
  asm("ld.shared.s8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds_v4f(uint32_t a) {
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void reds_add(uint32_t a, uint32_t by = 1u) {
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(by) : "memory");
}

// Sensor mosaic read in place of a float32 Bayer frame (SURVEY 8(f)-1): the dataset normalisation of
// data_process/yond_datasets.py:955-961 / :1053-1056, (float32(raw) - black) * ratio / (white - black) in float32 in that order,
// is applied on load, so the normalised frame never exists in memory (2 B/px instead of 4 per read).  base == nullptr: float source.
// per_img != nullptr: one yond_raw_norm per dataset image in device memory; a kernel's unit u (a box-filter image, a frame) belongs
// to image u / units_per_img, and raw_norm_at replaces the uniform fields with that image's entry, once per thread or CTA.
struct RawNorm {
  const uint16_t* base;
  float bl, ratio, denom;
  int clip;
  const yond_raw_norm* per_img;
  int units_per_img;
};
__device__ __forceinline__ float raw_norm(uint32_t v, const RawNorm& q) {
  float t = __fdiv_rn(__fmul_rn(__fsub_rn((float)v, q.bl), q.ratio), q.denom);
  if (q.clip) t = fminf(fmaxf(t, 0.f), 1.f);
  return t;
}
__device__ __forceinline__ RawNorm raw_norm_at(RawNorm q, int unit) {
  if (q.per_img) {
    const yond_raw_norm n = q.per_img[unit / q.units_per_img];
    q.bl = n.black;
    q.ratio = n.ratio;
    q.denom = __fsub_rn(n.white, n.black);  // the host's float32 white - black of make_raw_norm
    q.clip = n.clip;
  }
  return q;
}
static inline RawNorm make_raw_norm(const uint16_t* base, const yond_raw_norm* n, const yond_raw_norm* per_img = nullptr,
                                    int units_per_img = 1) {
  RawNorm q{};
  if (base && (n || per_img)) {
    q.base = base;
    if (n) {
      q.bl = n->black;
      q.ratio = n->ratio;
      q.denom = n->white - n->black;
      q.clip = n->clip;
    }
    q.per_img = per_img;
    q.units_per_img = units_per_img;
  }
  return q;
}

__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_stream_u2(const uint2* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float2 ldg_stream_f2(const float2* p) {
  float2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
}
