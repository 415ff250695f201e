// Shared device helpers for libssdgeom (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/ssdgeom.h"

#define SSDG_FULL 0xffffffffu

#define SSDG_CUDA_TRY(expr)                      \
  do {                                           \
    cudaError_t _e = (expr);                     \
    if (_e != cudaSuccess) return (int)_e;       \
  } while (0)

#define SSDG_LAUNCH_CHECK()                      \
  do {                                           \
    cudaError_t _e = cudaGetLastError();         \
    if (_e != cudaSuccess) return (int)_e;       \
  } while (0)

typedef unsigned long long u64;
typedef unsigned int u32;

namespace ssdg {

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int sm_count();          // cached multiprocessor count of the current device
int max_smem_optin();    // cached max dynamic shared memory per block (opt-in)

// Optional event bracketing of the dominant kernels (ssdg_profile_enable).
void prof_begin(int which, cudaStream_t st);
void prof_end(int which, cudaStream_t st);
const char* nccl_error_string(int nccl_result);   // comm.cu

// ---------------------------------------------------------------------------------------------
// Exactly-rounded arithmetic (never contracted into FMA, whatever the compiler flags).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float max_nn(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ float min_nn(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ double max_nn(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ double min_nn(double a, double b) { return fmin(a, b); }

// ---------------------------------------------------------------------------------------------
// Order-preserving keys.  key64(v) orders doubles like np.argmax does: NaN is the maximum
// (numpy's arg-max returns the first NaN), -0.0 == +0.0, ties compare equal.  Every finite or
// infinite value maps to a key > 0, so 0 can stand for "nothing seen".
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 key64(double v) {
  if (v != v) return ~0ull;
  if (v == 0.0) v = 0.0;  // canonical +0
  long long b = __double_as_longlong(v);
  return (u64)(b ^ ((b >> 63) | (long long)0x8000000000000000ull));
}
__device__ __forceinline__ double unkey64(u64 k) {
  long long b = (long long)k;
  b = (b < 0) ? (b ^ (long long)0x8000000000000000ull) : ~b;
  return __longlong_as_double(b);
}
#define SSDG_KEY_ZERO 0x8000000000000000ull /* key64(0.0) */

__device__ __forceinline__ u32 key32(float v) {
  if (v != v) return ~0u;
  if (v == 0.0f) v = 0.0f;
  int b = __float_as_int(v);
  return (u32)(b ^ ((b >> 31) | (int)0x80000000u));
}
__device__ __forceinline__ float unkey32(u32 k) {
  int b = (int)k;
  b = (b < 0) ? (b ^ (int)0x80000000u) : ~b;
  return __int_as_float(b);
}

// ---------------------------------------------------------------------------------------------
// Warp reductions on the REDUX unit (sm_80+: one instruction per 32-bit reduction).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 warp_max_u64(u64 k) {
  u32 hi = (u32)(k >> 32), lo = (u32)k;
  u32 mhi = __reduce_max_sync(SSDG_FULL, hi);
  u32 mlo = __reduce_max_sync(SSDG_FULL, hi == mhi ? lo : 0u);
  return ((u64)mhi << 32) | mlo;
}

// (max key, then min index) across the warp; lanes without a candidate pass key = 0.
__device__ __forceinline__ void warp_argmax_u64(u64& key, int& idx) {
  u64 m = warp_max_u64(key);
  int cand = (key == m) ? idx : 0x7fffffff;
  idx = (int)__reduce_min_sync(SSDG_FULL, (u32)cand);
  key = m;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SSDG_FULL, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SSDG_FULL, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------
// Box geometry in the reference's operation order.
// ---------------------------------------------------------------------------------------------
template <typename T>
struct Corners {
  T x1, y1, x2, y2, area;
};

// cx -/+ w/2 and w*h evaluated in the box's own dtype (utils/bbox.py:31-37).  w/2 == w*0.5
// bit for bit in IEEE arithmetic.
template <typename T>
__device__ __forceinline__ Corners<T> corners_of(T cx, T cy, T w, T h) {
  Corners<T> c;
  T hw = mul_rn(w, (T)0.5), hh = mul_rn(h, (T)0.5);
  c.x1 = sub_rn(cx, hw);
  c.y1 = sub_rn(cy, hh);
  c.x2 = add_rn(cx, hw);
  c.y2 = add_rn(cy, hh);
  c.area = mul_rn(w, h);
  return c;
}

// IoU of two corner sets already promoted to the result dtype R.  `eps` is the clamp of the
// intersection extents (1e-10 in iou_n utils/bbox.py:39, 0 in iou :23); the denominator always
// adds 1e-10 (:25,:41).  (a1 + a2) - inter + 1e-10, left to right.
template <typename R>
__device__ __forceinline__ R iou_corners(const Corners<R>& g, const Corners<R>& p, R eps) {
  R lox = max_nn(g.x1, p.x1), loy = max_nn(g.y1, p.y1);
  R hix = min_nn(g.x2, p.x2), hiy = min_nn(g.y2, p.y2);
  R ex = max_nn(eps, sub_rn(hix, lox)), ey = max_nn(eps, sub_rn(hiy, loy));
  R inter = mul_rn(ex, ey);
  R den = add_rn(sub_rn(add_rn(g.area, p.area), inter), (R)1e-10);
  return div_rn(inter, den);
}

// The helpers below are bit-exact only in units compiled with -fmad=false (match.cu, geom.cu): their plain
// operators must not be contracted into FMA.

// Result dtype of an IoU between a T1 and a T2 box (NumPy promotion): float only when both are float.
template <typename T1, typename T2>
struct Promote {
  typedef double type;
};
template <>
struct Promote<float, float> {
  typedef float type;
};

// Row i of a [n,4] float32 / float64 array.
template <typename T>
struct Vec4;
template <>
struct Vec4<float> {
  static __device__ __forceinline__ void load(const void* base, long long i, float& a, float& b, float& c,
                                              float& d) {
    float4 v = __ldg(reinterpret_cast<const float4*>(base) + i);
    a = v.x; b = v.y; c = v.z; d = v.w;
  }
};
template <>
struct Vec4<double> {
  static __device__ __forceinline__ void load(const void* base, long long i, double& a, double& b, double& c,
                                              double& d) {
    const double2* p = reinterpret_cast<const double2*>(base) + 2 * i;
    double2 u = __ldg(p), v = __ldg(p + 1);
    a = u.x; b = u.y; c = v.x; d = v.y;
  }
};

// Corners of (cx, cy, w, h) row i of a TIn array, computed in TIn and promoted to R.
template <typename TIn, typename R>
__device__ __forceinline__ Corners<R> load_corners(const void* base, long long i) {
  TIn cx, cy, w, h;
  Vec4<TIn>::load(base, i, cx, cy, w, h);
  const Corners<TIn> c = corners_of<TIn>(cx, cy, w, h);
  Corners<R> r;
  r.x1 = (R)c.x1; r.y1 = (R)c.y1; r.x2 = (R)c.x2; r.y2 = (R)c.y2; r.area = (R)c.area;
  return r;
}

// apply_anchor_box (utils/bbox.py:98-99) of box b against prior d in float64; callers cast the result.  The 1e-5
// clamp is applied in each operand's own dtype (NumPy promotes the Python scalar to the array dtype).
template <typename TB, typename TP>
__device__ __forceinline__ double4 anchor_offsets(TB bx, TB by, TB bw, TB bh, TP dx, TP dy, TP dw, TP dh) {
  const double tx = ((double)bx - (double)dx) / (double)dw;
  const double ty = ((double)by - (double)dy) / (double)dh;
  const double rw = (double)max_nn(bw, (TB)1e-5) / (double)max_nn(dw, (TP)1e-5);
  const double rh = (double)max_nn(bh, (TB)1e-5) / (double)max_nn(dh, (TP)1e-5);
  return make_double4(tx, ty, log(rw), log(rh));
}

// ---------------------------------------------------------------------------------------------
// mbarrier + 1-D bulk TMA (cp.async.bulk, SASS UBLKCP) for streaming contiguous tiles.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(u64* bar, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(u64* bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(u64* bar, u32 parity) {
  u32 ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy; dst, src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gsrc, u32 bytes, u64* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// exp(x - m) as FADD + FMUL + MUFU:  ex2.approx.ftz((x - m) * log2e)  -- __expf without its
// denormal-range fix-ups.  The subtraction comes first so the terms near the maximum (the ones that
// matter) carry no argument error; relative error ~2^-22 + 2^-24*|x-m|; flush-to-zero below 2^-126.
#define SSDG_LOG2E 1.4426950408889634f
__device__ __forceinline__ float exp2_ftz(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float exp_shifted(float x, float m) { return exp2_ftz((x - m) * SSDG_LOG2E); }

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (sm_90+): a kernel launched with launch_pdl is set up while its predecessor in the
// stream still runs and its CTAs are dispatched as soon as every CTA of the predecessor has exited (or called
// pdl_trigger()); it must call pdl_wait() before it touches anything the predecessor reads or writes -- pdl_wait()
// returns when the predecessor grid has completed and its memory is visible.  Takes the launch latency (and any
// prologue in front of pdl_wait) of the small kernels of a latency-bound chain off the critical path: loss tail
// 0.038 -> 0.034 ms, chained step 0.508 -> 0.504 ms (B=256), 0.305 -> 0.299 ms (B=128).  An EARLY pdl_trigger() is
// deliberately not used: the dependents' CTAs would sit on the SMs waiting, and in the chained step those are
// resources the concurrent NMS needs (measured: 0.508 -> 0.546 ms).  Without the launch attribute both calls are
// no-ops.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// streaming stores / loads that do not pollute L1
__device__ __forceinline__ void st_cs(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void st_cs(float4* p, float4 v) { __stcs(p, v); }

}  // namespace ssdg
