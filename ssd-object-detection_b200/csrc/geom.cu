// Small element-wise geometry kernels: anchors (A1), encode (A4), decode (A7), paired IoU (A2/A10).
#include "common.cuh"

namespace ssdg {

constexpr int kMaxLevels = 16;
constexpr int kMaxShapes = 16;  // 2 + 2 * ratios per level

struct PriorTable {
  int n_levels;
  int feat_h[kMaxLevels], feat_w[kMaxLevels], n_shapes[kMaxLevels];
  long long first[kMaxLevels + 1];          // first prior index of the level
  double shape_w[kMaxLevels][kMaxShapes];   // evaluated on the host with the same libm sqrt
  double shape_h[kMaxLevels][kMaxShapes];   // (correctly rounded) the reference uses
};

// models/ssd_model.py:178-192: one thread per prior; only the centre needs device arithmetic.
__global__ void prior_kernel(const __grid_constant__ PriorTable tab, double* __restrict__ out, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int l = 0;
  while (l + 1 < tab.n_levels && i >= tab.first[l + 1]) ++l;
  long long r = i - tab.first[l];
  int ns = tab.n_shapes[l];
  int s = (int)(r % ns);
  long long cell = r / ns;
  int x = (int)(cell % tab.feat_w[l]), y = (int)(cell / tab.feat_w[l]);
  double cx = __ddiv_rn(__dadd_rn((double)x, 0.5), (double)tab.feat_w[l]);
  double cy = __ddiv_rn(__dadd_rn((double)y, 0.5), (double)tab.feat_h[l]);
  double2* o = reinterpret_cast<double2*>(out) + 2 * i;
  o[0] = make_double2(cx, cy);
  o[1] = make_double2(tab.shape_w[l][s], tab.shape_h[l][s]);
}

// utils/bbox.py:98-99.
template <typename TB, typename TP, typename TO>
__global__ void encode_kernel(const void* __restrict__ boxes, const void* __restrict__ priors, TO* __restrict__ out,
                              long long n, int A) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  TB bx, by, bw, bh;
  TP dx, dy, dw, dh;
  Vec4<TB>::load(boxes, i, bx, by, bw, bh);
  Vec4<TP>::load(priors, i % A, dx, dy, dw, dh);
  const double4 t = anchor_offsets<TB, TP>(bx, by, bw, bh, dx, dy, dw, dh);
  out[4 * i + 0] = (TO)t.x; out[4 * i + 1] = (TO)t.y; out[4 * i + 2] = (TO)t.z; out[4 * i + 3] = (TO)t.w;
}

// models/ssd_model.py:466-467.
template <typename TP>
__global__ void decode_kernel(const float* __restrict__ loc, const void* __restrict__ priors, float* __restrict__ out,
                              long long n, int A, double scale) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 t = __ldg(reinterpret_cast<const float4*>(loc) + i);
  TP dx, dy, dw, dh;
  Vec4<TP>::load(priors, i % A, dx, dy, dw, dh);
  float4 o;
  o.x = (float)(((double)t.x * dw + dx) * scale);
  o.y = (float)(((double)t.y * dh + dy) * scale);
  o.z = (float)(exp((double)t.z) * dw * scale);
  o.w = (float)(exp((double)t.w) * dh * scale);
  reinterpret_cast<float4*>(out)[i] = o;
}

template <typename T1, typename T2>
__global__ void iou_pairs_kernel(const void* __restrict__ b1, const void* __restrict__ b2, void* __restrict__ out,
                                 long long n, int use_eps) {
  typedef typename Promote<T1, T2>::type R;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  reinterpret_cast<R*>(out)[i] =
      iou_corners<R>(load_corners<T1, R>(b1, i), load_corners<T2, R>(b2, i), use_eps ? (R)1e-10 : (R)0);
}

static inline unsigned blocks_for(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

}  // namespace ssdg

using namespace ssdg;

extern "C" int64_t ssdg_prior_count(const int32_t* feat_h, const int32_t* feat_w, const int32_t* ratio_offsets,
                                    int32_t n_levels) {
  if (!feat_h || !feat_w || !ratio_offsets || n_levels <= 0) return SSDG_ERR_ARG;
  int64_t n = 0;
  for (int l = 0; l < n_levels; ++l)
    n += (int64_t)feat_h[l] * feat_w[l] * (2 + 2 * (ratio_offsets[l + 1] - ratio_offsets[l]));
  return n;
}

extern "C" int ssdg_prior_boxes(const int32_t* feat_h, const int32_t* feat_w, const double* s_k,
                                const int32_t* ratio_offsets, const double* ratios, int32_t n_levels,
                                double input_size, double* out_priors, int64_t n_priors, void* stream) {
  if (!feat_h || !feat_w || !s_k || !ratio_offsets || !out_priors || n_levels <= 0) return SSDG_ERR_ARG;
  if (n_levels > kMaxLevels) return SSDG_ERR_LIMIT;
  if ((uintptr_t)out_priors & 15) return SSDG_ERR_ALIGN;
  PriorTable tab;
  tab.n_levels = n_levels;
  long long first = 0;
  for (int l = 0; l < n_levels; ++l) {
    int nr = ratio_offsets[l + 1] - ratio_offsets[l];
    if (nr < 0 || 2 + 2 * nr > kMaxShapes || feat_h[l] <= 0 || feat_w[l] <= 0) return SSDG_ERR_LIMIT;
    if (nr > 0 && !ratios) return SSDG_ERR_ARG;
    tab.feat_h[l] = feat_h[l]; tab.feat_w[l] = feat_w[l]; tab.n_shapes[l] = 2 + 2 * nr;
    tab.first[l] = first;
    first += (long long)feat_h[l] * feat_w[l] * tab.n_shapes[l];
    // models/ssd_model.py:184-192 -- scalar shape arithmetic, IEEE double, host libm sqrt
    volatile double s = s_k[l] / input_size;
    volatile double s_next = s_k[l + 1] / input_size;
    volatile double prod = s * s_next;
    double sp = sqrt(prod);
    tab.shape_w[l][0] = s; tab.shape_h[l][0] = s;
    tab.shape_w[l][1] = sp; tab.shape_h[l][1] = sp;
    for (int r = 0; r < nr; ++r) {
      volatile double q = sqrt(ratios[ratio_offsets[l] + r]);
      volatile double wide = s * q, tall = s / q;
      tab.shape_w[l][2 + 2 * r] = wide; tab.shape_h[l][2 + 2 * r] = tall;
      tab.shape_w[l][3 + 2 * r] = tall; tab.shape_h[l][3 + 2 * r] = wide;
    }
  }
  tab.first[n_levels] = first;
  if (first != n_priors) return SSDG_ERR_SHAPE;
  prior_kernel<<<blocks_for(first, 256), 256, 0, (cudaStream_t)stream>>>(tab, out_priors, first);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

extern "C" int ssdg_encode(const void* boxes, int32_t box_dtype, const void* priors, int32_t prior_dtype,
                           int64_t batch, int32_t n_priors, void* out, int32_t out_dtype, void* stream) {
  if (!boxes || !priors || !out || batch <= 0 || n_priors <= 0) return SSDG_ERR_ARG;
  if (((uintptr_t)boxes | (uintptr_t)priors | (uintptr_t)out) & 15) return SSDG_ERR_ALIGN;
  long long n = (long long)batch * n_priors;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned g = blocks_for(n, 256);
#define SSDG_ENC(TB, TP, TO) encode_kernel<TB, TP, TO><<<g, 256, 0, st>>>(boxes, priors, (TO*)out, n, n_priors)
  int sel = (box_dtype == SSDG_F64 ? 4 : 0) | (prior_dtype == SSDG_F64 ? 2 : 0) | (out_dtype == SSDG_F64 ? 1 : 0);
  switch (sel) {
    case 0: SSDG_ENC(float, float, float); break;
    case 1: SSDG_ENC(float, float, double); break;
    case 2: SSDG_ENC(float, double, float); break;
    case 3: SSDG_ENC(float, double, double); break;
    case 4: SSDG_ENC(double, float, float); break;
    case 5: SSDG_ENC(double, float, double); break;
    case 6: SSDG_ENC(double, double, float); break;
    default: SSDG_ENC(double, double, double); break;
  }
#undef SSDG_ENC
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

extern "C" int ssdg_decode(const float* loc, const void* priors, int32_t prior_dtype, int64_t batch,
                           int32_t n_priors, double scale, float* out, void* stream) {
  if (!loc || !priors || !out || batch <= 0 || n_priors <= 0) return SSDG_ERR_ARG;
  if (((uintptr_t)loc | (uintptr_t)priors | (uintptr_t)out) & 15) return SSDG_ERR_ALIGN;
  long long n = (long long)batch * n_priors;
  unsigned g = blocks_for(n, 256);
  if (prior_dtype == SSDG_F64) decode_kernel<double><<<g, 256, 0, (cudaStream_t)stream>>>(loc, priors, out, n, n_priors, scale);
  else decode_kernel<float><<<g, 256, 0, (cudaStream_t)stream>>>(loc, priors, out, n, n_priors, scale);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

extern "C" int ssdg_iou_pairs(const void* boxes_1, int32_t dtype_1, const void* boxes_2, int32_t dtype_2, int64_t n,
                              int32_t use_eps_clamp, void* out, void* stream) {
  if (!boxes_1 || !boxes_2 || !out || n <= 0) return SSDG_ERR_ARG;
  if (((uintptr_t)boxes_1 | (uintptr_t)boxes_2) & 15) return SSDG_ERR_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned g = blocks_for(n, 256);
  if (dtype_1 == SSDG_F32 && dtype_2 == SSDG_F32) iou_pairs_kernel<float, float><<<g, 256, 0, st>>>(boxes_1, boxes_2, out, n, use_eps_clamp);
  else if (dtype_1 == SSDG_F32) iou_pairs_kernel<float, double><<<g, 256, 0, st>>>(boxes_1, boxes_2, out, n, use_eps_clamp);
  else if (dtype_2 == SSDG_F32) iou_pairs_kernel<double, float><<<g, 256, 0, st>>>(boxes_1, boxes_2, out, n, use_eps_clamp);
  else iou_pairs_kernel<double, double><<<g, 256, 0, st>>>(boxes_1, boxes_2, out, n, use_eps_clamp);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}
