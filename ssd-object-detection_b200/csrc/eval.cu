// A11: detection evaluation.  COCOeval.evaluateImg / accumulate (iouType "bbox", area range "all", no crowd, no
// ignore flags) over the kept lists of ssdg_detect, on the device:
//   eval_match_kernel   per batch: one CTA per image matches each (image, class) kept list against the image's
//                       ground truth of that class and writes one fixed slot per (class, global image, rank) --
//                       a 64-bit sort key and a flag word -- plus the per-(class, image) ground-truth counts.
//                       Every slot has exactly one writer, so the kernel needs no global atomics on the slots, is
//                       deterministic, and re-running a batch with the same image_base overwrites it.
//   finalize            once per evaluation: a device-wide radix sort of each class's keys (flags as values), then
//                       one CTA per (class, IoU threshold) for the cumulative sums, the precision envelope and the
//                       recall-threshold lookup.  Every output is an IEEE function of integers and host doubles,
//                       so it is bit-identical to the NumPy restatement in tests/coco_eval_oracle.py.
// Compiled with -fmad=false; the IoU also uses the non-contractible intrinsics of common.cuh.
#include "common.cuh"

#include <cub/cub.cuh>

#include <cmath>

namespace ssdg {
namespace {

constexpr int kHdrWords = 64;          // int32 header in front of the flags (see EvalLayout)
constexpr u32 kPresent = 1u << 16;     // flag bit: the slot holds a detection (bits 0..15: TP at threshold k)
constexpr int kMaxThr = 16;
constexpr int kMaxRecall = 256;
constexpr int kMaxGt = 2048;
constexpr int kMaxDets = 1024;         // the rank takes 10 bits of the sort key
constexpr int64_t kMaxImages = 1ll << 22;   // the global image index takes the other 22
constexpr int kMatchThreads = 256;
constexpr int kCurveThreads = 256;
constexpr int kCurveItems = 4;

// header words (int32): additive, so a data-parallel sum of the int32 region keeps them meaningful
enum { HDR_BAD_CLASS = 0, HDR_TOO_MANY_GT = 1, HDR_DUPLICATE = 2, HDR_BAD_PRIOR = 3 };

// State: int32 hdr[64] | u32 flags[K][M][D] | int32 n_gt[K][M] | (256-aligned) u64 keys[K][M][D]
struct EvalLayout {
  int64_t K, M, D, slots;
  size_t ngt_off, keys_off, bytes;
};

int eval_layout(int32_t n_classes, int64_t max_images, int32_t max_dets, EvalLayout& L) {
  if (n_classes < 2 || max_images <= 0 || max_dets <= 0) return SSDG_ERR_ARG;
  if (max_images >= kMaxImages || max_dets > kMaxDets) return SSDG_ERR_LIMIT;
  L.K = n_classes - 1; L.M = max_images; L.D = max_dets;
  L.slots = L.K * L.M * L.D;
  if (L.slots >= (1ll << 31)) return SSDG_ERR_LIMIT;      // int32 item counts and slot offsets in the sorts
  L.ngt_off = (size_t)(kHdrWords + L.slots) * 4;
  L.keys_off = align_up(L.ngt_off + (size_t)(L.K * L.M) * 4, 256);
  L.bytes = align_up(L.keys_off + (size_t)L.slots * 8, 256);
  return SSDG_OK;
}

struct MatchParams {
  const int32_t* kept;
  const int32_t* count;
  const float* kept_score;
  const float4* boxes;
  const float* gt_boxes;
  const float* gt_cls;
  const int32_t* gt_off;
  int32_t top_k, n_priors, K, max_gt, n_thr, max_dets;
  int64_t image_base, max_images;
  double thr_min;         // min over k of min(thr[k], 1 - 1e-10)
  int32_t* hdr;
  u32* flags;
  int32_t* ngt;
  u64* keys;
  double thr[kMaxThr];
};

struct DBox {
  double x0, y0, x1, y1, area;
};

__device__ __forceinline__ DBox dbox(double cx, double cy, double w, double h) {
  DBox b;
  const double hw = mul_rn(0.5, w), hh = mul_rn(0.5, h);
  b.x0 = sub_rn(cx, hw); b.x1 = add_rn(cx, hw);
  b.y0 = sub_rn(cy, hh); b.y1 = add_rn(cy, hh);
  b.area = mul_rn(w, h);
  return b;
}

// iw = min(x1) - max(x0), ih likewise; 0 unless both > 0; inter / ((area_d + area_g) - inter)
__device__ __forceinline__ double eval_iou(const DBox& d, const DBox& g) {
  const double iw = sub_rn(fmin(d.x1, g.x1), fmax(d.x0, g.x0));
  const double ih = sub_rn(fmin(d.y1, g.y1), fmax(d.y0, g.y0));
  if (!(iw > 0.0) || !(ih > 0.0)) return 0.0;
  const double inter = mul_rn(iw, ih);
  return div_rn(inter, sub_rn(add_rn(d.area, g.area), inter));
}

__global__ void __launch_bounds__(kMatchThreads) eval_match_kernel(const MatchParams P) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int img = blockIdx.x, tid = threadIdx.x;
  const int K = P.K, MG = P.max_gt;
  DBox* gbox = (DBox*)smem;                       // [max_gt] bucketed by class, row order within a class
  int* gcls = (int*)(gbox + MG);                  // [max_gt] class of row t (-1: out of range)
  u32* gmatch = (u32*)(gcls + MG);                // [max_gt] bit k: matched at threshold k (bucketed order)
  int* cnt = (int*)(gmatch + MG);                 // [K]
  int* off = cnt + K;                             // [K+1]

  const int g0 = P.gt_off[img];
  int T = P.gt_off[img + 1] - g0;
  if (T < 0 || T > MG) {
    if (tid == 0) atomicAdd(&P.hdr[HDR_TOO_MANY_GT], 1);
    T = 0;
  }
  for (int c = tid; c < K; c += blockDim.x) cnt[c] = 0;
  __syncthreads();
  for (int t = tid; t < T; t += blockDim.x) {
    const float cf = P.gt_cls[g0 + t];
    const bool ok = cf > -1.0f && cf < (float)K;  // (int) truncates toward zero, as ssdg_match_encode
    const int c = ok ? (int)cf : -1;
    gcls[t] = c;
    if (ok) atomicAdd(&cnt[c], 1);
    else atomicAdd(&P.hdr[HDR_BAD_CLASS], 1);
  }
  __syncthreads();
  if (tid < 32) {                                 // exclusive scan of the class counts
    int run = 0;
    for (int base = 0; base < K; base += 32) {
      const int v = base + tid < K ? cnt[base + tid] : 0;
      int inc = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(SSDG_FULL, inc, o);
        if (tid >= o) inc += n;
      }
      if (base + tid < K) off[base + tid] = run + inc - v;
      run += __shfl_sync(SSDG_FULL, inc, 31);
    }
    if (tid == 0) off[K] = run;
  }
  __syncthreads();
  for (int t = tid; t < T; t += blockDim.x) {
    const int c = gcls[t];
    if (c < 0) continue;
    int r = 0;                                    // stable: rows of the same class keep their order
    for (int u = 0; u < t; ++u) r += gcls[u] == c;
    const float* g = P.gt_boxes + (int64_t)(g0 + t) * 4;
    gbox[off[c] + r] = dbox(g[0], g[1], g[2], g[3]);
    gmatch[off[c] + r] = 0u;
  }
  for (int c = tid; c < K; c += blockDim.x) P.ngt[(int64_t)c * P.max_images + P.image_base + img] = cnt[c];
  __syncthreads();

  // One warp per class list, 32 detections at a time: lane j gathers detection j and tests it against the class's
  // ground truth.  Only a detection with an IoU >= the lowest threshold against some row can take part in the greedy
  // rule (every other one skips every row at every threshold and changes no state), so only those are walked, one at
  // a time in list order, with lane k running the rule at threshold k.
  const int warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
  const double best0 = lane < P.n_thr ? fmin(P.thr[lane < kMaxThr ? lane : 0], 1.0 - 1e-10) : 0.0;
  const u32 gimg = (u32)(P.image_base + img) << 10;
  volatile u32* vmatch = gmatch;
  for (int c = warp; c < K; c += nwarps) {
    const int64_t li = (int64_t)img * K + c;
    const int nd = max(0, min(P.count[li], P.max_dets));
    const int gb = off[c], ge = off[c + 1];
    const int64_t sbase = ((int64_t)c * P.max_images + P.image_base + img) * P.max_dets;
    for (int d0 = 0; d0 < nd; d0 += 32) {
      const int d = d0 + lane;
      const bool live = d < nd;
      const int prior = live ? P.kept[li * P.top_k + d] : -1;
      const bool valid = live && (unsigned)prior < (unsigned)P.n_priors;
      float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
      bool cand = false;
      if (valid && gb < ge) {
        b = P.boxes[(int64_t)img * P.n_priors + prior];
        const DBox db = dbox(b.x, b.y, b.z, b.w);
        for (int g = gb; g < ge; ++g) cand |= !(eval_iou(db, gbox[g]) < P.thr_min);
      }
      u32 todo = __ballot_sync(SSDG_FULL, cand);
      u32 mytp = 0u;
      while (todo) {
        const int j = __ffs(todo) - 1;
        todo &= todo - 1;
        const float cx = __shfl_sync(SSDG_FULL, b.x, j), cy = __shfl_sync(SSDG_FULL, b.y, j);
        const float w = __shfl_sync(SSDG_FULL, b.z, j), h = __shfl_sync(SSDG_FULL, b.w, j);
        int m = -1;
        if (lane < P.n_thr) {
          const DBox db = dbox(cx, cy, w, h);
          double best = best0;
          for (int g = gb; g < ge; ++g) {
            if ((vmatch[g] >> lane) & 1u) continue;
            const double iou = eval_iou(db, gbox[g]);
            if (iou < best) continue;             // among equal IoUs the last ground truth wins
            best = iou;
            m = g;
          }
          if (m >= 0) atomicOr(&gmatch[m], 1u << lane);
        }
        const u32 tp = __ballot_sync(SSDG_FULL, m >= 0);
        if (lane == j) mytp = tp;
      }
      if (live) {
        if (!valid) atomicAdd(&P.hdr[HDR_BAD_PRIOR], 1);
        const u32 sb = __float_as_uint(P.kept_score[li * P.top_k + d]);
        P.keys[sbase + d] = ((u64)sb << 32) | (u64)(0xFFFFFFFFu - (gimg | (u32)d));
        P.flags[sbase + d] = kPresent | mytp;
      }
    }
    for (int d = nd + lane; d < P.max_dets; d += 32) {
      P.keys[sbase + d] = 0ull;
      P.flags[sbase + d] = 0u;
    }
  }
}

struct CurveParams {
  const u64* keys;        // sorted, [K][M*D] descending
  const u32* flags;       // sorted with the keys
  const int32_t* ngt;     // [K][M]
  int32_t* hdr;
  double* precision;      // [T][R][K]
  double* recall;         // [T][K]
  int64_t* n_gt;          // [K]
  int64_t* n_det;         // [K]
  int32_t K, n_thr, n_rec, seg, M;
  double rec[kMaxRecall];
};

struct DMax {
  __device__ __forceinline__ double operator()(double a, double b) const { return fmax(a, b); }
};

// One CTA per (class, threshold).  Records of the class are in COCO's order after the sort (score desc, global
// image asc, rank asc) and the present ones form a prefix of the segment.
__global__ void __launch_bounds__(kCurveThreads) eval_curve_kernel(const CurveParams P) {
  typedef cub::BlockReduce<long long, kCurveThreads> ReduceL;
  typedef cub::BlockScan<int, kCurveThreads> ScanI;
  typedef cub::BlockScan<double, kCurveThreads> ScanD;
  __shared__ union {
    typename ReduceL::TempStorage rl;
    typename ScanI::TempStorage si;
    typename ScanD::TempStorage sd;
  } tmp;
  __shared__ int s_nd;
  __shared__ long long s_npig, s_tp;
  const int c = blockIdx.x / P.n_thr, t = blockIdx.x % P.n_thr, tid = threadIdx.x;
  const u64* keys = P.keys + (int64_t)c * P.seg;
  const u32* flags = P.flags + (int64_t)c * P.seg;

  if (tid == 0) {                                 // first empty slot (key 0): the number of detections
    int lo = 0, hi = P.seg;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (keys[mid] != 0ull) lo = mid + 1; else hi = mid;
    }
    s_nd = lo;
  }
  long long g = 0;
  for (int i = tid; i < P.M; i += blockDim.x) g += P.ngt[(int64_t)c * P.M + i];
  g = ReduceL(tmp.rl).Sum(g);
  if (tid == 0) s_npig = g;
  __syncthreads();
  const int nd = s_nd;
  const long long npig = s_npig;
  long long tp_tot = 0;
  bool dup = false;
  for (int i = tid; i < nd; i += blockDim.x) {
    const u32 f = flags[i];
    tp_tot += (f >> t) & 1u;
    dup |= f >= 2 * kPresent;                     // two writers: the present bits carried
  }
  if (dup && t == 0) atomicOr(&P.hdr[HDR_DUPLICATE], 1);
  __syncthreads();
  tp_tot = ReduceL(tmp.rl).Sum(tp_tot);
  if (tid == 0) s_tp = tp_tot;
  __syncthreads();
  tp_tot = s_tp;
  if (t == 0 && tid == 0) {
    P.n_gt[c] = npig;
    P.n_det[c] = nd;
  }
  const int K = P.K, R = P.n_rec;
  double* prec = P.precision + (int64_t)t * R * K + c;
  if (npig == 0) {                                // COCO leaves -1 where a class has no ground truth
    for (int j = tid; j < R; j += blockDim.x) prec[(int64_t)j * K] = -1.0;
    if (tid == 0) P.recall[(int64_t)t * K + c] = -1.0;
    return;
  }
  for (int j = tid; j < R; j += blockDim.x) prec[(int64_t)j * K] = 0.0;
  if (tid == 0) P.recall[(int64_t)t * K + c] = nd ? (double)tp_tot / (double)npig : 0.0;
  __syncthreads();
  const double dn = (double)npig;
  const double eps = 2.220446049250313e-16;       // np.spacing(1)
  long long carry_tp = 0;                         // TP bits right of the chunk
  double carry_q = 0.0;                           // max precision right of the chunk
  constexpr int kChunk = kCurveThreads * kCurveItems;
  for (int hi = nd; hi > 0; hi -= kChunk) {       // right to left; the scans run over reversed positions
    int bits[kCurveItems], inc[kCurveItems];
#pragma unroll
    for (int j = 0; j < kCurveItems; ++j) {
      const int e = hi - 1 - (tid * kCurveItems + j);
      bits[j] = e >= 0 ? (int)((flags[e] >> t) & 1u) : 0;
    }
    int agg;
    ScanI(tmp.si).InclusiveSum(bits, inc, agg);
    __syncthreads();
    double pr[kCurveItems], q[kCurveItems];
    long long tp[kCurveItems];
#pragma unroll
    for (int j = 0; j < kCurveItems; ++j) {
      const int e = hi - 1 - (tid * kCurveItems + j);
      tp[j] = tp_tot - (carry_tp + inc[j]) + bits[j];
      const double dtp = (double)tp[j], dfp = (double)((long long)(e + 1) - tp[j]);
      pr[j] = e >= 0 ? div_rn(dtp, add_rn(add_rn(dfp, dtp), eps)) : 0.0;
    }
    double qagg;
    ScanD(tmp.sd).InclusiveScan(pr, q, DMax(), qagg);
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kCurveItems; ++j) {
      const int e = hi - 1 - (tid * kCurveItems + j);
      if (e < 0 || !(bits[j] || e == 0)) continue;
      // recall thresholds r with rc[e-1] < r <= rc[e]: searchsorted(rc, r, "left") == e
      const double qe = fmax(q[j], carry_q);
      const double rc = div_rn((double)tp[j], dn);
      const double rc_prev = e == 0 ? -INFINITY : div_rn((double)(tp[j] - 1), dn);
      for (int r = 0; r < R; ++r) {
        const double x = P.rec[r];
        if (rc_prev < x && x <= rc) prec[(int64_t)r * K] = qe;
      }
    }
    carry_tp += agg;
    carry_q = fmax(carry_q, qagg);
  }
}

}  // namespace
}  // namespace ssdg

using namespace ssdg;

extern "C" {

size_t ssdg_eval_state_bytes(int32_t n_classes, int64_t max_images, int32_t max_dets, int32_t n_thresholds) {
  EvalLayout L;
  if (n_thresholds <= 0 || n_thresholds > kMaxThr || eval_layout(n_classes, max_images, max_dets, L) != SSDG_OK) return 0;
  return L.bytes;
}

int ssdg_eval_reset(void* state, size_t state_bytes, void* stream) {
  if (!state || state_bytes == 0) return SSDG_ERR_ARG;
  return (int)cudaMemsetAsync(state, 0, state_bytes, (cudaStream_t)stream);
}

int ssdg_eval_accumulate(const int32_t* kept, const int32_t* count, const float* kept_score, int32_t top_k,
                         const float* boxes, int32_t batch, int32_t n_priors, int32_t n_classes,
                         const float* gt_boxes, const float* gt_cls, const int32_t* gt_offsets, int32_t max_gt,
                         const double* iou_thresholds, int32_t n_thresholds, int32_t max_dets, int64_t image_base,
                         int64_t max_images, void* state, size_t state_bytes, void* stream) {
  if (!kept || !count || !kept_score || !boxes || !gt_boxes || !gt_cls || !gt_offsets || !iou_thresholds || !state)
    return SSDG_ERR_ARG;
  if (batch <= 0 || n_priors <= 0 || top_k <= 0 || max_gt < 0 || n_thresholds <= 0 || image_base < 0)
    return SSDG_ERR_ARG;
  EvalLayout L;
  const int lst = eval_layout(n_classes, max_images, max_dets, L);
  if (lst != SSDG_OK) return lst;
  if (max_dets > top_k || image_base + batch > max_images) return SSDG_ERR_ARG;
  if (n_thresholds > kMaxThr || max_gt > kMaxGt) return SSDG_ERR_LIMIT;
  for (int k = 0; k < n_thresholds; ++k)
    if (iou_thresholds[k] != iou_thresholds[k]) return SSDG_ERR_ARG;     // NaN
  if (state_bytes < L.bytes || ((uintptr_t)state & 255)) return SSDG_ERR_WORKSPACE;
  if ((uintptr_t)boxes & 15) return SSDG_ERR_ALIGN;
  MatchParams P;
  P.kept = kept; P.count = count; P.kept_score = kept_score; P.boxes = (const float4*)boxes;
  P.gt_boxes = gt_boxes; P.gt_cls = gt_cls; P.gt_off = gt_offsets;
  P.top_k = top_k; P.n_priors = n_priors; P.K = (int32_t)L.K; P.max_gt = max_gt; P.n_thr = n_thresholds;
  P.max_dets = max_dets; P.image_base = image_base; P.max_images = max_images;
  char* base = (char*)state;
  P.hdr = (int32_t*)base;
  P.flags = (u32*)(base + kHdrWords * 4);
  P.ngt = (int32_t*)(base + L.ngt_off);
  P.keys = (u64*)(base + L.keys_off);
  P.thr_min = 1.0 - 1e-10;
  for (int k = 0; k < kMaxThr; ++k) {
    P.thr[k] = k < n_thresholds ? iou_thresholds[k] : 0.0;
    if (k < n_thresholds) P.thr_min = std::fmin(P.thr_min, iou_thresholds[k]);
  }
  const size_t smem = (size_t)max_gt * (sizeof(DBox) + 8) + (size_t)(2 * L.K + 1) * 4;
  if (smem > 48 * 1024) {
    if ((int)smem > max_smem_optin()) return SSDG_ERR_LIMIT;
    SSDG_CUDA_TRY(cudaFuncSetAttribute(eval_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  eval_match_kernel<<<batch, kMatchThreads, smem, (cudaStream_t)stream>>>(P);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

int ssdg_eval_exchange(void* state, int32_t n_classes, int64_t max_images, int32_t max_dets, int32_t which,
                       void** out_ptr, int64_t* out_count) {
  if (!state || !out_ptr || !out_count || which < 0 || which > 1) return SSDG_ERR_ARG;
  EvalLayout L;
  const int lst = eval_layout(n_classes, max_images, max_dets, L);
  if (lst != SSDG_OK) return lst;
  if (which == 0) { *out_ptr = (char*)state + L.keys_off; *out_count = L.slots; }            // int64 keys
  else { *out_ptr = state; *out_count = (int64_t)(L.ngt_off / 4) + L.K * L.M; }             // int32: header, flags, GT counts
  return SSDG_OK;
}

int ssdg_eval_status(const void* state, int32_t* status, void* stream) {
  if (!state || !status) return SSDG_ERR_ARG;
  int32_t h[4];
  SSDG_CUDA_TRY(cudaMemcpyAsync(h, state, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  SSDG_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  *status = (h[HDR_BAD_CLASS] ? 1 : 0) | (h[HDR_TOO_MANY_GT] ? 2 : 0) | (h[HDR_DUPLICATE] ? 4 : 0) |
            (h[HDR_BAD_PRIOR] ? 8 : 0);
  return SSDG_OK;
}

// workspace: sorted keys | sorted flags | the sort's temporary storage (one class at a time).  A device-wide sort per
// class rather than one segmented sort: the segmented sort gives a segment one CTA, and a class holds M*D slots
// (500 000 for COCO val).
static int eval_ws_layout(const EvalLayout& L, size_t* sort_bytes, size_t* total) {
  size_t tb = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairsDescending(nullptr, tb, (const u64*)nullptr, (u64*)nullptr,
                                                            (const u32*)nullptr, (u32*)nullptr, (int)(L.M * L.D), 0, 64);
  if (e != cudaSuccess) return (int)e;
  *sort_bytes = tb;
  *total = align_up((size_t)L.slots * 8, 256) + align_up((size_t)L.slots * 4, 256) + align_up(tb, 256);
  return SSDG_OK;
}

size_t ssdg_eval_finalize_workspace_bytes(int32_t n_classes, int64_t max_images, int32_t max_dets) {
  EvalLayout L;
  size_t tb = 0, total = 0;
  if (eval_layout(n_classes, max_images, max_dets, L) != SSDG_OK || eval_ws_layout(L, &tb, &total) != SSDG_OK) return 0;
  return total;
}

int ssdg_eval_finalize(void* state, size_t state_bytes, int32_t n_classes, int64_t max_images, int32_t max_dets,
                       int32_t n_thresholds, const double* recall_thresholds, int32_t n_recall,
                       double* out_precision, double* out_recall, int64_t* out_n_gt, int64_t* out_n_det,
                       void* workspace, size_t workspace_bytes, void* stream) {
  if (!state || !recall_thresholds || !out_precision || !out_recall || !out_n_gt || !out_n_det || n_thresholds <= 0 ||
      n_recall <= 0)
    return SSDG_ERR_ARG;
  EvalLayout L;
  const int lst = eval_layout(n_classes, max_images, max_dets, L);
  if (lst != SSDG_OK) return lst;
  if (n_thresholds > kMaxThr || n_recall > kMaxRecall) return SSDG_ERR_LIMIT;
  if (state_bytes < L.bytes || ((uintptr_t)state & 255)) return SSDG_ERR_WORKSPACE;
  if (!workspace || ((uintptr_t)workspace & 255)) return SSDG_ERR_WORKSPACE;
  size_t tb = 0, total = 0;
  const int wst = eval_ws_layout(L, &tb, &total);
  if (wst != SSDG_OK) return wst;
  if (workspace_bytes < total) return SSDG_ERR_WORKSPACE;
  const cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)state;
  char* w = (char*)workspace;
  u64* skeys = (u64*)w;
  w += align_up((size_t)L.slots * 8, 256);
  u32* sflags = (u32*)w;
  w += align_up((size_t)L.slots * 4, 256);
  const int32_t seg = (int32_t)(L.M * L.D);
  const u64* keys = (const u64*)(base + L.keys_off);
  const u32* flags = (const u32*)(base + kHdrWords * 4);
  for (int64_t c = 0; c < L.K; ++c) {
    size_t tbc = tb;
    SSDG_CUDA_TRY(cub::DeviceRadixSort::SortPairsDescending(w, tbc, keys + c * seg, skeys + c * seg, flags + c * seg,
                                                            sflags + c * seg, seg, 0, 64, st));
  }
  CurveParams P;
  P.keys = skeys; P.flags = sflags; P.ngt = (const int32_t*)(base + L.ngt_off); P.hdr = (int32_t*)base;
  P.precision = out_precision; P.recall = out_recall; P.n_gt = out_n_gt; P.n_det = out_n_det;
  P.K = (int32_t)L.K; P.n_thr = n_thresholds; P.n_rec = n_recall; P.seg = seg; P.M = (int32_t)L.M;
  for (int r = 0; r < kMaxRecall; ++r) P.rec[r] = r < n_recall ? recall_thresholds[r] : 0.0;
  eval_curve_kernel<<<(int)L.K * n_thresholds, kCurveThreads, 0, st>>>(P);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

}  // extern "C"
