// SSD training augmentation (A13, include/ssdgeom.h): the SSD paper's zoom-out, min-IoU crop and horizontal flip of a
// batch that is already on the device, with the decisions of torchvision's RandomZoomOut -> RandomIoUCrop ->
// RandomHorizontalFlip (spec: tests/augment_oracle.py).
//
//   aug_sample_kernel    one CTA per image: zoom draw, the crop rounds (warps over trials, lanes over rows, one ballot
//                        per trial), flip draw; writes the transform record and the survivor count into out_offsets
//   aug_scan_kernel      one CTA: the counts in out_offsets[1..B] become offsets in place
//   aug_compact_kernel   one CTA per image: the surviving rows in input order (block prefix over the within flags),
//                        mapped into the output image; rows past out_offsets[B] zeroed
//   aug_image_kernel     grid-stride bilinear resample of each record's crop of the virtual canvas back to H x W
//
// Every random number has a fixed Philox4x32-10 address (key = seed, counter = (g lo, g hi, stream, index), g the
// global image index), so trials are evaluated in parallel and an image's result depends only on (seed, g, config).
// Box tests and outputs are float64 from the exactly promoted float32 inputs (intrinsics, and -fmad=false for this
// unit); the integer decisions copy torchvision's float32 arithmetic.
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace ssdg {

constexpr int kAugMaxOptions = 16;
constexpr int kAugMaxGt = 2048;
constexpr int kAugThreads = 256;
constexpr int kAugScanThreads = 1024;
constexpr int kAugMaxSide = 16384;        // image height / width
constexpr double kAugMaxZoom = 64.0;      // side_hi: canvas sides stay below 2^20, exact in float32
// transform record words (out_transform int32 [B, SSDG_AUG_RECORD])
enum { R_CW = 0, R_CH, R_PL, R_PT, R_L, R_T, R_W, R_H, R_FLIP, R_ROUNDS };

struct AugConfig {
  u64 seed;
  long long image_base;
  int height, width, max_gt, n_options, trials, max_rounds;
  float zoom_p, side_lo, side_d, flip_p, min_s, scale_d;   // as torch sees them: float32
  double min_ar, max_ar;
  double options[kAugMaxOptions];
};

// Philox4x32-10 (Salmon et al., SC'11; Random123).
__device__ __forceinline__ uint4 philox(u64 key, u64 g, u32 stream, u32 index) {
  u32 c0 = (u32)g, c1 = (u32)(g >> 32), c2 = stream, c3 = index;
  u32 k0 = (u32)key, k1 = (u32)(key >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const u32 lo0 = 0xD2511F53u * c0, hi0 = __umulhi(0xD2511F53u, c0);
    const u32 lo1 = 0xCD9E8D57u * c2, hi1 = __umulhi(0xCD9E8D57u, c2);
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float unif(u32 x) { return (float)(x >> 8) * 0x1p-24f; }

// The min-IoU option of crop round q (torch.randint(0, n) as (x * n) >> 32).  `options`: c.options copied to shared
// memory (a dynamically indexed kernel parameter would be copied to the stack).
__device__ __forceinline__ double round_option(const AugConfig& c, const double* options, u64 g, int q) {
  const u32 x = philox(c.seed, g, 1u, (u32)q).x;
  return options[(int)(((u64)x * (u32)c.n_options) >> 32)];
}
// Whether a record with `rounds` crop rounds was cropped: its last round drew an option below 1 (and so had a
// successful trial).  The record itself then needs no separate flag.
__device__ __forceinline__ bool cropped(const AugConfig& c, const double* options, u64 g, int rounds) {
  return rounds > 0 && round_option(c, options, g, rounds - 1) < 1.0;
}
__device__ __forceinline__ void load_options(const AugConfig& c, double* s_options) {
#pragma unroll
  for (int k = 0; k < kAugMaxOptions; ++k)
    if (threadIdx.x == k) s_options[k] = c.options[k];
}

// A crop trial's rectangle on the canvas, or ok = false when torchvision's aspect / zero-area checks reject it.
struct Rect {
  int l, t, w, h;
  bool ok;
};
__device__ __forceinline__ Rect crop_trial(const AugConfig& c, u64 g, int q, int t, int cw, int ch) {
  const uint4 x = philox(c.seed, g, 2u + (u32)q, (u32)t);
  Rect r;
  r.w = (int)mul_rn((float)cw, add_rn(c.min_s, mul_rn(unif(x.x), c.scale_d)));
  r.h = (int)mul_rn((float)ch, add_rn(c.min_s, mul_rn(unif(x.y), c.scale_d)));
  r.l = (int)mul_rn((float)(cw - r.w), unif(x.z));
  r.t = (int)mul_rn((float)(ch - r.h), unif(x.w));
  r.ok = false;
  if (r.h == 0 || r.w == 0) return r;
  const double ar = div_rn((double)r.w, (double)r.h);
  r.ok = c.min_ar <= ar && ar <= c.max_ar;
  return r;
}

// Pixel corners of a relative cxcywh row on the canvas: (cx -/+ 0.5w) * W + pad.
__device__ __forceinline__ double4 canvas_corners(float4 b, int width, int height, int pl, int pt) {
  const double hw = mul_rn(0.5, (double)b.z), hh = mul_rn(0.5, (double)b.w);
  const double W = (double)width, H = (double)height;
  return make_double4(add_rn(mul_rn(sub_rn((double)b.x, hw), W), (double)pl),
                      add_rn(mul_rn(sub_rn((double)b.y, hh), H), (double)pt),
                      add_rn(mul_rn(add_rn((double)b.x, hw), W), (double)pl),
                      add_rn(mul_rn(add_rn((double)b.y, hh), H), (double)pt));
}

__device__ __forceinline__ bool centre_within(double4 k, int l, int t, int w, int h) {
  const double cx = mul_rn(0.5, add_rn(k.x, k.z)), cy = mul_rn(0.5, add_rn(k.y, k.w));
  return (double)l < cx && cx < (double)(l + w) && (double)t < cy && cy < (double)(t + h);
}

// torchvision's box_iou(row, crop) >= min_iou, written as !(iou < min_iou) so that a NaN IoU passes (torch.max
// propagates NaN and `NaN < m` is false).
__device__ __forceinline__ bool iou_passes(double4 k, int l, int t, int w, int h, double min_iou) {
  const double area1 = mul_rn(sub_rn(k.z, k.x), sub_rn(k.w, k.y));
  const double area2 = (double)w * (double)h;
  const double ex = fmax(sub_rn(fmin(k.z, (double)(l + w)), fmax(k.x, (double)l)), 0.0);
  const double ey = fmax(sub_rn(fmin(k.w, (double)(t + h)), fmax(k.y, (double)t)), 0.0);
  const double inter = mul_rn(ex, ey);
  const double iou = div_rn(inter, sub_rn(add_rn(area1, area2), inter));
  return !(iou < min_iou);
}

__global__ void __launch_bounds__(kAugThreads, 2) aug_sample_kernel(const float4* __restrict__ boxes,
                                                                 const int* __restrict__ offsets, AugConfig c,
                                                                 int* __restrict__ out_offsets,
                                                                 int* __restrict__ out_transform) {
  extern __shared__ double4 s_corner[];          // the first min(T, max_gt) rows' canvas corners
  __shared__ int s_best, s_count;
  __shared__ double s_options[kAugMaxOptions];
  load_options(c, s_options);
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const u64 g = (u64)(c.image_base + b);
  const int r0 = offsets[b], n = offsets[b + 1] - r0;
  const int staged = min(n, c.max_gt);

  const uint4 z = philox(c.seed, g, 0u, 0u);
  int cw = c.width, ch = c.height, pl = 0, pt = 0;
  if (unif(z.x) < c.zoom_p) {
    const float r = add_rn(c.side_lo, mul_rn(unif(z.y), c.side_d));
    cw = (int)mul_rn((float)c.width, r);
    ch = (int)mul_rn((float)c.height, r);
    pl = (int)mul_rn((float)(cw - c.width), unif(z.z));
    pt = (int)mul_rn((float)(ch - c.height), unif(z.w));
  }
  for (int i = tid; i < staged; i += blockDim.x) s_corner[i] = canvas_corners(boxes[r0 + i], c.width, c.height, pl, pt);
  __syncthreads();

  // crop rounds: round q draws an option; its trials run in parallel, the first success by trial index wins
  int rounds = c.n_options > 0 ? -1 : 0, best = -1, q_won = -1;
  for (int q = 0; c.n_options > 0 && q < c.max_rounds; ++q) {
    const double m = round_option(c, s_options, g, q);
    if (m >= 1.0) { rounds = q + 1; break; }
    if (tid == 0) s_best = 0x7fffffff;
    __syncthreads();
    for (int t = warp; t < c.trials; t += nwarps) {
      if (t > __shfl_sync(SSDG_FULL, *(volatile int*)&s_best, 0)) break;   // warp-uniform
      const Rect rc = crop_trial(c, g, q, t, cw, ch);
      if (!rc.ok) continue;
      bool pass = false;
      for (int i0 = 0; i0 < n && !pass; i0 += 32) {
        const int i = i0 + lane;
        bool p = false;
        if (i < n) {
          const double4 k = i < staged ? s_corner[i] : canvas_corners(boxes[r0 + i], c.width, c.height, pl, pt);
          p = centre_within(k, rc.l, rc.t, rc.w, rc.h) && iou_passes(k, rc.l, rc.t, rc.w, rc.h, m);
        }
        pass = __any_sync(SSDG_FULL, p);
      }
      if (pass && lane == 0) atomicMin(&s_best, t);
    }
    __syncthreads();
    best = s_best;
    __syncthreads();                              // everyone has read s_best before the next round resets it
    if (best != 0x7fffffff) { rounds = q + 1; q_won = q; break; }
    best = -1;
  }

  Rect crop{0, 0, cw, ch, false};
  if (q_won >= 0) crop = crop_trial(c, g, q_won, best, cw, ch);
  // survivors: the rows within the crop, or every row without one
  if (tid == 0) s_count = 0;
  __syncthreads();
  int cnt = 0;
  if (q_won >= 0) {
    for (int i = tid; i < n; i += blockDim.x) {
      const double4 k = i < staged ? s_corner[i] : canvas_corners(boxes[r0 + i], c.width, c.height, pl, pt);
      cnt += centre_within(k, crop.l, crop.t, crop.w, crop.h);
    }
    cnt = __reduce_add_sync(SSDG_FULL, cnt);
    if (lane == 0 && cnt) atomicAdd(&s_count, cnt);
  }
  __syncthreads();
  if (tid == 0) {
    const uint4 f = philox(c.seed, g, 0u, 1u);
    int* rec = out_transform + (size_t)b * SSDG_AUG_RECORD;
    rec[R_CW] = cw; rec[R_CH] = ch; rec[R_PL] = pl; rec[R_PT] = pt;
    rec[R_L] = crop.l; rec[R_T] = crop.t; rec[R_W] = crop.w; rec[R_H] = crop.h;
    rec[R_FLIP] = unif(f.x) < c.flip_p;
    rec[R_ROUNDS] = rounds;
    out_offsets[b + 1] = q_won >= 0 ? s_count : n;
    if (b == 0) out_offsets[0] = 0;
  }
}

__global__ void __launch_bounds__(kAugScanThreads) aug_scan_kernel(int* __restrict__ offsets, int batch) {
  typedef cub::BlockScan<int, kAugScanThreads> Scan;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int base = 1; base <= batch; base += kAugScanThreads) {
    const int i = base + threadIdx.x;
    int v = i <= batch ? offsets[i] : 0, total;
    Scan(tmp).InclusiveSum(v, v, total);
    const int carry = s_carry;
    if (i <= batch) offsets[i] = v + carry;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + total;
    __syncthreads();
  }
}

// A row mapped through a record: shifted into the crop, clamped to it when the image was cropped, relative cxcywh of
// the crop, cx -> 1 - cx under a flip; float64, rounded once.
__device__ __forceinline__ float4 map_row(float4 b, const int* rec, int width, int height, bool cropped) {
  double4 k = canvas_corners(b, width, height, rec[R_PL], rec[R_PT]);
  const double l = (double)rec[R_L], t = (double)rec[R_T], w = (double)rec[R_W], h = (double)rec[R_H];
  k.x = sub_rn(k.x, l); k.z = sub_rn(k.z, l); k.y = sub_rn(k.y, t); k.w = sub_rn(k.w, t);
  if (cropped) {
    k.x = fmin(fmax(k.x, 0.0), w); k.z = fmin(fmax(k.z, 0.0), w);
    k.y = fmin(fmax(k.y, 0.0), h); k.w = fmin(fmax(k.w, 0.0), h);
  }
  double cx = div_rn(mul_rn(add_rn(k.x, k.z), 0.5), w);
  const double cy = div_rn(mul_rn(add_rn(k.y, k.w), 0.5), h);
  if (rec[R_FLIP]) cx = sub_rn(1.0, cx);
  return make_float4(__double2float_rn(cx), __double2float_rn(cy), __double2float_rn(div_rn(sub_rn(k.z, k.x), w)),
                     __double2float_rn(div_rn(sub_rn(k.w, k.y), h)));
}

__global__ void __launch_bounds__(kAugThreads, 2) aug_compact_kernel(const float4* __restrict__ boxes,
                                                                  const float* __restrict__ cls,
                                                                  const int* __restrict__ offsets, int batch,
                                                                  AugConfig c, const int* __restrict__ out_offsets,
                                                                  const int* __restrict__ transform,
                                                                  float4* __restrict__ out_boxes,
                                                                  float* __restrict__ out_cls,
                                                                  int* __restrict__ out_src_row) {
  typedef cub::BlockScan<int, kAugThreads> Scan;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int s_rec[SSDG_AUG_RECORD];
  __shared__ double s_options[kAugMaxOptions];
  load_options(c, s_options);
  const int b = blockIdx.x, tid = threadIdx.x;
  if (tid < SSDG_AUG_RECORD) s_rec[tid] = transform[(size_t)b * SSDG_AUG_RECORD + tid];
  __syncthreads();
  const int r0 = offsets[b], n = offsets[b + 1] - r0;
  const bool crop = cropped(c, s_options, (u64)(c.image_base + b), s_rec[R_ROUNDS]);
  int o = out_offsets[b];
  for (int i0 = 0; i0 < n; i0 += blockDim.x) {
    const int i = i0 + tid;
    float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
    int keep = 0;
    if (i < n) {
      bx = boxes[r0 + i];
      keep = !crop || centre_within(canvas_corners(bx, c.width, c.height, s_rec[R_PL], s_rec[R_PT]), s_rec[R_L],
                                    s_rec[R_T], s_rec[R_W], s_rec[R_H]);
    }
    int pos, total;
    Scan(tmp).ExclusiveSum(keep, pos, total);
    if (keep) {
      out_boxes[o + pos] = map_row(bx, s_rec, c.width, c.height, crop);
      out_cls[o + pos] = cls[r0 + i];
      out_src_row[o + pos] = r0 + i;
    }
    o += total;
    __syncthreads();
  }
  // rows past out_offsets[B]: zero / -1
  const int rows = offsets[batch];
  const long long stride = (long long)batch * blockDim.x;
  for (long long i = out_offsets[batch] + (long long)b * blockDim.x + tid; i < rows; i += stride) {
    out_boxes[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    out_cls[i] = 0.f;
    out_src_row[i] = -1;
  }
}

// One output pixel of image b: bilinear (align_corners=False, no antialias) over the crop of the virtual canvas.
__device__ __forceinline__ float3 aug_pixel(const float* __restrict__ img, const int* rec, int i, int j, int H, int W,
                                            float3 fill) {
  if (rec[R_FLIP]) j = W - 1 - j;
  const int nw = rec[R_W], nh = rec[R_H];
  const float sx = fmaxf(0.f, sub_rn(mul_rn(div_rn((float)nw, (float)W), add_rn((float)j, 0.5f)), 0.5f));
  const float sy = fmaxf(0.f, sub_rn(mul_rn(div_rn((float)nh, (float)H), add_rn((float)i, 0.5f)), 0.5f));
  const int x0 = (int)sx, y0 = (int)sy;
  const int x1 = x0 + (x0 < nw - 1 ? 1 : 0), y1 = y0 + (y0 < nh - 1 ? 1 : 0);
  const float lx = sub_rn(sx, (float)x0), ly = sub_rn(sy, (float)y0);
  const float hx = sub_rn(1.f, lx), hy = sub_rn(1.f, ly);
  const int ox = rec[R_L] - rec[R_PL], oy = rec[R_T] - rec[R_PT];   // crop -> image coordinates
  float v[4][3];
  const int xs[2] = {x0 + ox, x1 + ox}, ys[2] = {y0 + oy, y1 + oy};
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int y = ys[a], x = xs[e];
      float* d = v[2 * a + e];
      if (0 <= x && x < W && 0 <= y && y < H) {
        const float* p = img + ((size_t)y * W + x) * 3;
        d[0] = __ldg(p); d[1] = __ldg(p + 1); d[2] = __ldg(p + 2);
      } else {
        d[0] = fill.x; d[1] = fill.y; d[2] = fill.z;
      }
    }
  float o[3];
#pragma unroll
  for (int ch = 0; ch < 3; ++ch)
    o[ch] = add_rn(mul_rn(hy, add_rn(mul_rn(hx, v[0][ch]), mul_rn(lx, v[1][ch]))),
                   mul_rn(ly, add_rn(mul_rn(hx, v[2][ch]), mul_rn(lx, v[3][ch]))));
  return make_float3(o[0], o[1], o[2]);
}

__device__ __forceinline__ float3 aug_out_pixel(const float* __restrict__ images, const int* __restrict__ transform,
                                                long long p, int H, int W, float3 fill) {
  const long long hw = (long long)H * W;
  const int b = (int)(p / hw), r = (int)(p - b * hw), i = r / W, j = r - i * W;
  const int* rec = transform + (size_t)b * SSDG_AUG_RECORD;
  const float* img = images + (size_t)b * hw * 3;
  if (rec[R_FLIP] == 0 && rec[R_W] == W && rec[R_H] == H && rec[R_L] == rec[R_PL] && rec[R_T] == rec[R_PT]) {
    const float* s = img + (size_t)r * 3;     // the crop is the image itself: a copy
    return make_float3(__ldg(s), __ldg(s + 1), __ldg(s + 2));
  }
  return aug_pixel(img, rec, i, j, H, W, fill);
}

__global__ void __launch_bounds__(256) aug_image_kernel(const float* __restrict__ images,
                                                        const int* __restrict__ transform, long long pixels, int H,
                                                        int W, float3 fill, float* __restrict__ out) {
  const long long groups = (pixels + 3) >> 2;
  const bool vec = ((uintptr_t)out & 15) == 0;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < groups;
       q += (long long)gridDim.x * blockDim.x) {
    const long long p0 = q << 2;
    if (vec && p0 + 4 <= pixels) {
      float3 v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = aug_out_pixel(images, transform, p0 + k, H, W, fill);
      float4* d = reinterpret_cast<float4*>(out + p0 * 3);
      __stcs(d, make_float4(v[0].x, v[0].y, v[0].z, v[1].x));
      __stcs(d + 1, make_float4(v[1].y, v[1].z, v[2].x, v[2].y));
      __stcs(d + 2, make_float4(v[2].z, v[3].x, v[3].y, v[3].z));
    } else {
      for (long long p = p0; p < p0 + 4 && p < pixels; ++p) {
        const float3 v = aug_out_pixel(images, transform, p, H, W, fill);
        out[p * 3] = v.x; out[p * 3 + 1] = v.y; out[p * 3 + 2] = v.z;
      }
    }
  }
}

static bool in01(double p) { return p >= 0.0 && p <= 1.0; }

}  // namespace ssdg

using namespace ssdg;

extern "C" int ssdg_augment_boxes(const float* gt_boxes, const float* gt_cls, const int32_t* gt_offsets, int32_t batch,
                                  int32_t max_gt, int32_t height, int32_t width, uint64_t seed, int64_t image_base,
                                  double zoom_p, double side_lo, double side_hi, const double* min_ious,
                                  int32_t n_options, double min_scale, double max_scale, double min_aspect,
                                  double max_aspect, int32_t trials, int32_t max_rounds, double flip_p,
                                  float* out_boxes, float* out_cls, int32_t* out_offsets, int32_t* out_src_row,
                                  int32_t* out_transform, void* stream) {
  if (!gt_boxes || !gt_cls || !gt_offsets || !out_boxes || !out_cls || !out_offsets || !out_src_row || !out_transform)
    return SSDG_ERR_ARG;
  if (batch <= 0 || max_gt < 0 || height <= 0 || width <= 0 || trials < 1 || max_rounds < 1) return SSDG_ERR_ARG;
  if (n_options < 0 || (n_options > 0 && !min_ious)) return SSDG_ERR_ARG;
  if (!in01(zoom_p) || !in01(flip_p) || !(side_lo >= 1.0 && side_lo <= side_hi)) return SSDG_ERR_ARG;
  if (!(min_scale >= 0.0 && min_scale <= max_scale && max_scale <= 1.0)) return SSDG_ERR_ARG;
  if (!(min_aspect > 0.0 && min_aspect <= max_aspect) || max_aspect != max_aspect) return SSDG_ERR_ARG;
  for (int k = 0; k < n_options && k < kAugMaxOptions; ++k)
    if (min_ious[k] != min_ious[k]) return SSDG_ERR_ARG;
  if (n_options > kAugMaxOptions || max_gt > kAugMaxGt || height > kAugMaxSide || width > kAugMaxSide ||
      side_hi > kAugMaxZoom)
    return SSDG_ERR_LIMIT;
  if (((uintptr_t)gt_boxes | (uintptr_t)out_boxes) & 15) return SSDG_ERR_ALIGN;
  if (((uintptr_t)gt_cls | (uintptr_t)gt_offsets | (uintptr_t)out_cls | (uintptr_t)out_offsets |
       (uintptr_t)out_src_row | (uintptr_t)out_transform) & 3)
    return SSDG_ERR_ALIGN;
  AugConfig c = {};
  c.seed = seed; c.image_base = image_base;
  c.height = height; c.width = width; c.max_gt = max_gt; c.n_options = n_options;
  c.trials = trials; c.max_rounds = max_rounds;
  c.zoom_p = (float)zoom_p; c.side_lo = (float)side_lo; c.side_d = (float)(side_hi - side_lo);
  c.flip_p = (float)flip_p; c.min_s = (float)min_scale; c.scale_d = (float)(max_scale - min_scale);
  c.min_ar = min_aspect; c.max_ar = max_aspect;
  for (int k = 0; k < n_options; ++k) c.options[k] = min_ious[k];
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)max_gt * sizeof(double4);
  if (smem > 48 * 1024) SSDG_CUDA_TRY(cudaFuncSetAttribute(aug_sample_kernel,
                                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  aug_sample_kernel<<<batch, kAugThreads, smem, st>>>((const float4*)gt_boxes, gt_offsets, c, out_offsets,
                                                      out_transform);
  SSDG_LAUNCH_CHECK();
  aug_scan_kernel<<<1, kAugScanThreads, 0, st>>>(out_offsets, batch);
  SSDG_LAUNCH_CHECK();
  aug_compact_kernel<<<batch, kAugThreads, 0, st>>>((const float4*)gt_boxes, gt_cls, gt_offsets, batch, c, out_offsets, out_transform, (float4*)out_boxes, out_cls,
                                                    out_src_row);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

extern "C" int ssdg_augment_images(const float* images, const int32_t* transform, int32_t batch, int32_t height,
                                   int32_t width, const float* fill, float* out_images, void* stream) {
  if (!images || !transform || !fill || !out_images || batch <= 0 || height <= 0 || width <= 0) return SSDG_ERR_ARG;
  if (height > kAugMaxSide || width > kAugMaxSide) return SSDG_ERR_LIMIT;
  if (((uintptr_t)images | (uintptr_t)transform | (uintptr_t)out_images) & 3) return SSDG_ERR_ALIGN;
  const long long pixels = (long long)batch * height * width;
  const uintptr_t a = (uintptr_t)images, o = (uintptr_t)out_images, n = (uintptr_t)(pixels * 3 * sizeof(float));
  if (a < o + n && o < a + n) return SSDG_ERR_ARG;          // in and out overlap
  long long blocks = ((pixels + 3) / 4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  aug_image_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(images, transform, pixels, height, width,
                                                                       make_float3(fill[0], fill[1], fill[2]),
                                                                       out_images);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}
