// Bounding-box evaluation on the device: compute_ats_bounding_boxes (src/utils/helper.py:33-72) with compute_iou (:79-83).
//   iou(i, j) = area(hull(box1_i) ^ hull(box2_j)) / area(hull(box1_i) u hull(box2_j))      for pairs whose axis-aligned
//   extents overlap (the reference's four strict conditions), 0 otherwise; iou_max_j = max_i iou(i, j);
//   for thresholds t in {0.5 .. 0.9}: tp = #(iou_max > t), ts = tp / (n1 + n2 - tp); result = sum(ts / t) / sum(1 / t).
// The reference walks the n1 x n2 pairs in a Python loop and builds two shapely polygons per pair (the convex hull of the
// four corners: the dataset's corner order fl, fr, bl, br is a bow-tie, hence the hull).  Here: one thread per pair,
// convex hull of 4 points (monotone chain), Sutherland-Hodgman clipping of one hull by the other, shoelace areas, all in
// float64 like shapely; the union is area1 + area2 - intersection.  The final score repeats the reference's float32
// arithmetic step by step (tensor ops on a 0-dim float32 tensor).  One CTA: box counts are tens, not thousands.
// Also the training target's rasteriser, box_raster_kernel (below).
#include "box_raster.cuh"
#include "dd_common.cuh"

namespace {

struct P2 { double x, y; };

__device__ __forceinline__ double cross(const P2& o, const P2& a, const P2& b) {
  return (a.x - o.x) * (b.y - o.y) - (a.y - o.y) * (b.x - o.x);
}

// convex hull of 4 points, counter-clockwise, collinear points dropped; returns the vertex count (0..4)
__device__ int hull4(const P2 (&in)[4], P2 (&out)[4]) {
  P2 p[4] = {in[0], in[1], in[2], in[3]};
  for (int i = 1; i < 4; ++i)                          // insertion sort by (x, y)
    for (int j = i; j > 0 && (p[j].x < p[j - 1].x || (p[j].x == p[j - 1].x && p[j].y < p[j - 1].y)); --j) {
      const P2 t = p[j]; p[j] = p[j - 1]; p[j - 1] = t;
    }
  P2 h[8];
  int k = 0;
  for (int i = 0; i < 4; ++i) {                        // lower hull
    while (k >= 2 && cross(h[k - 2], h[k - 1], p[i]) <= 0.0) --k;
    h[k++] = p[i];
  }
  for (int i = 2, t = k + 1; i >= 0; --i) {            // upper hull
    while (k >= t && cross(h[k - 2], h[k - 1], p[i]) <= 0.0) --k;
    h[k++] = p[i];
  }
  const int n = k - 1;                                 // last point repeats the first
  for (int i = 0; i < n && i < 4; ++i) out[i] = h[i];
  return n < 0 ? 0 : (n > 4 ? 4 : n);
}

__device__ double area_of(const P2* v, int n) {
  double s = 0.0;
  for (int i = 0; i < n; ++i) {
    const P2& a = v[i];
    const P2& b = v[(i + 1) % n];
    s += a.x * b.y - b.x * a.y;
  }
  return 0.5 * fabs(s);
}

// area of the intersection of two convex counter-clockwise polygons (<= 4 vertices each)
__device__ double clip_area(const P2* subj, int ns, const P2* clip, int nc) {
  P2 cur[16], nxt[16];
  int n = ns;
  for (int i = 0; i < ns; ++i) cur[i] = subj[i];
  for (int e = 0; e < nc && n > 0; ++e) {
    const P2 a = clip[e], b = clip[(e + 1) % nc];
    int m = 0;
    for (int i = 0; i < n; ++i) {
      const P2 p = cur[i], q = cur[(i + 1) % n];
      const double sp = cross(a, b, p), sq = cross(a, b, q);
      if (sp >= 0.0) nxt[m++] = p;
      if ((sp > 0.0 && sq < 0.0) || (sp < 0.0 && sq > 0.0)) {
        const double t = sp / (sp - sq);
        nxt[m].x = p.x + t * (q.x - p.x);
        nxt[m].y = p.y + t * (q.y - p.y);
        ++m;
      }
    }
    n = m;
    for (int i = 0; i < n; ++i) cur[i] = nxt[i];
  }
  return n >= 3 ? area_of(cur, n) : 0.0;
}

__global__ void __launch_bounds__(256) ats_kernel(const float* __restrict__ b1, int n1, const float* __restrict__ b2, int n2,
                                                  float* __restrict__ iou_out, float* __restrict__ ats) {
  extern __shared__ unsigned int s_max[];              // iou_max per box of boxes2, as float bits (iou >= 0: ordered like uints)
  for (int j = threadIdx.x; j < n2; j += blockDim.x) s_max[j] = 0u;
  __syncthreads();
  for (int pair = threadIdx.x; pair < n1 * n2; pair += blockDim.x) {
    const int i = pair / n2, j = pair - i * n2;
    const float* p = b1 + (size_t)i * 8;               // [2][4]: x row, y row
    const float* q = b2 + (size_t)j * 8;
    float ax0 = p[0], ax1 = p[0], ay0 = p[4], ay1 = p[4], bx0 = q[0], bx1 = q[0], by0 = q[4], by1 = q[4];
    for (int k = 1; k < 4; ++k) {
      ax0 = fminf(ax0, p[k]); ax1 = fmaxf(ax1, p[k]); ay0 = fminf(ay0, p[4 + k]); ay1 = fmaxf(ay1, p[4 + k]);
      bx0 = fminf(bx0, q[k]); bx1 = fmaxf(bx1, q[k]); by0 = fminf(by0, q[4 + k]); by1 = fmaxf(by1, q[4 + k]);
    }
    float iou = 0.f;
    if (ax1 > bx0 && ax0 < bx1 && ay1 > by0 && ay0 < by1) {       // helper.py:47-51
      P2 pa[4], pb[4], ha[4], hb[4];
      for (int k = 0; k < 4; ++k) { pa[k].x = p[k]; pa[k].y = p[4 + k]; pb[k].x = q[k]; pb[k].y = q[4 + k]; }
      const int na = hull4(pa, ha), nb = hull4(pb, hb);
      const double aa = na >= 3 ? area_of(ha, na) : 0.0, ab = nb >= 3 ? area_of(hb, nb) : 0.0;
      const double inter = (na >= 3 && nb >= 3) ? clip_area(ha, na, hb, nb) : 0.0;
      const double uni = aa + ab - inter;
      iou = (float)(inter / uni);                      // iou_matrix is a float32 tensor (helper.py:53,57); 0/0 -> nan like shapely
    }
    if (iou_out) iou_out[pair] = iou;
    if (iou > 0.f) atomicMax(&s_max[j], __float_as_uint(iou));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double thr[5] = {0.5, 0.6, 0.7, 0.8, 0.9};
    float total = 0.f;
    double weight = 0.0;
    for (int t = 0; t < 5; ++t) {
      long long tp = 0;
      for (int j = 0; j < n2; ++j) tp += __uint_as_float(s_max[j]) > (float)thr[t];     // float32 tensor > python float
      const float ts = __fdiv_rn((float)tp, (float)((long long)n1 + n2 - tp));          // tp * 1.0 / (n1 + n2 - tp)
      total = __fadd_rn(total, __fmul_rn((float)(1.0 / thr[t]), ts));                   // += 1.0 / threshold * threat_score
      weight += 1.0 / thr[t];
    }
    ats[0] = __fdiv_rn(total, (float)weight);
  }
}

}  // namespace

extern "C" int dd_ats_bounding_boxes(const float* boxes1, int n1, const float* boxes2, int n2, float* iou_matrix, float* ats,
                                     void* stream) {
  DD_REQUIRE(boxes1 && boxes2 && ats, DD_ERR_BAD_ARG, "dd_ats_bounding_boxes: null pointer");
  DD_REQUIRE(n1 >= 1 && n2 >= 1 && n2 <= 8192 && (long long)n1 * n2 <= (1 << 24), DD_ERR_BAD_ARG,
             "dd_ats_bounding_boxes: box counts %d x %d", n1, n2);
  ats_kernel<<<1, 256, (size_t)n2 * sizeof(unsigned int), dd::as_stream(stream)>>>(boxes1, n1, boxes2, n2, iou_matrix, ats);
  return dd::check_launch("ats_bounding_boxes");
}

// ---- box rasteriser: boxes_to_binary_map (src/utils/bb_to_img.py:5-21) for a batch of scenes -------------------------
// One CTA per (scene, band of kBand image rows).  The CTA converts its scene's boxes (in chunks of kChunk) to Pillow's
// integer corners and edge records in shared memory, ORs every (box, row) span into a bit row per image row (a union of
// ones: the result does not depend on the order), then writes the band's rows at their flipped positions as 16-byte
// stores of 0. / 1.  The corner arithmetic is the reference's own: metre * 10 + 400 in the boxes' dtype, each
// operation rounded separately (no FMA), truncated to int like Pillow.
namespace {

constexpr int kBand = 16;                            // image rows per CTA
constexpr int kChunk = 128;                          // boxes per shared-memory chunk
constexpr int kWords = box_raster::kMap / 32;        // 25 words of bits per row
constexpr int kRasterThreads = 256;

template <typename T>
__device__ __forceinline__ int to_pixel(T metre);
template <>
__device__ __forceinline__ int to_pixel<float>(float m) { return __float2int_rz(__fadd_rn(__fmul_rn(m, 10.f), 400.f)); }
template <>
__device__ __forceinline__ int to_pixel<double>(double m) { return __double2int_rz(__dadd_rn(__dmul_rn(m, 10.0), 400.0)); }

template <typename T>
__global__ void __launch_bounds__(kRasterThreads) box_raster_kernel(const T* __restrict__ boxes, const int* __restrict__ offsets,
                                                                    float* __restrict__ out) {
  using namespace box_raster;
  __shared__ Poly s_poly[kChunk];
  __shared__ unsigned int s_bits[kBand][kWords];
  __shared__ float s_xx[kMaxCross][kRasterThreads];
  constexpr int kBands = kMap / kBand;
  const int scene = blockIdx.x / kBands, y0 = (blockIdx.x % kBands) * kBand;
  for (int i = threadIdx.x; i < kBand * kWords; i += blockDim.x) (&s_bits[0][0])[i] = 0u;
  const int begin = offsets[scene], end = offsets[scene + 1];
  for (int c = begin; c < end; c += kChunk) {
    const int n = min(kChunk, end - c);
    __syncthreads();                                   // the previous chunk's rows are done (and the bits are zeroed)
    if (threadIdx.x < n) {
      const T* b = boxes + (size_t)(c + threadIdx.x) * 8;   // [2][4]: x row, y row; columns fl, fr, bl, br
      int x[4], y[4];
      const int col[4] = {0, 1, 3, 2};                 // drawn as fl, fr, br, bl
#pragma unroll
      for (int k = 0; k < 4; ++k) { x[k] = to_pixel<T>(b[col[k]]); y[k] = to_pixel<T>(b[4 + col[k]]); }
      build(s_poly[threadIdx.x], x, y);
    }
    __syncthreads();
    for (int p = threadIdx.x; p < n * kBand; p += blockDim.x) {
      const int r = p / n, box = p - r * n;
      row_spans(s_poly[box], y0 + r, &s_xx[0][threadIdx.x], kRasterThreads, [&](int a, int e) {
        for (int w = a >> 5; w <= (e >> 5); ++w) {
          const int lo = max(a - w * 32, 0), hi = min(e - w * 32, 31);
          const unsigned int m = (hi == 31 ? ~0u : ((1u << (hi + 1)) - 1u)) & (~0u << lo);
          atomicOr(&s_bits[r][w], m);
        }
      });
    }
  }
  __syncthreads();
  float* dst = out + (size_t)scene * kMap * kMap;
  for (int i = threadIdx.x; i < kBand * (kMap / 4); i += blockDim.x) {
    const int r = i / (kMap / 4), q = i - r * (kMap / 4);
    const unsigned int bits = s_bits[r][q >> 3] >> ((q & 7) * 4);
    const float4 v = make_float4((float)(bits & 1u), (float)((bits >> 1) & 1u), (float)((bits >> 2) & 1u),
                                 (float)((bits >> 3) & 1u));
    reinterpret_cast<float4*>(dst + (size_t)(kMap - 1 - (y0 + r)) * kMap)[q] = v;   // image row y -> output row 799 - y
  }
}

}  // namespace

extern "C" int dd_boxes_to_map(const void* boxes, int boxes_f64, const int* offsets, int B, float* out, void* stream) {
  DD_REQUIRE(B >= 0, DD_ERR_BAD_ARG, "dd_boxes_to_map: B = %d < 0", B);
  if (B == 0) return DD_OK;
  DD_REQUIRE(boxes && offsets && out, DD_ERR_BAD_ARG, "dd_boxes_to_map: null pointer (boxes %p, offsets %p, out %p)", boxes,
             (const void*)offsets, (void*)out);
  DD_REQUIRE(((uintptr_t)out & 15) == 0, DD_ERR_ALIGNMENT, "dd_boxes_to_map: out must be 16-byte aligned");
  const long long grid = (long long)B * (box_raster::kMap / kBand);
  DD_REQUIRE(grid <= 0x7fffffffLL, DD_ERR_BAD_ARG, "dd_boxes_to_map: B = %d is too large", B);
  if (boxes_f64)
    box_raster_kernel<double><<<(unsigned)grid, kRasterThreads, 0, dd::as_stream(stream)>>>(
        static_cast<const double*>(boxes), offsets, out);
  else
    box_raster_kernel<float><<<(unsigned)grid, kRasterThreads, 0, dd::as_stream(stream)>>>(
        static_cast<const float*>(boxes), offsets, out);
  return dd::check_launch("boxes_to_map");
}
