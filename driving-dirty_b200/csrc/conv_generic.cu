// Generic 2-D convolution / transposed convolution on the CUDA cores (fp32 accumulate, fp32 or bf16
// NHWC storage): any kernel size, stride, padding, dilation, channel counts.  This is the fp32
// parity path (and the on-device check for tensor-core versions) of every layer of the scene
// pipeline that is not one of the three encoder convs:
//   Decoder dc1..dc4            components.py:70-73,89-92   (ConvTranspose2d k3 p1, k3 p1, k2 s2, k1)
//   SpatialMappingCNN convs     spatial_bb/components.py:18-26,34-76 (1x50 / 52x1 stride (3,2), 3x3 valid)
//   RoadMapBoxesMergingCNN      spatial_bb/components.py:129-139,149-168 (1x24 s(1,7), k2 s2 deconv,
//                               k7 s3 d3 p1, k3 d3, four dilated ConvTranspose2d k7, k2 s2 deconv)
//
// Both directions are written as GATHERS over the output pixel:
//   conv : y[ho,wo,co] = sum_{kh,kw,ci} x[ho*sh - ph + kh*dh, wo*sw - pw + kw*dw, ci] * W[co,ci,kh,kw]
//   convT: y[ho,wo,co] = sum_{kh,kw,ci} x[(ho + ph - kh*dh)/sh, (wo + pw - kw*dw)/sw, ci] * W[ci,co,kh,kw]
//          (terms whose division is not exact are absent)
// so the input gradient of a conv is the convT gather over dy with the SAME weight tensor, and vice
// versa; the weight gradient of either is one "pivot x shifted" pixel contraction.
#include "dd_common.cuh"

namespace {

struct Geo {
  int B, Ci, Co;          // channels of the gathered tensor / of the produced tensor
  int Hi, Wi, Ho, Wo;     // gathered tensor grid / produced tensor grid
  int kh, kw, sh, sw, ph, pw, dh, dw;
  int transposed;         // gather form (see above)
};

// wg[t][a][b] = w[a][b][t] (swap = 0) or w[b][a][t] (swap = 1); A, Bc = sizes of a, b; T taps
__global__ void wprep_kernel(const float* __restrict__ w, float* __restrict__ wg, int A, int Bc, int T, int swap) {
  const int n = A * Bc * T;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int b = i % Bc, a = (i / Bc) % A, t = i / (A * Bc);
    wg[i] = swap ? w[((size_t)b * A + a) * T + t] : w[((size_t)a * Bc + b) * T + t];
  }
}

__device__ __forceinline__ bool tap_coord(const Geo& g, int o, int k, int s, int p, int d, int n, int& i) {
  if (!g.transposed) {
    i = o * s - p + k * d;
    return i >= 0 && i < n;
  }
  const int t = o + p - k * d;
  if (t < 0) return false;
  i = t / s;
  return (i * s == t) && i < n;
}

// ------------------------------------------------------------------------------------------------
// forward / input-gradient gather: thread = 1 output pixel x 16 output channels, CTA = 256 threads,
// weights of one tap staged in shared memory ([ci][CO_T]) and read as broadcast float4s.
// act: 0 none, 1 ReLU, 2 sigmoid.  mask (optional, same shape as y): y *= (mask > 0).
// Strided transposed gathers (the input gradient of a strided conv, a strided ConvTranspose2d): an output pixel only sees
// the taps of its residue class modulo the stride.  gridDim.z = sh * sw classes: a CTA's pixels all belong to ONE class, so
// the taps the class cannot see are skipped for the whole CTA (no staging, no barrier) and every thread works on the
// others -- ss_conv's input gradient (1x24 taps, stride 7: 3-4 of 24 taps per pixel) 6.6 -> ~1 ms.
// ------------------------------------------------------------------------------------------------
constexpr int MAX_CI = 128;

template <typename T, int CO_T>
__global__ void __launch_bounds__(256) conv2d_gather_kernel(const T* __restrict__ x, const float* __restrict__ wg,
                                                            const float* __restrict__ bias, const T* __restrict__ mask,
                                                            T* __restrict__ y, Geo g, int act) {
  constexpr int TPP = CO_T / 16;            // threads per pixel
  constexpr int PIX = 256 / TPP;
  __shared__ __align__(16) float s_w[MAX_CI * CO_T];
  const int tid = threadIdx.x;
  const int sub = tid % TPP;
  const bool by_class = gridDim.z > 1;                 // launch_gather: transposed with a stride
  const int rh = by_class ? (int)blockIdx.z / g.sw : 0, rw = by_class ? (int)blockIdx.z % g.sw : 0;
  const int ch = by_class ? g.sh : 1, cw = by_class ? g.sw : 1;
  const int Hc = g.Ho > rh ? (g.Ho - rh + ch - 1) / ch : 0, Wc = g.Wo > rw ? (g.Wo - rw + cw - 1) / cw : 0;   // pixels of the class
  const long long npix = (long long)g.B * Hc * Wc;
  const long long idx = (long long)blockIdx.x * PIX + tid / TPP;
  const bool live = idx < npix;
  const int co0 = blockIdx.y * CO_T;
  int wo = 0, ho = 0, b = 0;
  if (live) {
    wo = rw + (int)(idx % Wc) * cw;
    ho = rh + (int)((idx / Wc) % Hc) * ch;
    b = (int)(idx / ((long long)Wc * Hc));
  }
  const long long pix = ((long long)b * g.Ho + ho) * g.Wo + wo;
  float acc[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) acc[k] = 0.f;
  const bool vec = (g.Ci % 8) == 0;
  const T* img = x + (size_t)b * g.Hi * g.Wi * g.Ci;

  for (int t = 0; t < g.kh * g.kw; ++t) {
    if (by_class) {                                    // CTA-uniform: taps outside the residue class contribute nothing
      const int th = rh + g.ph - (t / g.kw) * g.dh, tw = rw + g.pw - (t % g.kw) * g.dw;
      if (((th % g.sh) + g.sh) % g.sh != 0 || ((tw % g.sw) + g.sw) % g.sw != 0) continue;
    }
    __syncthreads();
    for (int i = tid; i < g.Ci * CO_T; i += 256) {
      const int c = i % CO_T, ci = i / CO_T;
      s_w[i] = (co0 + c < g.Co) ? __ldg(wg + ((size_t)t * g.Ci + ci) * g.Co + co0 + c) : 0.f;
    }
    __syncthreads();
    int hi, wi;
    const bool ok = live && tap_coord(g, ho, t / g.kw, g.sh, g.ph, g.dh, g.Hi, hi) &&
                    tap_coord(g, wo, t % g.kw, g.sw, g.pw, g.dw, g.Wi, wi);
    if (!ok) continue;
    const T* px = img + ((size_t)hi * g.Wi + wi) * g.Ci;
    const float4* w4 = reinterpret_cast<const float4*>(s_w + sub * 16);
    if (vec) {
      for (int c8 = 0; c8 < g.Ci; c8 += 8) {
        float xv[8];
        dd::ld8<T>(px + c8, xv);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float4* wr = w4 + (size_t)(c8 + e) * (CO_T / 4);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 ww = wr[q];
            acc[4 * q + 0] = fmaf(xv[e], ww.x, acc[4 * q + 0]);
            acc[4 * q + 1] = fmaf(xv[e], ww.y, acc[4 * q + 1]);
            acc[4 * q + 2] = fmaf(xv[e], ww.z, acc[4 * q + 2]);
            acc[4 * q + 3] = fmaf(xv[e], ww.w, acc[4 * q + 3]);
          }
        }
      }
    } else {
      for (int ci = 0; ci < g.Ci; ++ci) {
        const float xv = dd::ld<T>(px + ci);
        const float4* wr = w4 + (size_t)ci * (CO_T / 4);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 ww = wr[q];
          acc[4 * q + 0] = fmaf(xv, ww.x, acc[4 * q + 0]);
          acc[4 * q + 1] = fmaf(xv, ww.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(xv, ww.z, acc[4 * q + 2]);
          acc[4 * q + 3] = fmaf(xv, ww.w, acc[4 * q + 3]);
        }
      }
    }
  }
  if (!live) return;
  const int cbase = co0 + sub * 16;
  T* out = y + (size_t)pix * g.Co + cbase;
  const T* mk = mask ? mask + (size_t)pix * g.Co + cbase : nullptr;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if (cbase + k >= g.Co) break;
    float v = acc[k] + (bias ? __ldg(bias + cbase + k) : 0.f);
    if (act == 1) v = fmaxf(v, 0.f);
    else if (act == 2) {
      const float e = expf(-fabsf(v));
      const float inv = __frcp_rn(1.0f + e);
      v = v >= 0.f ? inv : e * inv;
    }
    if (mk && !(dd::ld<T>(mk + k) > 0.f)) v = 0.f;
    dd::st<T>(out + k, v);
  }
}

// ------------------------------------------------------------------------------------------------
// weight gradient: out[t][cP][cQ] = sum_p P[p][cP] * Q[shift(p, t)][cQ]
//   conv : P = dy (pivot grid = output grid), Q = x       -> dW[co][ci][t]
//   convT: P = x  (pivot grid = input grid),  Q = dy      -> dW[ci][co][t]
// shift(p, t) = p*s - pad + k*d (both cases).  grid = (taps, splits); thread (i, j) of a 16x16
// layout owns cP in {i + 16a}, cQ in {j + 16b}; pixels staged 32 at a time through shared memory;
// per-(split) partials, folded in order by wgrad_fold_kernel.
// ------------------------------------------------------------------------------------------------
struct WGeo {
  int B, cP, cQ, Hp, Wp, Hq, Wq, kh, kw, sh, sw, ph, pw, dh, dw;
  long long pix_per_split;
};

template <typename T, int TP, int TQ>
__global__ void __launch_bounds__(256) conv2d_wgrad_kernel(const T* __restrict__ P, const T* __restrict__ Q,
                                                           float* __restrict__ partial, WGeo g) {
  constexpr int CH = 32;                       // pixels per stage
  constexpr int PP = TP * 16, QQ = TQ * 16;
  __shared__ float s_p[CH][PP + 1];
  __shared__ float s_q[CH][QQ + 1];
  const int tid = threadIdx.x, i = tid & 15, j = tid >> 4;
  const int t = blockIdx.x, kh_i = t / g.kw, kw_i = t % g.kw;
  const long long npix = (long long)g.B * g.Hp * g.Wp;
  const long long p_begin = (long long)blockIdx.y * g.pix_per_split;
  const long long p_end = p_begin + g.pix_per_split < npix ? p_begin + g.pix_per_split : npix;
  float acc[TP][TQ];
#pragma unroll
  for (int a = 0; a < TP; ++a)
#pragma unroll
    for (int b = 0; b < TQ; ++b) acc[a][b] = 0.f;

  for (long long p0 = p_begin; p0 < p_end; p0 += CH) {
    __syncthreads();
    for (int e = tid; e < CH * PP; e += 256) {
      const int c = e % PP, l = e / PP;
      const long long p = p0 + l;
      s_p[l][c] = (p < p_end && c < g.cP) ? dd::ld<T>(P + (size_t)p * g.cP + c) : 0.f;
    }
    for (int e = tid; e < CH * QQ; e += 256) {
      const int c = e % QQ, l = e / QQ;
      const long long p = p0 + l;
      float v = 0.f;
      if (p < p_end && c < g.cQ) {
        const int wp = (int)(p % g.Wp), hp = (int)((p / g.Wp) % g.Hp);
        const long long b = p / ((long long)g.Wp * g.Hp);
        const int hq = hp * g.sh - g.ph + kh_i * g.dh, wq = wp * g.sw - g.pw + kw_i * g.dw;
        if (hq >= 0 && hq < g.Hq && wq >= 0 && wq < g.Wq)
          v = dd::ld<T>(Q + (((size_t)b * g.Hq + hq) * g.Wq + wq) * g.cQ + c);
      }
      s_q[l][c] = v;
    }
    __syncthreads();
#pragma unroll 4
    for (int l = 0; l < CH; ++l) {
      float pv[TP], qv[TQ];
#pragma unroll
      for (int a = 0; a < TP; ++a) pv[a] = s_p[l][i + 16 * a];
#pragma unroll
      for (int b = 0; b < TQ; ++b) qv[b] = s_q[l][j + 16 * b];
#pragma unroll
      for (int a = 0; a < TP; ++a)
#pragma unroll
        for (int b = 0; b < TQ; ++b) acc[a][b] = fmaf(pv[a], qv[b], acc[a][b]);
    }
  }
  float* out = partial + ((size_t)blockIdx.y * gridDim.x + t) * g.cP * g.cQ;
#pragma unroll
  for (int a = 0; a < TP; ++a)
#pragma unroll
    for (int b = 0; b < TQ; ++b) {
      const int cp = i + 16 * a, cq = j + 16 * b;
      if (cp < g.cP && cq < g.cQ) out[cp * g.cQ + cq] = acc[a][b];
    }
}

// ------------------------------------------------------------------------------------------------
// weight gradient, second form: ALL taps per CTA.  The kernel above gives every (tap, pixel range) its own CTA, so the
// pivot tensor P is re-read once per tap (49 x for the 7 x 7 layers) through scalar loads: 0.3-6 TFLOP/s on the
// small-channel layers of the bounding-box model (up_conv_3 / 4, rm_conv_1, the strip convs, ss_conv), 150 of that
// model's 174 ms step.  Here a CTA walks row segments of the pivot grid; a segment's P pixels and the KH rows of Q it
// touches are staged in shared memory ONCE, and every thread owns a register tile acc[TT taps][TP cP][TQ cQ] that
// lives for the whole launch (thread = (pixel lane, tap group, cP group, cQ group)).  Per-(CTA, pixel lane) partials,
// folded in order by wgrad_fold_kernel (deterministic).
// ------------------------------------------------------------------------------------------------
struct WTile {
  int ntg, npg, nqg, lanes;     // tap / cP / cQ groups, pixel lanes; ntg * npg * nqg * lanes <= 256
  int seg, qw;                  // pivot pixels per row segment; staged Q pixels per row = (seg-1)*sw + (kw-1)*dw + 1
  int segs_per_row, nseg;       // segments per pivot row; total segments = B * Hp * segs_per_row
};

template <typename T, int TT, int TP, int TQ>
__global__ void __launch_bounds__(256) conv2d_wgrad_tile_kernel(const T* __restrict__ P, const T* __restrict__ Q,
                                                                float* __restrict__ partial, WGeo g, WTile c) {
  extern __shared__ float s_tile[];
  const int cPp = c.npg * TP, cQp = c.nqg * TQ;
  float* s_p = s_tile;                                  // [seg][cPp]
  float* s_q = s_tile + c.seg * cPp;                    // [kh][qw][cQp]
  const int tid = threadIdx.x;
  const int ngroups = c.ntg * c.npg * c.nqg;
  const int grp = tid % ngroups, pl = tid / ngroups;
  const int qg = grp % c.nqg, pg = (grp / c.nqg) % c.npg, tg = grp / (c.nqg * c.npg);
  const bool active = pl < c.lanes;
  const int taps = g.kh * g.kw;
  int qoff[TT];
#pragma unroll
  for (int tt = 0; tt < TT; ++tt) {
    const int tap = min(tg * TT + tt, taps - 1);        // (padding taps recompute the last one; never written out)
    qoff[tt] = ((tap / g.kw) * c.qw + (tap % g.kw) * g.dw) * cQp + qg * TQ;
  }
  float acc[TT][TP][TQ];
#pragma unroll
  for (int tt = 0; tt < TT; ++tt)
#pragma unroll
    for (int a = 0; a < TP; ++a)
#pragma unroll
      for (int b = 0; b < TQ; ++b) acc[tt][a][b] = 0.f;

  for (int sgi = blockIdx.x; sgi < c.nseg; sgi += gridDim.x) {
    const int ws = sgi % c.segs_per_row;
    const int hp = (sgi / c.segs_per_row) % g.Hp;
    const int b = sgi / (c.segs_per_row * g.Hp);
    const int wp0 = ws * c.seg;
    __syncthreads();
    for (int e = tid; e < c.seg * cPp; e += 256) {
      const int ch = e % cPp, px = e / cPp;
      s_p[e] = (wp0 + px < g.Wp && ch < g.cP) ? dd::ld<T>(P + (((size_t)b * g.Hp + hp) * g.Wp + wp0 + px) * g.cP + ch) : 0.f;
    }
    const int wq0 = wp0 * g.sw - g.pw;
    for (int e = tid; e < g.kh * c.qw * cQp; e += 256) {
      const int ch = e % cQp, x = (e / cQp) % c.qw, khi = e / (cQp * c.qw);
      const int hq = hp * g.sh - g.ph + khi * g.dh, wq = wq0 + x;
      s_q[e] = (ch < g.cQ && hq >= 0 && hq < g.Hq && wq >= 0 && wq < g.Wq)
                   ? dd::ld<T>(Q + (((size_t)b * g.Hq + hq) * g.Wq + wq) * g.cQ + ch) : 0.f;
    }
    __syncthreads();
    if (active) {
      for (int px = pl; px < c.seg; px += c.lanes) {
        float pv[TP];
#pragma unroll
        for (int a = 0; a < TP; ++a) pv[a] = s_p[px * cPp + pg * TP + a];
        const float* qrow = s_q + px * g.sw * cQp;
#pragma unroll
        for (int tt = 0; tt < TT; ++tt) {
          float qv[TQ];
#pragma unroll
          for (int bq = 0; bq < TQ; ++bq) qv[bq] = qrow[qoff[tt] + bq];
#pragma unroll
          for (int a = 0; a < TP; ++a)
#pragma unroll
            for (int bq = 0; bq < TQ; ++bq) acc[tt][a][bq] = fmaf(pv[a], qv[bq], acc[tt][a][bq]);
        }
      }
    }
  }
  if (active) {
    float* out = partial + ((size_t)blockIdx.x * c.lanes + pl) * taps * g.cP * g.cQ;
#pragma unroll
    for (int tt = 0; tt < TT; ++tt) {
      const int tap = tg * TT + tt;
      if (tap >= taps) continue;
#pragma unroll
      for (int a = 0; a < TP; ++a)
#pragma unroll
        for (int bq = 0; bq < TQ; ++bq) {
          const int cp = pg * TP + a, cq = qg * TQ + bq;
          if (cp < g.cP && cq < g.cQ) out[((size_t)tap * g.cP + cp) * g.cQ + cq] = acc[tt][a][bq];
        }
    }
  }
}

// picks a register tiling for the all-taps form; false: this layer keeps the per-tap kernel
static bool wtile_config(const WGeo& g, int taps, int& TT, int& TP, int& TQ, WTile& c, size_t& smem, int& grid) {
  if (g.cP % 4 != 0 && g.cP > 4) return false;
  TP = 4;
  TQ = g.cQ % 4 == 0 ? 4 : (g.cQ == 3 ? 3 : (g.cQ == 1 ? 1 : 0));
  if (TQ == 0) return false;
  TT = taps % 7 == 0 ? 7 : (taps <= 4 ? 4 : (taps % 8 == 0 ? 8 : 7));
  if (TT == 4 && TQ == 3) return false;     // not instantiated (launch_wgrad_cc): e.g. the decoder's dc4, 32 -> 3, 1 tap
  c.ntg = (taps + TT - 1) / TT; c.npg = (g.cP + TP - 1) / TP; c.nqg = (g.cQ + TQ - 1) / TQ;
  const int ngroups = c.ntg * c.npg * c.nqg;
  if (ngroups > 256) return false;
  c.lanes = 256 / ngroups;
  c.seg = 64;
  while (true) {
    c.qw = (c.seg - 1) * g.sw + (g.kw - 1) * g.dw + 1;
    smem = ((size_t)c.seg * c.npg * TP + (size_t)g.kh * c.qw * c.nqg * TQ) * sizeof(float);
    if (smem <= 96 * 1024 || c.seg <= 16) break;
    c.seg /= 2;
  }
  if (smem > 200 * 1024) return false;
  if (c.lanes > c.seg) c.lanes = c.seg;
  c.segs_per_row = (g.Wp + c.seg - 1) / c.seg;
  const long long nseg = (long long)g.B * g.Hp * c.segs_per_row;
  if (nseg > 0x7fffffff) return false;
  c.nseg = (int)nseg;
  grid = (int)(nseg < 2 * dd::kSMs ? nseg : 2 * dd::kSMs);
  return true;
}

// dw[cP][cQ][t] = sum over splits (in order) of partial[split][t][cP][cQ]
__global__ void wgrad_fold_kernel(const float* __restrict__ partial, float* __restrict__ dw, int taps, int cPQ, int splits) {
  const int n = taps * cPQ;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const int pq = e % cPQ, t = e / cPQ;
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += partial[(size_t)k * n + e];
    dw[(size_t)pq * taps + t] = s;
  }
}

// db[c] = sum over pixels of dy[p][c]: per-CTA partials then an ordered fold.  Accumulated in double:
// a bias gradient is a long mixed-sign sum ((p - t)/N terms) and fp32 partials lose ~1e-4 of it.
template <typename T>
__global__ void __launch_bounds__(256) chansum_kernel(const T* __restrict__ dy, long long npix, int Cn, double* __restrict__ partial) {
  __shared__ double red[256];
  const int tid = threadIdx.x;
  const int lanes = 256 / Cn > 0 ? 256 / Cn : 1;     // pixel lanes per CTA (Cn <= 256)
  const int c = tid % Cn, pl = tid / Cn;
  double s = 0.0;
  if (pl < lanes)
    for (long long p = (long long)blockIdx.x * lanes + pl; p < npix; p += (long long)gridDim.x * lanes)
      s += (double)dd::ld<T>(dy + (size_t)p * Cn + c);
  red[tid] = (pl < lanes) ? s : 0.0;
  __syncthreads();
  if (tid < Cn) {
    double tsum = 0.0;
    for (int l = 0; l < lanes; ++l) tsum += red[l * Cn + tid];
    partial[(size_t)blockIdx.x * Cn + tid] = tsum;
  }
}
__global__ void chansum_fold_kernel(const double* __restrict__ partial, int nblk, int Cn, float* __restrict__ db) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cn) return;
  double s = 0.0;
  for (int k = 0; k < nblk; ++k) s += partial[(size_t)k * Cn + c];
  db[c] = (float)s;
}

constexpr int kChanBlocks = dd::kSMs * 2;

bool desc_ok(const dd_conv_desc* d) {
  return d && d->B >= 0 && d->Cin > 0 && d->Cout > 0 && d->Hi > 0 && d->Wi > 0 && d->Ho > 0 && d->Wo > 0 && d->kh > 0 &&
         d->kw > 0 && d->sh > 0 && d->sw > 0 && d->ph >= 0 && d->pw >= 0 && d->dh > 0 && d->dw > 0;
}

size_t wg_bytes(const dd_conv_desc* d) { return ((size_t)d->kh * d->kw * d->Cin * d->Cout * sizeof(float) + 255) / 256 * 256; }

int wgrad_splits(const dd_conv_desc* d, long long npix) {
  const int taps = d->kh * d->kw;
  int s = (dd::kSMs * 4 + taps - 1) / taps;
  const long long maxs = (npix + 255) / 256;
  if (s > maxs) s = (int)maxs;
  return s < 1 ? 1 : s;
}

template <typename T>
int launch_gather(const T* x, const float* wg, const float* bias, const T* mask, T* y, const Geo& g, int act, cudaStream_t st) {
  if (g.Ci > MAX_CI) return dd::fail(DD_ERR_UNSUPPORTED, "conv2d: %d input channels > %d", g.Ci, MAX_CI);
  const bool by_class = g.transposed && (g.sh > 1 || g.sw > 1) && g.sh * g.sw <= 64;
  const int ch = by_class ? g.sh : 1, cw = by_class ? g.sw : 1;
  const long long npix = (long long)g.B * ((g.Ho + ch - 1) / ch) * ((g.Wo + cw - 1) / cw);     // of the largest class
  const unsigned classes = by_class ? (unsigned)(g.sh * g.sw) : 1u;
  if (g.Co > 16) {
    dim3 grid((unsigned)((npix + 127) / 128), (g.Co + 31) / 32, classes);
    conv2d_gather_kernel<T, 32><<<grid, 256, 0, st>>>(x, wg, bias, mask, y, g, act);
  } else {
    dim3 grid((unsigned)((npix + 255) / 256), 1, classes);
    conv2d_gather_kernel<T, 16><<<grid, 256, 0, st>>>(x, wg, bias, mask, y, g, act);
  }
  return dd::check_launch("conv2d_gather");
}

template <typename T>
int launch_wgrad(const T* P, const T* Q, float* partial, const WGeo& g, int taps, int splits, cudaStream_t st) {
  dim3 grid(taps, splits);
  const int tp = (g.cP + 15) / 16, tq = (g.cQ + 15) / 16;
#define DD_WG(TPv, TQv) conv2d_wgrad_kernel<T, TPv, TQv><<<grid, 256, 0, st>>>(P, Q, partial, g)
  if (tp <= 1 && tq <= 1) DD_WG(1, 1);
  else if (tp <= 2 && tq <= 1) DD_WG(2, 1);
  else if (tp <= 1 && tq <= 2) DD_WG(1, 2);
  else if (tp <= 2 && tq <= 2) DD_WG(2, 2);
  else if (tp <= 4 && tq <= 2) DD_WG(4, 2);
  else if (tp <= 2 && tq <= 4) DD_WG(2, 4);
  else if (tp <= 4 && tq <= 4) DD_WG(4, 4);
  else if (tp <= 6 && tq <= 4) DD_WG(6, 4);
  else if (tp <= 4 && tq <= 6) DD_WG(4, 6);
  else return dd::fail(DD_ERR_UNSUPPORTED, "conv2d wgrad: channel tile %dx%d", g.cP, g.cQ);
#undef DD_WG
  return dd::check_launch("conv2d_wgrad");
}

// CUDA-core weight-gradient partials: the all-taps register-tiled form where wtile_config finds a tiling (small channel
// counts), else one CTA per (tap, pixel range).  slots = partial buffers written, for wgrad_fold_kernel.
template <typename T>
int launch_wgrad_cc(const T* P, const T* Q, float* partial, const WGeo& g, int taps, int splits, int& slots, cudaStream_t st) {
  int TT, TP, TQ, grid;
  WTile c;
  size_t smem;
  if (!wtile_config(g, taps, TT, TP, TQ, c, smem, grid)) {
    slots = splits;
    return launch_wgrad(P, Q, partial, g, taps, splits, st);
  }
  slots = grid * c.lanes;
#define DD_WT(a, b, q)                                                                                             \
  if (TT == a && TP == b && TQ == q) {                                                                             \
    auto k = conv2d_wgrad_tile_kernel<T, a, b, q>;                                                                 \
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "conv2d wgrad tile")) return e;                      \
    k<<<grid, 256, smem, st>>>(P, Q, partial, g, c);                                                               \
    return dd::check_launch("conv2d_wgrad_tile");                                                                  \
  }
  DD_WT(7, 4, 4) DD_WT(7, 4, 1) DD_WT(7, 4, 3) DD_WT(8, 4, 4) DD_WT(4, 4, 4) DD_WT(4, 4, 1) DD_WT(8, 4, 3) DD_WT(8, 4, 1)
#undef DD_WT
  return dd::fail(DD_ERR_UNSUPPORTED, "conv2d wgrad tile: no instantiation for %d taps x %d x %d", TT, TP, TQ);
}
}  // namespace

// tcgen05 kernels for the stride-1 (dilated) layers: conv_dil_tc.cu, conv_dil_wgrad_tc.cu.  K / N: gathered / produced
// channels per pixel as launched, of which the first Kreal / Nreal exist in the weights (the rest are zero padding).
namespace dd {
bool conv_dil_tc_supported(int K, int N, int KT, int D);
int conv_dil_tc(const void* in, const float* w, long long sn, long long sk, int flip, const float* bias, const void* mask, void* out,
                void* pack_ws, int B, int Hi, int Wi, int Ho, int Wo, int K, int N, int KT, int D, int sign, int off, int relu,
                cudaStream_t st, int Kreal, int Nreal);
bool conv_dil_wgrad_tc_supported(int K, int N, int KT, int D);
size_t conv_dil_wgrad_tc_ws_bytes(int K, int N, int KT);
int conv_dil_wgrad_tc(const void* in, const void* dout, float* dw, long long sn, long long sk, void* ws, size_t ws_bytes, int B,
                      int Hi, int Wi, int Ho, int Wo, int K, int N, int KT, int D, int sign, int off, cudaStream_t st, int Kreal,
                      int Nreal);
}  // namespace dd

// ---- narrow layers on the tensor-core kernels: 8- / 16-channel pixels zero-padded to the kernels' 32 ------------------------
// up_conv_3 (32 -> 16) and up_conv_4 (16 -> 8) of RoadMapBoxesMergingCNN (spatial_bb/components.py:137-138) gather or
// contract over tensors with 8 or 16 channels; the tcgen05 kernels want whole 64-byte pixels.  One pass copies the narrow
// tensor into 32-channel pixels (zeros above), the weights of the missing channels are packed as zeros (Kreal) and the
// weight-gradient fold drops them (Kreal / Nreal): up_conv_3 input gradient 6.9 -> 0.7 ms, weight gradient 12.4 -> 2.1.
namespace {
__global__ void chan_pad32_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long npix, int cs) {
  const long long total = npix * 4;                       // four 16-byte pieces per padded pixel
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long pix = i >> 2;
    const int c8 = (int)(i & 3) * 8;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (c8 < cs) v = *reinterpret_cast<const uint4*>(src + pix * cs + c8);
    *reinterpret_cast<uint4*>(dst + pix * 32 + c8) = v;
  }
}
int pad32(const void* src, void* dst, long long npix, int cs, cudaStream_t st) {
  const long long want = (npix * 4 + 255) / 256;
  chan_pad32_kernel<<<(int)(want < dd::kSMs * 16 ? want : dd::kSMs * 16), 256, 0, st>>>((const __nv_bfloat16*)src, (__nv_bfloat16*)dst, npix, cs);
  return dd::check_launch("conv2d_chan_pad");
}
// forward of a layer that PRODUCES 8 channels: the kernel's narrowest instantiation writes 16-channel pixels; drop the upper 8
__global__ void chan_unpad16to8_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long npix) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (long long)gridDim.x * blockDim.x)
    reinterpret_cast<uint4*>(dst)[i] = *reinterpret_cast<const uint4*>(src + i * 16);
}
__global__ void bias_pad_kernel(const float* __restrict__ b, float* __restrict__ out, int n, int npad) {
  const int i = threadIdx.x;
  if (i < npad) out[i] = (b != nullptr && i < n) ? b[i] : 0.f;
}
inline bool narrow(int c) { return c == 8 || c == 16; }
inline int padded(int c) { return narrow(c) ? 32 : c; }
size_t pad_slot(long long npix) { return ((size_t)npix * 64 + 1023) / 1024 * 1024; }   // one tensor in 32-channel bf16 pixels

// ---- which engine runs a pass ------------------------------------------------------------------------------------------------
// A pass (0 forward, 1 input gradient, 2 weight gradient) runs on the tensor cores when the layer is bf16, stride 1, a square
// filter with one dilation and padding for both axes, and its channel counts, after the padding below, are ones the kernels
// take.  Everything else, and fp32 (the parity path), runs on the CUDA-core kernels above.
struct TcPlan {
  bool ok = false;
  int K = 0, N = 0;             // gathered / produced channels as launched: x / y, dy / dx, x / dy
  int Kreal = 0, Nreal = 0;     // as in the layer; K > Kreal or N > Nreal: that tensor goes through a padded copy
  long long sn = 0, sk = 0;     // strides of the produced / gathered channel index in the torch-layout weights
  int flip = 0, sign = 0, off = 0;
  // workspace: [core_ws_bytes | dy's copy, or the forward's 16-channel y | x's copy | padded bias]; offsets past core_ws_bytes
  size_t x_pad = 0, bias_pad = 0;
  bool padded() const { return ok && (K != Kreal || N != Nreal); }
};

TcPlan tc_plan(const dd_conv_desc* d, int dtype, int pass, int act) {
  TcPlan p;
  if (dtype != DD_BF16 || d->sh != 1 || d->sw != 1 || d->kh != d->kw || d->dh != d->dw || d->ph != d->pw) return p;
  if (pass == 0 && act == 2) return p;                  // the kernels' epilogue has bias and ReLU, no sigmoid
  const bool dgrad = pass == 1;
  p.Kreal = dgrad ? d->Cout : d->Cin;
  p.Nreal = dgrad ? d->Cin : d->Cout;
  p.K = padded(p.Kreal);                                // 8 / 16 gathered channels -> 32 in every pass
  // produced channels: the weight gradient pads 8 / 16 -> 32 (its kernel takes 32 or 64); the forward pads 8 -> 16 (the
  // narrowest instantiation) and narrows the result; the input gradient pads none (no layer here needs an 8-channel dx)
  p.N = pass == 2 ? padded(p.Nreal) : (pass == 0 && p.Nreal == 8 ? 16 : p.Nreal);
  p.ok = pass == 2 ? dd::conv_dil_wgrad_tc_supported(p.K, p.N, d->kh, d->dh) : dd::conv_dil_tc_supported(p.K, p.N, d->kh, d->dh);
  // Conv2d weights are [Cout][Cin][t], ConvTranspose2d [Cin][Cout][t].  The ConvT forward and the Conv input gradient gather
  // from h - D*kh + p (flip 0, sign -1); the Conv forward and the ConvT input gradient from h + D*kh - p (flip 1, sign +1).
  // The weight gradient takes the forward's strides, sign and offset.
  const bool convT_gather = d->transposed != dgrad;
  const long long T = (long long)d->kh * d->kw;
  p.sn = convT_gather ? T : p.Kreal * T;
  p.sk = convT_gather ? p.Nreal * T : T;
  p.flip = !convT_gather;
  p.sign = convT_gather ? -1 : +1;
  p.off = convT_gather ? d->ph : -d->ph;
  const size_t y_slot = narrow(d->Cout) ? pad_slot((long long)d->B * d->Ho * d->Wo) : 0;
  p.x_pad = y_slot;
  p.bias_pad = y_slot + (narrow(d->Cin) ? pad_slot((long long)d->B * d->Hi * d->Wi) : 0);
  return p;
}
}  // namespace

extern "C" int dd_conv2d_tc_supported(const dd_conv_desc* d, int dtype, int pass) {
  return desc_ok(d) && tc_plan(d, dtype, pass, 0).ok;
}

// CUDA-core weights / weight-gradient partials or the tensor-core weight gradient's partials, then the bias gradient's
// channel sums; the padded copies sit behind all of it (1024-byte aligned)
static size_t core_ws_bytes(const dd_conv_desc* d) {
  const long long np_out = (long long)d->B * d->Ho * d->Wo, np_in = (long long)d->B * d->Hi * d->Wi;
  const long long pivot = d->transposed ? np_in : np_out;
  const size_t partial = (size_t)wgrad_splits(d, pivot) * d->kh * d->kw * d->Cin * d->Cout * sizeof(float);
  const size_t chan = (size_t)kChanBlocks * d->Cout * sizeof(double) + 8;
  const size_t tile_partial = (size_t)2 * dd::kSMs * 256 * 128 * sizeof(float);   // all-taps form: slots x taps x cP x cQ <= CTAs x 256 threads x 128 accumulators
  const size_t a = wg_bytes(d), b = (partial > tile_partial ? partial : tile_partial) + chan;
  const TcPlan wgrad = tc_plan(d, DD_BF16, 2, 0);
  const size_t c = wgrad.ok ? dd::conv_dil_wgrad_tc_ws_bytes(wgrad.K, wgrad.N, d->kh) + chan : 0;
  const size_t m = a > b ? a : b;
  return ((m > c ? m : c) + 256 + 1023) / 1024 * 1024;
}

extern "C" size_t dd_conv2d_workspace_bytes(const dd_conv_desc* d) {
  if (!desc_ok(d)) return 256;
  size_t pad = 0;
  if (tc_plan(d, DD_BF16, 0, 0).padded() || tc_plan(d, DD_BF16, 1, 0).padded() || tc_plan(d, DD_BF16, 2, 0).padded()) {
    // room for the copies at the offsets tc_plan gives
    const size_t np_out = (size_t)d->B * d->Ho * d->Wo, np_in = (size_t)d->B * d->Hi * d->Wi;
    pad = (narrow(d->Cout) ? np_out * 64 + 1024 : 0) + (narrow(d->Cin) ? np_in * 64 + 1024 : 0) + 2048;
  }
  return core_ws_bytes(d) + pad;
}

extern "C" int dd_conv2d_fwd(const void* x, const float* w, const float* bias, void* y, const dd_conv_desc* d, int dtype,
                             int act, void* workspace, size_t ws_bytes, void* stream) {
  DD_REQUIRE(desc_ok(d), DD_ERR_BAD_ARG, "dd_conv2d_fwd: bad descriptor");
  if (d->B == 0) return 0;
  DD_REQUIRE(x && w && y && workspace, DD_ERR_BAD_ARG, "dd_conv2d_fwd: null pointer");
  DD_REQUIRE(ws_bytes >= wg_bytes(d), DD_ERR_WORKSPACE, "dd_conv2d_fwd: workspace %zu < %zu", ws_bytes, wg_bytes(d));
  DD_REQUIRE(act >= 0 && act <= 2, DD_ERR_BAD_ARG, "dd_conv2d_fwd: act %d", act);
  cudaStream_t st = dd::as_stream(stream);
  const TcPlan p = tc_plan(d, dtype, 0, act);
  if (p.ok) {
    if (p.padded())
      DD_REQUIRE(ws_bytes >= dd_conv2d_workspace_bytes(d), DD_ERR_WORKSPACE, "dd_conv2d_fwd: workspace %zu < %zu", ws_bytes,
                 dd_conv2d_workspace_bytes(d));
    uint8_t* pad = p.padded() ? (uint8_t*)workspace + core_ws_bytes(d) : nullptr;
    const void* xin = x;
    if (p.K != p.Kreal) {
      if (int e = pad32(x, pad + p.x_pad, (long long)d->B * d->Hi * d->Wi, d->Cin, st)) return e;
      xin = pad + p.x_pad;
    }
    void* yt = p.N != p.Nreal ? (void*)pad : y;          // 8 produced channels: 16-channel pixels first, narrowed below
    const float* bptr = bias;
    if (p.N != p.Nreal && bias) {
      bias_pad_kernel<<<1, 32, 0, st>>>(bias, (float*)(pad + p.bias_pad), d->Cout, p.N);
      if (int e = dd::check_launch("conv2d_bias_pad")) return e;
      bptr = (const float*)(pad + p.bias_pad);
    }
    if (int e = dd::conv_dil_tc(xin, w, p.sn, p.sk, p.flip, bptr, nullptr, yt, workspace, d->B, d->Hi, d->Wi, d->Ho, d->Wo, p.K, p.N,
                                d->kh, d->dh, p.sign, p.off, act == 1, st, p.Kreal, p.Nreal))
      return e;
    if (p.N == p.Nreal) return 0;
    const long long np_out = (long long)d->B * d->Ho * d->Wo, want = (np_out + 255) / 256;
    chan_unpad16to8_kernel<<<(int)(want < dd::kSMs * 16 ? want : dd::kSMs * 16), 256, 0, st>>>((const __nv_bfloat16*)yt, (__nv_bfloat16*)y, np_out);
    return dd::check_launch("conv2d_chan_unpad");
  }
  float* wg = (float*)workspace;
  const int taps = d->kh * d->kw;
  // conv weights are [Cout][Cin][t] (need wg[t][ci][co] = w[co][ci][t]: swap); convT weights are [Cin][Cout][t]
  wprep_kernel<<<64, 256, 0, st>>>(w, wg, d->Cin, d->Cout, taps, d->transposed ? 0 : 1);
  if (int e = dd::check_launch("conv2d_wprep")) return e;
  Geo g{d->B, d->Cin, d->Cout, d->Hi, d->Wi, d->Ho, d->Wo, d->kh, d->kw, d->sh, d->sw, d->ph, d->pw, d->dh, d->dw, d->transposed};
  if (dtype == DD_F32) return launch_gather<float>((const float*)x, wg, bias, nullptr, (float*)y, g, act, st);
  if (dtype == DD_BF16)
    return launch_gather<__nv_bfloat16>((const __nv_bfloat16*)x, wg, bias, nullptr, (__nv_bfloat16*)y, g, act, st);
  return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv2d_fwd: dtype %d", dtype);
}

extern "C" int dd_conv2d_dgrad(const void* dy, const float* w, const void* x_mask, void* dx, const dd_conv_desc* d, int dtype,
                               void* workspace, size_t ws_bytes, void* stream) {
  DD_REQUIRE(desc_ok(d), DD_ERR_BAD_ARG, "dd_conv2d_dgrad: bad descriptor");
  if (d->B == 0) return 0;
  DD_REQUIRE(dy && w && dx && workspace, DD_ERR_BAD_ARG, "dd_conv2d_dgrad: null pointer");
  DD_REQUIRE(ws_bytes >= wg_bytes(d), DD_ERR_WORKSPACE, "dd_conv2d_dgrad: workspace %zu < %zu", ws_bytes, wg_bytes(d));
  cudaStream_t st = dd::as_stream(stream);
  const TcPlan p = tc_plan(d, dtype, 1, 0);
  if (p.ok) {
    const void* dyin = dy;
    if (p.K != p.Kreal) {
      DD_REQUIRE(ws_bytes >= dd_conv2d_workspace_bytes(d), DD_ERR_WORKSPACE, "dd_conv2d_dgrad: workspace %zu < %zu", ws_bytes,
                 dd_conv2d_workspace_bytes(d));
      uint8_t* dyp = (uint8_t*)workspace + core_ws_bytes(d);
      if (int e = pad32(dy, dyp, (long long)d->B * d->Ho * d->Wo, d->Cout, st)) return e;
      dyin = dyp;
    }
    return dd::conv_dil_tc(dyin, w, p.sn, p.sk, p.flip, nullptr, x_mask, dx, workspace, d->B, d->Ho, d->Wo, d->Hi, d->Wi, p.K, p.N,
                           d->kh, d->dh, p.sign, p.off, 0, st, p.Kreal, p.Nreal);
  }
  float* wg = (float*)workspace;
  const int taps = d->kh * d->kw;
  // gathered tensor = dy (Cout channels), produced = dx (Cin channels): wg[t][co][ci]
  wprep_kernel<<<64, 256, 0, st>>>(w, wg, d->Cout, d->Cin, taps, d->transposed ? 1 : 0);
  if (int e = dd::check_launch("conv2d_wprep")) return e;
  Geo g{d->B, d->Cout, d->Cin, d->Ho, d->Wo, d->Hi, d->Wi, d->kh, d->kw, d->sh, d->sw, d->ph, d->pw, d->dh, d->dw, !d->transposed};
  if (dtype == DD_F32) return launch_gather<float>((const float*)dy, wg, nullptr, (const float*)x_mask, (float*)dx, g, 0, st);
  if (dtype == DD_BF16)
    return launch_gather<__nv_bfloat16>((const __nv_bfloat16*)dy, wg, nullptr, (const __nv_bfloat16*)x_mask, (__nv_bfloat16*)dx, g, 0, st);
  return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv2d_dgrad: dtype %d", dtype);
}

extern "C" int dd_conv2d_wgrad(const void* x, const void* dy, float* dw, float* db, const dd_conv_desc* d, int dtype,
                               void* workspace, size_t ws_bytes, void* stream) {
  DD_REQUIRE(desc_ok(d), DD_ERR_BAD_ARG, "dd_conv2d_wgrad: bad descriptor");
  DD_REQUIRE(d->B > 0, DD_ERR_BAD_ARG, "dd_conv2d_wgrad: empty batch");
  DD_REQUIRE(x && dy && dw && workspace, DD_ERR_BAD_ARG, "dd_conv2d_wgrad: null pointer");
  DD_REQUIRE(ws_bytes >= dd_conv2d_workspace_bytes(d), DD_ERR_WORKSPACE, "dd_conv2d_wgrad: workspace %zu < %zu", ws_bytes,
             dd_conv2d_workspace_bytes(d));
  DD_REQUIRE(d->Cout <= 256, DD_ERR_UNSUPPORTED, "dd_conv2d_wgrad: Cout %d > 256", d->Cout);
  cudaStream_t st = dd::as_stream(stream);
  const int taps = d->kh * d->kw;
  const long long np_out = (long long)d->B * d->Ho * d->Wo, np_in = (long long)d->B * d->Hi * d->Wi;
  const TcPlan p = tc_plan(d, dtype, 2, 0);
  void* chan;                                                // the bias gradient's per-CTA sums, behind the partials
  if (p.ok) {
    const size_t tcb = dd::conv_dil_wgrad_tc_ws_bytes(p.K, p.N, d->kh);
    uint8_t* pad = (uint8_t*)workspace + core_ws_bytes(d);
    const void *xin = x, *dout = dy;
    if (p.N != p.Nreal) {
      if (int e = pad32(dy, pad, np_out, d->Cout, st)) return e;
      dout = pad;
    }
    if (p.K != p.Kreal) {
      if (int e = pad32(x, pad + p.x_pad, np_in, d->Cin, st)) return e;
      xin = pad + p.x_pad;
    }
    if (int e = dd::conv_dil_wgrad_tc(xin, dout, dw, p.sn, p.sk, workspace, tcb, d->B, d->Hi, d->Wi, d->Ho, d->Wo, p.K, p.N, d->kh,
                                      d->dh, p.sign, p.off, st, p.Kreal, p.Nreal))
      return e;
    chan = (uint8_t*)workspace + tcb;
  } else {
    const long long pivot = d->transposed ? np_in : np_out;
    const int splits = wgrad_splits(d, pivot);
    WGeo g;
    g.B = d->B;
    g.kh = d->kh; g.kw = d->kw; g.sh = d->sh; g.sw = d->sw; g.ph = d->ph; g.pw = d->pw; g.dh = d->dh; g.dw = d->dw;
    g.pix_per_split = ((pivot + splits - 1) / splits + 31) / 32 * 32;
    const void *Pp, *Qp;
    if (!d->transposed) { g.cP = d->Cout; g.cQ = d->Cin; g.Hp = d->Ho; g.Wp = d->Wo; g.Hq = d->Hi; g.Wq = d->Wi; Pp = dy; Qp = x; }
    else { g.cP = d->Cin; g.cQ = d->Cout; g.Hp = d->Hi; g.Wp = d->Wi; g.Hq = d->Ho; g.Wq = d->Wo; Pp = x; Qp = dy; }
    float* partial = (float*)workspace;
    int slots;
    if (dtype != DD_F32 && dtype != DD_BF16) return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv2d_wgrad: dtype %d", dtype);
    const int e = dtype == DD_F32
                      ? launch_wgrad_cc<float>((const float*)Pp, (const float*)Qp, partial, g, taps, splits, slots, st)
                      : launch_wgrad_cc<__nv_bfloat16>((const __nv_bfloat16*)Pp, (const __nv_bfloat16*)Qp, partial, g, taps, splits, slots, st);
    if (e) return e;
    const int n = taps * d->Cin * d->Cout;
    wgrad_fold_kernel<<<(n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184, 256, 0, st>>>(partial, dw, taps, d->Cin * d->Cout, slots);
    if (int e2 = dd::check_launch("conv2d_wgrad_fold")) return e2;
    chan = partial + (size_t)slots * n;
  }
  if (!db) return 0;
  double* cpart = reinterpret_cast<double*>(((uintptr_t)chan + 7) & ~(uintptr_t)7);
  const int lanes = 256 / d->Cout > 0 ? 256 / d->Cout : 1;
  const long long want = (np_out + lanes - 1) / lanes;
  const int nblk = (int)(want < kChanBlocks ? want : kChanBlocks);
  if (dtype == DD_F32) chansum_kernel<float><<<nblk, 256, 0, st>>>((const float*)dy, np_out, d->Cout, cpart);
  else chansum_kernel<__nv_bfloat16><<<nblk, 256, 0, st>>>((const __nv_bfloat16*)dy, np_out, d->Cout, cpart);
  if (int e = dd::check_launch("conv2d_chansum")) return e;
  chansum_fold_kernel<<<(d->Cout + 255) / 256, 256, 0, st>>>(cpart, nblk, d->Cout, db);
  return dd::check_launch("conv2d_chansum_fold");
}

// ================================================================================================
// Data movement around the bounding-box CNNs (spatial_bb/components.py:34-73,156) and the prob-space
// loss of spatial_w_rm.py:128-131.
// ================================================================================================
namespace {

// one camera of each scene as an NHWC image, with the rot90 / flip of SpatialMappingCNN.forward folded
// into the indexing.  mode 0: as is; 1: rot90(k=1,[2,3]) out[i,j] = x[j, W-1-i]; 2: rot90(k=1,[3,2])
// out[i,j] = x[H-1-j, i]; 3: flip([2,3]) out[i,j] = x[H-1-i, W-1-j].  views fp32 [B,6,3,H,W].
template <typename T>
__global__ void view_extract_kernel(const float* __restrict__ views, T* __restrict__ out, int B, int H, int W, int view,
                                    int mode, int Ho, int Wo) {
  const long long total = (long long)B * Ho * Wo * 3;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % 3);
    const int j = (int)((idx / 3) % Wo);
    const int i = (int)((idx / (3LL * Wo)) % Ho);
    const long long b = idx / (3LL * Wo * Ho);
    int h, w;
    if (mode == 0) { h = i; w = j; }
    else if (mode == 1) { h = j; w = W - 1 - i; }
    else if (mode == 2) { h = H - 1 - j; w = i; }
    else { h = H - 1 - i; w = W - 1 - j; }
    dd::st<T>(out + idx, __ldg(views + (((b * 6 + view) * 3 + c) * H + h) * (size_t)W + w));
  }
}

// backward of view_extract_kernel: thread = element of view `view` of the views gradient (each written once; the other
// five views are not touched); it reads the extracted image's gradient at the transformed position
template <typename T>
__global__ void view_extract_bwd_kernel(const T* __restrict__ dout, float* __restrict__ dviews, int B, int H, int W,
                                        int view, int mode, int Ho, int Wo) {
  const long long total = (long long)B * 3 * H * W;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int w = (int)(idx % W);
    const int h = (int)((idx / W) % H);
    const int c = (int)((idx / ((long long)W * H)) % 3);
    const long long b = idx / (3LL * W * H);
    int i, j;
    if (mode == 0) { i = h; j = w; }
    else if (mode == 1) { i = W - 1 - w; j = h; }
    else if (mode == 2) { i = w; j = H - 1 - h; }
    else { i = H - 1 - h; j = W - 1 - w; }
    dviews[(((b * 6 + view) * 3 + c) * H + h) * (size_t)W + w] = dd::ld<T>(dout + ((b * Ho + i) * Wo + j) * 3 + c);
  }
}

// dir 0: big[b, oy+i, ox+j, oc+k] = small[b,i,j,k];  dir 1: small[b,i,j,k] = big[b, oy+i, ox+j, oc+k]
template <typename T>
__global__ void nhwc_place_kernel(T* __restrict__ small_, T* __restrict__ big, int B, int h, int w, int c, int H, int W,
                                  int C, int oy, int ox, int oc, int dir) {
  const long long total = (long long)B * h * w * c;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx % c);
    const int j = (int)((idx / c) % w);
    const int i = (int)((idx / ((long long)c * w)) % h);
    const long long b = idx / ((long long)c * w * h);
    const size_t o = (((size_t)b * H + oy + i) * W + ox + j) * C + oc + k;
    if (dir == 0) big[o] = small_[idx];
    else small_[idx] = big[o];
  }
}

// dpre = dy * (1 - y) * y   (torch's sigmoid backward)
template <typename T>
__global__ void sigmoid_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ y, T* __restrict__ out, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float yy = dd::ld<T>(y + i);
    dd::st<T>(out + i, dd::ld<T>(dy + i) * (1.0f - yy) * yy);
  }
}

// F.binary_cross_entropy(p, t) (spatial_w_rm.py:131): -(t * max(log p, -100) + (1-t) * max(log(1-p), -100)), mean
struct BceProbWs {
  double partial[dd::kSMs * 4];
  unsigned int ticket, pad[3];
};
__global__ void __launch_bounds__(256) bce_prob_kernel(const float* __restrict__ p, const float* __restrict__ t,
                                                       float* __restrict__ loss, BceProbWs* __restrict__ ws, long long n) {
  float s = 0.f;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float pv = p[i], tv = t[i];
    s -= tv * fmaxf(logf(pv), -100.f) + (1.0f - tv) * fmaxf(log1pf(-pv), -100.f);
  }
  __shared__ double red[8];
  double v = dd::warp_sum((double)s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int k = 0; k < 8; ++k) tot += red[k];
    ws->partial[blockIdx.x] = tot;
    __threadfence();
    last = atomicAdd(&ws->ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last || threadIdx.x != 0) return;
  __threadfence();
  double tot = 0.0;
  for (unsigned int k = 0; k < gridDim.x; ++k) tot += __ldcg(&ws->partial[k]);
  loss[0] = (float)(tot / (double)n);
  ws->ticket = 0;
}
// dp = g * (p - t) / max((1 - p) * p, 1e-12) / n   (aten's binary_cross_entropy_backward, mean reduction)
__global__ void bce_prob_bwd_kernel(const float* __restrict__ p, const float* __restrict__ t, const float* __restrict__ g,
                                    float* __restrict__ dp, long long n) {
  const float go = g ? __ldg(g) : 1.0f;
  const float fn = (float)n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float pv = p[i];
    dp[i] = __fdiv_rn(__fdiv_rn(go * (pv - t[i]), fmaxf((1.0f - pv) * pv, 1e-12f)), fn);
  }
}

int grid_elems(long long total) {
  long long g = (total + 255) / 256;
  return (int)(g < 1 ? 1 : (g < dd::kSMs * 16 ? g : dd::kSMs * 16));
}
}  // namespace

extern "C" int dd_view_extract(const float* views, void* out, int out_dtype, int B, int H, int W, int view, int mode,
                               void* stream) {
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_view_extract: bad shape");
  DD_REQUIRE(view >= 0 && view < 6 && mode >= 0 && mode <= 3, DD_ERR_BAD_ARG, "dd_view_extract: view %d mode %d", view, mode);
  if (B == 0) return 0;
  DD_REQUIRE(views && out, DD_ERR_BAD_ARG, "dd_view_extract: null pointer");
  const bool rot = mode == 1 || mode == 2;
  const int Ho = rot ? W : H, Wo = rot ? H : W;
  const long long total = (long long)B * Ho * Wo * 3;
  cudaStream_t st = dd::as_stream(stream);
  if (out_dtype == DD_F32) view_extract_kernel<float><<<grid_elems(total), 256, 0, st>>>(views, (float*)out, B, H, W, view, mode, Ho, Wo);
  else if (out_dtype == DD_BF16)
    view_extract_kernel<__nv_bfloat16><<<grid_elems(total), 256, 0, st>>>(views, (__nv_bfloat16*)out, B, H, W, view, mode, Ho, Wo);
  else return dd::fail(DD_ERR_UNSUPPORTED, "dd_view_extract: dtype %d", out_dtype);
  return dd::check_launch("view_extract");
}

extern "C" int dd_view_extract_bwd(const void* dout, int dtype, float* dviews, int B, int H, int W, int view, int mode,
                                   void* stream) {
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_view_extract_bwd: bad shape");
  DD_REQUIRE(view >= 0 && view < 6 && mode >= 0 && mode <= 3, DD_ERR_BAD_ARG, "dd_view_extract_bwd: view %d mode %d", view, mode);
  if (B == 0) return 0;
  DD_REQUIRE(dout && dviews, DD_ERR_BAD_ARG, "dd_view_extract_bwd: null pointer");
  const bool rot = mode == 1 || mode == 2;
  const int Ho = rot ? W : H, Wo = rot ? H : W;
  const long long total = (long long)B * 3 * H * W;
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_F32)
    view_extract_bwd_kernel<float><<<grid_elems(total), 256, 0, st>>>((const float*)dout, dviews, B, H, W, view, mode, Ho, Wo);
  else if (dtype == DD_BF16)
    view_extract_bwd_kernel<__nv_bfloat16><<<grid_elems(total), 256, 0, st>>>((const __nv_bfloat16*)dout, dviews, B, H, W, view,
                                                                                mode, Ho, Wo);
  else return dd::fail(DD_ERR_UNSUPPORTED, "dd_view_extract_bwd: dtype %d", dtype);
  return dd::check_launch("view_extract_bwd");
}

extern "C" int dd_nhwc_place(void* small_, void* big, int dtype, int B, int h, int w, int c, int H, int W, int C, int oy,
                             int ox, int oc, int dir, void* stream) {
  DD_REQUIRE(B >= 0 && h > 0 && w > 0 && c > 0, DD_ERR_BAD_ARG, "dd_nhwc_place: bad shape");
  DD_REQUIRE(oy >= 0 && ox >= 0 && oc >= 0 && oy + h <= H && ox + w <= W && oc + c <= C, DD_ERR_BAD_ARG,
             "dd_nhwc_place: window [%d+%d, %d+%d, %d+%d] outside [%d,%d,%d]", oy, h, ox, w, oc, c, H, W, C);
  if (B == 0) return 0;
  DD_REQUIRE(small_ && big, DD_ERR_BAD_ARG, "dd_nhwc_place: null pointer");
  const long long total = (long long)B * h * w * c;
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_F32) nhwc_place_kernel<float><<<grid_elems(total), 256, 0, st>>>((float*)small_, (float*)big, B, h, w, c, H, W, C, oy, ox, oc, dir);
  else if (dtype == DD_BF16)
    nhwc_place_kernel<__nv_bfloat16><<<grid_elems(total), 256, 0, st>>>((__nv_bfloat16*)small_, (__nv_bfloat16*)big, B, h, w, c, H, W, C, oy, ox, oc, dir);
  else return dd::fail(DD_ERR_UNSUPPORTED, "dd_nhwc_place: dtype %d", dtype);
  return dd::check_launch("nhwc_place");
}

extern "C" int dd_sigmoid_bwd(const void* dy, const void* y, void* out, int dtype, long long n, void* stream) {
  DD_REQUIRE(n >= 0, DD_ERR_BAD_ARG, "dd_sigmoid_bwd: n=%lld", n);
  if (n == 0) return 0;
  DD_REQUIRE(dy && y && out, DD_ERR_BAD_ARG, "dd_sigmoid_bwd: null pointer");
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_F32) sigmoid_bwd_kernel<float><<<grid_elems(n), 256, 0, st>>>((const float*)dy, (const float*)y, (float*)out, n);
  else if (dtype == DD_BF16)
    sigmoid_bwd_kernel<__nv_bfloat16><<<grid_elems(n), 256, 0, st>>>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)y, (__nv_bfloat16*)out, n);
  else return dd::fail(DD_ERR_UNSUPPORTED, "dd_sigmoid_bwd: dtype %d", dtype);
  return dd::check_launch("sigmoid_bwd");
}

extern "C" size_t dd_bce_prob_workspace_bytes(void) { return sizeof(BceProbWs); }

extern "C" int dd_bce_prob_fwd(const float* probs, const float* target, float* loss, void* workspace, size_t ws_bytes,
                               long long n, void* stream) {
  DD_REQUIRE(probs && target && loss && workspace, DD_ERR_BAD_ARG, "dd_bce_prob_fwd: null pointer");
  DD_REQUIRE(n > 0, DD_ERR_BAD_ARG, "dd_bce_prob_fwd: n=%lld", n);
  DD_REQUIRE(ws_bytes >= sizeof(BceProbWs), DD_ERR_WORKSPACE, "dd_bce_prob_fwd: workspace too small");
  long long want = (n + 1023) / 1024;
  const int grid = (int)(want < dd::kSMs * 4 ? want : dd::kSMs * 4);
  bce_prob_kernel<<<grid, 256, 0, dd::as_stream(stream)>>>(probs, target, loss, (BceProbWs*)workspace, n);
  return dd::check_launch("bce_prob_fwd");
}

extern "C" int dd_bce_prob_bwd(const float* probs, const float* target, const float* grad_out, float* dprobs, long long n,
                               void* stream) {
  DD_REQUIRE(probs && target && dprobs, DD_ERR_BAD_ARG, "dd_bce_prob_bwd: null pointer");
  DD_REQUIRE(n > 0, DD_ERR_BAD_ARG, "dd_bce_prob_bwd: n=%lld", n);
  bce_prob_bwd_kernel<<<grid_elems(n), 256, 0, dd::as_stream(stream)>>>(probs, target, grad_out, dprobs, n);
  return dd::check_launch("bce_prob_bwd");
}
