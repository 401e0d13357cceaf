// Encoder convolutions on the CUDA cores (fp32 accumulate, fp32 or bf16 storage).
//
// This is the fp32 parity path (1e-5 contract against the reference's fp32 torch convs,
// components.py:19-21,41-43) and the reference implementation the tcgen05 kernels in
// conv_tc.cu are checked against on the device.  Layout: activations NHWC [B][H][W][32].
//
//   c1   : 3->32 3x3 pad 1 from NCHW fp32 input (views with the stitch folded in, or a mosaic)
//   c2/c3: 32->32 3x3 pad 1 stride 1/2, bias+ReLU epilogue
//   dgrad: stride 1 = same kernel with the flipped/transposed filter and a (x>0) mask epilogue;
//          stride 2 = gather form over parity classes
//   wgrad: per-CTA [tap][ci][co] partials over a persistent pixel-tile loop, then an ordered
//          reduction kernel (deterministic; no atomics)
#include "dd_common.cuh"

namespace {

constexpr int C = 32;        // channels of every encoder activation
constexpr int PADC = 33;     // smem pixel stride in floats (bank-conflict-free across pixels)

// ------------------------------------------------------------------------------------------
// cooperative tile load: NHWC global -> smem [pix][PADC] fp32, zero outside the image
// ------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void load_tile_nhwc(const T* __restrict__ img, int H, int W, int h_base,
                                               int w_base, int th, int tw, float* __restrict__ s,
                                               int tid, int nthreads) {
  const int chunks = th * tw * 4;  // 8-channel chunks
  for (int i = tid; i < chunks; i += nthreads) {
    const int cg = i & 3;
    const int pix = i >> 2;
    const int r = pix / tw, c = pix - r * tw;
    const int h = h_base + r, w = w_base + c;
    float v[8];
    if (h >= 0 && h < H && w >= 0 && w < W) {
      dd::ld8<T>(img + ((size_t)h * W + w) * C + cg * 8, v);
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = 0.f;
    }
    float* d = s + pix * PADC + cg * 8;
#pragma unroll
    for (int k = 0; k < 8; ++k) d[k] = v[k];
  }
}

// acc[0..31] += xv * w[0..31]   (w: 32 consecutive floats in smem, 16-byte aligned, broadcast)
__device__ __forceinline__ void fma_row32(float (&acc)[C], float xv, const float* __restrict__ w) {
  const float4* w4 = reinterpret_cast<const float4*>(w);
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 ww = w4[q];
    acc[4 * q + 0] = fmaf(xv, ww.x, acc[4 * q + 0]);
    acc[4 * q + 1] = fmaf(xv, ww.y, acc[4 * q + 1]);
    acc[4 * q + 2] = fmaf(xv, ww.z, acc[4 * q + 2]);
    acc[4 * q + 3] = fmaf(xv, ww.w, acc[4 * q + 3]);
  }
}

template <typename T>
__device__ __forceinline__ void store_pixel32(T* __restrict__ p, const float (&acc)[C]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = acc[g * 8 + k];
    dd::st8<T>(p + g * 8, v);
  }
}

// ------------------------------------------------------------------------------------------
// 32->32 3x3 conv, pad 1.  MODE 0: forward (bias + ReLU).  MODE 1: stride-1 dgrad (flipped,
// transposed filter; epilogue multiplies by mask_act > 0 when mask_act != nullptr).
// CTA = TH x TW output pixels, one thread per pixel, 32 accumulators per thread.
// ------------------------------------------------------------------------------------------
template <typename T, int STRIDE, int MODE, int TH, int TW>
__global__ void __launch_bounds__(TH * TW) conv3x3_c32_simt(const T* __restrict__ in,
                                                            const float* __restrict__ w_oihw,
                                                            const float* __restrict__ bias,
                                                            const T* __restrict__ mask_act,
                                                            T* __restrict__ out, int H, int W, int Ho,
                                                            int Wo) {
  constexpr int NT = TH * TW;
  constexpr int IH = (TH - 1) * STRIDE + 3, IW = (TW - 1) * STRIDE + 3;
  extern __shared__ __align__(16) float smem[];
  float* s_w = smem;                 // [9][32 in][32 out]
  float* s_in = smem + 9 * C * C;    // [IH*IW][PADC]
  const int tid = threadIdx.x;
  const int b = blockIdx.z;
  const int ho0 = blockIdx.y * TH, wo0 = blockIdx.x * TW;

  for (int i = tid; i < 9 * C * C; i += NT) {
    const int o = i & 31, ii = (i >> 5) & 31, tap = i >> 10;
    float v;
    if (MODE == 0) v = w_oihw[(o * C + ii) * 9 + tap];            // W[co=o][ci=ii][tap]
    else v = w_oihw[(ii * C + o) * 9 + (8 - tap)];                // W[co=ii][ci=o][flipped tap]
    s_w[i] = v;
  }
  load_tile_nhwc<T>(in + (size_t)b * H * W * C, H, W, ho0 * STRIDE - 1, wo0 * STRIDE - 1, IH, IW, s_in, tid, NT);
  __syncthreads();

  const int py = tid / TW, px = tid - py * TW;
  float acc[C];
#pragma unroll
  for (int k = 0; k < C; ++k) acc[k] = (MODE == 0) ? __ldg(bias + k) : 0.f;

#pragma unroll 1
  for (int tap = 0; tap < 9; ++tap) {
    const int kh = tap / 3, kw = tap - kh * 3;
    const float* xin = s_in + ((py * STRIDE + kh) * IW + px * STRIDE + kw) * PADC;
    const float* wt = s_w + tap * C * C;
#pragma unroll 4
    for (int ci = 0; ci < C; ++ci) fma_row32(acc, xin[ci], wt + ci * C);
  }

  const int ho = ho0 + py, wo = wo0 + px;
  if (ho < Ho && wo < Wo) {
    const size_t off = (((size_t)b * Ho + ho) * Wo + wo) * C;
    if (MODE == 0) {
#pragma unroll
      for (int k = 0; k < C; ++k) acc[k] = fmaxf(acc[k], 0.f);
    } else if (mask_act) {
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float m[8];
        dd::ld8<T>(mask_act + off + g * 8, m);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[g * 8 + k] = m[k] > 0.f ? acc[g * 8 + k] : 0.f;
      }
    }
    store_pixel32<T>(out + off, acc);
  }
}

// ------------------------------------------------------------------------------------------
// stride-2 dgrad: dx[h,w,ci] = sum_{kh,kw,co} dy[(h+1-kh)/2,(w+1-kw)/2,co] W[co,ci,kh,kw] over the
// taps whose numerators are even and in range.  CTA = 8 rows x 64 cols of dx; a thread owns the
// horizontal pair (w even, w+1 odd) so that every lane of a warp runs the same taps.
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) conv3x3_c32_dgrad_s2_simt(const T* __restrict__ dy,
                                                                 const float* __restrict__ w_oihw,
                                                                 const T* __restrict__ mask_act,
                                                                 T* __restrict__ dx, int H, int W, int Ho,
                                                                 int Wo) {
  constexpr int TH = 8, TWP = 32;          // 32 pairs = 64 columns
  constexpr int DH = TH / 2 + 1, DW = TWP + 1;
  extern __shared__ __align__(16) float smem[];
  float* s_w = smem;                       // [9][32 co][32 ci]
  float* s_dy = smem + 9 * C * C;          // [DH*DW][PADC]
  const int tid = threadIdx.x;
  const int b = blockIdx.z;
  const int h0 = blockIdx.y * TH, w0 = blockIdx.x * (2 * TWP);

  for (int i = tid; i < 9 * C * C; i += 256) {
    const int ci = i & 31, co = (i >> 5) & 31, tap = i >> 10;
    s_w[i] = w_oihw[(co * C + ci) * 9 + tap];
  }
  // dy rows h0/2 .. h0/2+4, cols w0/2 .. w0/2+32
  load_tile_nhwc<T>(dy + (size_t)b * Ho * Wo * C, Ho, Wo, h0 / 2, w0 / 2, DH, DW, s_dy, tid, 256);
  __syncthreads();

  const int r = tid >> 5, j = tid & 31;
  const int h = h0 + r, we = w0 + 2 * j;   // even column; odd column is we+1
  float acc_e[C], acc_o[C];
#pragma unroll
  for (int k = 0; k < C; ++k) { acc_e[k] = 0.f; acc_o[k] = 0.f; }

#pragma unroll 1
  for (int kh = 0; kh < 3; ++kh) {
    if (((h + 1 - kh) & 1) != 0) continue;           // warp-uniform (h is per warp)
    const int dr = ((h + 1 - kh) >> 1) - h0 / 2;     // row inside the dy tile (0..4)
    // even column we: kw = 1 -> dy col we/2 ; odd column we+1: kw = 0 -> (we+2)/2, kw = 2 -> we/2
    const float* d0 = s_dy + (dr * DW + j) * PADC;        // dy col we/2
    const float* d1 = s_dy + (dr * DW + j + 1) * PADC;    // dy col we/2 + 1
    const float* w_k0 = s_w + (kh * 3 + 0) * C * C;
    const float* w_k1 = s_w + (kh * 3 + 1) * C * C;
    const float* w_k2 = s_w + (kh * 3 + 2) * C * C;
#pragma unroll 2
    for (int co = 0; co < C; ++co) {
      const float a = d0[co], bq = d1[co];
      fma_row32(acc_e, a, w_k1 + co * C);
      fma_row32(acc_o, bq, w_k0 + co * C);
      fma_row32(acc_o, a, w_k2 + co * C);
    }
  }
  if (h < H) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int w = we + half;
      if (w >= W) continue;
      float (&acc)[C] = half ? acc_o : acc_e;
      const size_t off = (((size_t)b * H + h) * W + w) * C;
      if (mask_act) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float m[8];
          dd::ld8<T>(mask_act + off + g * 8, m);
#pragma unroll
          for (int k = 0; k < 8; ++k) acc[g * 8 + k] = m[k] > 0.f ? acc[g * 8 + k] : 0.f;
        }
      }
      store_pixel32<T>(dx + off, acc);
    }
  }
}

// ------------------------------------------------------------------------------------------
// wgrad: dW[co][ci][tap] = sum_pix x[pix*S + tap - 1][ci] * dy[pix][co];  db[co] = sum dy.
// CTA = 288 threads (warp = tap, lane = ci), 32 co accumulators per thread, persistent loop over
// TH x TW tiles of dy; partial[blk][tap][ci][co] (+ db) to the workspace, then reduce kernel.
// ------------------------------------------------------------------------------------------
template <typename T, int STRIDE, int TH, int TW>
__global__ void __launch_bounds__(288) conv3x3_c32_wgrad_simt(const T* __restrict__ x,
                                                              const T* __restrict__ dy,
                                                              float* __restrict__ partial, int B, int H,
                                                              int W, int Ho, int Wo) {
  constexpr int IH = (TH - 1) * STRIDE + 3, IW = (TW - 1) * STRIDE + 3;
  extern __shared__ __align__(16) float smem[];
  float* s_dy = smem;                       // [TH*TW][32] (broadcast reads, no padding needed)
  float* s_x = smem + TH * TW * C;          // [IH*IW][PADC]
  const int tid = threadIdx.x;
  const int tap = tid >> 5, ci = tid & 31;
  const int kh = tap / 3, kw = tap - kh * 3;
  const int tiles_x = (Wo + TW - 1) / TW, tiles_y = (Ho + TH - 1) / TH;
  const int tiles = B * tiles_y * tiles_x;

  float acc[C], db = 0.f;
#pragma unroll
  for (int k = 0; k < C; ++k) acc[k] = 0.f;

  for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int tx = t % tiles_x, ty = (t / tiles_x) % tiles_y, b = t / (tiles_x * tiles_y);
    const int ho0 = ty * TH, wo0 = tx * TW;
    __syncthreads();  // previous tile fully consumed
    load_tile_nhwc<T>(x + (size_t)b * H * W * C, H, W, ho0 * STRIDE - 1, wo0 * STRIDE - 1, IH, IW, s_x, tid, 288);
    // dy tile, zero outside the image
    for (int i = tid; i < TH * TW * 4; i += 288) {
      const int cg = i & 3, pix = i >> 2;
      const int r = pix / TW, c = pix - r * TW;
      float v[8];
      if (ho0 + r < Ho && wo0 + c < Wo) {
        dd::ld8<T>(dy + ((((size_t)b * Ho + ho0 + r) * Wo + wo0 + c) * C) + cg * 8, v);
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = 0.f;
      }
      float4* d = reinterpret_cast<float4*>(s_dy + pix * C + cg * 8);
      d[0] = make_float4(v[0], v[1], v[2], v[3]);
      d[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    __syncthreads();
#pragma unroll 2
    for (int p = 0; p < TH * TW; ++p) {
      const int py = p / TW, px = p - py * TW;
      const float xv = s_x[((py * STRIDE + kh) * IW + px * STRIDE + kw) * PADC + ci];
      fma_row32(acc, xv, s_dy + p * C);
      if (tap == 0) db += s_dy[p * C + ci];   // warp 0: lane doubles as co for the bias grad
    }
  }
  float* out = partial + (size_t)blockIdx.x * (9 * C * C + C);
#pragma unroll
  for (int g = 0; g < 8; ++g)
    reinterpret_cast<float4*>(out + (tap * C + ci) * C)[g] =
        make_float4(acc[4 * g], acc[4 * g + 1], acc[4 * g + 2], acc[4 * g + 3]);
  if (tap == 0) out[9 * C * C + ci] = db;
}

// dw[co][ci][tap] (OIHW) = sum_blk partial[blk][tap][ci][co];  db[co] likewise.  K = 9*Cin.
__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, int nblk, int cin, float* __restrict__ dw,
                                    float* __restrict__ db) {
  const int K = 9 * cin;
  const int stride = K * C + C;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= stride) return;
  float s = 0.f;
  for (int blk = 0; blk < nblk; ++blk) s += partial[(size_t)blk * stride + i];
  if (i < K * C) {
    const int co = i & 31, k = i >> 5;        // k = tap*cin + ci
    const int ci = k % cin, tap = k / cin;
    dw[(co * cin + ci) * 9 + tap] = s;
  } else {
    db[i - K * C] = s;
  }
}

// ------------------------------------------------------------------------------------------
// c1: 3->32 from NCHW fp32.  IS_VIEWS folds the stitch (mosaic column wm -> view, column).
// ------------------------------------------------------------------------------------------
template <bool IS_VIEWS>
__device__ __forceinline__ float c1_input(const float* __restrict__ in, int b, int c, int h, int wm, int H,
                                          int Wm) {
  if (h < 0 || h >= H || wm < 0 || wm >= Wm) return 0.f;
  if (IS_VIEWS) {
    const int W = Wm / 6;
    const int j = wm / W, w = wm - j * W;
    return __ldg(in + ((((size_t)b * 6 + dd::view_of_slot(j)) * 3 + c) * H + h) * W + w);
  }
  return __ldg(in + (((size_t)b * 3 + c) * H + h) * Wm + wm);
}

template <typename T, bool IS_VIEWS>
__global__ void __launch_bounds__(256) conv_c1_fwd_simt(const float* __restrict__ in,
                                                        const float* __restrict__ w_oihw,
                                                        const float* __restrict__ bias, T* __restrict__ out,
                                                        int H, int Wm) {
  constexpr int TH = 8, TW = 32, IH = TH + 2, IW = TW + 2;
  __shared__ __align__(16) float s_w[27 * C];      // [k = ci*9+tap][co]
  __shared__ float s_in[3 * IH * IW];
  const int tid = threadIdx.x, b = blockIdx.z;
  const int h0 = blockIdx.y * TH, w0 = blockIdx.x * TW;
  for (int i = tid; i < 27 * C; i += 256) {
    const int co = i & 31, k = i >> 5;
    s_w[i] = w_oihw[co * 27 + k];
  }
  for (int i = tid; i < 3 * IH * IW; i += 256) {
    const int c = i / (IH * IW), rem = i - c * IH * IW;
    const int r = rem / IW, cc = rem - r * IW;
    s_in[i] = c1_input<IS_VIEWS>(in, b, c, h0 + r - 1, w0 + cc - 1, H, Wm);
  }
  __syncthreads();
  const int py = tid / TW, px = tid - py * TW;
  float acc[C];
#pragma unroll
  for (int k = 0; k < C; ++k) acc[k] = __ldg(bias + k);
#pragma unroll
  for (int ci = 0; ci < 3; ++ci)
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int kh = tap / 3, kw = tap % 3;
      fma_row32(acc, s_in[(ci * IH + py + kh) * IW + px + kw], s_w + (ci * 9 + tap) * C);
    }
  const int h = h0 + py, w = w0 + px;
  if (h < H && w < Wm) {
#pragma unroll
    for (int k = 0; k < C; ++k) acc[k] = fmaxf(acc[k], 0.f);
    store_pixel32<T>(out + (((size_t)b * H + h) * Wm + w) * C, acc);
  }
}

// c1 input gradient on the CUDA cores (the fp32 parity path; bf16 with DD_IMPL_SIMT): thread = image pixel, reading the
// whole 32-channel da1 pixel of each of its 9 taps; fp32 dx stored into the NCHW mosaic or, IS_VIEWS, the views
// (mosaic column w of slot j = w / Wv lands in view dd::view_of_slot(j)).  Fixed summation order: kh, kw, o.
template <typename T, bool IS_VIEWS>
__global__ void __launch_bounds__(256) conv_c1_dgrad_simt(const T* __restrict__ dy, const float* __restrict__ w_oihw,
                                                          float* __restrict__ dx, int H, int Wm) {
  constexpr int TH = 8, TW = 32;
  __shared__ float s_w[9 * C * 3];                 // [tap][o][c]
  const int tid = threadIdx.x, b = blockIdx.z;
  for (int i = tid; i < 9 * C * 3; i += 256) {
    const int c = i % 3, o = (i / 3) % C, tap = i / (3 * C);
    s_w[i] = w_oihw[(o * 3 + c) * 9 + tap];
  }
  __syncthreads();
  const int h = blockIdx.y * TH + tid / TW, w = blockIdx.x * TW + tid % TW;
  if (h >= H || w >= Wm) return;
  float acc[3] = {0.f, 0.f, 0.f};
  for (int kh = 0; kh < 3; ++kh) {
    const int y = h + 1 - kh;
    if (y < 0 || y >= H) continue;
    for (int kw = 0; kw < 3; ++kw) {
      const int x = w + 1 - kw;
      if (x < 0 || x >= Wm) continue;
      const T* p = dy + (((size_t)b * H + y) * Wm + x) * C;
      const float* wt = s_w + (kh * 3 + kw) * C * 3;
#pragma unroll
      for (int g = 0; g < C / 8; ++g) {
        float v[8];
        dd::ld8<T>(p + 8 * g, v);
#pragma unroll
        for (int k = 0; k < 8; ++k)
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[c] = fmaf(v[k], wt[(8 * g + k) * 3 + c], acc[c]);
      }
    }
  }
  float* dst;
  size_t cs;
  if (IS_VIEWS) {
    const int Wv = Wm / 6, j = w / Wv;
    dst = dx + ((size_t)(6 * b + dd::view_of_slot(j)) * 3 * H + h) * Wv + (w - j * Wv);
    cs = (size_t)H * Wv;
  } else {
    dst = dx + ((size_t)3 * b * H + h) * Wm + w;
    cs = (size_t)H * Wm;
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) dst[c * cs] = acc[c];
}

// c1 wgrad: lane k<27 owns filter tap k = ci*9+tap for all 32 co; the 8 warps split the tile's
// pixels; CTA partial [27][32] + db[32] to the workspace (persistent tile loop).
template <typename T, bool IS_VIEWS>
__global__ void __launch_bounds__(256) conv_c1_wgrad_simt(const float* __restrict__ in,
                                                          const T* __restrict__ dy,
                                                          float* __restrict__ partial, int B, int H, int Wm) {
  constexpr int TH = 8, TW = 32, IH = TH + 2, IW = TW + 2;
  __shared__ __align__(16) float s_dy[TH * TW * C];
  __shared__ float s_in[3 * IH * IW];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int k = lane < 27 ? lane : 26;
  const int ci = k / 9, tap = k - ci * 9, kh = tap / 3, kw = tap - kh * 3;
  const int tiles_x = (Wm + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
  const int tiles = B * tiles_y * tiles_x;
  float acc[C], db = 0.f;
#pragma unroll
  for (int q = 0; q < C; ++q) acc[q] = 0.f;
  for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int tx = t % tiles_x, ty = (t / tiles_x) % tiles_y, b = t / (tiles_x * tiles_y);
    const int h0 = ty * TH, w0 = tx * TW;
    __syncthreads();
    for (int i = tid; i < 3 * IH * IW; i += 256) {
      const int c = i / (IH * IW), rem = i - c * IH * IW;
      const int r = rem / IW, cc = rem - r * IW;
      s_in[i] = c1_input<IS_VIEWS>(in, b, c, h0 + r - 1, w0 + cc - 1, H, Wm);
    }
    for (int i = tid; i < TH * TW * 4; i += 256) {
      const int cg = i & 3, pix = i >> 2;
      const int r = pix / TW, c = pix - r * TW;
      float v[8];
      if (h0 + r < H && w0 + c < Wm) {
        dd::ld8<T>(dy + ((((size_t)b * H + h0 + r) * Wm + w0 + c) * C) + cg * 8, v);
      } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = 0.f;
      }
      float4* d = reinterpret_cast<float4*>(s_dy + pix * C + cg * 8);
      d[0] = make_float4(v[0], v[1], v[2], v[3]);
      d[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    __syncthreads();
    for (int p = warp; p < TH * TW; p += 8) {
      const int py = p / TW, px = p - py * TW;
      fma_row32(acc, s_in[(ci * IH + py + kh) * IW + px + kw], s_dy + p * C);
      db += s_dy[p * C + lane];
    }
  }
  // fold the 8 warps through smem (reuse s_dy: 8 * (27*32+32) floats = 7168 <= 8192)
  __syncthreads();
  float* red = s_dy;
  if (lane < 27) {
#pragma unroll
    for (int q = 0; q < C; ++q) red[warp * 896 + lane * C + q] = acc[q];
  }
  red[warp * 896 + 864 + lane] = db;
  __syncthreads();
  float* out = partial + (size_t)blockIdx.x * 896;
  for (int i = tid; i < 896; i += 256) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w * 896 + i];
    out[i] = s;
  }
}

// c1 reduce: partial[blk][k=ci*9+tap][co] -> dw[co][ci][tap] = dw[co*27 + k]
__global__ void c1_wgrad_reduce_kernel(const float* __restrict__ partial, int nblk, float* __restrict__ dw,
                                       float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 896) return;
  float s = 0.f;
  for (int blk = 0; blk < nblk; ++blk) s += partial[(size_t)blk * 896 + i];
  if (i < 864) dw[(i & 31) * 27 + (i >> 5)] = s;
  else db[i - 864] = s;
}

template <typename T>
__global__ void relu_mask_kernel(const T* __restrict__ g, const T* __restrict__ act, T* __restrict__ out,
                                 long long n8, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float a[8], b[8];
    dd::ld8<T>(g + i * 8, a);
    dd::ld8<T>(act + i * 8, b);
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = b[k] > 0.f ? a[k] : 0.f;
    dd::st8<T>(out + i * 8, a);
  }
  // ragged tail (n % 8), first CTA
  if (blockIdx.x == 0)
    for (long long i = n8 * 8 + threadIdx.x; i < n; i += blockDim.x)
      dd::st<T>(out + i, dd::ld<T>(act + i) > 0.f ? dd::ld<T>(g + i) : 0.f);
}

constexpr int kWgradBlocks = dd::kSMs * 2;
constexpr size_t kWgradWsBytes = (size_t)12 << 20;   // >= SIMT partials (296 x 9248 floats) and tcgen05 partials (148 x 18432 + 592 x 32)

template <typename T>
int conv_fwd_simt(const T* in, const float* w, const float* bias, T* out, int B, int H, int W, int stride,
                  cudaStream_t st) {
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  if (stride == 1) {
    constexpr int TH = 8, TW = 32;
    const size_t smem = (9 * C * C + (TH + 2) * (TW + 2) * PADC) * sizeof(float);
    auto k = conv3x3_c32_simt<T, 1, 0, TH, TW>;
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "conv3x3_c32_fwd_simt")) return e;
    k<<<dim3((Wo + TW - 1) / TW, (Ho + TH - 1) / TH, B), TH * TW, smem, st>>>(in, w, bias, nullptr, out, H, W, Ho, Wo);
  } else {
    constexpr int TH = 8, TW = 16;
    const size_t smem = (9 * C * C + (2 * TH + 1) * (2 * TW + 1) * PADC) * sizeof(float);
    auto k = conv3x3_c32_simt<T, 2, 0, TH, TW>;
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "conv3x3_c32_fwd_simt")) return e;
    k<<<dim3((Wo + TW - 1) / TW, (Ho + TH - 1) / TH, B), TH * TW, smem, st>>>(in, w, bias, nullptr, out, H, W, Ho, Wo);
  }
  return dd::check_launch("conv3x3_c32_fwd_simt");
}

template <typename T>
int conv_dgrad_simt(const T* dy, const float* w, const T* x, T* dx, int B, int H, int W, int stride,
                    cudaStream_t st) {
  if (stride == 1) {
    constexpr int TH = 8, TW = 32;
    const size_t smem = (9 * C * C + (TH + 2) * (TW + 2) * PADC) * sizeof(float);
    auto k = conv3x3_c32_simt<T, 1, 1, TH, TW>;
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "conv3x3_c32_dgrad_simt")) return e;
    k<<<dim3((W + TW - 1) / TW, (H + TH - 1) / TH, B), TH * TW, smem, st>>>(dy, w, nullptr, x, dx, H, W, H, W);
  } else {
    const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
    const size_t smem = (9 * C * C + 5 * 33 * PADC) * sizeof(float);
    auto k = conv3x3_c32_dgrad_s2_simt<T>;
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "conv3x3_c32_dgrad_simt")) return e;
    k<<<dim3((W + 63) / 64, (H + 7) / 8, B), 256, smem, st>>>(dy, w, x, dx, H, W, Ho, Wo);
  }
  return dd::check_launch("conv3x3_c32_dgrad_simt");
}

template <typename T>
int conv_wgrad_simt(const T* x, const T* dy, float* dw, float* db, float* ws, int B, int H, int W, int stride,
                    cudaStream_t st) {
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  int nblk;
  if (stride == 1) {
    constexpr int TH = 8, TW = 32;
    const int tiles = B * ((Ho + TH - 1) / TH) * ((Wo + TW - 1) / TW);
    nblk = tiles < kWgradBlocks ? tiles : kWgradBlocks;
    const size_t smem = (TH * TW * C + (TH + 2) * (TW + 2) * PADC) * sizeof(float);
    auto k = conv3x3_c32_wgrad_simt<T, 1, TH, TW>;
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "conv3x3_c32_wgrad_simt")) return e;
    k<<<nblk, 288, smem, st>>>(x, dy, ws, B, H, W, Ho, Wo);
  } else {
    constexpr int TH = 8, TW = 16;
    const int tiles = B * ((Ho + TH - 1) / TH) * ((Wo + TW - 1) / TW);
    nblk = tiles < kWgradBlocks ? tiles : kWgradBlocks;
    const size_t smem = (TH * TW * C + (2 * TH + 1) * (2 * TW + 1) * PADC) * sizeof(float);
    auto k = conv3x3_c32_wgrad_simt<T, 2, TH, TW>;
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "conv3x3_c32_wgrad_simt")) return e;
    k<<<nblk, 288, smem, st>>>(x, dy, ws, B, H, W, Ho, Wo);
  }
  if (int e = dd::check_launch("conv3x3_c32_wgrad_simt")) return e;
  wgrad_reduce_kernel<<<(9 * C * C + C + 255) / 256, 256, 0, st>>>(ws, nblk, C, dw, db);
  return dd::check_launch("wgrad_reduce");
}

}  // namespace

// tcgen05 implementations live in conv_tc.cu
namespace dd {
int conv3x3_c32_fwd_tc(const void* in, const float* w, const float* bias, void* out, int B, int H, int W,
                       int stride, int mode, const void* mask, uint32_t* bits, cudaStream_t st);
int conv3x3_c32_wgrad_tc(const void* x, const void* dy, float* dw, float* db, void* ws, size_t ws_bytes, int B,
                         int H, int W, int stride, cudaStream_t st);
int conv_c1_fwd_tc(const void* in, int in_flags, const float* w, const float* bias, void* out, uint32_t* bits, int B, int H,
                   int Wm, cudaStream_t st);
int enc_c1c2_fused_fwd_tc(const void* in, int in_flags, const float* w1, const float* b1, const float* w2, const float* b2,
                          void* out, int B, int H, int Wm, cudaStream_t st);
int conv_c1_wgrad_tc(const void* in, int in_flags, const void* dy, float* dw, float* db, void* ws, size_t ws_bytes,
                     int B, int H, int Wm, cudaStream_t st);
int conv_c1_dgrad_tc(const void* dy, const float* w, float* dx, bool views, int B, int H, int Wm, cudaStream_t st);
}  // namespace dd

extern "C" size_t dd_conv_wgrad_workspace_bytes(void) { return kWgradWsBytes; }

extern "C" int dd_conv3x3_c32_fwd(const void* in, const float* w_oihw, const float* bias, void* out, int dtype,
                                  int B, int H, int W, int stride, int impl, void* stream) {
  DD_REQUIRE(in && w_oihw && bias && out, DD_ERR_BAD_ARG, "dd_conv3x3_c32_fwd: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_conv3x3_c32_fwd: bad shape");
  DD_REQUIRE(stride == 1 || stride == 2, DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_fwd: stride %d", stride);
  DD_REQUIRE((uintptr_t)in % 16 == 0 && (uintptr_t)out % 16 == 0, DD_ERR_ALIGNMENT, "dd_conv3x3_c32_fwd: alignment");
  if (B == 0) return 0;
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_BF16 && impl != DD_IMPL_SIMT)
    return dd::conv3x3_c32_fwd_tc(in, w_oihw, bias, out, B, H, W, stride, 0, nullptr, nullptr, st);
  DD_REQUIRE(!(dtype == DD_F32 && impl == DD_IMPL_TCGEN05), DD_ERR_UNSUPPORTED, "tcgen05 conv is bf16 only");
  if (dtype == DD_F32) return conv_fwd_simt<float>((const float*)in, w_oihw, bias, (float*)out, B, H, W, stride, st);
  if (dtype == DD_BF16)
    return conv_fwd_simt<__nv_bfloat16>((const __nv_bfloat16*)in, w_oihw, bias, (__nv_bfloat16*)out, B, H, W, stride, st);
  return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_fwd: dtype %d", dtype);
}

extern "C" int dd_conv3x3_c32_dgrad(const void* dy, const float* w_oihw, const void* x, void* dx, int dtype, int B,
                                    int H, int W, int stride, int impl, void* stream) {
  DD_REQUIRE(dy && w_oihw && dx, DD_ERR_BAD_ARG, "dd_conv3x3_c32_dgrad: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_conv3x3_c32_dgrad: bad shape");
  DD_REQUIRE(stride == 1 || stride == 2, DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_dgrad: stride %d", stride);
  if (B == 0) return 0;
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_BF16 && impl != DD_IMPL_SIMT)
    return dd::conv3x3_c32_fwd_tc(dy, w_oihw, nullptr, dx, B, H, W, stride, 1, x, nullptr, st);
  DD_REQUIRE(!(dtype == DD_F32 && impl == DD_IMPL_TCGEN05), DD_ERR_UNSUPPORTED, "tcgen05 conv is bf16 only");
  if (dtype == DD_F32)
    return conv_dgrad_simt<float>((const float*)dy, w_oihw, (const float*)x, (float*)dx, B, H, W, stride, st);
  if (dtype == DD_BF16)
    return conv_dgrad_simt<__nv_bfloat16>((const __nv_bfloat16*)dy, w_oihw, (const __nv_bfloat16*)x,
                                          (__nv_bfloat16*)dx, B, H, W, stride, st);
  return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_dgrad: dtype %d", dtype);
}

// the ReLU sign-word forms (conv_tc.cu, relu_bits): bf16 tensor-core kernels only; every check runs before the launch
extern "C" int dd_conv3x3_c32_fwd_bits(const void* in, const float* w_oihw, const float* bias, void* out, uint32_t* bits,
                                       int dtype, int B, int H, int W, int stride, int impl, void* stream) {
  DD_REQUIRE(in && w_oihw && bias && out && bits, DD_ERR_BAD_ARG, "dd_conv3x3_c32_fwd_bits: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_conv3x3_c32_fwd_bits: bad shape");
  DD_REQUIRE(stride == 1, DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_fwd_bits: stride %d (sign words are kept for stride 1 only)", stride);
  DD_REQUIRE(dtype == DD_BF16 && impl != DD_IMPL_SIMT, DD_ERR_UNSUPPORTED,
             "dd_conv3x3_c32_fwd_bits: sign words come from the bf16 tensor-core kernel only (dtype %d, impl %d)", dtype, impl);
  if (B == 0) return 0;
  return dd::conv3x3_c32_fwd_tc(in, w_oihw, bias, out, B, H, W, stride, 0, nullptr, bits, dd::as_stream(stream));
}

extern "C" int dd_conv3x3_c32_dgrad_bits(const void* dy, const float* w_oihw, const uint32_t* x_bits, void* dx, int dtype,
                                         int B, int H, int W, int stride, int impl, void* stream) {
  DD_REQUIRE(dy && w_oihw && x_bits && dx, DD_ERR_BAD_ARG, "dd_conv3x3_c32_dgrad_bits: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_conv3x3_c32_dgrad_bits: bad shape");
  DD_REQUIRE(stride == 1 || stride == 2, DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_dgrad_bits: stride %d", stride);
  DD_REQUIRE(dtype == DD_BF16 && impl != DD_IMPL_SIMT, DD_ERR_UNSUPPORTED,
             "dd_conv3x3_c32_dgrad_bits: sign words are read by the bf16 tensor-core kernels only (dtype %d, impl %d)", dtype, impl);
  if (B == 0) return 0;
  return dd::conv3x3_c32_fwd_tc(dy, w_oihw, nullptr, dx, B, H, W, stride, 1, nullptr, const_cast<uint32_t*>(x_bits),
                                dd::as_stream(stream));
}

extern "C" int dd_conv3x3_c32_wgrad(const void* x, const void* dy, float* dw, float* db, void* workspace,
                                    size_t ws_bytes, int dtype, int B, int H, int W, int stride, int impl,
                                    void* stream) {
  DD_REQUIRE(x && dy && dw && db && workspace, DD_ERR_BAD_ARG, "dd_conv3x3_c32_wgrad: null pointer");
  DD_REQUIRE(B > 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_conv3x3_c32_wgrad: bad shape");
  DD_REQUIRE(stride == 1 || stride == 2, DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_wgrad: stride %d", stride);
  DD_REQUIRE(ws_bytes >= kWgradWsBytes, DD_ERR_WORKSPACE, "dd_conv3x3_c32_wgrad: workspace %zu < %zu", ws_bytes, kWgradWsBytes);
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_BF16 && impl != DD_IMPL_SIMT)
    return dd::conv3x3_c32_wgrad_tc(x, dy, dw, db, workspace, ws_bytes, B, H, W, stride, st);
  DD_REQUIRE(!(dtype == DD_F32 && impl == DD_IMPL_TCGEN05), DD_ERR_UNSUPPORTED, "tcgen05 conv is bf16 only");
  if (dtype == DD_F32)
    return conv_wgrad_simt<float>((const float*)x, (const float*)dy, dw, db, (float*)workspace, B, H, W, stride, st);
  if (dtype == DD_BF16)
    return conv_wgrad_simt<__nv_bfloat16>((const __nv_bfloat16*)x, (const __nv_bfloat16*)dy, dw, db,
                                          (float*)workspace, B, H, W, stride, st);
  return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv3x3_c32_wgrad: dtype %d", dtype);
}

extern "C" int dd_encoder_c1c2_fused_fwd(const void* in_, int in_flags, const float* w1_oihw, const float* bias1,
                                         const float* w2_oihw, const float* bias2, void* a2, int B, int H, int Wm,
                                         void* stream) {
  DD_REQUIRE(in_ && w1_oihw && bias1 && w2_oihw && bias2 && a2, DD_ERR_BAD_ARG, "dd_encoder_c1c2_fused_fwd: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && Wm > 0, DD_ERR_BAD_ARG, "dd_encoder_c1c2_fused_fwd: bad shape");
  DD_REQUIRE((in_flags & ~3) == 0, DD_ERR_BAD_ARG, "dd_encoder_c1c2_fused_fwd: in_flags %d", in_flags);
  DD_REQUIRE(!(in_flags & DD_IN_VIEWS) || Wm % 6 == 0, DD_ERR_BAD_ARG, "dd_encoder_c1c2_fused_fwd: mosaic width %d not a multiple of 6", Wm);
  if (B == 0) return 0;
  return dd::enc_c1c2_fused_fwd_tc(in_, in_flags, w1_oihw, bias1, w2_oihw, bias2, a2, B, H, Wm, dd::as_stream(stream));
}

extern "C" int dd_conv_c1_fwd(const void* in_, int in_flags, const float* w_oihw, const float* bias, void* out,
                              int out_dtype, int B, int H, int Wm, int impl, void* stream) {
  DD_REQUIRE(in_ && w_oihw && bias && out, DD_ERR_BAD_ARG, "dd_conv_c1_fwd: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && Wm > 0, DD_ERR_BAD_ARG, "dd_conv_c1_fwd: bad shape");
  DD_REQUIRE((in_flags & ~3) == 0, DD_ERR_BAD_ARG, "dd_conv_c1_fwd: in_flags %d", in_flags);
  const int in_is_views = in_flags & DD_IN_VIEWS;
  DD_REQUIRE(!in_is_views || Wm % 6 == 0, DD_ERR_BAD_ARG, "dd_conv_c1_fwd: mosaic width %d not a multiple of 6", Wm);
  if (B == 0) return 0;
  cudaStream_t st = dd::as_stream(stream);
  DD_REQUIRE(!(out_dtype == DD_F32 && impl == DD_IMPL_TCGEN05), DD_ERR_UNSUPPORTED, "tcgen05 conv is bf16 only");
  if (out_dtype == DD_BF16 && impl != DD_IMPL_SIMT) return dd::conv_c1_fwd_tc(in_, in_flags, w_oihw, bias, out, nullptr, B, H, Wm, st);
  DD_REQUIRE(!(in_flags & DD_IN_U8), DD_ERR_UNSUPPORTED, "dd_conv_c1_fwd: raw-byte input runs on the bf16 tensor-core path only "
             "(fp32 parity path: dd_stitch_u8 first)");
  const float* in = (const float*)in_;
  dim3 grid((Wm + 31) / 32, (H + 7) / 8, B);
  if (out_dtype == DD_F32) {
    if (in_is_views) conv_c1_fwd_simt<float, true><<<grid, 256, 0, st>>>(in, w_oihw, bias, (float*)out, H, Wm);
    else conv_c1_fwd_simt<float, false><<<grid, 256, 0, st>>>(in, w_oihw, bias, (float*)out, H, Wm);
  } else if (out_dtype == DD_BF16) {
    if (in_is_views) conv_c1_fwd_simt<__nv_bfloat16, true><<<grid, 256, 0, st>>>(in, w_oihw, bias, (__nv_bfloat16*)out, H, Wm);
    else conv_c1_fwd_simt<__nv_bfloat16, false><<<grid, 256, 0, st>>>(in, w_oihw, bias, (__nv_bfloat16*)out, H, Wm);
  } else {
    return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv_c1_fwd: dtype %d", out_dtype);
  }
  return dd::check_launch("conv_c1_fwd");
}

extern "C" int dd_conv_c1_fwd_bits(const void* in_, int in_flags, const float* w_oihw, const float* bias, void* out,
                                   uint32_t* bits, int out_dtype, int B, int H, int Wm, int impl, void* stream) {
  DD_REQUIRE(in_ && w_oihw && bias && out && bits, DD_ERR_BAD_ARG, "dd_conv_c1_fwd_bits: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && Wm > 0, DD_ERR_BAD_ARG, "dd_conv_c1_fwd_bits: bad shape");
  DD_REQUIRE((in_flags & ~3) == 0, DD_ERR_BAD_ARG, "dd_conv_c1_fwd_bits: in_flags %d", in_flags);
  DD_REQUIRE(!(in_flags & DD_IN_VIEWS) || Wm % 6 == 0, DD_ERR_BAD_ARG, "dd_conv_c1_fwd_bits: mosaic width %d not a multiple of 6", Wm);
  DD_REQUIRE(out_dtype == DD_BF16 && impl != DD_IMPL_SIMT, DD_ERR_UNSUPPORTED,
             "dd_conv_c1_fwd_bits: sign words come from the bf16 tensor-core kernel only (dtype %d, impl %d)", out_dtype, impl);
  if (B == 0) return 0;
  return dd::conv_c1_fwd_tc(in_, in_flags, w_oihw, bias, out, bits, B, H, Wm, dd::as_stream(stream));
}

extern "C" int dd_conv_c1_wgrad(const void* in_, int in_flags, const void* dy, int dtype, float* dw, float* db,
                                void* workspace, size_t ws_bytes, int B, int H, int Wm, int impl, void* stream) {
  DD_REQUIRE(in_ && dy && dw && db && workspace, DD_ERR_BAD_ARG, "dd_conv_c1_wgrad: null pointer");
  DD_REQUIRE((in_flags & ~3) == 0, DD_ERR_BAD_ARG, "dd_conv_c1_wgrad: in_flags %d", in_flags);
  const int in_is_views = in_flags & DD_IN_VIEWS;
  DD_REQUIRE(B > 0 && H > 0 && Wm > 0, DD_ERR_BAD_ARG, "dd_conv_c1_wgrad: bad shape");
  DD_REQUIRE(ws_bytes >= kWgradWsBytes, DD_ERR_WORKSPACE, "dd_conv_c1_wgrad: workspace too small");
  cudaStream_t st = dd::as_stream(stream);
  DD_REQUIRE(!(dtype == DD_F32 && impl == DD_IMPL_TCGEN05), DD_ERR_UNSUPPORTED, "tcgen05 conv is bf16 only");
  DD_REQUIRE(!in_is_views || Wm % 6 == 0, DD_ERR_BAD_ARG, "dd_conv_c1_wgrad: mosaic width %d not a multiple of 6", Wm);
  if (dtype == DD_BF16 && impl != DD_IMPL_SIMT)
    return dd::conv_c1_wgrad_tc(in_, in_flags, dy, dw, db, workspace, ws_bytes, B, H, Wm, st);
  DD_REQUIRE(!(in_flags & DD_IN_U8), DD_ERR_UNSUPPORTED, "dd_conv_c1_wgrad: raw-byte input runs on the bf16 tensor-core path only");
  const float* in = (const float*)in_;
  const int tiles = B * ((H + 7) / 8) * ((Wm + 31) / 32);
  const int nblk = tiles < kWgradBlocks ? tiles : kWgradBlocks;
  float* ws = (float*)workspace;
  if (dtype == DD_F32) {
    if (in_is_views) conv_c1_wgrad_simt<float, true><<<nblk, 256, 0, st>>>(in, (const float*)dy, ws, B, H, Wm);
    else conv_c1_wgrad_simt<float, false><<<nblk, 256, 0, st>>>(in, (const float*)dy, ws, B, H, Wm);
  } else if (dtype == DD_BF16) {
    if (in_is_views) conv_c1_wgrad_simt<__nv_bfloat16, true><<<nblk, 256, 0, st>>>(in, (const __nv_bfloat16*)dy, ws, B, H, Wm);
    else conv_c1_wgrad_simt<__nv_bfloat16, false><<<nblk, 256, 0, st>>>(in, (const __nv_bfloat16*)dy, ws, B, H, Wm);
  } else {
    return dd::fail(DD_ERR_UNSUPPORTED, "dd_conv_c1_wgrad: dtype %d", dtype);
  }
  if (int e = dd::check_launch("conv_c1_wgrad")) return e;
  c1_wgrad_reduce_kernel<<<4, 256, 0, st>>>(ws, nblk, dw, db);
  return dd::check_launch("c1_wgrad_reduce");
}

extern "C" int dd_conv_c1_dgrad(const void* dy, int dtype, const float* w_oihw, float* dx, int out_flags, int B, int H,
                                int Wm, int impl, void* stream) {
  DD_REQUIRE(B >= 0 && H > 0 && Wm > 0, DD_ERR_BAD_ARG, "dd_conv_c1_dgrad: bad shape");
  DD_REQUIRE((out_flags & ~3) == 0, DD_ERR_BAD_ARG, "dd_conv_c1_dgrad: out_flags %d", out_flags);
  DD_REQUIRE(!(out_flags & DD_IN_U8), DD_ERR_UNSUPPORTED, "dd_conv_c1_dgrad: raw camera bytes have no gradient");
  const bool views = out_flags & DD_IN_VIEWS;
  DD_REQUIRE(!views || Wm % 6 == 0, DD_ERR_BAD_ARG, "dd_conv_c1_dgrad: mosaic width %d not a multiple of 6", Wm);
  DD_REQUIRE(dtype == DD_F32 || dtype == DD_BF16, DD_ERR_UNSUPPORTED, "dd_conv_c1_dgrad: dtype %d", dtype);
  DD_REQUIRE(!(dtype == DD_F32 && impl == DD_IMPL_TCGEN05), DD_ERR_UNSUPPORTED, "tcgen05 conv is bf16 only");
  if (B == 0) return 0;
  DD_REQUIRE(dy && w_oihw && dx, DD_ERR_BAD_ARG, "dd_conv_c1_dgrad: null pointer");
  DD_REQUIRE((uintptr_t)dy % 16 == 0 && (uintptr_t)dx % 4 == 0, DD_ERR_ALIGNMENT,
             "dd_conv_c1_dgrad: dy %p must be 16-byte aligned, dx %p 4-byte aligned", dy, dx);
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_BF16 && impl != DD_IMPL_SIMT) return dd::conv_c1_dgrad_tc(dy, w_oihw, dx, views, B, H, Wm, st);
  dim3 grid((Wm + 31) / 32, (H + 7) / 8, B);
  if (dtype == DD_F32) {
    if (views) conv_c1_dgrad_simt<float, true><<<grid, 256, 0, st>>>((const float*)dy, w_oihw, dx, H, Wm);
    else conv_c1_dgrad_simt<float, false><<<grid, 256, 0, st>>>((const float*)dy, w_oihw, dx, H, Wm);
  } else {
    if (views) conv_c1_dgrad_simt<__nv_bfloat16, true><<<grid, 256, 0, st>>>((const __nv_bfloat16*)dy, w_oihw, dx, H, Wm);
    else conv_c1_dgrad_simt<__nv_bfloat16, false><<<grid, 256, 0, st>>>((const __nv_bfloat16*)dy, w_oihw, dx, H, Wm);
  }
  return dd::check_launch("conv_c1_dgrad");
}

extern "C" int dd_relu_mask(const void* g, const void* act, void* out, int dtype, long long n, void* stream) {
  DD_REQUIRE(n >= 0, DD_ERR_BAD_ARG, "dd_relu_mask: n=%lld", n);
  if (n == 0) return 0;
  DD_REQUIRE(g && act && out, DD_ERR_BAD_ARG, "dd_relu_mask: null pointer");
  const long long n8 = n / 8;
  long long want = (n8 + 255) / 256;
  if (want < 1) want = 1;
  const int grid = (int)(want < dd::kSMs * 8 ? want : dd::kSMs * 8);
  cudaStream_t st = dd::as_stream(stream);
  if (dtype == DD_F32) relu_mask_kernel<float><<<grid, 256, 0, st>>>((const float*)g, (const float*)act, (float*)out, n8, n);
  else if (dtype == DD_BF16)
    relu_mask_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)g, (const __nv_bfloat16*)act, (__nv_bfloat16*)out, n8, n);
  else return dd::fail(DD_ERR_UNSUPPORTED, "dd_relu_mask: dtype %d", dtype);
  return dd::check_launch("relu_mask");
}
