// Stride-1 (dilated) convolutions and transposed convolutions with wide filters as implicit GEMMs on the 5th-gen tensor
// cores: the merging CNN's up_conv_1..3 (ConvTranspose2d k7, dilation 7: 64.9 of the bounding-box model's 80.8 GFLOP per
// scene; spatial_bb/components.py:135-137,164-166), rm_conv_2 and out_conv (k3, dilation 3 / 1; :26,133), the decoder's
// dc1 / dc2 (ConvTranspose2d k3 p1; autoencoder/components.py:70-71,89-90) -- forward passes and input gradients.
//
// One form covers all of them (KT x KT taps, dilation D, sign s, offset o):
//      out[h, w, n] = sum_{kh, kw, k}  in[h + s*D*kh + o, w + s*D*kw + o, k] * W[kh][kw][n][k]          (in = 0 outside)
//   transposed conv forward: s = -1, o = +pad;  conv forward and transposed-conv input gradient: s = +1, o = -pad;
//   conv input gradient: s = -1, o = +pad.
//
// Output rows h = D*t + rho of one residue class rho depend on input rows of ONE class only, D*(t + s*kh) + rho + o: along
// the class the dilated filter is a dense KT-tap one.  A CTA takes G consecutive class rows t0..t0+G-1 of a 128-pixel
// column strip (G accumulators of N columns in TMEM) and the G + KT - 1 input rows they need; an input row r feeds the
// outputs i in [r-KT+1, r] through taps kappa = i - r + KT - 1 that sit side by side in the packed weights, so ONE
// tcgen05.mma of N-extent n*N (n outputs, up to 256 columns) covers them: the A tile (128 pixels x 16 channels, the
// shared-memory hog at small N) is read once per row instead of once per tap -- the row-scatter idea of the 3x3 kernel,
// over 7 taps.  Horizontal taps are shifts of the A start address by D*kw pixels (64-byte-swizzled K-major rows: the swizzle
// follows the absolute address, profiles/r2_tma_layout_probe.txt).  Loop nest per item: 32-channel chunk -> kw -> row ->
// K half; the rows of a chunk stay resident, the (chunk, kw) weight slabs (KT x N rows of 64 B) stream through a
// double buffer from a packed bf16 copy that a small kernel writes per call (L2 resident).
// Warps: 0 = TMA producer for input rows, 1 = TMA producer for weight slabs, 2 = MMA issuer, 4..11 = epilogue
// (TMEM -> bias / ReLU or ReLU mask -> bf16 NHWC).
#include "dd_common.cuh"
#include "tma_host.h"
#include "umma.cuh"

namespace {

constexpr int TM = 128;                       // output pixels per strip (M)
constexpr int TILE_PX = 170;                  // input pixels per row tile: 128 + 6 * 7
constexpr int ROWPITCH = 22 * 512;            // 170 px x 64 B = 10880, rounded up to the swizzle period
constexpr int ROW_TX = TILE_PX * 64;
constexpr int DT_THREADS = 384;               // 12 warps
constexpr int EPI_WARP0 = 4;

struct DilGeo {
  int B, Hi, Wi, Ho, Wo;
  int KT, D, sign, off;                       // taps per axis, dilation, s, o
  int relu, has_bias, has_mask;
  int items, strips, groups_max;              // work decomposition
};

template <int KC, int N, int G>
struct DT {
  static constexpr int R = G + 6;                               // row slots (KT <= 7)
  static constexpr int RP = (R + 1) / 2;                        // row-pair barriers
  static constexpr int SLAB = 7 * N * 64;                       // one (chunk, kw) weight slab: [kappa][n][32 k] bf16
  static constexpr int ROWS_BYTES = R * ROWPITCH;
  static constexpr int SMEM = ROWS_BYTES + 2 * SLAB + 512;
  static constexpr int NBUF = 2 * G * N <= 512 ? 2 : 1;         // accumulator sets in TMEM
  static constexpr int COLS = G * N * NBUF <= 128 ? 128 : (G * N * NBUF <= 256 ? 256 : 512);
  static constexpr int NMAX = 256 / N;                          // outputs one MMA can cover
  static_assert(SMEM <= 227 * 1024, "shared memory");
  static_assert(G * N * NBUF <= 512, "TMEM");
  static_assert(SLAB % 512 == 0, "slab alignment");
};

struct DilBars {
  uint64_t row_full[8], row_empty[8], w_full[2], w_empty[2], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

// item -> (b, class rho, first class row t0, strip); strips vary fastest so that neighbouring CTAs share input rows in L2
struct Item { int b, rho, t0, w0, nrows; };
__device__ __forceinline__ Item decode(const DilGeo& g, int it, int G_) {
  Item o;
  const int strip = it % g.strips;
  int rest = it / g.strips;
  const int grp = rest % g.groups_max;
  rest /= g.groups_max;
  o.rho = rest % g.D;
  o.b = rest / g.D;
  o.t0 = grp * G_;
  o.w0 = strip * TM;
  const int T = (g.Ho - o.rho + g.D - 1) / g.D;                  // class rows of this class
  o.nrows = min(G_, T - o.t0);                                   // <= 0: nothing to do (classes differ by one row)
  return o;
}

template <int KC, int N, int G>
__global__ void __launch_bounds__(DT_THREADS, 1) conv_dil_tc_kernel(const __grid_constant__ CUtensorMap map_in,
                                                                    const __grid_constant__ CUtensorMap map_w,
                                                                    const float* __restrict__ bias,
                                                                    const __nv_bfloat16* __restrict__ mask,
                                                                    __nv_bfloat16* __restrict__ out, const DilGeo g) {
  using T = DT<KC, N, G>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_rows = smem;
  uint8_t* s_w = smem + T::ROWS_BYTES;
  DilBars* bars = reinterpret_cast<DilBars*>(smem + T::ROWS_BYTES + 2 * T::SLAB);
  __shared__ float s_bias[N];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int KT = g.KT, R = G + KT - 1, RP = (R + 1) / 2;

  if (tid < N) s_bias[tid] = g.has_bias ? bias[tid] : 0.f;
  if (tid == 0) {
    for (int i = 0; i < T::RP; ++i) { umma::mbar_init(&bars->row_full[i], 1); umma::mbar_init(&bars->row_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      umma::mbar_init(&bars->w_full[i], 1); umma::mbar_init(&bars->w_empty[i], 1);
      umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], 8);
    }
    umma::fence_mbar_init();
  }
  if (warp == 2) umma::tmem_alloc(&bars->tmem_base, T::COLS);
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp == 0) {
    // =========================== producer: input rows (one thread, TMA) ============================
    if (lane == 0) {
      umma::tma_prefetch_desc(&map_in);
      uint32_t q = 0;                                         // (item, chunk) counter = use index of every row slot
      for (int it = blockIdx.x; it < g.items; it += gridDim.x) {
        const Item im = decode(g, it, G);
        if (im.nrows <= 0) continue;
        const int u0 = g.sign < 0 ? im.t0 - (KT - 1) : im.t0;   // first input class row
        const int x0 = im.w0 + g.off - (g.sign < 0 ? (KT - 1) * g.D : 0);
        for (int c = 0; c < KC; ++c, ++q) {
          for (int rp = 0; rp < RP; ++rp) {
            umma::mbar_wait(&bars->row_empty[rp], (q & 1) ^ 1);
            const int nr = min(2, R - 2 * rp);
            umma::mbar_expect_tx(&bars->row_full[rp], (uint32_t)(nr * ROW_TX));
            for (int k = 0; k < nr; ++k) {
              const int r = 2 * rp + k;
              umma::tma_load_4d(umma::smem_u32(s_rows) + r * ROWPITCH, &map_in, c * 32, x0, g.D * (u0 + r) + im.rho + g.off, im.b,
                                &bars->row_full[rp]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== producer: weight slabs (one thread, TMA) ==========================
    if (lane == 0) {
      umma::tma_prefetch_desc(&map_w);
      uint32_t wu = 0;
      for (int it = blockIdx.x; it < g.items; it += gridDim.x) {
        const Item im = decode(g, it, G);
        if (im.nrows <= 0) continue;
        for (int c = 0; c < KC; ++c)
          for (int kw = 0; kw < KT; ++kw, ++wu) {
            const uint32_t slot = wu & 1;
            umma::mbar_wait(&bars->w_empty[slot], ((wu >> 1) & 1) ^ 1);
            umma::mbar_expect_tx(&bars->w_full[slot], (uint32_t)(KT * N * 64));
            for (int ka = 0; ka < KT; ++ka)                    // one box per kappa: N rows of 64 B
              umma::tma_load_2d(umma::smem_u32(s_w) + slot * T::SLAB + ka * N * 64, &map_w, 0, ((c * KT + kw) * KT + ka) * N,
                                &bars->w_full[slot]);
          }
      }
    }
  } else if (warp == 2) {
    // =========================== MMA issuer (whole warp loops, elected lane issues) ================
    constexpr uint32_t ab_hi = umma::desc_hi_sw64(512);                         // K-major SWIZZLE_64B, 8-row groups of 512 B
    constexpr uint32_t idesc1 = umma::make_idesc_bf16(TM, N, false, false);
    constexpr uint32_t IDESC_NSTEP = ((uint32_t)N >> 3) << 17;                   // + N columns
    const uint32_t rows_lo = umma::desc_lo(umma::smem_u32(s_rows), 0);
    const uint32_t w_lo = umma::desc_lo(umma::smem_u32(s_w), 0);
    uint32_t q = 0, wu = 0, ic = 0;
    for (int it = blockIdx.x; it < g.items; it += gridDim.x) {
      const Item im = decode(g, it, G);
      if (im.nrows <= 0) continue;
      const uint32_t buf = T::NBUF == 2 ? (ic & 1) : 0;
      umma::mbar_wait(&bars->acc_empty[buf], (((ic / T::NBUF) & 1) ^ 1));
      umma::tc_fence_after_sync();
      const uint32_t d_base = tmem + buf * (G * N);
      for (int c = 0; c < KC; ++c, ++q) {
        for (int kw = 0; kw < KT; ++kw, ++wu) {
          const uint32_t slot = wu & 1;
          umma::mbar_wait(&bars->w_full[slot], (wu >> 1) & 1);
          const uint32_t pxoff = (uint32_t)((g.sign < 0 ? (KT - 1 - kw) : kw) * g.D) * 64u;
          const uint32_t b_slab = w_lo + ((slot * T::SLAB) >> 4);
          for (int r = 0; r < R; ++r) {
            if (kw == 0 && (r & 1) == 0) umma::mbar_wait(&bars->row_full[r >> 1], q & 1);
            umma::tc_fence_after_sync();
            const int ilo = max(0, r - (KT - 1)), ihi = min(G - 1, r);
            const uint32_t a_row = rows_lo + ((r * ROWPITCH + pxoff) >> 4);
            if (umma::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) {
                const uint32_t a = a_row + ks * 2;             // K half: +32 B
                if (c == 0 && kw == 0 && ks == 0) {
                  // the item's first pass: output i gets its first contribution from row r = i -> overwrite there
                  for (int i = ilo; i <= ihi; ++i)
                    umma::mma_bf16_lohi(d_base + i * N, a, ab_hi, b_slab + (((i - r + KT - 1) * N * 64) >> 4), ab_hi, idesc1,
                                        r > i ? 1u : 0u);
                } else {
                  for (int i0 = ilo; i0 <= ihi; i0 += T::NMAX) {
                    const int n = min(T::NMAX, ihi - i0 + 1);
                    umma::mma_bf16_lohi(d_base + i0 * N, a, ab_hi, b_slab + (((i0 - r + KT - 1) * N * 64 + ks * 32) >> 4), ab_hi,
                                        idesc1 + (uint32_t)(n - 1) * IDESC_NSTEP, 1u);
                  }
                }
              }
              if (kw == KT - 1 && ((r & 1) == 1 || r == R - 1)) umma::mma_commit(&bars->row_empty[r >> 1]);
            }
            __syncwarp();
          }
          if (umma::elect_one()) umma::mma_commit(&bars->w_empty[slot]);
          __syncwarp();
        }
      }
      if (umma::elect_one()) umma::mma_commit(&bars->acc_full[buf]);
      __syncwarp();
      ++ic;
    }
  } else if (warp >= EPI_WARP0) {
    // =========================== epilogue (warps 4..11) =============================================
    // thread = output pixel (TMEM lane); two warps per lane quarter take alternate output rows
    const int ew = warp - EPI_WARP0;
    const int quarter = warp & 3;
    const int half = ew >> 2;
    uint32_t ic = 0;
    for (int it = blockIdx.x; it < g.items; it += gridDim.x) {
      const Item im = decode(g, it, G);
      if (im.nrows <= 0) continue;
      const uint32_t buf = T::NBUF == 2 ? (ic & 1) : 0;
      umma::mbar_wait_sleep(&bars->acc_full[buf], (ic / T::NBUF) & 1);
      umma::tc_fence_after_sync();
      const int w = im.w0 + quarter * 32 + lane;
      for (int i = half; i < G; i += 2) {
        const int h = g.D * (im.t0 + i) + im.rho;
        const bool ok = i < im.nrows && h < g.Ho && w < g.Wo;      // (warp-uniform except for w)
        const size_t off = (((size_t)im.b * g.Ho + (ok ? h : 0)) * g.Wo + (ok ? w : 0)) * N;
#pragma unroll
        for (int c0 = 0; c0 < N; c0 += 32) {
          constexpr int CW = N < 32 ? N : 32;
          uint32_t rr[32];
          if (N >= 32) {
            umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + buf * (G * N) + i * N + c0, rr);
          } else {
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                         : "=r"(rr[0]), "=r"(rr[1]), "=r"(rr[2]), "=r"(rr[3]), "=r"(rr[4]), "=r"(rr[5]), "=r"(rr[6]), "=r"(rr[7]),
                           "=r"(rr[8]), "=r"(rr[9]), "=r"(rr[10]), "=r"(rr[11]), "=r"(rr[12]), "=r"(rr[13]), "=r"(rr[14]), "=r"(rr[15])
                         : "r"(tmem + ((uint32_t)(quarter * 32) << 16) + buf * (G * N) + i * N + c0)
                         : "memory");
          }
          umma::tmem_ld_wait();
          if (ok) {
            uint32_t pk[CW / 2];
#pragma unroll
            for (int k = 0; k < CW / 2; ++k) {
              float x0 = __uint_as_float(rr[2 * k]) + s_bias[c0 + 2 * k], x1 = __uint_as_float(rr[2 * k + 1]) + s_bias[c0 + 2 * k + 1];
              if (g.relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
              __nv_bfloat162 hh = __floats2bfloat162_rn(x0, x1);
              pk[k] = *reinterpret_cast<uint32_t*>(&hh);
            }
            if (g.has_mask) {
#pragma unroll
              for (int k8 = 0; k8 < CW / 16; ++k8) {
                uint32_t mk[8];
                umma::ldg256(mask + off + c0 + 16 * k8, mk);
                const __nv_bfloat162 zero = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
                for (int k = 0; k < 8; ++k) pk[8 * k8 + k] &= __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&mk[k]), zero);
              }
            }
#pragma unroll
            for (int k8 = 0; k8 < CW / 16; ++k8) umma::stg256(out + off + c0 + 16 * k8, pk + 8 * k8);
          }
        }
      }
      umma::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) umma::mbar_arrive_relaxed(&bars->acc_empty[buf]);   // relaxed: a release arrive would first drain this warp's outstanding global stores
      ++ic;
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) umma::tmem_dealloc(tmem, T::COLS);
}

// packed weights [chunk][kw][kappa][n][32 k] bf16 from a torch-layout fp32 tensor: element (n, k, kh, kw) sits at
// w[n * sn + k * sk + kh * KT + kw]; kh = flip ? KT-1-kappa : kappa.  Channels k >= Kreal / n >= Nreal are zero.
__global__ void dil_pack_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wp, int KC, int KT, int N, int Kreal,
                                int Nreal, long long sn, long long sk, int flip) {
  const long long total = (long long)KC * KT * KT * N * 32;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k32 = (int)(i & 31);
    long long rest = i >> 5;
    const int n = (int)(rest % N); rest /= N;
    const int ka = (int)(rest % KT); rest /= KT;
    const int kw = (int)(rest % KT);
    const int c = (int)(rest / KT);
    const int k = c * 32 + k32;
    const int kh = flip ? KT - 1 - ka : ka;
    wp[i] = __float2bfloat16_rn(k < Kreal && n < Nreal ? w[n * sn + k * sk + (long long)kh * KT + kw] : 0.f);
  }
}

template <int KC, int N, int G>
int launch_dil(const void* in, const __nv_bfloat16* wp, const float* bias, const void* mask, void* out, DilGeo g, int K,
               cudaStream_t st) {
  using T = DT<KC, N, G>;
  g.strips = (g.Wo + TM - 1) / TM;
  const int Tmax = (g.Ho + g.D - 1) / g.D;
  g.groups_max = (Tmax + G - 1) / G;
  g.items = g.B * g.D * g.groups_max * g.strips;
  auto k = conv_dil_tc_kernel<KC, N, G>;
  if (int e = dd::set_smem(k, T::SMEM, dd::Carveout::kMaxShared, "conv_dil_tc")) return e;
  CUtensorMap min_, mw;
  char msg[256];
  if (dd::tma_map_nhwc_sw64(&min_, in, g.B, g.Hi, g.Wi, K, TILE_PX, 1, msg, sizeof msg))
    return dd::fail(DD_ERR_UNSUPPORTED, "conv_dil_tc: in: %s", msg);
  if (dd::tma_map_2d(&mw, wp, 2, (uint64_t)KC * g.KT * g.KT * N, 32, 32, 32, N, CU_TENSOR_MAP_SWIZZLE_64B, msg, sizeof msg))
    return dd::fail(DD_ERR_UNSUPPORTED, "conv_dil_tc: w: %s", msg);
  const int grid = g.items < dd::kSMs ? g.items : dd::kSMs;
  k<<<grid, DT_THREADS, T::SMEM, st>>>(min_, mw, bias, (const __nv_bfloat16*)mask, (__nv_bfloat16*)out, g);
  return dd::check_launch("conv_dil_tc");
}

}  // namespace

namespace dd {

// K = channels of the gathered tensor, N = channels produced.  Supported: square KT in {3, 7} taps, one dilation for both
// axes, stride 1, K in {32, 64, 96}, N in {16, 32, 64, 96} with an instantiated (K, N) pair.
bool conv_dil_tc_supported(int K, int N, int KT, int D) {
  if (!(KT == 3 || KT == 7) || D < 1 || D > 7) return false;
  return (K == 96 && N == 64) || (K == 64 && N == 32) || (K == 32 && N == 16) || (K == 32 && N == 32) || (K == 64 && N == 96) ||
         (K == 32 && N == 64);
}

// w: torch-layout fp32 weights; (sn, sk): strides of the produced / gathered channel index in it; flip: kh = KT-1-kappa
int conv_dil_tc(const void* in, const float* w, long long sn, long long sk, int flip, const float* bias, const void* mask, void* out,
                void* pack_ws, int B, int Hi, int Wi, int Ho, int Wo, int K, int N, int KT, int D, int sign, int off, int relu,
                cudaStream_t st, int Kreal, int Nreal) {
  // Kreal < K: `in` carries K channels per pixel of which only the first Kreal exist in the weights (zero-padded pixels);
  // Nreal < N: the weights have Nreal produced channels, `out` / bias / mask carry N (the caller drops the padding)
  if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(mask) |
        reinterpret_cast<uintptr_t>(pack_ws)) & 31) != 0)
    return fail(DD_ERR_ALIGNMENT, "conv_dil_tc: pointers must be 32-byte aligned");
  const int KC = K / 32;
  __nv_bfloat16* wp = (__nv_bfloat16*)pack_ws;
  const long long total = (long long)KC * KT * KT * N * 32;
  dil_pack_kernel<<<(int)((total + 255) / 256 < 592 ? (total + 255) / 256 : 592), 256, 0, st>>>(w, wp, KC, KT, N, Kreal, Nreal, sn, sk, flip);
  if (int e = check_launch("conv_dil_pack")) return e;
  DilGeo g = {};
  g.B = B; g.Hi = Hi; g.Wi = Wi; g.Ho = Ho; g.Wo = Wo; g.KT = KT; g.D = D; g.sign = sign; g.off = off;
  g.relu = relu; g.has_bias = bias != nullptr; g.has_mask = mask != nullptr;
  if (K == 96 && N == 64) return launch_dil<3, 64, 4>(in, wp, bias, mask, out, g, K, st);
  if (K == 64 && N == 32) return launch_dil<2, 32, 8>(in, wp, bias, mask, out, g, K, st);
  if (K == 32 && N == 16) return launch_dil<1, 16, 8>(in, wp, bias, mask, out, g, K, st);
  if (K == 32 && N == 32) return launch_dil<1, 32, 8>(in, wp, bias, mask, out, g, K, st);
  if (K == 64 && N == 96) return launch_dil<2, 96, 4>(in, wp, bias, mask, out, g, K, st);
  if (K == 32 && N == 64) return launch_dil<1, 64, 4>(in, wp, bias, mask, out, g, K, st);
  return fail(DD_ERR_UNSUPPORTED, "conv_dil_tc: K %d N %d", K, N);
}

}  // namespace dd
