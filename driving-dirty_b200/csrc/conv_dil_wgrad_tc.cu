// Weight gradients of the wide stride-1 (dilated) convs / transposed convs on the tensor cores (up_conv_1 / up_conv_2 of the
// merging CNN, rm_conv_2, out_conv, the decoder's dc1 / dc2): the companion of conv_dil_tc.cu.  With the forward written as
//      out[h, w, n] = sum_{kh, kw, k}  in[h + s*D*kh + o, w + s*D*kw + o, k] * W(n, k, kh, kw)
// the gradient is      dW(n, k, kh, kw) = sum_{b, h, w}  in[h + s*D*kh + o, w + s*D*kw + o, k] * dout[h, w, n]:
// a contraction over PIXELS, operands MN-major like csrc/conv_wgrad_tc.cu (whole-pixel TMA boxes, 64-byte swizzle; the tap
// kw is a shift of the A start address by D*kw pixels).  KT*KT taps x K x N accumulators (4704 x 64 fp32 for up_conv_1 =
// 1.2 MB) do not fit the 256 KB of TMEM, so the taps are split over CTA TYPES: a type owns one 32-channel chunk of `in` and
// up to four kw; a CTA of that type marches down the class rows (rows h = D*t + rho of one residue class: the dilated
// filter is dense along a class) of its share of (image, class, column strip) items.  Per step (one dout row t) and kw:
//       A = 4 consecutive class rows of `in` out of the last 8 (two groups: M = 4 x 32 k),   B = the dout row (N columns)
// -> block r of a group is tap kh = 3 - r + 4*group (s < 0; mirrored for s > 0); 7 of the 8 blocks are taps.  One TMEM
// accumulator per (kw, group) for the whole launch, written once as partials that a fold kernel sums per type in a
// fixed order (deterministic).  The ring keeps every `in` row until the seven later steps have used it; three mirror
// slots behind the ring keep any 4 consecutive rows contiguous.
// Warps: 0 = TMA producer, 4 = MMA issuer, 0-3 write the accumulators out at the end.
#include "dd_common.cuh"
#include "tma_host.h"
#include "umma.cuh"

namespace {

constexpr int KPX = 128;                   // dout pixels per strip = K extent of a step
constexpr int XTILE_PX = 170;              // 128 + 6 * 7
constexpr int XS = 22 * 512;               // `in` row tile pitch (170 px x 64 B = 10880, rounded up to the swizzle period)
constexpr int DHALF = KPX * 64;            // one 32-channel half of a dout row
constexpr int WGD_THREADS = 160;

struct WgdGeo {
  int B, Ho, Wo;                // dout size (the `in` size only enters through the tensor map)
  int KT, D, sign, off;
  int NG;                       // row groups per step: 2 for 7 taps, 1 for 3
  int RX, RD;                   // ring depths (`in` rows, dout rows); RX - RD = rows a step still needs = 4*NG - 1
  int nchunks, nkwsets, kws;    // types = nchunks * nkwsets; kw per set (the last set may hold fewer)
  int ctas_per_type;
  int strips, segs, seg_rows;   // items of a type: (b, rho, seg, strip)
  int items;
};

struct WgdBars {
  uint64_t full[8], done[8], fin;
  uint32_t tmem_base;
};

struct WItem { int b, rho, ta, tb, w0; };
__device__ __forceinline__ WItem wdecode(const WgdGeo& g, int it) {
  WItem o;
  const int strip = it % g.strips;
  int rest = it / g.strips;
  const int seg = rest % g.segs;
  rest /= g.segs;
  o.rho = rest % g.D;
  o.b = rest / g.D;
  const int T = (g.Ho - o.rho + g.D - 1) / g.D;
  o.ta = seg * g.seg_rows;
  o.tb = min(T, o.ta + g.seg_rows);
  o.w0 = strip * KPX;
  return o;
}

template <int N>
__global__ void __launch_bounds__(WGD_THREADS, 1) conv_dil_wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                           const __grid_constant__ CUtensorMap map_dy,
                                                                           float* __restrict__ partial, const WgdGeo g) {
  constexpr int DS = (N / 32) * DHALF;                       // dout ring slot
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_x = smem;
  uint8_t* s_d = smem + (g.RX + 3) * XS;
  WgdBars* bars = reinterpret_cast<WgdBars*>(s_d + g.RD * DS);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int type = blockIdx.x % (g.nchunks * g.nkwsets), slot_in_type = blockIdx.x / (g.nchunks * g.nkwsets);
  const int chunk = type % g.nchunks, kwset = type / g.nchunks;
  const int kw0 = kwset * g.kws, nkw = min(g.kws, g.KT - kw0);
  const int KT = g.KT;

  if (tid == 0) {
    for (int i = 0; i < g.RD; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->done[i], 1); }
    umma::mbar_init(&bars->fin, 1);
    umma::fence_mbar_init();
  }
  if (warp == 4) umma::tmem_alloc(&bars->tmem_base, 512);
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp == 0) {
    // =========================== producer (one thread): stage = {one `in` class row, one dout class row} ==========
    if (lane == 0) {
      umma::tma_prefetch_desc(&map_x);
      umma::tma_prefetch_desc(&map_dy);
      uint32_t gs = 0;
      for (int it = slot_in_type; it < g.items; it += g.ctas_per_type) {
        const WItem im = wdecode(g, it);
        if (im.tb <= im.ta) continue;
        const int nst = im.tb - im.ta + KT - 1;
        const int x0 = im.w0 + g.off - (g.sign < 0 ? (KT - 1) * g.D : 0);
        for (int i = 0; i < nst; ++i, ++gs) {
          const uint32_t sd = gs % g.RD, sx = gs % g.RX;
          umma::mbar_wait(&bars->done[sd], ((gs / g.RD) & 1) ^ 1);        // step gs - RD finished: dout slot and `in` slot free
          const int u = g.sign < 0 ? im.ta - (KT - 1) + i : im.ta + i;        // `in` class row of this stage
          const int t = im.ta + i - (KT - 1);                                  // dout class row processed at this stage
          const bool has_d = t >= im.ta;
          const uint32_t copies = sx < 3 ? 2u : 1u;
          umma::mbar_expect_tx(&bars->full[sd], copies * (uint32_t)(XTILE_PX * 64) + (has_d ? (uint32_t)DS : 0u));
          const int xrow = g.D * u + im.rho + g.off;
          umma::tma_load_4d(umma::smem_u32(s_x) + sx * XS, &map_x, chunk * 32, x0, xrow, im.b, &bars->full[sd]);
          if (copies == 2) umma::tma_load_4d(umma::smem_u32(s_x) + (g.RX + sx) * XS, &map_x, chunk * 32, x0, xrow, im.b, &bars->full[sd]);
          if (has_d) {
#pragma unroll
            for (int hh = 0; hh < N / 32; ++hh)
              umma::tma_load_4d(umma::smem_u32(s_d) + sd * DS + hh * DHALF, &map_dy, hh * 32, im.w0, g.D * t + im.rho, im.b, &bars->full[sd]);
          }
        }
      }
    }
  } else if (warp == 4) {
    // =========================== MMA issuer ===================================================================
    constexpr uint32_t idesc = umma::make_idesc_bf16(128, N, true, true);
    constexpr uint32_t ab_hi = umma::desc_hi_sw64(512);
    const uint32_t x_lo0 = umma::desc_lo(umma::smem_u32(s_x), XS);         // LBO: next `in` row = next 32-k block of M
    const uint32_t d_lo0 = umma::desc_lo(umma::smem_u32(s_d), DHALF);      // LBO: next 32-channel half of N
    uint32_t gs = 0, fresh = 1;
    for (int it = slot_in_type; it < g.items; it += g.ctas_per_type) {
      const WItem im = wdecode(g, it);
      if (im.tb <= im.ta) continue;
      const int nst = im.tb - im.ta + KT - 1;
      for (int i = 0; i < nst; ++i, ++gs) {
        const uint32_t sd = gs % g.RD;
        umma::mbar_wait(&bars->full[sd], (gs / g.RD) & 1);
        umma::tc_fence_after_sync();
        const uint32_t first = fresh;
        if (i >= KT - 1) fresh = 0;
        if (umma::elect_one()) {
          if (i >= KT - 1) {
            const uint32_t b0 = d_lo0 + ((sd * DS) >> 4);
            for (int j = 0; j < nkw; ++j) {
              const int kw = kw0 + j;
              const uint32_t pxoff = (uint32_t)((g.sign < 0 ? (KT - 1 - kw) : kw) * g.D) * 64u;
              for (int gi = 0; gi < g.NG; ++gi) {
                // group gi = the 4 ring rows ending 4*gi rows before the newest one (3 mirror slots keep them contiguous)
                const uint32_t start = (gs + (uint32_t)g.RX * 4u - 3u - 4u * gi) % g.RX;
                const uint32_t a0 = x_lo0 + ((start * XS + pxoff) >> 4);
                const uint32_t d_t = tmem + (j * g.NG + gi) * N;
#pragma unroll
                for (int ks = 0; ks < KPX / 16; ++ks)
                  umma::mma_bf16_lohi(d_t, a0 + ((ks * 1024) >> 4), ab_hi, b0 + ((ks * 1024) >> 4), ab_hi, idesc,
                                      (first && ks == 0) ? 0u : 1u);
              }
            }
          }
          umma::mma_commit(&bars->done[sd]);
        }
        __syncwarp();
      }
    }
    if (umma::elect_one()) umma::mma_commit(&bars->fin);
    __syncwarp();
  }
  // =========================== epilogue: TMEM -> this CTA's partials [kw][kh][k 32][n] ===================================
  __syncwarp();
  if (warp < 4) {
    umma::mbar_wait_sleep(&bars->fin, 0);
    umma::tc_fence_after_sync();
    const int r = warp;                                    // TMEM lane quarter = row r of the group; lane = channel k
    float* outp = partial + (size_t)blockIdx.x * (g.kws * KT * 32 * N);
    for (int j = 0; j < nkw; ++j)
      for (int gi = 0; gi < g.NG; ++gi) {
        const int kh = g.sign < 0 ? 3 - r + 4 * gi : (KT - 1) - 3 + r - 4 * gi;
#pragma unroll
        for (int c0 = 0; c0 < N; c0 += 32) {
          uint32_t v[32];
          umma::tmem_ld_32x32(tmem + ((uint32_t)(r * 32) << 16) + (j * g.NG + gi) * N + c0, v);
          umma::tmem_ld_wait();
          if (kh >= 0 && kh < KT) {
            float4* dst = reinterpret_cast<float4*>(outp + ((size_t)(j * KT + kh) * 32 + lane) * N + c0);
#pragma unroll
            for (int g4 = 0; g4 < 8; ++g4)
              dst[g4] = make_float4(__uint_as_float(v[4 * g4]), __uint_as_float(v[4 * g4 + 1]), __uint_as_float(v[4 * g4 + 2]),
                                    __uint_as_float(v[4 * g4 + 3]));
          }
        }
      }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) umma::tmem_dealloc(tmem, 512);
}

// dw(n, k, kh, kw) at dw[n*sn + k*sk + kh*KT + kw] = sum over the CTAs of the type that owns (chunk of k, kw), fixed order
__global__ void wgd_fold_kernel(const float* __restrict__ partial, float* __restrict__ dw, WgdGeo g, int N, int Kreal, int Nreal,
                                long long sn, long long sk) {
  const int ntypes = g.nchunks * g.nkwsets;
  const long long total = (long long)g.nchunks * 32 * g.KT * g.KT * N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i % N);
    long long rest = i / N;
    const int k32 = (int)(rest % 32); rest /= 32;
    const int kh = (int)(rest % g.KT); rest /= g.KT;
    const int kw = (int)(rest % g.KT);
    const int chunk = (int)(rest / g.KT);
    const int k = chunk * 32 + k32;
    if (k >= Kreal || n >= Nreal) continue;
    const int kwset = kw / g.kws, j = kw - kwset * g.kws;
    const int type = kwset * g.nchunks + chunk;
    float s = 0.f;
    for (int c = 0; c < g.ctas_per_type; ++c) {
      const size_t cta = (size_t)c * ntypes + type;
      s += partial[cta * ((size_t)g.kws * g.KT * 32 * N) + ((size_t)(j * g.KT + kh) * 32 + k32) * N + n];
    }
    dw[n * sn + k * sk + (long long)kh * g.KT + kw] = s;
  }
}

WgdGeo make_geo(int B, int Ho, int Wo, int K, int N, int KT, int D, int sign, int off) {
  WgdGeo g = {};
  g.B = B; g.Ho = Ho; g.Wo = Wo; g.KT = KT; g.D = D; g.sign = sign; g.off = off;
  g.NG = KT > 4 ? 2 : 1;
  g.RD = 3;
  g.RX = g.RD + 4 * g.NG - 1;                      // a row is needed by the 4*NG - 1 steps after its own
  g.nchunks = K / 32;
  const int max_combos = 512 / (g.NG * N);         // accumulators of N columns that fit TMEM
  g.kws = KT < max_combos ? KT : max_combos;
  if (g.kws > 4 && KT > 4 && N > 32) g.kws = 4;
  g.nkwsets = (KT + g.kws - 1) / g.kws;
  const int ntypes = g.nchunks * g.nkwsets;
  g.ctas_per_type = dd::kSMs / ntypes;
  g.strips = (Wo + KPX - 1) / KPX;
  const int Tmax = (Ho + D - 1) / D;
  // enough items per type to balance its CTAs: split the class rows into segments when the classes are few (D = 1)
  g.seg_rows = Tmax;
  while ((long long)B * D * g.strips * ((Tmax + g.seg_rows - 1) / g.seg_rows) < 6LL * g.ctas_per_type && g.seg_rows > 16) g.seg_rows = (g.seg_rows + 1) / 2;
  g.segs = (Tmax + g.seg_rows - 1) / g.seg_rows;
  const int Tmin = Ho / D;                          // the class with the fewest rows: no segment may be empty for it
  while (g.segs > 1 && (g.segs - 1) * g.seg_rows >= Tmin) { --g.segs; g.seg_rows = (Tmax + g.segs - 1) / g.segs; }
  g.items = B * D * g.segs * g.strips;
  if (g.items < g.ctas_per_type) g.ctas_per_type = g.items;      // every CTA must accumulate at least one item
  return g;
}

}  // namespace

namespace dd {

bool conv_dil_wgrad_tc_supported(int K, int N, int KT, int D) {
  return (KT == 3 || KT == 7) && D >= 1 && D <= 7 && (K == 32 || K == 64 || K == 96) && (N == 32 || N == 64);
}

size_t conv_dil_wgrad_tc_ws_bytes(int K, int N, int KT) {
  (void)K;
  return (size_t)kSMs * 4 * KT * 32 * N * sizeof(float) * (N == 32 && KT == 7 ? 2 : 1) + 256;
}

// `in` [B,Hi,Wi,K] and `dout` [B,Ho,Wo,N] bf16 NHWC; dw: torch-layout fp32 weights with the produced / gathered channel
// strides (sn, sk) -- the same convention as dd::conv_dil_tc.
int conv_dil_wgrad_tc(const void* in, const void* dout, float* dw, long long sn, long long sk, void* ws, size_t ws_bytes, int B,
                      int Hi, int Wi, int Ho, int Wo, int K, int N, int KT, int D, int sign, int off, cudaStream_t st, int Kreal,
                      int Nreal) {
  // Kreal < K / Nreal < N: zero-padded pixels; only dw[n < Nreal][k < Kreal] exists
  if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(dout)) & 15) != 0)
    return fail(DD_ERR_ALIGNMENT, "conv_dil_wgrad_tc: operands must be 16-byte aligned");
  WgdGeo g = make_geo(B, Ho, Wo, K, N, KT, D, sign, off);
  const int grid = g.ctas_per_type * g.nchunks * g.nkwsets;
  const size_t need = (size_t)grid * g.kws * KT * 32 * N * sizeof(float);
  if (ws_bytes < need) return fail(DD_ERR_WORKSPACE, "conv_dil_wgrad_tc: workspace %zu < %zu", ws_bytes, need);
  CUtensorMap mx, md;
  char msg[256];
  if (tma_map_nhwc_sw64(&mx, in, B, Hi, Wi, K, XTILE_PX, 1, msg, sizeof msg)) return fail(DD_ERR_UNSUPPORTED, "conv_dil_wgrad_tc: in: %s", msg);
  if (tma_map_nhwc_sw64(&md, dout, B, Ho, Wo, N, KPX, 1, msg, sizeof msg)) return fail(DD_ERR_UNSUPPORTED, "conv_dil_wgrad_tc: dout: %s", msg);
  const int smem = (g.RX + 3) * XS + g.RD * (N / 32) * DHALF + 256;
  if (N == 64) {
    if (int e = set_smem(conv_dil_wgrad_tc_kernel<64>, smem, Carveout::kMaxShared, "conv_dil_wgrad_tc")) return e;
    conv_dil_wgrad_tc_kernel<64><<<grid, WGD_THREADS, smem, st>>>(mx, md, (float*)ws, g);
  } else {
    if (int e = set_smem(conv_dil_wgrad_tc_kernel<32>, smem, Carveout::kMaxShared, "conv_dil_wgrad_tc")) return e;
    conv_dil_wgrad_tc_kernel<32><<<grid, WGD_THREADS, smem, st>>>(mx, md, (float*)ws, g);
  }
  if (int err = check_launch("conv_dil_wgrad_tc")) return err;
  const long long total = (long long)g.nchunks * 32 * KT * KT * N;
  wgd_fold_kernel<<<(int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184), 256, 0, st>>>((const float*)ws, dw, g, N, Kreal, Nreal, sn, sk);
  return check_launch("conv_dil_wgrad_fold");
}

}  // namespace dd
