// Weight gradients of the 32->32 3x3 encoder convs (c2: stride 1, c3: stride 2; components.py:20-21) on the 5th-gen
// tensor cores, fed by whole-pixel TMA boxes through a rolling row ring.
//
//   dW[co][ci][kh][kw] = sum_{b,h,w} x[b, S*h+kh-1, S*w+kw-1, ci] * dy[b,h,w,co],     db[co] = sum dy[b,h,w,co]
//
// The contraction runs over PIXELS (K), the channels are the M / N index: an NHWC row "[pixel][32 ch]" (64-byte rows) is
// exactly the canonical MN-major 64-byte-swizzle operand layout (atoms of 8 K-rows x 64 B).  So every x row and every dy
// row of a 128-pixel column strip is ONE TMA box of whole pixels (CU_TENSOR_MAP_SWIZZLE_64B): full 32-byte sectors from
// L2 and one request per row, where round 1's four [pixel][8 ch] boxes per row (16-byte inner extent) read half sectors
// and four times the requests (ncu: L2 75 % busy at 36 % of DRAM bandwidth).  The horizontal tap kw is a shift of the A
// start address by kw pixels (kw * 64 B): the swizzle follows the absolute shared-memory address, so any start works
// with base_offset 0 (tools/tma_sw64_mn_probe.cu, profiles/r2_tma_sw64_mn_probe.txt).  Stride 2 loads the even and the
// odd pixels of an x row as two planes with a TMA element stride of 2 (same probe).
//
// A CTA owns a column strip and marches DOWN the image: per step it takes 2 new x rows and NQ new dy rows (stride 1:
// NQ = 2; stride 2: NQ = 1) and issues, per kw, 8 tcgen05.mma (K = 16 pixels each) of
//       A = the 4 x rows  S*h-1 .. S*h+2   (M = 4 x 32 ci, LBO = the ring's row pitch)
//       B = the NQ dy rows h .. h+NQ-1      (N = NQ x 32 co)
// into one TMEM accumulator per kw that lives for the whole launch.  Block (r, q) of D is tap kh = r - S*q; 6 of 8
// (stride 2: 3 of 4) blocks are taps, the others are never read.  Each x row is loaded ONCE per strip (round 1: 1.5x):
// the ring keeps the two rows a step shares with the next one.  The 4 rows of A must be contiguous, so the ring has two
// extra slots at its end that mirror slots 0-1 (the rows that land there are loaded twice, from L2).
// One stage = {2 x rows, NQ dy rows}, one mbarrier pair per stage: the MMA thread waits once per step.
// Warps: 0 = TMA producer (one thread), 1-2 = bias gradient (sum the dy rows out of shared memory, swizzle-aware),
// 4 = MMA issuer; 0-3 write the accumulators out once, as [cta][q][tap][ci][co] partials folded in a fixed order.
#include "dd_common.cuh"
#include "tma_host.h"
#include "umma.cuh"

namespace {

constexpr int C = 32;
constexpr int KP = 128;               // dy pixels of a strip = K extent of a step (8 x K16)
constexpr int DROW = KP * 64;         // dy row tile [128 px][32 ch] bf16: 8192 B
constexpr int XPAD = 17 * 512;        // x row tile pitch: 130 (129) pixels of 64 B, rounded up to the 512-byte swizzle period
constexpr int WGT_THREADS = 160;

template <int STRIDE>
struct WG {
  static constexpr int NQ = STRIDE == 1 ? 2 : 1;                     // dy rows per step
  static constexpr int XS = STRIDE == 1 ? XPAD : DROW + XPAD;        // x ring slot = one row (stride 2: [even plane | odd plane])
  static constexpr int NS = STRIDE == 1 ? 6 : 4;                     // stages in the ring
  static constexpr int X_BYTES = (2 * NS + 2) * XS;                  // + the two mirror slots
  static constexpr int D_BYTES = NS * NQ * DROW;
  static constexpr int SMEM = X_BYTES + D_BYTES + 256;
  static constexpr int HSEG = STRIDE == 1 ? 64 : 32;                 // dy rows per work item
  static constexpr int N = 32 * NQ;
  static constexpr int PARTIAL = NQ * 9 * C * C;                     // floats per CTA
  static constexpr uint32_t XROW_TX = STRIDE == 1 ? 130 * 64 : (128 + 128 + 1) * 64;   // bytes one x row's boxes deliver
  static_assert(X_BYTES % 512 == 0 && XS % 512 == 0, "tiles must sit on the 64-byte-swizzle period");
  static_assert(SMEM <= 227 * 1024, "shared memory");
};

struct RingBars {
  uint64_t full[8], empty[8], done;
  uint32_t tmem_base;
};

template <int STRIDE>
__global__ void __launch_bounds__(WGT_THREADS, 1) conv3x3_c32_wgrad_ring_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                                const __grid_constant__ CUtensorMap map_x1,
                                                                                const __grid_constant__ CUtensorMap map_dy,
                                                                                float* __restrict__ partial,
                                                                                float* __restrict__ db_partial, int B, int Ho,
                                                                                int Wo) {
  using G = WG<STRIDE>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_x = smem;
  uint8_t* s_d = smem + G::X_BYTES;
  RingBars* bars = reinterpret_cast<RingBars*>(smem + G::X_BYTES + G::D_BYTES);
  __shared__ float s_db[2][C];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wtiles = (Wo + KP - 1) / KP;
  const int hsegs = (Ho + G::HSEG - 1) / G::HSEG;
  const int items = B * wtiles * hsegs;

  if (tid == 0) {
    for (int i = 0; i < G::NS; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 3); }
    umma::mbar_init(&bars->done, 1);
    umma::fence_mbar_init();
  }
  if (warp == 4) umma::tmem_alloc(&bars->tmem_base, 256);
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp == 0) {
    // =========================== producer: one thread, TMA ========================================
    // Out-of-image rows / columns (the conv padding, the ragged last strip, the odd last dy row of a stride-1 item) are
    // zero-filled by the TMA unit and count towards the transaction bytes.
    if (lane == 0) {
      umma::tma_prefetch_desc(&map_x);
      umma::tma_prefetch_desc(&map_dy);
      if (STRIDE == 2) umma::tma_prefetch_desc(&map_x1);
      uint32_t g = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
        const int h0 = hs * G::HSEG, w0 = wt * KP;
        const int rows = min(G::HSEG, Ho - h0);
        const int P = (rows + G::NQ - 1) / G::NQ;                  // steps of this item; stages 0..P
        for (int i = 0; i <= P; ++i, ++g) {
          const uint32_t s = g % G::NS;
          uint64_t* full = &bars->full[s];
          umma::mbar_wait(&bars->empty[s], ((g / G::NS) & 1) ^ 1);
          const uint32_t copies = s == 0 ? 2u : 1u;
          umma::mbar_expect_tx(full, copies * 2u * G::XROW_TX + (i < P ? (uint32_t)(G::NQ * DROW) : 0u));
          const int xr0 = STRIDE * h0 - 1 + 2 * i;                 // first of the stage's two x rows
          for (uint32_t cp = 0; cp < copies; ++cp) {
            const uint32_t dst0 = umma::smem_u32(s_x) + (cp ? 2 * G::NS : 2 * s) * G::XS;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const uint32_t dst = dst0 + r * G::XS;
              if (STRIDE == 1) {
                umma::tma_load_4d(dst, &map_x, 0, w0 - 1, xr0 + r, b, full);
              } else {
                umma::tma_load_4d(dst, &map_x, 0, 2 * w0, xr0 + r, b, full);                       // even pixels 2w0, 2w0+2, ...
                umma::tma_load_4d(dst + DROW, &map_x, 0, 2 * w0 - 1, xr0 + r, b, full);            // odd pixels 2w0-1, ... (128)
                umma::tma_load_4d(dst + DROW + KP * 64, &map_x1, 0, 2 * w0 + 2 * KP - 1, xr0 + r, b, full);   // ... and the 129th
              }
            }
          }
          if (i < P) {
#pragma unroll
            for (int q = 0; q < G::NQ; ++q)
              umma::tma_load_4d(umma::smem_u32(s_d) + (s * G::NQ + q) * DROW, &map_dy, 0, w0, h0 + G::NQ * i + q, b, full);
          }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // =========================== bias gradient: db[co] = sum of dy over pixels ======================
    // The dy rows are in shared memory anyway.  Lane = (pixel lane >> 2, 16-byte channel chunk lane & 3): a warp reads 8
    // whole pixels (512 contiguous bytes) per instruction; the chunk's physical position inside its 64-byte row is
    // chunk ^ ((pixel >> 1) & 3) (64-byte swizzle: address bits 4-5 ^= bits 7-8).
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    const int chunk = lane & 3;
    const int px0 = (warp - 1) * 64 + (lane >> 2);          // this warp's half of the strip
    uint32_t g = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(G::HSEG, Ho - hs * G::HSEG);
      const int P = (rows + G::NQ - 1) / G::NQ;
      for (int i = 0; i <= P; ++i, ++g) {
        const uint32_t s = g % G::NS;
        umma::mbar_wait_sleep(&bars->full[s], (g / G::NS) & 1);
        if (i < P) {
          const uint32_t base = umma::smem_u32(s_d) + s * G::NQ * DROW;
#pragma unroll
          for (int q = 0; q < G::NQ; ++q)
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              const int p = px0 + 8 * t;
              uint32_t w0, w1, w2, w3;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3)
                           : "r"(base + q * DROW + p * 64 + ((chunk ^ ((p >> 1) & 3)) << 4)));
              const uint32_t ww[4] = {w0, w1, w2, w3};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ww[k]));
                acc[2 * k] += f.x;
                acc[2 * k + 1] += f.y;
              }
            }
        }
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&bars->empty[s]);
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float v = acc[k];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      if (lane < 4) s_db[warp - 1][chunk * 8 + k] = v;
    }
  } else if (warp == 4) {
    // =========================== MMA issuer (whole warp loops, elected lane issues) ================
    constexpr uint32_t idesc = umma::make_idesc_bf16(128, G::N, true, true);
    constexpr uint32_t ab_hi = ((512u >> 4) & 0x3FFF) | (1u << 14) | (4u << 29);     // SBO = 512 B (next 8-pixel group), SWIZZLE_64B
    const uint32_t x_lo0 = umma::desc_lo(umma::smem_u32(s_x), G::XS);                // LBO = next x row (next 32-ci block of M)
    const uint32_t d_lo0 = umma::desc_lo(umma::smem_u32(s_d), DROW);                 // LBO = next dy row (next 32-co block of N)
    uint32_t g = 0, waited = 0, fresh = 1;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(G::HSEG, Ho - hs * G::HSEG);
      const int P = (rows + G::NQ - 1) / G::NQ;
      for (int j = 0; j < P; ++j, ++g) {
        // step j reads the x rows of stages g and g + 1 and the dy rows of stage g
        for (; waited < g + 2; ++waited) umma::mbar_wait(&bars->full[waited % G::NS], (waited / G::NS) & 1);
        umma::tc_fence_after_sync();
        const uint32_t s = g % G::NS;
        const uint32_t a0 = x_lo0 + ((2 * s * G::XS) >> 4);
        const uint32_t b0 = d_lo0 + ((s * G::NQ * DROW) >> 4);
        if (umma::elect_one()) {
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            // stride 1: x column w+kw-1 = tile pixel (w-w0)+kw.  stride 2: kw 0 -> odd[i], 1 -> even[i], 2 -> odd[i+1]
            const uint32_t koff = STRIDE == 1 ? kw * 64 : (kw == 1 ? 0 : DROW + (kw == 2 ? 64 : 0));
#pragma unroll
            for (int ks = 0; ks < KP / 16; ++ks)
              umma::mma_bf16_lohi(tmem + kw * 64, a0 + ((koff + ks * 1024) >> 4), ab_hi, b0 + ((ks * 1024) >> 4), ab_hi, idesc,
                                  (fresh && ks == 0) ? 0u : 1u);
          }
          umma::mma_commit(&bars->empty[s]);
          if (j == P - 1) umma::mma_commit(&bars->empty[(g + 1) % G::NS]);     // the item's last stage holds x rows only
        }
        fresh = 0;
        __syncwarp();
      }
      ++g;            // the x-only stage
    }
    if (umma::elect_one()) umma::mma_commit(&bars->done);
    __syncwarp();
  }
  // =========================== epilogue: TMEM -> per-CTA partials (warps 0..3) ========================
  __syncwarp();
  if (warp < 4) {
    umma::mbar_wait_sleep(&bars->done, 0);
    umma::tc_fence_after_sync();
    const int r = warp;                      // TMEM lane quarter = x row r of the group; lane = ci
    float* out = partial + (size_t)blockIdx.x * G::PARTIAL;
#pragma unroll 1
    for (int kw = 0; kw < 3; ++kw) {
#pragma unroll 1
      for (int q = 0; q < G::NQ; ++q) {
        uint32_t v[32];
        umma::tmem_ld_32x32(tmem + ((uint32_t)(r * 32) << 16) + kw * 64 + q * 32, v);
        umma::tmem_ld_wait();
        const int kh = r - STRIDE * q;
        if (kh >= 0 && kh <= 2) {
          float4* dst = reinterpret_cast<float4*>(out + (size_t)q * 9 * C * C + ((kh * 3 + kw) * C + lane) * C);
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
  if (tid < C) db_partial[(size_t)blockIdx.x * C + tid] = s_db[0][tid] + s_db[1][tid];
  if (warp == 4) umma::tmem_dealloc(tmem, 256);
}

// dw[co][ci][tap] = sum over CTAs and their q slots (nslots = CTAs x NQ) of partial[slot][tap][ci][co];
// db[co] = sum of the per-CTA sums -- fixed order: deterministic
__global__ void wgrad_ring_reduce_kernel(const float* __restrict__ partial, int nslots, const float* __restrict__ dbp, int ndb,
                                         float* __restrict__ dw, float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 9 * C * C) {
    float s = 0.f;
    for (int blk = 0; blk < nslots; ++blk) s += partial[(size_t)blk * (9 * C * C) + i];
    const int co = i & 31, ci = (i >> 5) & 31, tap = i >> 10;
    dw[(co * C + ci) * 9 + tap] = s;
  } else if (i < 9 * C * C + C) {
    const int co = i - 9 * C * C;
    float s = 0.f;
    for (int blk = 0; blk < ndb; ++blk) s += dbp[(size_t)blk * C + co];
    db[co] = s;
  }
}

// ================================================================================================
// Weight gradient of the first conv (3 -> 32, components.py:19,41), stitch (and the ToTensor /255 of raw camera
// bytes) folded into the loads:
//   dW[co][c][kh][kw] = sum_{b,h,w} in[b,c,h+kh-1,w+kw-1] * dy[b,h,w,co],   db[co] = sum dy[b,h,w,co]
// Same march as above (pixels = K, a CTA walks down a 128-pixel column strip), with
//   B = 4 dy rows per step, whole-pixel TMA boxes, 64-byte swizzle (N = 4 x 32 co = 128);
//   A = 8 x rows of "tap-packed" pixels built by four converter warps from the fp32 / u8 image: 16 channels per pixel,
//       channel j = kw*3 + c (j < 9) = in[c][p + kw - 1], j = 9 is 1.0 (-> the bias gradient rides along), rest 0 --
//       the three horizontal taps sit in the M dimension instead of costing three MMAs.  SWIZZLE_NONE MN-major:
//       two [pixel][8 ch] planes per row.  Each image row is read and converted ONCE per strip (thread = pixel column;
//       the left / right neighbours come from the adjacent lanes by shuffle), round 1 re-read 8 rows per 6.
// Block (r, q) of D = tap kh = r - q.  One stage = {4 x rows, 4 dy rows}; a step reads the x rows of two stages.
// Warps 0-3 converters (+ the final epilogue), 4 = MMA issuer, 5 = TMA producer for dy.
// ================================================================================================
constexpr int C1_RB = 4;                       // dy rows (and new x rows) per stage
constexpr int C1_NS = 4;                       // stages
constexpr int C1_PL = KP * 16;                 // one [128 px][8 ch] plane: 2048 B
constexpr int C1_XROW = 2 * C1_PL;             // x ring slot = one row = two planes
constexpr int C1_XBYTES = (C1_RB * C1_NS + C1_RB) * C1_XROW;     // + mirror of stage slot 0
constexpr int C1_DBYTES = C1_NS * C1_RB * DROW;
constexpr int C1_SMEM = C1_XBYTES + C1_DBYTES + 256;
constexpr int C1_HSEG = 64;
constexpr int C1_PARTIAL = C1_RB * 3 * 10 * C;  // floats per CTA: [q][kh][j][co]
constexpr int C1_THREADS = 192;
static_assert(C1_SMEM <= 227 * 1024, "shared memory");

template <bool IS_VIEWS, typename TIN>
__global__ void __launch_bounds__(C1_THREADS, 1) conv_c1_wgrad_ring_kernel(const TIN* __restrict__ in,
                                                                           const __grid_constant__ CUtensorMap map_dy,
                                                                           float* __restrict__ partial, int B, int H, int Wm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_x = smem;
  uint8_t* s_d = smem + C1_XBYTES;
  RingBars* bars = reinterpret_cast<RingBars*>(smem + C1_XBYTES + C1_DBYTES);
  __shared__ float s_lut[256];
  dd::c1_fill_lut(s_lut);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wtiles = (Wm + KP - 1) / KP;
  const int hsegs = (H + C1_HSEG - 1) / C1_HSEG;
  const int items = B * wtiles * hsegs;

  if (tid == 0) {
    // per stage: 128 converter arrivals (planes written and fenced) + the producer's expect_tx arrival (dy rows)
    for (int i = 0; i < C1_NS; ++i) { umma::mbar_init(&bars->full[i], 129); umma::mbar_init(&bars->empty[i], 1); }
    umma::mbar_init(&bars->done, 1);
    umma::fence_mbar_init();
  }
  if (warp == 4) umma::tmem_alloc(&bars->tmem_base, 128);
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp < 4) {
    // =========================== converters: thread = pixel column of the strip ====================
    // The image loads of stage g + 1 are issued BEFORE stage g is packed and stored (register double buffer): a stage's
    // global-load latency is hidden behind the previous stage's work instead of sitting on the ring's critical path.
    const int Wv = IS_VIEWS ? Wm / 6 : Wm;
    const size_t cstride = (size_t)H * Wv;
    const bool has_edge = lane == 0 || lane == 31;
    struct Cur { int it, i, P, xr0; size_t coff, eoff; bool cok, eok, valid; };
    auto open_item = [&](Cur& c) {
      c.valid = c.it < items;
      if (!c.valid) return;
      const int wt = c.it % wtiles, hs = (c.it / wtiles) % hsegs, b = c.it / (wtiles * hsegs);
      const int h0 = hs * C1_HSEG, w0 = wt * KP;
      c.P = (min(C1_HSEG, H - h0) + C1_RB - 1) / C1_RB;
      c.i = 0;
      c.xr0 = h0 - 1;
      // this thread's column, and for the warp's edge lanes the column just outside the warp (lane 0: left, 31: right)
      const int col = w0 + tid;
      const int ecol = lane == 0 ? col - 1 : col + 1;
      auto col_off = [&](int cc, bool& ok) -> size_t {
        ok = cc >= 0 && cc < Wm;
        const int c2 = ok ? cc : 0;
        if (IS_VIEWS) {
          const int j = c2 / Wv, w = c2 - j * Wv;
          return (((size_t)b * 6 + dd::view_of_slot(j)) * 3) * cstride + w;
        }
        return ((size_t)b * 3) * cstride + c2;
      };
      c.coff = col_off(col, c.cok);
      c.eoff = col_off(ecol, c.eok);
    };
    auto advance = [&](Cur& c) {
      if (c.i < c.P) { ++c.i; c.xr0 += C1_RB; return; }
      c.it += gridDim.x;
      open_item(c);
    };
    auto load_rows = [&](const Cur& c, TIN (&v)[C1_RB][3], TIN (&e)[C1_RB][3]) {      // raw values; 0 where there is no pixel
#pragma unroll
      for (int r = 0; r < C1_RB; ++r) {
        const int row = c.xr0 + r;
        const bool row_ok = row >= 0 && row < H;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          v[r][ch] = (row_ok && c.cok) ? __ldg(in + c.coff + ch * cstride + (size_t)row * Wv) : TIN(0);
          e[r][ch] = (has_edge && row_ok && c.eok) ? __ldg(in + c.eoff + ch * cstride + (size_t)row * Wv) : TIN(0);
        }
      }
    };
    Cur cur;
    cur.it = blockIdx.x;
    open_item(cur);
    TIN rv[C1_RB][3], re[C1_RB][3], vn[C1_RB][3], en[C1_RB][3];
    if (cur.valid) load_rows(cur, rv, re);
    uint32_t g = 0;
    while (cur.valid) {
      Cur nxt = cur;
      advance(nxt);
      if (nxt.valid) load_rows(nxt, vn, en);
      const uint32_t s = g % C1_NS;
      umma::mbar_wait(&bars->empty[s], ((g / C1_NS) & 1) ^ 1);
      float v[C1_RB][3], e[C1_RB][3];
#pragma unroll
      for (int r = 0; r < C1_RB; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) { v[r][c] = dd::c1_cvt<TIN>(rv[r][c], s_lut); e[r][c] = dd::c1_cvt<TIN>(re[r][c], s_lut); }
#pragma unroll
      for (int r = 0; r < C1_RB; ++r) {
        float lf[3], rt[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          lf[c] = __shfl_up_sync(0xffffffffu, v[r][c], 1);
          rt[c] = __shfl_down_sync(0xffffffffu, v[r][c], 1);
          if (lane == 0) lf[c] = e[r][c];
          if (lane == 31) rt[c] = e[r][c];
        }
        uint4 lo, hi;
        __nv_bfloat162 t;
        t = __floats2bfloat162_rn(lf[0], lf[1]);           lo.x = *reinterpret_cast<uint32_t*>(&t);
        t = __floats2bfloat162_rn(lf[2], v[r][0]);         lo.y = *reinterpret_cast<uint32_t*>(&t);
        t = __floats2bfloat162_rn(v[r][1], v[r][2]);       lo.z = *reinterpret_cast<uint32_t*>(&t);
        t = __floats2bfloat162_rn(rt[0], rt[1]);           lo.w = *reinterpret_cast<uint32_t*>(&t);
        t = __floats2bfloat162_rn(rt[2], 1.0f);            hi.x = *reinterpret_cast<uint32_t*>(&t);
        hi.y = hi.z = hi.w = 0u;
        uint8_t* dst = s_x + (size_t)(C1_RB * s + r) * C1_XROW + tid * 16;
        *reinterpret_cast<uint4*>(dst) = lo;
        *reinterpret_cast<uint4*>(dst + C1_PL) = hi;
        if (s == 0) {                                    // mirror of stage slot 0 behind the ring's last slot
          uint8_t* dm = s_x + (size_t)(C1_RB * C1_NS + r) * C1_XROW + tid * 16;
          *reinterpret_cast<uint4*>(dm) = lo;
          *reinterpret_cast<uint4*>(dm + C1_PL) = hi;
        }
      }
      umma::fence_proxy_async_smem();        // generic-proxy stores -> visible to the tensor core's reads
      umma::mbar_arrive(&bars->full[s]);
      ++g;
#pragma unroll
      for (int r = 0; r < C1_RB; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) { rv[r][c] = vn[r][c]; re[r][c] = en[r][c]; }
      cur = nxt;
    }
  } else if (warp == 5) {
    // =========================== producer: dy rows by TMA (one thread) ================================
    if (lane == 0) {
      umma::tma_prefetch_desc(&map_dy);
      uint32_t g = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
        const int h0 = hs * C1_HSEG, w0 = wt * KP;
        const int rows = min(C1_HSEG, H - h0);
        const int P = (rows + C1_RB - 1) / C1_RB;
        for (int i = 0; i <= P; ++i, ++g) {
          const uint32_t s = g % C1_NS;
          umma::mbar_wait(&bars->empty[s], ((g / C1_NS) & 1) ^ 1);
          if (i < P) {
            umma::mbar_expect_tx(&bars->full[s], C1_RB * DROW);
#pragma unroll
            for (int q = 0; q < C1_RB; ++q)
              umma::tma_load_4d(umma::smem_u32(s_d) + (s * C1_RB + q) * DROW, &map_dy, 0, w0, h0 + C1_RB * i + q, b, &bars->full[s]);
          } else {
            umma::mbar_arrive(&bars->full[s]);             // the item's last stage carries x rows only
          }
        }
      }
    }
  } else {
    // =========================== MMA issuer (warp 4) ===================================================
    constexpr uint32_t idesc = umma::make_idesc_bf16(128, C1_RB * 32, true, true);
    constexpr uint32_t a_hi = umma::desc_hi(C1_PL);                                   // A: SBO = next 8-channel chunk (plane), no swizzle
    constexpr uint32_t b_hi = ((512u >> 4) & 0x3FFF) | (1u << 14) | (4u << 29);       // B: SBO = 512 B, SWIZZLE_64B
    const uint32_t x_lo0 = umma::desc_lo(umma::smem_u32(s_x), 128);                   // A: LBO = next 8-pixel group
    const uint32_t d_lo0 = umma::desc_lo(umma::smem_u32(s_d), DROW);                  // B: LBO = next dy row
    uint32_t g = 0, waited = 0, fresh = 1;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(C1_HSEG, H - hs * C1_HSEG);
      const int P = (rows + C1_RB - 1) / C1_RB;
      for (int j = 0; j < P; ++j, ++g) {
        for (; waited < g + 2; ++waited) umma::mbar_wait(&bars->full[waited % C1_NS], (waited / C1_NS) & 1);
        umma::tc_fence_after_sync();
        const uint32_t s = g % C1_NS;
        const uint32_t a0 = x_lo0 + ((C1_RB * s * C1_XROW) >> 4);
        const uint32_t b0 = d_lo0 + ((s * C1_RB * DROW) >> 4);
        if (umma::elect_one()) {
#pragma unroll
          for (int ks = 0; ks < KP / 16; ++ks)
            umma::mma_bf16_lohi(tmem, a0 + ks * 16, a_hi, b0 + ((ks * 1024) >> 4), b_hi, idesc, (fresh && ks == 0) ? 0u : 1u);
          umma::mma_commit(&bars->empty[s]);
          if (j == P - 1) umma::mma_commit(&bars->empty[(g + 1) % C1_NS]);
        }
        fresh = 0;
        __syncwarp();
      }
      ++g;
    }
    if (umma::elect_one()) umma::mma_commit(&bars->done);
    __syncwarp();
  }
  // =========================== epilogue: TMEM -> per-CTA partials (warps 0..3) ==========================
  __syncwarp();
  if (warp < 4) {
    umma::mbar_wait_sleep(&bars->done, 0);
    umma::tc_fence_after_sync();
    const int r = 2 * warp + (lane >> 4), j = lane & 15;     // TMEM lane = r*16 + j
    float* out = partial + (size_t)blockIdx.x * C1_PARTIAL;
#pragma unroll 1
    for (int q = 0; q < C1_RB; ++q) {
      uint32_t v[32];
      umma::tmem_ld_32x32(tmem + ((uint32_t)(warp * 32) << 16) + q * 32, v);
      umma::tmem_ld_wait();
      const int kh = r - q;
      if (kh >= 0 && kh <= 2 && j < 10) {
        float4* dst = reinterpret_cast<float4*>(out + ((q * 3 + kh) * 10 + j) * C);
#pragma unroll
        for (int g4 = 0; g4 < 8; ++g4)
          dst[g4] = make_float4(__uint_as_float(v[4 * g4]), __uint_as_float(v[4 * g4 + 1]), __uint_as_float(v[4 * g4 + 2]),
                                __uint_as_float(v[4 * g4 + 3]));
      }
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) umma::tmem_dealloc(tmem, 128);
}

// block (kh, j): sums partial[slot][kh][j][co] over the nslots = CTAs x 4 (cta, q) slots in a fixed order
__global__ void __launch_bounds__(256) c1_wgrad_ring_reduce_kernel(const float* __restrict__ partial, int nslots,
                                                                   float* __restrict__ dw, float* __restrict__ db) {
  __shared__ float red[8][C];
  const int kh = blockIdx.x / 10, j = blockIdx.x % 10;
  const int co = threadIdx.x & 31, g = threadIdx.x >> 5;
  float s = 0.f;
  for (int slot = g; slot < nslots; slot += 8) s += partial[(((size_t)slot * 3 + kh) * 10 + j) * C + co];
  red[g][co] = s;
  __syncthreads();
  if (g == 0) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][co];
    if (j < 9) dw[((co * 3 + j % 3) * 3 + kh) * 3 + j / 3] = t;
    else if (kh == 1) db[co] = t;
  }
}

template <int STRIDE>
int wgrad_ring_launch(const void* x, const void* dy, float* dw, float* db, void* ws, size_t ws_bytes, int B, int H, int W,
                      cudaStream_t st) {
  using G = WG<STRIDE>;
  const int Ho = (H - 1) / STRIDE + 1, Wo = (W - 1) / STRIDE + 1;
  const int items = B * ((Wo + KP - 1) / KP) * ((Ho + G::HSEG - 1) / G::HSEG);
  const int grid = items < dd::kSMs ? items : dd::kSMs;
  const size_t need = ((size_t)grid * G::PARTIAL + (size_t)grid * C) * sizeof(float);
  if (ws_bytes < need) return dd::fail(DD_ERR_WORKSPACE, "tcgen05 wgrad: workspace %zu < %zu", ws_bytes, need);
  if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy)) & 15) != 0)
    return dd::fail(DD_ERR_ALIGNMENT, "tcgen05 wgrad: x / dy are not 16-byte aligned");
  float* partial = (float*)ws;
  float* dbp = partial + (size_t)grid * G::PARTIAL;
  auto k = conv3x3_c32_wgrad_ring_kernel<STRIDE>;
  if (int e = dd::set_smem(k, G::SMEM, dd::Carveout::kMaxShared, "wgrad_tc")) return e;
  CUtensorMap mx = {}, mx1 = {}, mdy = {};
  char msg[256];
  int r;
  if (STRIDE == 1) {
    r = dd::tma_map_nhwc_sw64(&mx, x, B, H, W, C, 130, 1, msg, sizeof msg);
  } else {
    r = dd::tma_map_nhwc_sw64(&mx, x, B, H, W, C, 255, 2, msg, sizeof msg);          // 255 source pixels -> 128 loaded
    if (!r) r = dd::tma_map_nhwc_sw64(&mx1, x, B, H, W, C, 1, 1, msg, sizeof msg);
  }
  if (r) return dd::fail(DD_ERR_UNSUPPORTED, "tcgen05 wgrad: x: %s", msg);
  if (dd::tma_map_nhwc_sw64(&mdy, dy, B, Ho, Wo, C, KP, 1, msg, sizeof msg))
    return dd::fail(DD_ERR_UNSUPPORTED, "tcgen05 wgrad: dy: %s", msg);
  k<<<grid, WGT_THREADS, G::SMEM, st>>>(mx, mx1, mdy, partial, dbp, B, Ho, Wo);
  if (int err = dd::check_launch("conv3x3_c32_wgrad_ring")) return err;
  wgrad_ring_reduce_kernel<<<(9 * C * C + C + 255) / 256, 256, 0, st>>>(partial, grid * G::NQ, dbp, grid, dw, db);
  return dd::check_launch("wgrad_ring_reduce");
}

}  // namespace

namespace dd {

int conv3x3_c32_wgrad_tc(const void* x, const void* dy, float* dw, float* db, void* ws, size_t ws_bytes, int B, int H,
                         int W, int stride, cudaStream_t st) {
  if (stride == 1) return wgrad_ring_launch<1>(x, dy, dw, db, ws, ws_bytes, B, H, W, st);
  if (stride == 2) return wgrad_ring_launch<2>(x, dy, dw, db, ws, ws_bytes, B, H, W, st);
  return fail(DD_ERR_UNSUPPORTED, "tcgen05 wgrad: stride %d", stride);
}


// in_flags: bit 0 = `in` holds the six views [B,6,3,H,W] (stitch folded in), else a mosaic [B,3,H,Wm]; bit 1 = raw bytes (u8)
int conv_c1_wgrad_tc(const void* in, int in_flags, const void* dy, float* dw, float* db, void* ws, size_t ws_bytes, int B,
                     int H, int Wm, cudaStream_t st) {
  const int items = B * ((Wm + KP - 1) / KP) * ((H + C1_HSEG - 1) / C1_HSEG);
  const int grid = items < kSMs ? items : kSMs;
  const size_t need = (size_t)grid * C1_PARTIAL * sizeof(float);
  if (ws_bytes < need) return fail(DD_ERR_WORKSPACE, "tcgen05 c1 wgrad: workspace %zu < %zu", ws_bytes, need);
  if ((reinterpret_cast<uintptr_t>(dy) & 15) != 0) return fail(DD_ERR_ALIGNMENT, "tcgen05 c1 wgrad: dy is not 16-byte aligned");
  CUtensorMap mdy;
  char msg[256];
  if (tma_map_nhwc_sw64(&mdy, dy, B, H, Wm, C, KP, 1, msg, sizeof msg)) return fail(DD_ERR_UNSUPPORTED, "tcgen05 c1 wgrad: dy: %s", msg);
  auto launch1 = [&](auto k, auto* typed_in) {
    if (int e = set_smem(k, C1_SMEM, Carveout::kMaxShared, "conv_c1_wgrad_tc")) return e;
    k<<<grid, C1_THREADS, C1_SMEM, st>>>(typed_in, mdy, (float*)ws, B, H, Wm);
    return check_launch("conv_c1_wgrad_ring");
  };
  int err;
  const bool views = in_flags & 1, u8 = in_flags & 2;
  if (u8) err = views ? launch1(conv_c1_wgrad_ring_kernel<true, uint8_t>, (const uint8_t*)in)
                      : launch1(conv_c1_wgrad_ring_kernel<false, uint8_t>, (const uint8_t*)in);
  else err = views ? launch1(conv_c1_wgrad_ring_kernel<true, float>, (const float*)in)
                   : launch1(conv_c1_wgrad_ring_kernel<false, float>, (const float*)in);
  if (err) return err;
  c1_wgrad_ring_reduce_kernel<<<30, 256, 0, st>>>((const float*)ws, grid * C1_RB, dw, db);
  return check_launch("c1_wgrad_ring_reduce");
}

}  // namespace dd
