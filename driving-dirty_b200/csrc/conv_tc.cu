// 32->32 3x3 convolutions of the encoder as implicit GEMMs on the 5th-gen tensor cores
// (tcgen05.mma, accumulators in TMEM), bf16 NHWC activations, fp32 accumulate.
// Reference ops: components.py:20-21,42-43 (c2, c3) and their input gradients.
//
// Formulation ("row marching"): a CTA owns a strip of 128 output pixels of one image and walks
// down ROWS output rows.  GEMM per output row:  D[128 pix x 32 co] = sum over 9 taps of
// A_tap[128 pix x 32 ci] * W_tap[32 ci x 32 co]  -> 18 tcgen05.mma (M=128, N=32, K=16) into one
// 32-column TMEM accumulator.
//
// Shared-memory layout of an input row ("slab"): four channel-group planes, each [pixel][8 ch] =
// 16 B per pixel (core matrices of the SWIZZLE_NONE K-major canonical layout: 8 pixels x 16 B).
// Because the layout is unswizzled, the A operand of tap kw is the SAME slab addressed kw*16 B
// further on: every input row is loaded ONCE per strip and reused by 9 taps / 3 output rows
// (verified on hardware by tools/umma_probe.cu, profiles/r1_umma_descriptor_probe.txt).
// Stride 2 keeps even and odd input pixels in separate planes so that consecutive output pixels
// still read consecutive 16-byte rows.
//
// Warp roles (288 threads): warps 0..3 = producers (cp.async 16 B, zero-fill = conv padding; one
// warp cannot issue the ~520 copies per input row fast enough -- ncu showed the MMA thread starved),
// warp 4 = MMA issuer (one lane) + TMEM owner, warps 5..8 = epilogue (tcgen05.ld -> bias/ReLU or
// ReLU-mask -> bf16 -> global).  mbarrier rings: slab full/empty (8 deep), accumulator
// full/empty (4 x 32 TMEM columns), so loads, MMAs and epilogues of different rows overlap.
#include "dd_common.cuh"

#include "tma_host.h"
#include "umma.cuh"

namespace {

constexpr int C = 32;
constexpr int TILE_M = 128;
constexpr int ROWS = 32;            // output rows per work item
constexpr int RING = 8;             // slab ring depth
constexpr int NACC = 4;             // TMEM accumulator buffers (32 columns each)
constexpr int NPAD = 136;           // pixels per plane (>= 130, and 129 per parity plane for stride 2)
constexpr int PS = NPAD * 16;       // plane stride in bytes
constexpr int W_BYTES = 9 * 4 * 512;  // bf16 weights [tap][cg][co][8 ci]
constexpr int NPROD = 4;             // producer warps (0..3); warp 4 issues MMAs; warps 5..8 run the epilogue
constexpr int MMA_WARP = NPROD;
constexpr int NTHREADS = 32 * (NPROD + 1 + 4);

// ReLU sign words: the ReLU mask of a1 / a2 as the c2 / c3 input gradients need it, 4 bytes per pixel instead of the
// 64-byte activation.  One uint32 per pixel, NHWC pixel order [B][H][W]; bit c is 1 exactly when the STORED bf16
// activation of channel c is > 0 -- the comparison the input-gradient epilogues apply to the activation itself, so a
// positive fp32 value that rounds to bf16 zero and a -0 both give 0, and either form of the mask yields the same bits.
// Written by the c1 and stride-1 forward epilogues beside the activation (thread = pixel: a warp stores 128 contiguous
// bytes), read by the stride-1 and stride-2 input-gradient epilogues.
// (c1's four epilogue warps are one per scheduler, so every instruction and dependent step here is time of that kernel:
// one masked OR per half, in four independent chains, instead of shifting each bit into place)
__device__ __forceinline__ uint32_t relu_bits(const uint32_t (&pk)[16]) {
  const __nv_bfloat162 zero = __floats2bfloat162_rn(0.f, 0.f);
  uint32_t a[2] = {0u, 0u}, r[2] = {0u, 0u};
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    // m: 0xffff in the half of each channel (2k low, 2k+1 high) that is > 0.  Of bits 2k and 2k+1 one lies in its own
    // channel's half and is taken in place (a); the other is taken 16 places away (r), and r is rotated by 16 at the end
    const uint32_t m = __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&pk[k]), zero);
    if (k < 8) { a[k & 1] |= m & (1u << (2 * k)); r[k & 1] |= m & (1u << (2 * k + 17)); }
    else { a[k & 1] |= m & (1u << (2 * k + 1)); r[k & 1] |= m & (1u << (2 * k - 16)); }
  }
  const uint32_t rr = r[0] | r[1];
  return a[0] | a[1] | __funnelshift_l(rr, rr, 16);
}

// Sign word -> masks of channel pairs (0xffff per half whose bit is set, as __hgt2_mask gives).  r[s] = bits << s puts
// channel c at the top bit of byte c / 8 of r[7 - c % 8]; a byte permute with sign replication (prmt selector bit 3)
// spreads that bit over two bytes, so a pair costs one prmt.
__device__ __forceinline__ void relu_mask_prep(uint32_t bits, uint32_t (&r)[8]) {
#pragma unroll
  for (int s = 0; s < 8; ++s) r[s] = bits << s;
}
__device__ __forceinline__ uint32_t relu_mask2(const uint32_t (&r)[8], int k) {
  const int j = k >> 2, sa = 7 - ((2 * k) & 7);           // channel 2k: top of byte j of r[sa]; 2k+1: of r[sa - 1]
  const uint32_t sel = (8u | j) * 0x11u | ((8u | (4 + j)) * 0x11u) << 8;
  uint32_t m;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(m) : "r"(r[sa]), "r"(r[sa - 1]), "r"(sel));
  return m;
}

// one pixel's 32 channels (fp32 in registers) -> bf16 -> two 32-byte stores (64-byte aligned destination): whole sectors
// per lane instead of four half-sector 16-byte stores.  Returns the stored pixel's sign word (compiled away where unused).
__device__ __forceinline__ uint32_t store_pixel32(__nv_bfloat16* dst, const float (&v)[C]) {
  uint32_t pk[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
    pk[k] = *reinterpret_cast<uint32_t*>(&h);
  }
  umma::stg256(dst, pk);
  umma::stg256(dst + 16, pk + 8);
  return relu_bits(pk);
}

struct Bars {
  uint64_t full[RING], empty[RING], acc_full[NACC], acc_empty[NACC];
  uint32_t tmem_base;
};

// ================================================================================================
// Stride-2 32->32 3x3 conv (c3 forward, components.py:21,43), "row marching" gather form: 18 tcgen05.mma (M = 128 output
// pixels, N = 32, K = 16) per output row into a 32-column TMEM accumulator; every input row is loaded once per strip and
// used by the three output rows it feeds.  The input row lands as two whole-pixel planes through TMA boxes with an
// ELEMENT STRIDE of 2 along w (64-byte-swizzled K-major operand layout, profiles/r2_tma_layout_probe.txt): plane 0 =
// pixels c0, c0+2, ... (129 of them: taps kw = 0 and, one pixel on, kw = 2), plane 1 = pixels c0+1, c0+3, ... (kw = 1), so
// consecutive output pixels read consecutive 64-byte rows.  Rows / columns outside the image are zero-filled by the TMA
// unit (= the padding).  Round 1 fed this kernel with cp.async (16-byte pieces, four producer warps): 53 % of the HBM roof.
// Warps: 0 = TMA producer (one thread), 4 = MMA issuer, 5..8 = epilogue.
// ================================================================================================
constexpr int S2_P0 = 17 * 512;                 // plane 0: 129 pixels of 64 B, rounded up to the 512-byte swizzle period
constexpr int S2_P1 = TILE_M * 64;              // plane 1: 128 pixels
constexpr int S2_SLAB = S2_P0 + S2_P1;
constexpr int S2_SLAB_TX = (129 + 128) * 64;
constexpr int S2_SMEM = W_BYTES + RING * S2_SLAB + 1024;

__global__ void __launch_bounds__(NTHREADS, 1) conv3x3_c32_s2_tc_kernel(const __grid_constant__ CUtensorMap map_in2,
                                                                        const __grid_constant__ CUtensorMap map_in1,
                                                                        const float* __restrict__ w_oihw,
                                                                        const float* __restrict__ bias,
                                                                        __nv_bfloat16* __restrict__ out, int B, int H, int W,
                                                                        int Ho, int Wo) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_w = smem;
  uint8_t* s_slab = smem + W_BYTES;
  Bars* bars = reinterpret_cast<Bars*>(smem + W_BYTES + RING * S2_SLAB);
  __shared__ float s_bias[C];

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler: role code stays on the uniform datapath
  const int wtiles = (Wo + TILE_M - 1) / TILE_M;
  const int hsegs = (Ho + ROWS - 1) / ROWS;
  const int items = B * wtiles * hsegs;

  // ---- one-time setup: weights -> bf16 UMMA layout [tap][cg][co][8 ci], barriers, TMEM ----------
  for (int i = tid; i < 9 * C * C; i += NTHREADS) {
    const int ci = i & 31, co = (i >> 5) & 31, tap = i >> 10;
    *reinterpret_cast<__nv_bfloat16*>(s_w + (tap * 4 + (ci >> 3)) * 512 + co * 16 + (ci & 7) * 2) =
        __float2bfloat16_rn(w_oihw[(co * C + ci) * 9 + tap]);
  }
  if (tid < C) s_bias[tid] = bias[tid];
  if (tid == 0) {
    for (int i = 0; i < RING; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], 4); }
    umma::fence_mbar_init();
  }
  if (warp == MMA_WARP) umma::tmem_alloc(&bars->tmem_base, NACC * 32);
  umma::fence_proxy_async_smem();      // weights were written with generic stores
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp == 0) {
    // =========================== producer: one thread, TMA =====================================
    if (lane == 0) {
      umma::tma_prefetch_desc(&map_in2);
      umma::tma_prefetch_desc(&map_in1);
      uint32_t g = 0;                      // global slab counter
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
        const int ho0 = hs * ROWS;
        const int rows = min(ROWS, Ho - ho0);
        const int nslabs = (rows - 1) * 2 + 3;
        const int r0 = ho0 * 2 - 1;                      // first input row
        const int c0 = wt * TILE_M * 2 - 1;              // first input column
        for (int s = 0; s < nslabs; ++s, ++g) {
          const uint32_t slot = g % RING;
          umma::mbar_wait(&bars->empty[slot], ((g / RING) & 1) ^ 1);
          umma::mbar_expect_tx(&bars->full[slot], S2_SLAB_TX);
          const uint32_t dst = umma::smem_u32(s_slab + slot * S2_SLAB);
          umma::tma_load_4d(dst, &map_in2, 0, c0, r0 + s, b, &bars->full[slot]);                       // c0, c0+2, ... (128)
          umma::tma_load_4d(dst + TILE_M * 64, &map_in1, 0, c0 + 2 * TILE_M, r0 + s, b, &bars->full[slot]);   // ... and the 129th
          umma::tma_load_4d(dst + S2_P0, &map_in2, 0, c0 + 1, r0 + s, b, &bars->full[slot]);           // c0+1, c0+3, ... (128)
        }
      }
    }
  } else if (warp == MMA_WARP) {
    // =========================== MMA issuer (whole warp loops, elected lane issues) ===============
    constexpr uint32_t idesc = umma::make_idesc_bf16(TILE_M, C, false, false);
    constexpr uint32_t a_hi = umma::desc_hi_sw64(512), b_hi = umma::desc_hi(128);
    const uint32_t a_lo0 = umma::desc_lo(umma::smem_u32(s_slab), 0);        // A: K-major SWIZZLE_64B (one span covers K = 32)
    const uint32_t b_lo0 = umma::desc_lo(umma::smem_u32(s_w), 512);         // B: LBO = 512, SBO = 128
    uint32_t g0 = 0;            // slab counter at the start of the current item
    uint32_t waited = 0;        // slabs [0, waited) are known to be full
    uint32_t row_ctr = 0;       // global output-row counter (accumulator ring)
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(ROWS, Ho - hs * ROWS);
      const int nslabs = (rows - 1) * 2 + 3;
      for (int j = 0; j < rows; ++j, ++row_ctr) {
        const uint32_t need = g0 + j * 2 + 3;
        for (; waited < need; ++waited) umma::mbar_wait(&bars->full[waited % RING], (waited / RING) & 1);
        const uint32_t buf = row_ctr % NACC;
        umma::mbar_wait(&bars->acc_empty[buf], ((row_ctr / NACC) & 1) ^ 1);
        umma::tc_fence_after_sync();
        const uint32_t d_tmem = tmem + buf * 32;
        if (umma::elect_one()) {
#pragma unroll
          for (int kh = 0; kh < 3; ++kh) {
            const uint32_t slab_lo = a_lo0 + ((g0 + j * 2 + kh) % RING) * (S2_SLAB >> 4);
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
              // kw 0 -> plane 0 [i], 1 -> plane 1 [i], 2 -> plane 0 [i + 1]
              const int a_off = (kw == 1 ? S2_P0 : 0) + (kw == 2 ? 64 : 0);
#pragma unroll
              for (int ks = 0; ks < 2; ++ks)
                umma::mma_bf16_lohi(d_tmem, slab_lo + ((a_off + ks * 32) >> 4), a_hi,
                                    b_lo0 + (((kh * 3 + kw) * 4 + 2 * ks) * 512 >> 4), b_hi, idesc, (kh | kw | ks) ? 1u : 0u);
            }
          }
          umma::mma_commit(&bars->acc_full[buf]);
          // input rows that no later output row of this item reads
          const int nrel = (j == rows - 1) ? 3 : 2;
          for (int q = 0; q < nrel; ++q) umma::mma_commit(&bars->empty[(g0 + j * 2 + q) % RING]);
        }
        __syncwarp();
      }
      g0 += nslabs;
    }
  } else if (warp > MMA_WARP) {
    // =========================== epilogue (warps 5..8) =========================================
    const int quarter = warp & 3;                 // TMEM lanes [32*quarter, +32) belong to this warp
    uint32_t row_ctr = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
      const int ho0 = hs * ROWS;
      const int rows = min(ROWS, Ho - ho0);
      const int wo = wt * TILE_M + quarter * 32 + lane;
      for (int j = 0; j < rows; ++j, ++row_ctr) {
        const uint32_t buf = row_ctr % NACC;
        const size_t off = (((size_t)b * Ho + ho0 + j) * Wo + (wo < Wo ? wo : 0)) * C;
        umma::mbar_wait_sleep(&bars->acc_full[buf], (row_ctr / NACC) & 1);
        umma::tc_fence_after_sync();
        uint32_t r[32];
        umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + buf * 32, r);
        umma::tmem_ld_wait();
        umma::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive_relaxed(&bars->acc_empty[buf]);   // relaxed: a release arrive would first drain this warp's outstanding global stores
        if (wo < Wo) {
          float v[C];
#pragma unroll
          for (int k = 0; k < C; ++k) v[k] = fmaxf(__uint_as_float(r[k]) + s_bias[k], 0.f);
          store_pixel32(out + off, v);
        }
      }
    }
  }
  // ---- teardown ---------------------------------------------------------------------------------
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == MMA_WARP) umma::tmem_dealloc(tmem, NACC * 32);
}

int launch_s2_fwd(const void* in, const float* w, const float* bias, void* out, int B, int H, int W, cudaStream_t st) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const int items = B * ((Wo + TILE_M - 1) / TILE_M) * ((Ho + ROWS - 1) / ROWS);
  if (int e = dd::set_smem(conv3x3_c32_s2_tc_kernel, S2_SMEM, dd::Carveout::kMaxShared, "conv_tc s2")) return e;
  CUtensorMap m2, m1;
  char msg[256];
  if (dd::tma_map_nhwc_sw64(&m2, in, B, H, W, C, 255, 2, msg, sizeof msg) ||      // 255 source pixels -> 128 loaded
      dd::tma_map_nhwc_sw64(&m1, in, B, H, W, C, 1, 1, msg, sizeof msg))
    return dd::fail(DD_ERR_UNSUPPORTED, "conv_tc s2: %s", msg);
  const int grid = items < dd::kSMs ? items : dd::kSMs;
  conv3x3_c32_s2_tc_kernel<<<grid, NTHREADS, S2_SMEM, st>>>(m2, m1, w, bias, (__nv_bfloat16*)out, B, H, W, Ho, Wo);
  return dd::check_launch("conv3x3_c32_s2_tc");
}


// ================================================================================================
// Stride-1 32->32 3x3 conv (c2 forward, c2 input gradient), "row scatter" formulation; also the image gradient of c1
// (MODE 2, see below).
//
// An SS tcgen05.mma with N = 32 is bound by the shared-memory reads of its operands, not by the tensor
// pipe (tools/umma_rate2.cu: 40 cycles per M128 N32 K16 against a 16-cycle tensor floor; the 4 KB A
// tile dominates).  So instead of gathering 9 taps per OUTPUT row (18 MMAs of N = 32, every A tile read
// three times), each INPUT row is read once per (kw, K half) and scattered to the three output rows it
// feeds: B = [W(kh=2) | W(kh=1) | W(kh=0)] (N = 96) and D = the accumulators of output rows i-1, i, i+1,
// which sit in CONSECUTIVE 32-column slots of a TMEM ring -- accumulators are addressed by column, so
// the scatter costs nothing.  6 MMAs of N = 96 per input row (7 where the newest row needs its
// accumulate flag cleared or the ring wraps) instead of 18 of N = 32: 2.1x fewer operand bytes.
//
// The tensor pipe's queue is about one MMA deep (tools/umma_rate3.cu): whatever the issuing thread does
// between two tcgen05.mma -- an mbarrier wait costs ~100 cycles even when the phase is complete, a
// tcgen05.commit ~50 -- is time the pipe idles.  Hence all hand-shakes are per QUAD of rows: slabs are
// published and released four at a time (one per producer warp), accumulators are committed to / freed
// by the epilogue four at a time (16-slot ring = all 512 TMEM columns), and the D / B / instruction
// descriptor words of a batch are computed once per row.
// Warp roles (416 threads): 0..3 producers (cp.async, zero fill = padding), 4 MMA issuer,
// 5..12 epilogue (two warps per TMEM lane quarter, alternating output rows).
// ================================================================================================
constexpr int S1_ROWS = 64;         // output rows per work item (66 input rows)
#ifndef S1_NQUAD_V
#define S1_NQUAD_V 5
#endif
constexpr int S1_NQUAD = S1_NQUAD_V;   // slab ring: 5 quads = 20 input rows
constexpr int S1_RING = 4 * S1_NQUAD;
constexpr int S1_NACC = 16;         // accumulator ring: 16 x 32 TMEM columns, in 4 groups of 4 rows
constexpr int S1_NGRP = S1_NACC / 4;
constexpr int S1_EPI = 8;           // epilogue warps
constexpr int S1_SLAB = 17 * 512;   // one input row = ONE whole-pixel TMA box [130 px][32 ch] (8320 B), pitch rounded up to the 512-byte swizzle period
constexpr int S1_SLAB_TX = 130 * 64;       // bytes one input row's box delivers
constexpr int S1_WN = 96 * 16;      // bytes per (kw, channel group) weight block: [3 kh slots x 32 co][8 ci]
constexpr int S1_SMEM = W_BYTES + S1_RING * S1_SLAB + 1024;
constexpr int S1_THREADS = 32 * (NPROD + 1 + S1_EPI);
static_assert(NPROD == 4, "one slab of every quad per producer warp");

struct S1Bars {
  uint64_t full[S1_NQUAD], empty[S1_NQUAD], acc_full[S1_NGRP], acc_empty[S1_NGRP];
  uint32_t tmem_base;
};

// MODE 0: forward (bias + ReLU), MODE 1: input gradient (ReLU mask of the layer input), MODE 2: input gradient of c1
// (components.py:19,41), dx[c,h,w] = sum over o, kh, kw of da1[o, h+1-kh, w+1-kw] * W1[o,c,kh,kw].  MODE 2 reads the same
// operand as MODE 1 (da1, a [B,H,W,32] bf16 gradient) and issues the same MMAs: the B operand is W1 flipped, its 3 image
// channels zero-padded to the 32-column slot (as conv_generic.cu pads narrow layers).  Only the epilogue differs: 3 of the
// 32 accumulator columns, no mask (the images have no activation), fp32 stores into the NCHW mosaic [B,3,H,W] or, with
// Wv > 0, straight into the views [B,6,3,H,Wv] (W = 6 Wv; mosaic slot j -> view dd::view_of_slot(j)), `out` then being float*.
// BITS: MODE 0 also writes the output's ReLU sign words to `bits`; MODE 1 takes the ReLU mask from the sign words in `bits`
// instead of the activation `mask`
template <int MODE, bool BITS>
__global__ void __launch_bounds__(S1_THREADS, 1) conv3x3_c32_s1_tc_kernel(const __grid_constant__ CUtensorMap map_in,
                                                                           const float* __restrict__ w_oihw,
                                                                           const float* __restrict__ bias,
                                                                           const __nv_bfloat16* __restrict__ mask,
                                                                           __nv_bfloat16* __restrict__ out, int B, int H,
                                                                           int W, uint32_t* __restrict__ bits, int Wv) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_w = smem;
  uint8_t* s_slab = smem + W_BYTES;
  S1Bars* bars = reinterpret_cast<S1Bars*>(smem + W_BYTES + S1_RING * S1_SLAB);
  __shared__ float s_bias[C];

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wtiles = (W + TILE_M - 1) / TILE_M;
  const int hsegs = (H + S1_ROWS - 1) / S1_ROWS;
  const int items = B * wtiles * hsegs;

  // weights -> bf16 B operands [kw][cg][slot = 2 - kh][co][8 ci]: slot order = ascending output row
  for (int i = tid; i < 9 * C * C; i += S1_THREADS) {
    const int ci = i & 31, co = (i >> 5) & 31, tap = i >> 10;
    const int kh = tap / 3, kw = tap - 3 * kh;
    float v;
    if (MODE == 0) v = w_oihw[(co * C + ci) * 9 + tap];
    else if (MODE == 1) v = w_oihw[(ci * C + co) * 9 + (8 - tap)];  // dgrad: W[co=in][ci=out][flipped tap]
    else v = co < 3 ? w_oihw[(ci * 3 + co) * 9 + (8 - tap)] : 0.f;   // c1 dgrad: W1 [32 out][3 in], columns 3..31 zero
    *reinterpret_cast<__nv_bfloat16*>(s_w + (kw * 4 + (ci >> 3)) * S1_WN + ((2 - kh) * 32 + co) * 16 + (ci & 7) * 2) =
        __float2bfloat16_rn(v);
  }
  if (tid < C) s_bias[tid] = (MODE == 0) ? bias[tid] : 0.f;
  if (tid == 0) {
    for (int i = 0; i < S1_NQUAD; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 1); }
    for (int i = 0; i < S1_NGRP; ++i) { umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], S1_EPI); }
    umma::fence_mbar_init();
  }
  if (warp == MMA_WARP) umma::tmem_alloc(&bars->tmem_base, S1_NACC * 32);
  umma::fence_proxy_async_smem();
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp < NPROD) {
    // =========================== producer: one thread of warp 0, TMA (warps 1..3 idle) ============
    // cp.async (LDGSTS) tops out near 25-30 KB in flight per SM (every conv kernel fed that way sat at 35-50 % of
    // HBM bandwidth with its producer warps stalled issuing copies); TMA takes a whole input row per instruction
    // and keeps the full ring in flight.  ONE box of whole pixels per row ([130 px][32 ch], 64-byte swizzle: the K-major
    // SWIZZLE_64B operand layout; round 1's four [130 px][8 ch] boxes read half sectors from L2, four requests per row);
    // coordinates outside the image are zero-filled by the TMA unit = the conv padding.  One mbarrier per quad of
    // rows: expect_tx for the 4 boxes, then the loads.
    if (warp == 0 && lane == 0) {
      umma::tma_prefetch_desc(&map_in);
      uint32_t g = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
        const int h0 = hs * S1_ROWS;
        const int rows = min(S1_ROWS, H - h0);
        const int c0 = wt * TILE_M - 1;
        const bool last_item = it + (int)gridDim.x >= items;
        for (int s = 0; s < rows + 2; ++s, ++g) {
          const uint32_t quad = g >> 2;
          uint64_t* full = &bars->full[quad % S1_NQUAD];
          if ((g & 3) == 0) {
            umma::mbar_wait(&bars->empty[quad % S1_NQUAD], ((quad / S1_NQUAD) & 1) ^ 1);
            // slabs of this quad that exist: all four unless the CTA's work ends inside it
            const int left = last_item ? rows + 2 - s : 4;
            umma::mbar_expect_tx(full, (uint32_t)(min(left, 4) * S1_SLAB_TX));
          }
          umma::tma_load_4d(umma::smem_u32(s_slab + (g % S1_RING) * S1_SLAB), &map_in, 0, c0, h0 - 1 + s, b, full);
        }
      }
    }
  } else if (warp == MMA_WARP) {
    // =========================== MMA issuer (whole warp loops, elected lane issues) ===============
    constexpr uint32_t idesc32 = umma::make_idesc_bf16(TILE_M, 32, false, false);
    constexpr uint32_t IDESC_NSTEP = (32u >> 3) << 17;                        // +32 columns of N
    constexpr uint32_t b_hi = umma::desc_hi(128);
    constexpr uint32_t a_hi = umma::desc_hi_sw64(512);                        // A: K-major SWIZZLE_64B, SBO = 8 pixels x 64 B
    const uint32_t a_lo0 = umma::desc_lo(umma::smem_u32(s_slab), 0);          // (LBO unused: one swizzle span covers K = 32)
    const uint32_t b_lo0 = umma::desc_lo(umma::smem_u32(s_w), S1_WN);         // B: LBO = channel-group block, SBO = 128
    uint32_t g = 0;             // slab counter
    uint32_t rc0 = 0;           // output-row counter at the start of the item (accumulator ring position)
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(S1_ROWS, H - hs * S1_ROWS);
      const bool last_item = it + (int)gridDim.x >= items;
      for (int s = 0; s < rows + 2; ++s, ++g) {
        // input row s of the item feeds output rows s-2 (kh = 2), s-1 (kh = 1), s (kh = 0)
        const bool is_new = s < rows;                     // output row s receives its first contribution
        if ((g & 3) == 0) {                               // first slab of a quad
          const uint32_t quad = g >> 2;
          umma::mbar_wait(&bars->full[quad % S1_NQUAD], (quad / S1_NQUAD) & 1);   // TMA writes: async proxy, no fence needed
        }
        if (is_new && ((rc0 + s) & 3) == 0) {             // first row of an accumulator group
          const uint32_t grp = (rc0 + s) >> 2;
          umma::mbar_wait(&bars->acc_empty[grp % S1_NGRP], ((grp / S1_NGRP) & 1) ^ 1);
          umma::tc_fence_after_sync();
        }
        const uint32_t slab_lo = a_lo0 + (g % S1_RING) * (S1_SLAB >> 4);
        const uint32_t rc_done = rc0 + s - 2;             // output row completed by this batch (s >= 2)
        if (umma::elect_one()) {
          if (s >= 2 && is_new) {
            // ---- interior row (62 of 66): three output rows in ring slots sl, sl+1, sl+2; straight-line issue ----
            const uint32_t sl = rc_done % S1_NACC;
            const uint32_t d0 = tmem + sl * 32;
            constexpr uint32_t i32 = idesc32, i64 = idesc32 + IDESC_NSTEP, i96 = idesc32 + 2 * IDESC_NSTEP;
#define S1_AT(t) (slab_lo + (((((t) >> 1) * 64) + ((t) & 1) * 32) >> 4))      /* tap kw = t >> 1: +kw pixels; K half: +32 B */
#define S1_BT(t) (b_lo0 + ((((((t) >> 1) * 4) + 2 * ((t) & 1)) * S1_WN) >> 4))
            if (sl <= S1_NACC - 3) {
              umma::mma_bf16_lohi(d0, S1_AT(0), a_hi, S1_BT(0), b_hi, i64, 1u);
              umma::mma_bf16_lohi(d0 + 64, S1_AT(0), a_hi, S1_BT(0) + 64, b_hi, i32, 0u);
#pragma unroll
              for (int t = 1; t < 6; ++t) umma::mma_bf16_lohi(d0, S1_AT(t), a_hi, S1_BT(t), b_hi, i96, 1u);
            } else if (sl == S1_NACC - 2) {               // newest row wraps to slot 0
              umma::mma_bf16_lohi(d0, S1_AT(0), a_hi, S1_BT(0), b_hi, i64, 1u);
              umma::mma_bf16_lohi(tmem, S1_AT(0), a_hi, S1_BT(0) + 64, b_hi, i32, 0u);
#pragma unroll
              for (int t = 1; t < 6; ++t) {
                umma::mma_bf16_lohi(d0, S1_AT(t), a_hi, S1_BT(t), b_hi, i64, 1u);
                umma::mma_bf16_lohi(tmem, S1_AT(t), a_hi, S1_BT(t) + 64, b_hi, i32, 1u);
              }
            } else {                                      // slots 15, 0, 1
              umma::mma_bf16_lohi(d0, S1_AT(0), a_hi, S1_BT(0), b_hi, i32, 1u);
              umma::mma_bf16_lohi(tmem, S1_AT(0), a_hi, S1_BT(0) + 32, b_hi, i32, 1u);
              umma::mma_bf16_lohi(tmem + 32, S1_AT(0), a_hi, S1_BT(0) + 64, b_hi, i32, 0u);
#pragma unroll
              for (int t = 1; t < 6; ++t) {
                umma::mma_bf16_lohi(d0, S1_AT(t), a_hi, S1_BT(t), b_hi, i32, 1u);
                umma::mma_bf16_lohi(tmem, S1_AT(t), a_hi, S1_BT(t) + 32, b_hi, i64, 1u);
              }
            }
          } else {
            // ---- first / last two input rows of an item (or a very short item): general form ----
            const int jlo = max(s - 2, 0), jhi = min(s, rows - 1);
            const int n = jhi - jlo + 1;                      // output rows fed: 1..3
            const int blk = jlo - (s - 2);                    // their first kh slot in B
            const uint32_t sl = (rc0 + jlo) % S1_NACC;
            const int n1 = min(n, (int)(S1_NACC - sl));       // rows before the accumulator ring wraps
            const uint32_t d0 = tmem + sl * 32;
            const uint32_t i0 = idesc32 + (n1 - 1) * IDESC_NSTEP, i1 = idesc32 + (n - n1 - 1) * IDESC_NSTEP;
            const uint32_t bo0 = blk * 32, bo1 = (blk + n1) * 32;   // B start offsets (16-byte units): 32 co rows x 16 B per slot
            const bool two = n > n1;
            const int no = is_new ? n - 1 : n;                // rows that already hold partial sums
            const int no1 = min(no, n1), no2 = no - no1;
            // (kw 0, K half 0): accumulate into the older rows, overwrite the newest
            if (no1 > 0) umma::mma_bf16_lohi(d0, slab_lo, a_hi, b_lo0 + bo0, b_hi, idesc32 + (no1 - 1) * IDESC_NSTEP, 1u);
            if (no2 > 0) umma::mma_bf16_lohi(tmem, slab_lo, a_hi, b_lo0 + bo1, b_hi, idesc32 + (no2 - 1) * IDESC_NSTEP, 1u);
            if (is_new)
              umma::mma_bf16_lohi(tmem + ((rc0 + jhi) % S1_NACC) * 32, slab_lo, a_hi, b_lo0 + (blk + n - 1) * 32, b_hi, idesc32, 0u);
#pragma unroll
            for (int t = 1; t < 6; ++t) {
              umma::mma_bf16_lohi(d0, S1_AT(t), a_hi, S1_BT(t) + bo0, b_hi, i0, 1u);
              if (two) umma::mma_bf16_lohi(tmem, S1_AT(t), a_hi, S1_BT(t) + bo1, b_hi, i1, 1u);
            }
          }
#undef S1_AT
#undef S1_BT
          if ((g & 3) == 3) umma::mma_commit(&bars->empty[(g >> 2) % S1_NQUAD]);          // quad of slabs consumed
          if (s >= 2 && ((rc_done & 3) == 3 || (last_item && s == rows + 1)))              // group of output rows complete
            umma::mma_commit(&bars->acc_full[(rc_done >> 2) % S1_NGRP]);
        }
        __syncwarp();
      }
      rc0 += rows;
    }
  } else {
    // =========================== epilogue (warps 5..12) ===========================================
    // TMEM -> registers (thread = pixel) -> bias/ReLU (or ReLU mask) -> bf16 -> two 32-byte stores per thread.
    // Shared memory is the scarce resource of this kernel (the MMA operand reads use its full bandwidth), so the
    // epilogue stays out of it: bias lives in registers and there is no staging tile; 32-byte accesses keep
    // every global sector whole.
    const int quarter = warp & 3;                          // TMEM lanes [32*quarter, +32) belong to this warp
    const int ew = warp - (NPROD + 1);
    const uint32_t half = (uint32_t)ew >> 2;               // this warp takes output rows with (counter & 1) == half
    float bs[C];
#pragma unroll
    for (int k = 0; k < C; ++k) bs[k] = s_bias[k];
    uint32_t rc0 = 0;
    uint32_t cur_grp = 0xffffffffu;                        // accumulator group this warp is reading
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
      const int h0 = hs * S1_ROWS;
      const int rows = min(S1_ROWS, H - h0);
      const int wo = wt * TILE_M + quarter * 32 + lane;
      const bool ok = wo < W;
      const int j0 = (int)((rc0 ^ half) & 1);
      // MODE 2: this pixel's channel-0 element in row h0 of the image gradient; row and channel strides
      float* dx = nullptr;
      const int Wr = Wv > 0 ? Wv : W;
      const size_t cstride = (size_t)H * Wr;
      if (MODE == 2 && ok) {
        int img = 3 * b, col = wo;
        if (Wv > 0) {
          const int sj = wo / Wv;
          img = 3 * (6 * b + dd::view_of_slot(sj));
          col = wo - sj * Wv;
        }
        dx = reinterpret_cast<float*>(out) + ((size_t)img * H + h0) * Wr + col;
      }
      // sign words: this warp's next row is loaded while the current one is processed -- one 4-byte load issued just before
      // the wait for the MMAs leaves its DRAM round trip exposed on every row
      uint32_t mb_next = 0;
      if (MODE == 1 && BITS && ok && j0 < rows) mb_next = __ldg(bits + ((size_t)b * H + h0 + j0) * W + wo);
      for (int j = j0; j < rows; j += 2) {
        const uint32_t rc = rc0 + j;
        const uint32_t buf = rc % S1_NACC;
        const uint32_t grp = rc >> 2;
        const size_t off = (((size_t)b * H + h0 + j) * W + (ok ? wo : 0)) * C;
        uint32_t mk[16], mb = mb_next;
        if (MODE == 1 && BITS && ok && j + 2 < rows) mb_next = __ldg(bits + off / C + 2 * (size_t)W);
        if (MODE == 1 && !BITS && mask != nullptr && ok) {
          umma::ldg256(mask + off, mk);
          umma::ldg256(mask + off + 16, mk + 8);
        }
        if (grp != cur_grp) {
          if (cur_grp != 0xffffffffu) {          // both rows of the previous group are in registers
            umma::tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) umma::mbar_arrive_relaxed(&bars->acc_empty[cur_grp % S1_NGRP]);
          }
          umma::mbar_wait(&bars->acc_full[grp % S1_NGRP], (grp / S1_NGRP) & 1);
          umma::tc_fence_after_sync();
          cur_grp = grp;
        }
        if (MODE == 2) {
          uint32_t r[4];
          umma::tmem_ld_32x4(tmem + ((uint32_t)(quarter * 32) << 16) + buf * 32, r);
          umma::tmem_ld_wait();
          if (ok) {
            float* d = dx + (size_t)j * Wr;
#pragma unroll
            for (int c = 0; c < 3; ++c) d[c * cstride] = __uint_as_float(r[c]);
          }
          continue;
        }
        uint32_t r[32];
        umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + buf * 32, r);
        umma::tmem_ld_wait();
        if (ok) {
          uint32_t pk[16], mr[8];
          if (MODE == 1 && BITS) relu_mask_prep(mb, mr);
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            float x0 = __uint_as_float(r[2 * k]), x1 = __uint_as_float(r[2 * k + 1]);
            if (MODE == 0) { x0 = fmaxf(x0 + bs[2 * k], 0.f); x1 = fmaxf(x1 + bs[2 * k + 1], 0.f); }
            __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
            pk[k] = *reinterpret_cast<uint32_t*>(&h);
            if (MODE == 1 && BITS) {
              pk[k] &= relu_mask2(mr, k);
            } else if (MODE == 1 && mask != nullptr) {
              const __nv_bfloat162 zero = __floats2bfloat162_rn(0.f, 0.f);
              pk[k] &= __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&mk[k]), zero);
            }
          }
          umma::stg256(out + off, pk);
          umma::stg256(out + off + 16, pk + 8);
          if (MODE == 0 && BITS) bits[off / C] = relu_bits(pk);
        }
      }
      rc0 += rows;
    }
    // (the last group is never waited for by the MMA warp: no arrival owed)
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == MMA_WARP) umma::tmem_dealloc(tmem, S1_NACC * 32);
}

template <int MODE, bool BITS>
int launch_s1(const void* in, const float* w, const float* bias, const void* mask, void* out, int B, int H, int W,
              uint32_t* bits, cudaStream_t st, int Wv = 0) {
  const int items = B * ((W + TILE_M - 1) / TILE_M) * ((H + S1_ROWS - 1) / S1_ROWS);
  auto k = conv3x3_c32_s1_tc_kernel<MODE, BITS>;
  if (int e = dd::set_smem(k, S1_SMEM, dd::Carveout::kMaxShared, "conv_tc s1")) return e;
  const int grid = items < dd::kSMs ? items : dd::kSMs;
  if ((reinterpret_cast<uintptr_t>(in) & 15) != 0) return dd::fail(DD_ERR_ALIGNMENT, "conv_tc s1: input is not 16-byte aligned");
  CUtensorMap map;
  char msg[256];
  if (dd::tma_map_nhwc_sw64(&map, in, B, H, W, C, 130, 1, msg, sizeof msg)) return dd::fail(DD_ERR_UNSUPPORTED, "conv_tc s1: %s", msg);
  k<<<grid, S1_THREADS, S1_SMEM, st>>>(map, w, bias, (const __nv_bfloat16*)mask, (__nv_bfloat16*)out, B, H, W, bits, Wv);
  return dd::check_launch("conv3x3_c32_s1_tc");
}

// ================================================================================================
// Input gradient of the stride-2 conv (c3) = stride-2 transposed conv, on the tensor cores.
//   dx[h,w,ci] = sum over taps with (h+1-kh), (w+1-kw) even of dy[(h+1-kh)/2,(w+1-kw)/2,:] . W[:,ci,kh,kw]
// A CTA marches down dy rows m for a strip of 128 column PAIRS i (dx columns 2i, 2i+1).  Each m
// yields dx rows 2m and 2m+1; even and odd columns are separate GEMMs over the same dy slabs
// (plane layout, tap = 16-byte start shift), 9 taps = 18 MMAs per m into four 32-column TMEM
// accumulators {row 2m, 2m+1} x {even, odd}; the epilogue interleaves even/odd so that each thread
// stores two adjacent pixels (128 contiguous bytes) after the ReLU mask of the layer input.
// ================================================================================================
constexpr int DG_MROWS = 16;      // dy rows per work item (32 dx rows)
constexpr int DG_SMEM = W_BYTES + RING * 4 * PS + 1024;
constexpr int DG_THREADS = 32 * (NPROD + 1 + 8);      // 8 epilogue warps: two per TMEM lane quarter, one per dx row of the pair

struct DgBars {
  uint64_t full[RING], empty[RING], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

// (96 registers x 416 threads + the optimizer's 96 x 256 update CTA = 64.5 K: both fit one SM's register file, which the
// overlapped data-parallel update needs -- see csrc/adam.cu)
// BITS: the ReLU mask comes from the sign words in `bits` (8-byte aligned) instead of the activation `mask`
template <bool BITS>
__global__ void __maxnreg__(96) conv3x3_c32_dgrad_s2_tc_kernel(const __grid_constant__ CUtensorMap map_dy,
                                                                               const float* __restrict__ w_oihw,
                                                                               const __nv_bfloat16* __restrict__ mask,
                                                                               __nv_bfloat16* __restrict__ dx, int B,
                                                                               int H, int W, int Ho, int Wo,
                                                                               const uint32_t* __restrict__ bits) {
  constexpr int SLAB = 4 * PS;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_w = smem;
  uint8_t* s_slab = smem + W_BYTES;
  DgBars* bars = reinterpret_cast<DgBars*>(smem + W_BYTES + RING * SLAB);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler: role code stays on the uniform datapath
  const int Hp = (H + 1) / 2, Wp = (W + 1) / 2;
  const int wtiles = (Wp + TILE_M - 1) / TILE_M;
  const int hsegs = (Hp + DG_MROWS - 1) / DG_MROWS;
  const int items = B * wtiles * hsegs;

  // B operand of tap t: [n = ci][k = co] = W[co][ci][t]
  for (int i = tid; i < 9 * C * C; i += DG_THREADS) {
    const int co = i & 31, ci = (i >> 5) & 31, tap = i >> 10;
    *reinterpret_cast<__nv_bfloat16*>(s_w + (tap * 4 + (co >> 3)) * 512 + ci * 16 + (co & 7) * 2) =
        __float2bfloat16_rn(w_oihw[(co * C + ci) * 9 + tap]);
  }
  if (tid == 0) {
    for (int i = 0; i < RING; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 1); }
    for (int i = 0; i < 2; ++i) { umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], 8); }
    umma::fence_mbar_init();
  }
  if (warp == MMA_WARP) umma::tmem_alloc(&bars->tmem_base, 256);
  umma::fence_proxy_async_smem();
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp < NPROD) {
    // =========================== producer: dy rows m0 .. m0+rows, one thread, TMA ===============
    // ONE whole-pixel box [129 px][32 ch] per dy row (64-byte swizzle: the K-major SWIZZLE_64B operand; full sectors from L2,
    // one request per row); rows >= Ho and columns >= Wo are zero-filled by the TMA unit
    if (warp == 0 && lane == 0) {
      umma::tma_prefetch_desc(&map_dy);
      uint32_t g = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
        const int m0 = hs * DG_MROWS;
        const int rows = min(DG_MROWS, Hp - m0);
        const int i0 = wt * TILE_M;
        for (int s = 0; s <= rows; ++s, ++g) {
          const uint32_t slot = g % RING;
          umma::mbar_wait(&bars->empty[slot], ((g / RING) & 1) ^ 1);
          umma::mbar_expect_tx(&bars->full[slot], 129 * 64);
          umma::tma_load_4d(umma::smem_u32(s_slab + slot * SLAB), &map_dy, 0, i0, m0 + s, b, &bars->full[slot]);
        }
      }
    }
  } else if (warp == MMA_WARP) {
    {
      // =========================== MMA issuer (whole warp, elected lane issues) =================
      constexpr uint32_t idesc = umma::make_idesc_bf16(TILE_M, C, false, false);
      const uint32_t a_lo0 = umma::desc_lo(umma::smem_u32(s_slab), 0);          // A: K-major SWIZZLE_64B
      const uint32_t b_lo0 = umma::desc_lo(umma::smem_u32(s_w), 512);
      constexpr uint32_t a_hi = umma::desc_hi_sw64(512), b_hi = umma::desc_hi(128);
      // {accumulator (0: row 2m even, 1: row 2m odd, 2: row 2m+1 even, 3: row 2m+1 odd), kh, kw, slab (0: m, 1: m+1), shift}
      constexpr int T[9][5] = {{0, 1, 1, 0, 0}, {1, 1, 0, 0, 1}, {1, 1, 2, 0, 0}, {2, 0, 1, 1, 0}, {2, 2, 1, 0, 0},
                               {3, 0, 0, 1, 1}, {3, 0, 2, 1, 0}, {3, 2, 0, 0, 1}, {3, 2, 2, 0, 0}};
      uint32_t g0 = 0, waited = 0, mctr = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int hs = (it / wtiles) % hsegs;
        const int rows = min(DG_MROWS, Hp - hs * DG_MROWS);
        for (int j = 0; j < rows; ++j, ++mctr) {
          const uint32_t need = g0 + j + 2;
          for (; waited < need; ++waited) umma::mbar_wait(&bars->full[waited % RING], (waited / RING) & 1);   // TMA writes: no proxy fence
          const uint32_t set = mctr & 1;
          umma::mbar_wait(&bars->acc_empty[set], ((mctr >> 1) & 1) ^ 1);
          umma::tc_fence_after_sync();
          const uint32_t slab_lo[2] = {a_lo0 + ((g0 + j) % RING) * (SLAB >> 4), a_lo0 + ((g0 + j + 1) % RING) * (SLAB >> 4)};
          const uint32_t d0 = tmem + set * 128;
          if (umma::elect_one())
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            const int a = T[t][0], tap = T[t][1] * 3 + T[t][2];
            const bool first_of_acc = (t == 0) || (T[t][0] != T[t - (t > 0 ? 1 : 0)][0]);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks)
              umma::mma_bf16_lohi(d0 + a * 32, slab_lo[T[t][3]] + ((T[t][4] * 64 + ks * 32) >> 4), a_hi,
                                  b_lo0 + ((tap * 4 + 2 * ks) * 512 >> 4), b_hi, idesc,
                                  (first_of_acc && ks == 0) ? 0u : 1u);
          }
          if (umma::elect_one()) {
            umma::mma_commit(&bars->acc_full[set]);
            umma::mma_commit(&bars->empty[(g0 + j) % RING]);
            if (j == rows - 1) umma::mma_commit(&bars->empty[(g0 + j + 1) % RING]);
          }
          __syncwarp();
        }
        g0 += rows + 1;
      }
    }
  } else {
    // =========================== epilogue (warps 5..12) ========================================
    // two warps per TMEM lane quarter: warp `half` takes dx row 2m + half (accumulators 2*half: even columns, 2*half + 1: odd),
    // so that each thread stores two adjacent pixels (128 contiguous bytes) after the ReLU mask of the layer input
    const int quarter = warp & 3;
    const int half = (warp - (NPROD + 1)) >> 2;
    uint32_t mctr = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
      const int m0 = hs * DG_MROWS;
      const int rows = min(DG_MROWS, Hp - m0);
      const int i = wt * TILE_M + quarter * 32 + lane;
      for (int j = 0; j < rows; ++j, ++mctr) {
        const uint32_t set = mctr & 1;
        uint4 mk[2][4];
        uint32_t mb[2];
        if (BITS) {
          // this warp's dx row, pixels 2i and 2i+1: one 8-byte load where W is even (the pair is 8-byte aligned), two 4-byte
          // loads where it is odd; the odd-W edge and out-of-image pixels are clamped as below and never stored
          const int h = 2 * (m0 + j) + half, w = 2 * i;
          const size_t p = ((size_t)b * H + (h < H ? h : 0)) * W + (w < W ? w : 0);
          if ((W & 1) == 0) {
            const uint2 q = __ldg(reinterpret_cast<const uint2*>(bits + p));
            mb[0] = q.x; mb[1] = q.y;
          } else {
            mb[0] = __ldg(bits + p);
            mb[1] = __ldg(bits + p + (w + 1 < W ? 1 : 0));
          }
        } else if (mask != nullptr) {
#pragma unroll
          for (int aa = 0; aa < 2; ++aa) {
            const int a = 2 * half + aa;
            const int h = 2 * (m0 + j) + (a >> 1), w = 2 * i + (a & 1);
            const size_t moff = (((size_t)b * H + (h < H ? h : 0)) * W + (w < W ? w : 0)) * C;
#pragma unroll
            for (int gq = 0; gq < 4; ++gq) mk[aa][gq] = __ldg(reinterpret_cast<const uint4*>(mask + moff) + gq);
          }
        }
        umma::mbar_wait_sleep(&bars->acc_full[set], (mctr >> 1) & 1);
        umma::tc_fence_after_sync();
#pragma unroll
        for (int aa = 0; aa < 2; ++aa) {
          const int a = 2 * half + aa;
          uint32_t r[32];
          umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + set * 128 + a * 32, r);
          umma::tmem_ld_wait();
          if (aa == 1) {           // both accumulators of this warp's dx row are in registers / stored
            umma::tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) umma::mbar_arrive_relaxed(&bars->acc_empty[set]);
          }
          const int h = 2 * (m0 + j) + (a >> 1), w = 2 * i + (a & 1);
          if (h < H && w < W) {
            const size_t off = (((size_t)b * H + h) * W + w) * C;
            float v[C];
#pragma unroll
            for (int k = 0; k < C; ++k) v[k] = __uint_as_float(r[k]);
            if (BITS) {
#pragma unroll
              for (int k = 0; k < C; ++k) v[k] = (mb[aa] >> k) & 1u ? v[k] : 0.f;
            } else if (mask) {
#pragma unroll
              for (int gq = 0; gq < 4; ++gq) {
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&mk[aa][gq]);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float2 m = __bfloat1622float2(h2[k]);
                  v[gq * 8 + 2 * k] = m.x > 0.f ? v[gq * 8 + 2 * k] : 0.f;
                  v[gq * 8 + 2 * k + 1] = m.y > 0.f ? v[gq * 8 + 2 * k + 1] : 0.f;
                }
              }
            }
            store_pixel32(dx + off, v);
          }
        }
      }
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == MMA_WARP) umma::tmem_dealloc(tmem, 256);
}

// (the weight gradients of c1 / c2 / c3 live in conv_wgrad_tc.cu: rolling row rings fed by whole-pixel TMA boxes)

// ================================================================================================
// First encoder conv (3 -> 32, components.py:19,41) on the tensor cores, stitch folded in.
// The fp32 input (six views or a mosaic, NCHW) is converted by the producer warps into ONE plane
// per input row: [pixel][8 ch] bf16 = 16 B per pixel with channels 0..2 = image, 3 = 1.0 (used by
// the weight-gradient kernel for the bias gradient), 4..7 = 0.  With K = 8 real channels per tap a
// K = 16 MMA covers TWO horizontally adjacent taps by giving the A descriptor LBO = 16 B (the second
// K chunk is the same plane one pixel further on): 6 MMAs (M=128, N=32) per output row.
// ================================================================================================
constexpr int C1_NPROD = 6;
constexpr int C1_MMA_WARP = C1_NPROD;
constexpr int C1_THREADS = 32 * (C1_NPROD + 1 + 4);
constexpr int C1_RING = 12;
constexpr int C1_WBYTES = 6 * 1024;                 // [kh][pair][kchunk][co][8 ch] bf16
constexpr int C1_SMEM = C1_WBYTES + C1_RING * PS + 1024;

struct C1Bars {
  uint64_t full[C1_RING], empty[C1_RING], acc_full[NACC], acc_empty[NACC];
  uint32_t tmem_base;
};

// pointer to channel 0 of (b, mosaic row h, mosaic column wm); channel stride returned in cstride
template <bool IS_VIEWS, typename TIN>
__device__ __forceinline__ const TIN* c1_src(const TIN* __restrict__ in, int b, int h, int wm, int H, int Wm,
                                             size_t& cstride) {
  if (IS_VIEWS) {
    const int W = Wm / 6;
    const int j = wm / W, w = wm - j * W;
    cstride = (size_t)H * W;
    return in + (((size_t)b * 6 + dd::view_of_slot(j)) * 3) * cstride + (size_t)h * W + w;
  }
  cstride = (size_t)H * Wm;
  return in + ((size_t)b * 3) * cstride + (size_t)h * Wm + wm;
}

// one input row -> [pixel][8 ch] bf16 plane (130 pixels), by one warp
template <bool IS_VIEWS, typename TIN>
__device__ __forceinline__ void c1_load_row(uint8_t* __restrict__ slab, const TIN* __restrict__ in, int b, int r, int c0,
                                            int H, int Wm, int lane, const float* lut) {
  // all 15 global loads of the lane first, conversions afterwards: with the byte -> float table look-up inside the per-pixel
  // branch the compiler issued the loads three at a time, each group waiting for its own round trip (5 serialised global
  // latencies per row made the raw-byte converters the limit of the fused kernel)
  TIN raw[5][3];
  float v[5][3];
  bool ok[5];
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const int li = lane + 32 * k, col = c0 + li;
    ok[k] = li < 130 && r >= 0 && r < H && col >= 0 && col < Wm;
    raw[k][0] = raw[k][1] = raw[k][2] = TIN(0);
    if (ok[k]) {
      size_t cs;
      const TIN* p = c1_src<IS_VIEWS, TIN>(in, b, r, col, H, Wm, cs);
      raw[k][0] = __ldg(p); raw[k][1] = __ldg(p + cs); raw[k][2] = __ldg(p + 2 * cs);
    }
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) {
#pragma unroll
    for (int c = 0; c < 3; ++c) v[k][c] = ok[k] ? dd::c1_cvt<TIN>(raw[k][c], lut) : 0.f;
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const int li = lane + 32 * k;
    if (li < 130) {
      uint4 q;
      __nv_bfloat162 a = __floats2bfloat162_rn(v[k][0], v[k][1]);
      __nv_bfloat162 c = __floats2bfloat162_rn(v[k][2], ok[k] ? 1.0f : 0.0f);
      q.x = *reinterpret_cast<uint32_t*>(&a); q.y = *reinterpret_cast<uint32_t*>(&c); q.z = 0u; q.w = 0u;
      *reinterpret_cast<uint4*>(slab + li * 16) = q;
    }
  }
}

// BITS: also write the output's ReLU sign words to `bits`
template <bool IS_VIEWS, typename TIN, bool BITS>
__global__ void __launch_bounds__(C1_THREADS, 1) conv_c1_tc_kernel(const TIN* __restrict__ in,
                                                                    const float* __restrict__ w_oihw,
                                                                    const float* __restrict__ bias,
                                                                    __nv_bfloat16* __restrict__ out, int B, int H, int Wm,
                                                                    uint32_t* __restrict__ bits) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_w = smem;
  uint8_t* s_slab = smem + C1_WBYTES;
  C1Bars* bars = reinterpret_cast<C1Bars*>(smem + C1_WBYTES + C1_RING * PS);
  __shared__ float s_bias[C];
  __shared__ float s_lut[256];
  dd::c1_fill_lut(s_lut);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wtiles = (Wm + TILE_M - 1) / TILE_M;
  const int hsegs = (H + ROWS - 1) / ROWS;
  const int items = B * wtiles * hsegs;

  // weights: B operand of (kh, pair p): K chunk kc holds tap kw = 2p + kc, channels 0..7 (3 real)
  for (int i = tid; i < C1_WBYTES / 2; i += C1_THREADS) {
    const int ch = i & 7, co = (i >> 3) & 31, kc = (i >> 8) & 1, p = (i >> 9) & 1, kh = i >> 10;
    const int kw = 2 * p + kc;
    const float v = (kw < 3 && ch < 3) ? w_oihw[((co * 3 + ch) * 3 + kh) * 3 + kw] : 0.f;
    reinterpret_cast<__nv_bfloat16*>(s_w)[i] = __float2bfloat16_rn(v);
  }
  for (int i = tid; i < C1_RING * PS / 16; i += C1_THREADS) reinterpret_cast<uint4*>(s_slab)[i] = make_uint4(0, 0, 0, 0);
  if (tid < C) s_bias[tid] = bias[tid];
  if (tid == 0) {
    for (int i = 0; i < C1_RING; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], 4); }
    umma::fence_mbar_init();
  }
  if (warp == C1_MMA_WARP) umma::tmem_alloc(&bars->tmem_base, NACC * 32);
  umma::fence_proxy_async_smem();
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp < C1_NPROD) {
    // =========================== producers: slab g -> warp g % C1_NPROD =========================
    uint32_t g = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
      const int h0 = hs * ROWS;
      const int rows = min(ROWS, H - h0);
      for (int sidx = 0; sidx < rows + 2; ++sidx, ++g) {
        if ((g % C1_NPROD) != (uint32_t)warp) continue;
        const uint32_t slot = g % C1_RING;
        umma::mbar_wait(&bars->empty[slot], ((g / C1_RING) & 1) ^ 1);
        c1_load_row<IS_VIEWS, TIN>(s_slab + slot * PS, in, b, h0 - 1 + sidx, wt * TILE_M - 1, H, Wm, lane, s_lut);
        umma::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&bars->full[slot]);
      }
    }
  } else if (warp == C1_MMA_WARP) {
    // =========================== MMA issuer (whole warp, elected lane issues) ===================
    constexpr uint32_t idesc = umma::make_idesc_bf16(TILE_M, C, false, false);
    const uint32_t a_lo0 = umma::desc_lo(umma::smem_u32(s_slab), 16);       // second K chunk = next pixel
    const uint32_t b_lo0 = umma::desc_lo(umma::smem_u32(s_w), 512);
    constexpr uint32_t ab_hi = umma::desc_hi(128);
    uint32_t g0 = 0, waited = 0, row_ctr = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(ROWS, H - hs * ROWS);
      for (int j = 0; j < rows; ++j, ++row_ctr) {
        const uint32_t need = g0 + j + 3;
        for (; waited < need; ++waited) umma::mbar_wait(&bars->full[waited % C1_RING], (waited / C1_RING) & 1);
        const uint32_t buf = row_ctr % NACC;
        umma::mbar_wait(&bars->acc_empty[buf], ((row_ctr / NACC) & 1) ^ 1);
        umma::tc_fence_after_sync();
        if (umma::elect_one()) {
#pragma unroll
          for (int kh = 0; kh < 3; ++kh) {
            const uint32_t slab_lo = a_lo0 + ((g0 + j + kh) % C1_RING) * (PS >> 4);
#pragma unroll
            for (int p = 0; p < 2; ++p)
              umma::mma_bf16_lohi(tmem + buf * 32, slab_lo + 2 * p, ab_hi, b_lo0 + ((kh * 2 + p) * 1024 >> 4), ab_hi, idesc,
                                  (kh | p) ? 1u : 0u);
          }
          umma::mma_commit(&bars->acc_full[buf]);
          const int nrel = (j == rows - 1) ? 3 : 1;
          for (int q = 0; q < nrel; ++q) umma::mma_commit(&bars->empty[(g0 + j + q) % C1_RING]);
        }
        __syncwarp();
      }
      g0 += rows + 2;
    }
  } else {
    // =========================== epilogue: bias + ReLU -> bf16 NHWC ==============================
    const int quarter = warp & 3;
    uint32_t row_ctr = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
      const int h0 = hs * ROWS;
      const int rows = min(ROWS, H - h0);
      const int wo = wt * TILE_M + quarter * 32 + lane;
      for (int j = 0; j < rows; ++j, ++row_ctr) {
        const uint32_t buf = row_ctr % NACC;
        umma::mbar_wait_sleep(&bars->acc_full[buf], (row_ctr / NACC) & 1);
        umma::tc_fence_after_sync();
        uint32_t r[32];
        umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + buf * 32, r);
        umma::tmem_ld_wait();
        umma::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive_relaxed(&bars->acc_empty[buf]);   // relaxed: a release arrive would first drain this warp's outstanding global stores
        if (wo < Wm) {
          __nv_bfloat16* dst = out + (((size_t)b * H + h0 + j) * Wm + wo) * C;
          float v[C];
#pragma unroll
          for (int k = 0; k < C; ++k) v[k] = fmaxf(__uint_as_float(r[k]) + s_bias[k], 0.f);
          const uint32_t sign = store_pixel32(dst, v);
          if (BITS) bits[((size_t)b * H + h0 + j) * Wm + wo] = sign;
        }
      }
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == C1_MMA_WARP) umma::tmem_dealloc(tmem, NACC * 32);
}


// ================================================================================================
// Fused inference front of the encoder (components.py:41-43): relu(c1(x)) -> relu(c2(.)) in ONE kernel.
// The first activation (963 MB per 32 scenes as bf16) never touches HBM: a CTA walks a strip of 126 output
// pixels down 64 rows; per row
//   converter warps   views / mosaic row (fp32 or raw bytes) -> [130 px][8 ch] bf16 plane      (as conv_c1_tc_kernel)
//   two MMA warps     c1: row-scatter MMAs (N = 96, two taps per K = 16) over the planes -> TMEM;  c2: row-scatter MMAs over
//                     the a1 slab the first epilogue wrote.  Two issuing threads because every mbarrier wait and
//                     tcgen05.commit costs its thread 100-200 cycles: one thread doing both batches left the pipe idle
//                     60 % of the time (0.76 ms per 32 scenes; two issuers + 8-warp epilogues: 0.50)
//   epilogue 1        TMEM -> bias + ReLU -> bf16 -> shared memory, in the K-major SWIZZLE_64B layout the c2 MMAs read
//                     ([130 px][32 ch], 64-byte rows, 16-byte chunk ^= (px >> 1) & 3); pixels / rows outside the image
//                     are written as ZERO (c2's padding), not as relu(bias)
//   epilogue 2        TMEM -> bias + ReLU -> bf16 -> a2 in HBM (bit-identical to the two-kernel path: a1 is rounded to
//                     bf16 at the same point, the MMAs see the same operands in the same order)
// Halo recompute: 128 a1 pixels per 126 outputs, 66 a1 rows per 64.  Hand-shakes: the MMA warp publishes ONE commit
// per c1 batch (c1_done: a1 row v-2 complete + plane v free) and ONE per c2 batch (c2_done: output row j-2 complete +
// a1 slab free); ring indices are global plane / row counters.
// ================================================================================================
constexpr int E_STRIP = 126;
constexpr int E_ROWS = 64;
constexpr int E_NCONV = 6;                           // converter warps 0..5
constexpr int E_MMA_WARP = E_NCONV;                  // warp 6 issues the c1 MMAs, warp 7 the c2 MMAs: every mbarrier wait and
constexpr int E_MMA2_WARP = E_NCONV + 1;             // tcgen05.commit costs the issuing thread 100-200 cycles, and one thread
                                                     // doing both batches' hand-shakes left the tensor pipe idle 60 % of the time
constexpr int E_EPI1 = 8, E_EPI2 = 8;                // warps 8..15: a1 rows; warps 16..23: a2 rows (two warps per TMEM lane
                                                     // quarter each, alternating rows)
constexpr int E_THREADS = 32 * (E_NCONV + 2 + E_EPI1 + E_EPI2);
constexpr int E_VRING = 12;                          // view planes
constexpr int E_VS = 17 * 128;                       // [130 px][16 B]
constexpr int E_ARING = 8;                           // a1 slabs (S1_SLAB bytes each)
constexpr int E_NACC1 = 8, E_NACC2 = 8;              // TMEM: two rings of 8 x 32 columns (both layers scatter into three slots)
constexpr int E_W1N = 96 * 16;                       // c1 B operand: bytes per K chunk block [3 kh slots x 32 co][8 ch]
constexpr int E_DONE = 16;
constexpr int E_OFF_W1 = W_BYTES;
constexpr int E_OFF_A1 = W_BYTES + 6 * 1024;
constexpr int E_OFF_V = E_OFF_A1 + E_ARING * S1_SLAB;
constexpr int E_OFF_BARS = E_OFF_V + E_VRING * E_VS;
constexpr int E_SMEM = E_OFF_BARS + 1024;
static_assert(E_OFF_A1 % 1024 == 0, "a1 slabs need the 512-byte swizzle period");

struct EBars {
  uint64_t v_full[E_VRING], a1_full[E_ARING], acc1_empty[E_NACC1], acc2_empty[E_NACC2], c1_done[E_DONE], c2_done[E_DONE];
  uint32_t tmem_base;
};

template <bool IS_VIEWS, typename TIN>
__global__ void __maxnreg__(80) enc_c1c2_fused_kernel(const TIN* __restrict__ in, const float* __restrict__ w1_oihw,
                                                      const float* __restrict__ bias1, const float* __restrict__ w2_oihw,
                                                      const float* __restrict__ bias2, __nv_bfloat16* __restrict__ out,
                                                      int B, int H, int Wm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_w2 = smem;
  uint8_t* s_w1 = smem + E_OFF_W1;
  uint8_t* s_a1 = smem + E_OFF_A1;
  uint8_t* s_v = smem + E_OFF_V;
  EBars* bars = reinterpret_cast<EBars*>(smem + E_OFF_BARS);
  __shared__ float s_b1[C], s_b2[C];
  __shared__ float s_lut[256];
  dd::c1_fill_lut(s_lut);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int wtiles = (Wm + E_STRIP - 1) / E_STRIP;
  const int hsegs = (H + E_ROWS - 1) / E_ROWS;
  const int items = B * wtiles * hsegs;

  // c2 weights: [kw][cg][slot = 2 - kh][co][8 ci] (the s1 kernel's B operand); c1 weights: [pair][kchunk][slot = 2 - kh][co][8 ch]
  for (int i = tid; i < 9 * C * C; i += E_THREADS) {
    const int ci = i & 31, co = (i >> 5) & 31, tap = i >> 10;
    const int kh = tap / 3, kw = tap - 3 * kh;
    *reinterpret_cast<__nv_bfloat16*>(s_w2 + (kw * 4 + (ci >> 3)) * S1_WN + ((2 - kh) * 32 + co) * 16 + (ci & 7) * 2) =
        __float2bfloat16_rn(w2_oihw[(co * C + ci) * 9 + tap]);
  }
  for (int i = tid; i < 6 * 1024 / 2; i += E_THREADS) {           // [pair][kchunk][slot = 2 - kh][co][8 ch]
    const int ch = i & 7, co = (i >> 3) & 31;
    const int slot = (i >> 8) % 3, kc = ((i >> 8) / 3) & 1, pr = (i >> 8) / 6;
    const int kh = 2 - slot, kw = 2 * pr + kc;
    const float v = (kw < 3 && ch < 3) ? w1_oihw[((co * 3 + ch) * 3 + kh) * 3 + kw] : 0.f;
    reinterpret_cast<__nv_bfloat16*>(s_w1)[i] = __float2bfloat16_rn(v);
  }
  for (int i = tid; i < (E_ARING * S1_SLAB + E_VRING * E_VS) / 16; i += E_THREADS)      // slab pixels 128, 129 stay zero
    reinterpret_cast<uint4*>(s_a1)[i] = make_uint4(0, 0, 0, 0);
  if (tid < C) { s_b1[tid] = bias1[tid]; s_b2[tid] = bias2[tid]; }
  if (tid == 0) {
    for (int i = 0; i < E_VRING; ++i) umma::mbar_init(&bars->v_full[i], 1);
    for (int i = 0; i < E_ARING; ++i) umma::mbar_init(&bars->a1_full[i], 4);
    for (int i = 0; i < E_NACC1; ++i) umma::mbar_init(&bars->acc1_empty[i], 4);
    for (int i = 0; i < E_NACC2; ++i) umma::mbar_init(&bars->acc2_empty[i], 4);
    for (int i = 0; i < E_DONE; ++i) { umma::mbar_init(&bars->c1_done[i], 1); umma::mbar_init(&bars->c2_done[i], 1); }
    umma::fence_mbar_init();
  }
  if (warp == E_MMA_WARP) umma::tmem_alloc(&bars->tmem_base, 512);
  umma::fence_proxy_async_smem();
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);
  const uint32_t tmem2 = tmem + E_NACC1 * 32;

  if (warp < E_NCONV) {
    // =========================== converters: plane gv -> warp gv % E_NCONV ==========================
    uint32_t gvb = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
      const int h0 = hs * E_ROWS;
      const int rows = min(E_ROWS, H - h0);
      for (int v = 0; v < rows + 4; ++v) {
        const uint32_t gv = gvb + v;
        if ((gv % E_NCONV) != (uint32_t)warp) continue;
        if (gv >= E_VRING) {                                 // the c1 batch that last read this slot's previous plane
          const uint32_t d = gv - E_VRING;
          umma::mbar_wait(&bars->c1_done[d % E_DONE], (d / E_DONE) & 1);
        }
        c1_load_row<IS_VIEWS, TIN>(s_v + (gv % E_VRING) * E_VS, in, b, h0 - 2 + v, wt * E_STRIP - 2, H, Wm, lane, s_lut);
        umma::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&bars->v_full[gv % E_VRING]);
      }
      gvb += rows + 4;
    }
  } else if (warp == E_MMA_WARP) {
    // =========================== c1 issuer: plane v feeds a1 rows v-2 (kh = 2), v-1 (kh = 1), v (kh = 0) ==========
    // Row scatter here too: ONE plane is read by two MMAs of N = 96 (K = 16 = two horizontal taps) instead of six MMAs of
    // N = 32 per a1 row re-reading three planes (112 instead of 240 cycles of the shared tensor pipe per row).  Per a1 row
    // the accumulation order stays kh = 0, 1, 2 with the pairs inside: the same bits as conv_c1_tc_kernel.
    constexpr uint32_t idesc32 = umma::make_idesc_bf16(TILE_M, 32, false, false);
    constexpr uint32_t IDESC_NSTEP = (32u >> 3) << 17;
    constexpr uint32_t ab_hi = umma::desc_hi(128);                            // A and B: SWIZZLE_NONE, SBO = 128
    const uint32_t v_lo0 = umma::desc_lo(umma::smem_u32(s_v), 16);            // A: second K chunk = next pixel
    const uint32_t w1_lo0 = umma::desc_lo(umma::smem_u32(s_w1), E_W1N);       // B: LBO = K chunk block
    constexpr uint32_t W1_PAIR = (2 * E_W1N) >> 4;                            // second tap pair
    uint32_t gvb = 0, gab = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(E_ROWS, H - hs * E_ROWS);
      const int na = rows + 2;
      for (int v = 0; v < na + 2; ++v) {
        const uint32_t gv = gvb + v;
        umma::mbar_wait(&bars->v_full[gv % E_VRING], (gv / E_VRING) & 1);
        const bool is_new = v < na;                         // a1 row v receives its first contribution
        if (is_new) {
          const uint32_t a = gab + v;
          umma::mbar_wait(&bars->acc1_empty[a % E_NACC1], ((a / E_NACC1) & 1) ^ 1);
        }
        umma::tc_fence_after_sync();
        if (umma::elect_one()) {
          const uint32_t pl = v_lo0 + (gv % E_VRING) * (E_VS >> 4);
          const int jlo = max(v - 2, 0), jhi = min(v, na - 1);
          const int n = jhi - jlo + 1;                      // a1 rows fed: 1..3
          const int blk = jlo - (v - 2);                    // their first kh slot in B
          const uint32_t sl = (gab + jlo) % E_NACC1;
          const int n1 = min(n, (int)(E_NACC1 - sl));       // rows before the accumulator ring wraps
          const uint32_t d0 = tmem + sl * 32;
          const uint32_t bo0 = blk * 32, bo1 = (blk + n1) * 32;
          const int no = is_new ? n - 1 : n;                // rows that already hold partial sums
          const int no1 = min(no, n1), no2 = no - no1;
          // pair 0: accumulate into the older rows, overwrite the newest; pair 1: accumulate into all
          if (no1 > 0) umma::mma_bf16_lohi(d0, pl, ab_hi, w1_lo0 + bo0, ab_hi, idesc32 + (no1 - 1) * IDESC_NSTEP, 1u);
          if (no2 > 0) umma::mma_bf16_lohi(tmem, pl, ab_hi, w1_lo0 + bo1, ab_hi, idesc32 + (no2 - 1) * IDESC_NSTEP, 1u);
          if (is_new)
            umma::mma_bf16_lohi(tmem + ((gab + jhi) % E_NACC1) * 32, pl, ab_hi, w1_lo0 + (blk + n - 1) * 32, ab_hi, idesc32, 0u);
          umma::mma_bf16_lohi(d0, pl + 2, ab_hi, w1_lo0 + W1_PAIR + bo0, ab_hi, idesc32 + (n1 - 1) * IDESC_NSTEP, 1u);
          if (n > n1) umma::mma_bf16_lohi(tmem, pl + 2, ab_hi, w1_lo0 + W1_PAIR + bo1, ab_hi, idesc32 + (n - n1 - 1) * IDESC_NSTEP, 1u);
          umma::mma_commit(&bars->c1_done[gv % E_DONE]);   // plane gv is free; a1 row v-2 is complete
        }
        __syncwarp();
      }
      gvb += rows + 4; gab += na;
    }
  } else if (warp == E_MMA2_WARP) {
    // =========================== c2 issuer: a1 row s feeds output rows s-2 (kh = 2), s-1 (kh = 1), s (kh = 0) =====
    constexpr uint32_t idesc32 = umma::make_idesc_bf16(TILE_M, 32, false, false);
    constexpr uint32_t IDESC_NSTEP = (32u >> 3) << 17;
    constexpr uint32_t b_hi = umma::desc_hi(128);
    constexpr uint32_t a2_hi = umma::desc_hi_sw64(512);                       // A: K-major SWIZZLE_64B
    const uint32_t a1_lo0 = umma::desc_lo(umma::smem_u32(s_a1), 0);
    const uint32_t w2_lo0 = umma::desc_lo(umma::smem_u32(s_w2), S1_WN);
    uint32_t gab = 0, grb = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int hs = (it / wtiles) % hsegs;
      const int rows = min(E_ROWS, H - hs * E_ROWS);
      const int na = rows + 2;
      for (int s = 0; s < na; ++s) {
        const uint32_t a = gab + s;
        umma::mbar_wait(&bars->a1_full[a % E_ARING], (a / E_ARING) & 1);
        const bool is_new = s < rows;
        if (is_new) {
          const uint32_t rr = grb + s;
          umma::mbar_wait(&bars->acc2_empty[rr % E_NACC2], ((rr / E_NACC2) & 1) ^ 1);
        }
        umma::tc_fence_after_sync();
        if (umma::elect_one()) {
          const uint32_t slab_lo = a1_lo0 + (a % E_ARING) * (S1_SLAB >> 4);
#define E_AT(t) (slab_lo + (((((t) >> 1) * 64) + ((t) & 1) * 32) >> 4))
#define E_BT(t) (w2_lo0 + ((((((t) >> 1) * 4) + 2 * ((t) & 1)) * S1_WN) >> 4))
          if (s >= 2 && is_new) {
            // ---- interior row (62 of 66): three output rows in ring slots sl, sl+1, sl+2; straight-line issue, only the
            //      slab and the slot change from row to row (the general form below costs ~110 uniform instructions of
            //      descriptor arithmetic per row on the thread that is the kernel's critical path) ----
            const uint32_t sl = (grb + s - 2) % E_NACC2;
            const uint32_t d0 = tmem2 + sl * 32;
            constexpr uint32_t i32 = idesc32, i64 = idesc32 + IDESC_NSTEP, i96 = idesc32 + 2 * IDESC_NSTEP;
            if (sl <= E_NACC2 - 3) {
              umma::mma_bf16_lohi(d0, E_AT(0), a2_hi, E_BT(0), b_hi, i64, 1u);
              umma::mma_bf16_lohi(d0 + 64, E_AT(0), a2_hi, E_BT(0) + 64, b_hi, i32, 0u);
#pragma unroll
              for (int t = 1; t < 6; ++t) umma::mma_bf16_lohi(d0, E_AT(t), a2_hi, E_BT(t), b_hi, i96, 1u);
            } else if (sl == E_NACC2 - 2) {               // newest row wraps to slot 0
              umma::mma_bf16_lohi(d0, E_AT(0), a2_hi, E_BT(0), b_hi, i64, 1u);
              umma::mma_bf16_lohi(tmem2, E_AT(0), a2_hi, E_BT(0) + 64, b_hi, i32, 0u);
#pragma unroll
              for (int t = 1; t < 6; ++t) {
                umma::mma_bf16_lohi(d0, E_AT(t), a2_hi, E_BT(t), b_hi, i64, 1u);
                umma::mma_bf16_lohi(tmem2, E_AT(t), a2_hi, E_BT(t) + 64, b_hi, i32, 1u);
              }
            } else {                                      // last slot, then slots 0 and 1
              umma::mma_bf16_lohi(d0, E_AT(0), a2_hi, E_BT(0), b_hi, i32, 1u);
              umma::mma_bf16_lohi(tmem2, E_AT(0), a2_hi, E_BT(0) + 32, b_hi, i32, 1u);
              umma::mma_bf16_lohi(tmem2 + 32, E_AT(0), a2_hi, E_BT(0) + 64, b_hi, i32, 0u);
#pragma unroll
              for (int t = 1; t < 6; ++t) {
                umma::mma_bf16_lohi(d0, E_AT(t), a2_hi, E_BT(t), b_hi, i32, 1u);
                umma::mma_bf16_lohi(tmem2, E_AT(t), a2_hi, E_BT(t) + 32, b_hi, i64, 1u);
              }
            }
          } else {
            // ---- first / last two a1 rows of an item (or a very short item): general form ----
            const int jlo = max(s - 2, 0), jhi = min(s, rows - 1);
            const int n = jhi - jlo + 1;                      // output rows fed: 1..3
            const int blk = jlo - (s - 2);                    // their first kh slot in B
            const uint32_t sl = (grb + jlo) % E_NACC2;
            const int n1 = min(n, (int)(E_NACC2 - sl));       // rows before the accumulator ring wraps
            const uint32_t d0 = tmem2 + sl * 32;
            const uint32_t i0 = idesc32 + (n1 - 1) * IDESC_NSTEP, i1 = idesc32 + (n - n1 - 1) * IDESC_NSTEP;
            const uint32_t bo0 = blk * 32, bo1 = (blk + n1) * 32;
            const bool two = n > n1;
            const int no = is_new ? n - 1 : n;                // rows that already hold partial sums
            const int no1 = min(no, n1), no2 = no - no1;
            if (no1 > 0) umma::mma_bf16_lohi(d0, slab_lo, a2_hi, w2_lo0 + bo0, b_hi, idesc32 + (no1 - 1) * IDESC_NSTEP, 1u);
            if (no2 > 0) umma::mma_bf16_lohi(tmem2, slab_lo, a2_hi, w2_lo0 + bo1, b_hi, idesc32 + (no2 - 1) * IDESC_NSTEP, 1u);
            if (is_new)
              umma::mma_bf16_lohi(tmem2 + ((grb + jhi) % E_NACC2) * 32, slab_lo, a2_hi, w2_lo0 + (blk + n - 1) * 32, b_hi, idesc32, 0u);
#pragma unroll
            for (int t = 1; t < 6; ++t) {
              umma::mma_bf16_lohi(d0, E_AT(t), a2_hi, E_BT(t) + bo0, b_hi, i0, 1u);
              if (two) umma::mma_bf16_lohi(tmem2, E_AT(t), a2_hi, E_BT(t) + bo1, b_hi, i1, 1u);
            }
          }
#undef E_AT
#undef E_BT
          umma::mma_commit(&bars->c2_done[a % E_DONE]);
        }
        __syncwarp();
      }
      gab += na; grb += rows;
    }
  } else if (warp < E_MMA2_WARP + 1 + E_EPI1) {
    // =========================== epilogue 1: a1 row TMEM -> bias + ReLU -> bf16 -> swizzled slab ====
    const int quarter = warp & 3;
    const uint32_t half = (uint32_t)(warp - (E_MMA2_WARP + 1)) >> 2;     // this warp takes a1 rows with (counter & 1) == half
    const int m = quarter * 32 + lane;                       // a1 pixel of the strip: mosaic column x0 - 1 + m
    const uint32_t sw = (uint32_t)((m >> 1) & 3);
    const uint32_t a1_base = umma::smem_u32(s_a1) + m * 64;
    float bs[C];
#pragma unroll
    for (int k = 0; k < C; ++k) bs[k] = s_b1[k];
    uint32_t gvb = 0, gab = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs;
      const int h0 = hs * E_ROWS;
      const int rows = min(E_ROWS, H - h0);
      const int col = wt * E_STRIP - 1 + m;
      const bool col_ok = col >= 0 && col < Wm;
      for (int t = (int)((gab ^ half) & 1); t < rows + 2; t += 2) {
        const uint32_t a = gab + t, buf = a % E_NACC1, dv = gvb + t + 2;      // complete after plane t+2's batch
        umma::mbar_wait(&bars->c1_done[dv % E_DONE], (dv / E_DONE) & 1);
        umma::tc_fence_after_sync();
        uint32_t r[32];
        umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + buf * 32, r);
        umma::tmem_ld_wait();
        umma::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive_relaxed(&bars->acc1_empty[buf]);
        if (a >= E_ARING) {                                  // the c2 batch that read this slab's previous row
          const uint32_t d = a - E_ARING;
          umma::mbar_wait(&bars->c2_done[d % E_DONE], (d / E_DONE) & 1);
        }
        const int ha = h0 - 1 + t;
        const uint32_t keep = (col_ok && ha >= 0 && ha < H) ? 0xffffffffu : 0u;     // outside the image a1 is c2's zero padding
        const uint32_t dst = a1_base + (a % E_ARING) * S1_SLAB;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t pk[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            __nv_bfloat162 h = __floats2bfloat162_rn(fmaxf(__uint_as_float(r[8 * c + 2 * k]) + bs[8 * c + 2 * k], 0.f),
                                                     fmaxf(__uint_as_float(r[8 * c + 2 * k + 1]) + bs[8 * c + 2 * k + 1], 0.f));
            pk[k] = *reinterpret_cast<uint32_t*>(&h) & keep;
          }
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + ((c ^ sw) << 4)), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]),
                       "r"(pk[3]) : "memory");
        }
        umma::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&bars->a1_full[a % E_ARING]);
      }
      gvb += rows + 4; gab += rows + 2;
    }
  } else {
    // =========================== epilogue 2: a2 row TMEM -> bias + ReLU -> bf16 -> HBM ==============
    const int quarter = warp & 3;
    const uint32_t half = (uint32_t)(warp - (E_MMA2_WARP + 1 + E_EPI1)) >> 2;
    const int m = quarter * 32 + lane;
    float bs[C];
#pragma unroll
    for (int k = 0; k < C; ++k) bs[k] = s_b2[k];
    uint32_t gab = 0, grb = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x) {
      const int wt = it % wtiles, hs = (it / wtiles) % hsegs, b = it / (wtiles * hsegs);
      const int h0 = hs * E_ROWS;
      const int rows = min(E_ROWS, H - h0);
      const int wo = wt * E_STRIP + m;
      const bool ok = m < E_STRIP && wo < Wm;
      for (int j = (int)((grb ^ half) & 1); j < rows; j += 2) {
        const uint32_t rr = grb + j, slot = rr % E_NACC2, d = gab + j + 2;
        umma::mbar_wait_sleep(&bars->c2_done[d % E_DONE], (d / E_DONE) & 1);
        umma::tc_fence_after_sync();
        uint32_t r[32];
        umma::tmem_ld_32x32(tmem2 + ((uint32_t)(quarter * 32) << 16) + slot * 32, r);
        umma::tmem_ld_wait();
        umma::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive_relaxed(&bars->acc2_empty[slot]);
        if (ok) {
          uint32_t pk[16];
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            __nv_bfloat162 h = __floats2bfloat162_rn(fmaxf(__uint_as_float(r[2 * k]) + bs[2 * k], 0.f),
                                                     fmaxf(__uint_as_float(r[2 * k + 1]) + bs[2 * k + 1], 0.f));
            pk[k] = *reinterpret_cast<uint32_t*>(&h);
          }
          __nv_bfloat16* dst = out + (((size_t)b * H + h0 + j) * Wm + wo) * C;
          umma::stg256(dst, pk);
          umma::stg256(dst + 16, pk + 8);
        }
      }
      gab += rows + 2; grb += rows;
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == E_MMA_WARP) umma::tmem_dealloc(tmem, 512);
}


}  // namespace


namespace dd {

// bits (may be NULL): the ReLU sign words (see relu_bits), written by mode 0 stride 1, read instead of `mask` by mode 1
int conv3x3_c32_fwd_tc(const void* in, const float* w, const float* bias, void* out, int B, int H, int W, int stride,
                       int mode, const void* mask, uint32_t* bits, cudaStream_t st) {
  // the epilogues store (and read the ReLU mask) in 32-byte pieces; the producers read 16-byte pieces
  if (((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(mask)) & 31) != 0 || (reinterpret_cast<uintptr_t>(in) & 15) != 0)
    return fail(DD_ERR_ALIGNMENT, "conv_tc: activations must be 32-byte aligned (in %p, out %p, mask %p)", in, out, mask);
  if ((reinterpret_cast<uintptr_t>(bits) & 7) != 0) return fail(DD_ERR_ALIGNMENT, "conv_tc: sign words %p are not 8-byte aligned", bits);
  if (bits && mode == 0 && stride != 1) return fail(DD_ERR_UNSUPPORTED, "conv_tc: sign words are written by the stride-1 forward only");
  if (mode == 0 && stride == 1)
    return bits ? launch_s1<0, true>(in, w, bias, nullptr, out, B, H, W, bits, st) : launch_s1<0, false>(in, w, bias, nullptr, out, B, H, W, nullptr, st);
  if (mode == 0 && stride == 2) return launch_s2_fwd(in, w, bias, out, B, H, W, st);
  if (mode == 1 && stride == 1)
    return bits ? launch_s1<1, true>(in, w, nullptr, nullptr, out, B, H, W, bits, st) : launch_s1<1, false>(in, w, nullptr, mask, out, B, H, W, nullptr, st);
  if (mode == 1 && stride == 2) {
    // here `in` = dy [B,Ho,Wo,32], `out` = dx [B,H,W,32]
    const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
    const int items = B * (((W + 1) / 2 + TILE_M - 1) / TILE_M) * (((H + 1) / 2 + DG_MROWS - 1) / DG_MROWS);
    auto k = bits ? conv3x3_c32_dgrad_s2_tc_kernel<true> : conv3x3_c32_dgrad_s2_tc_kernel<false>;
    if (int e = set_smem(k, DG_SMEM, Carveout::kMaxShared, "dgrad_s2_tc")) return e;
    if ((reinterpret_cast<uintptr_t>(in) & 15) != 0) return fail(DD_ERR_ALIGNMENT, "dgrad_s2_tc: dy is not 16-byte aligned");
    CUtensorMap mdy;
    char msg[256];
    if (tma_map_nhwc_sw64(&mdy, in, B, Ho, Wo, C, 129, 1, msg, sizeof msg)) return fail(DD_ERR_UNSUPPORTED, "dgrad_s2_tc: %s", msg);
    k<<<items < kSMs ? items : kSMs, DG_THREADS, DG_SMEM, st>>>(mdy, w, bits ? nullptr : (const __nv_bfloat16*)mask,
                                                                 (__nv_bfloat16*)out, B, H, W, Ho, Wo, bits);
    return check_launch("conv3x3_c32_dgrad_s2_tc");
  }
  return fail(DD_ERR_UNSUPPORTED, "conv_tc: mode %d stride %d", mode, stride);
}

// image gradient of c1 from da1 (bf16 NHWC [B,H,Wm,32]) -> fp32 dx: the views [B,6,3,H,Wm/6] when `views`, else the
// mosaic [B,3,H,Wm]
int conv_c1_dgrad_tc(const void* dy, const float* w, float* dx, bool views, int B, int H, int Wm, cudaStream_t st) {
  return launch_s1<2, false>(dy, w, nullptr, nullptr, dx, B, H, Wm, nullptr, st, views ? Wm / 6 : 0);
}

// in_flags: bit 0 = six views [B,6,3,H,W] (stitch folded in), else a mosaic [B,3,H,Wm]; bit 1 = raw camera bytes (u8, /255 folded in)
// bits (may be NULL): also write a1's ReLU sign words (see relu_bits)
int conv_c1_fwd_tc(const void* in, int in_flags, const float* w, const float* bias, void* out, uint32_t* bits, int B, int H,
                   int Wm, cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(out) & 31) != 0) return fail(DD_ERR_ALIGNMENT, "conv_c1_tc: out %p is not 32-byte aligned", out);
  if ((reinterpret_cast<uintptr_t>(bits) & 7) != 0) return fail(DD_ERR_ALIGNMENT, "conv_c1_tc: sign words %p are not 8-byte aligned", bits);
  const int items = B * ((Wm + TILE_M - 1) / TILE_M) * ((H + ROWS - 1) / ROWS);
  const int grid = items < kSMs ? items : kSMs;
  auto launch1 = [&](auto k, auto* typed_in) {
    if (int e = set_smem(k, C1_SMEM, Carveout::kMaxShared, "conv_c1_tc")) return e;
    k<<<grid, C1_THREADS, C1_SMEM, st>>>(typed_in, w, bias, (__nv_bfloat16*)out, B, H, Wm, bits);
    return check_launch("conv_c1_tc");
  };
  auto launch = [&](auto typed_in, auto k_plain, auto k_bits) { return bits ? launch1(k_bits, typed_in) : launch1(k_plain, typed_in); };
  const bool views = in_flags & 1, u8 = in_flags & 2;
  const uint8_t* in8 = (const uint8_t*)in;
  const float* in32 = (const float*)in;
  if (u8)
    return views ? launch(in8, conv_c1_tc_kernel<true, uint8_t, false>, conv_c1_tc_kernel<true, uint8_t, true>)
                 : launch(in8, conv_c1_tc_kernel<false, uint8_t, false>, conv_c1_tc_kernel<false, uint8_t, true>);
  return views ? launch(in32, conv_c1_tc_kernel<true, float, false>, conv_c1_tc_kernel<true, float, true>)
               : launch(in32, conv_c1_tc_kernel<false, float, false>, conv_c1_tc_kernel<false, float, true>);
}

// relu(c1) -> relu(c2) of the encoder in one kernel (inference: the first activation is not kept); out = a2, bf16 NHWC
int enc_c1c2_fused_fwd_tc(const void* in, int in_flags, const float* w1, const float* b1, const float* w2, const float* b2,
                          void* out, int B, int H, int Wm, cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(out) & 31) != 0) return fail(DD_ERR_ALIGNMENT, "enc_c1c2_fused: out %p is not 32-byte aligned", out);
  const int items = B * ((Wm + E_STRIP - 1) / E_STRIP) * ((H + E_ROWS - 1) / E_ROWS);
  const int grid = items < kSMs ? items : kSMs;
  auto launch1 = [&](auto k, auto* typed_in) {
    if (int e = set_smem(k, E_SMEM, Carveout::kMaxShared, "enc_c1c2_fused")) return e;
    k<<<grid, E_THREADS, E_SMEM, st>>>(typed_in, w1, b1, w2, b2, (__nv_bfloat16*)out, B, H, Wm);
    return check_launch("enc_c1c2_fused");
  };
  const bool views = in_flags & 1, u8 = in_flags & 2;
  if (u8) return views ? launch1(enc_c1c2_fused_kernel<true, uint8_t>, (const uint8_t*)in) : launch1(enc_c1c2_fused_kernel<false, uint8_t>, (const uint8_t*)in);
  return views ? launch1(enc_c1c2_fused_kernel<true, float>, (const float*)in) : launch1(enc_c1c2_fused_kernel<false, float>, (const float*)in);
}

}  // namespace dd
