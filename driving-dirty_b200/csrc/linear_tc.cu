// Skinny, weight-streaming linear layers on the 5th-gen tensor cores: fp32 weights go HBM -> TMA
// (128-byte-swizzled boxes) -> shared memory -> tcgen05.mma kind::tf32 -> TMEM, once per pass.
//   Encoder.fc1.fc1  Linear(940,032 -> hidden)   components.py:26,105
//   roadmap head     Linear(latent -> 640,000)   roadmap_bce_v2.py:50,75
//   Decoder.fc2.fc1  Linear(hidden -> 1,253,376) components.py:69
// All three passes are HBM-bound (the weight, or its gradient, crosses HBM exactly once per pass over
// the batch); the batch is the narrow MMA dimension: 32 rows per pass in the training step (forward,
// dgrad, wgrad), up to 256 rows per pass in the forward (inference batches; SCfg below).
//
//   fwd   y[b][n]  = sum_k x[b][k] W[n][k]     D[128 n x 32 b]:  A = W tile, K-major (SWIZZLE_128B);
//                                              B = x tile, K-major
//   dgrad dx[b][k] = sum_n dy[b][n] W[n][k]    D[128 k x 32 b]:  A = W^T tile, MN-major -- for tf32 that
//                                              is SWIZZLE_128B_BASE32B (TMA ..._ATOM_32B);  B = dy, K-major
//   wgrad dW[n][k] = sum_b dy[b][n] x[b][k]    D[128 n x 256 k]: A = dy^T, B = x, both MN-major
//   bwd + Adam (world size 1): dgrad as above and G^T[k][n] = sum_b x[b][k] dy[b][n] (A = x, B = dy, both MN-major) per
//                              weight tile, whose Adam update is applied on chip: one pass over W, m and v
// Operand descriptors were verified on hardware with tools/umma_tf32_probe.cu
// (profiles/r1_umma_tf32_tma_probe.txt).
//
// Warp roles (192 threads): warp 0 = TMA producer (one lane), warp 1 = MMA issuer + TMEM owner,
// warps 2..5 = epilogue (TMEM -> registers -> global).  Persistent CTAs walk (tile, split) work items;
// split contractions go to ordered partial buffers folded by a second kernel (deterministic).
#include "adam.cuh"
#include "dd_common.cuh"
#include "tma_host.h"
#include "umma.cuh"

namespace {

constexpr int NB = 32;                    // batch rows per launch (MMA N, or K for wgrad)
constexpr int kLinearTcMaxRows = 256;     // forward only: rows per pass (SCfg below)
constexpr int THREADS = 192;
constexpr int BOX = 32 * 128;             // a 32-row x 128-byte TMA box
constexpr int kChunk = 32;                // contraction elements per stage (one 128-byte swizzle span)

__device__ __forceinline__ uint8_t* align1024(uint8_t* p) {
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 1023) & ~static_cast<uintptr_t>(1023));
}
// ------------------------------------------------------------------------------------------------
// fwd (MODE 0) and dgrad (MODE 1): out[b * LD + r] = sum over the contraction, r = row of the 128-row tile
// ------------------------------------------------------------------------------------------------
// NBT = batch rows per pass (the MMA N): 32 for the training step; the inference front end sends up to 256 scenes per
// call, and with NBT = 256 the weights still cross HBM once (they were re-read for every 32 rows: 8 passes over the
// 0.96 GB of Encoder.fc1 at batch 256)
template <int NBT> struct SCfg {
  static constexpr int STAGES = NBT <= 32 ? 8 : NBT <= 64 ? 8 : NBT <= 128 ? 6 : 4;
  static constexpr int STAGE_BYTES = 4 * BOX + NBT * 128;      // A: 128 x 128 B (fwd) or 4 boxes (dgrad); B: NBT rows x 128 B
  static constexpr int SMEM = STAGES * STAGE_BYTES + 2048;
};
constexpr int S_MAX_STAGES = 8;

struct StreamBars {
  uint64_t full[S_MAX_STAGES], empty[S_MAX_STAGES], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

struct StreamGeo {
  int B, LD;                // batch rows; output leading dimension (N for fwd, K for dgrad)
  int tiles, splits;        // 128-row output tiles; contraction splits
  int chunks, chunks_per_split;
};

template <int MODE, typename TOUT, int NBT = NB>
__global__ void __launch_bounds__(THREADS, 1) linear_stream_tc_kernel(const __grid_constant__ CUtensorMap map_w,
                                                                       const __grid_constant__ CUtensorMap map_v,
                                                                       const float* __restrict__ bias,
                                                                       TOUT* __restrict__ out, float* __restrict__ partial,
                                                                       StreamGeo g) {
  constexpr int S_STAGES = SCfg<NBT>::STAGES, S_STAGE_BYTES = SCfg<NBT>::STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  StreamBars* bars = reinterpret_cast<StreamBars*>(smem + S_STAGES * S_STAGE_BYTES);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int items = g.tiles * g.splits;

  if (tid == 0) {
    for (int i = 0; i < S_STAGES; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 1); }
    for (int i = 0; i < 2; ++i) { umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], 4); }
    umma::fence_mbar_init();
    umma::tma_prefetch_desc(&map_w);
    umma::tma_prefetch_desc(&map_v);
  }
  if (warp == 1) umma::tmem_alloc(&bars->tmem_base, 2 * NBT);
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp == 0) {
    // =========================== TMA producer ===================================================
    if (umma::elect_one()) {
      uint32_t c = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int ti = it % g.tiles, si = it / g.tiles;
        const int c0 = si * g.chunks_per_split;
        const int c1 = min(c0 + g.chunks_per_split, g.chunks);
        for (int ch = c0; ch < c1; ++ch, ++c) {
          const uint32_t s = c % S_STAGES;
          umma::mbar_wait(&bars->empty[s], ((c / S_STAGES) & 1) ^ 1);
          const uint32_t dst = umma::smem_u32(smem + s * S_STAGE_BYTES);
          umma::mbar_expect_tx(&bars->full[s], S_STAGE_BYTES);
          if (MODE == 0) {
            umma::tma_load_2d(dst, &map_w, ch * kChunk, ti * 128, &bars->full[s]);             // W[n tile][k chunk]
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)                                                         // W[n chunk][k tile], 4 x 32 k
              umma::tma_load_2d(dst + i * BOX, &map_w, ti * 128 + 32 * i, ch * kChunk, &bars->full[s]);
          }
          umma::tma_load_2d(dst + 4 * BOX, &map_v, ch * kChunk, 0, &bars->full[s]);             // x / dy [b][chunk]
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer =======================================================
    constexpr uint32_t idesc = umma::make_idesc_tf32(128, NBT, MODE == 1, false);
    uint32_t c = 0, n_item = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x, ++n_item) {
      const int si = it / g.tiles;
      const int c0 = si * g.chunks_per_split;
      const int c1 = min(c0 + g.chunks_per_split, g.chunks);
      const uint32_t a = n_item & 1;
      umma::mbar_wait(&bars->acc_empty[a], ((n_item >> 1) & 1) ^ 1);
      umma::tc_fence_after_sync();
      for (int ch = c0; ch < c1; ++ch, ++c) {
        const uint32_t s = c % S_STAGES;
        umma::mbar_wait(&bars->full[s], (c / S_STAGES) & 1);
        umma::tc_fence_after_sync();
        const uint32_t base = umma::smem_u32(smem + s * S_STAGE_BYTES);
        if (umma::elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint32_t a_lo, a_hi;
            if (MODE == 0) { a_lo = umma::desc_lo(base + k * 32, 16); a_hi = umma::desc_hi_sw128(1024); }
            else { a_lo = umma::desc_lo(base + k * 1024, BOX); a_hi = umma::desc_hi_sw128_base32(512); }
            umma::mma_tf32_lohi(tmem + a * NBT, a_lo, a_hi, umma::desc_lo(base + 4 * BOX + k * 32, 16), umma::desc_hi_sw128(1024),
                                idesc, (ch > c0 || k > 0) ? 1u : 0u);
          }
          umma::mma_commit(&bars->empty[s]);
          if (ch == c1 - 1) umma::mma_commit(&bars->acc_full[a]);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== epilogue (warps 2..5) =============================================
    const int quarter = warp & 3;
    uint32_t n_item = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x, ++n_item) {
      const int ti = it % g.tiles, si = it / g.tiles;
      const uint32_t a = n_item & 1;
      umma::mbar_wait_sleep(&bars->acc_full[a], (n_item >> 1) & 1);
      umma::tc_fence_after_sync();
      const int r = ti * 128 + quarter * 32 + lane;
      const float bv = (g.splits == 1 && bias && r < g.LD) ? __ldg(bias + r) : 0.f;
#pragma unroll 1
      for (int nb = 0; nb < NBT; nb += 32) {
        uint32_t v[32];
        umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + a * NBT + nb, v);
        umma::tmem_ld_wait();
        const bool last = nb + 32 >= NBT || nb + 32 >= g.B;
        if (last) {                                      // last group read: hand the accumulator back before the stores
          umma::tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) umma::mbar_arrive(&bars->acc_empty[a]);
        }
        if (r < g.LD) {
          if (g.splits == 1) {
#pragma unroll
            for (int b = 0; b < 32; ++b)
              if (nb + b < g.B) dd::st<TOUT>(out + (size_t)(nb + b) * g.LD + r, __uint_as_float(v[b]) + bv);
          } else {
            float* p = partial + (size_t)si * g.B * g.LD + (size_t)nb * g.LD + r;
#pragma unroll
            for (int b = 0; b < 32; ++b)
              if (nb + b < g.B) p[(size_t)b * g.LD] = __uint_as_float(v[b]);
          }
        }
        if (last) break;
      }
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) umma::tmem_dealloc(tmem, 2 * NBT);
}

// out[i] = sum over splits (in order) of partial[s][i] (+ bias[i % LD])
template <typename TOUT>
__global__ void split_fold_kernel(const float* __restrict__ partial, const float* __restrict__ bias, TOUT* __restrict__ out,
                                  int splits, long long n, int LD) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int k = 0;
  for (; k + 4 <= splits; k += 4) {       // four independent chains: the loads overlap, the order stays fixed
    s0 += partial[(size_t)k * n + i];
    s1 += partial[(size_t)(k + 1) * n + i];
    s2 += partial[(size_t)(k + 2) * n + i];
    s3 += partial[(size_t)(k + 3) * n + i];
  }
  for (; k < splits; ++k) s0 += partial[(size_t)k * n + i];
  dd::st<TOUT>(out + i, ((s0 + s1) + (s2 + s3)) + (bias ? __ldg(bias + (i % LD)) : 0.f));
}

// ------------------------------------------------------------------------------------------------
// wgrad: dW[n][k] (+)= sum_b dy[b][n] x[b][k]; one 128 x KT output tile per stage (no accumulation across
// stages), written straight from TMEM to HBM.
// MULTI (dd_linear_wgrad_acc, B > 32): every 32-row batch chunk of an item gets a stage and a TMEM accumulator of its own;
// the epilogue sums the chunks in fp32 in the order of the chunked plain launches (D = D_0, then D = D_j + D) and only
// then adds the stored gradient: dw_old + D, not the (dw_old + D_0) + D_1 of accumulating chunk by chunk.
// ------------------------------------------------------------------------------------------------
constexpr int W_STAGES = 3;
constexpr int W_STAGE_BYTES = 4 * BOX + 8 * BOX;     // dy^T: 4 boxes of 32 n; x: up to 8 boxes of 32 k
constexpr int W_TPAD = 36;                           // floats per row of a warp's 32 x 32 transpose block
constexpr int W_EPI = 4;                             // epilogue warps (192 threads x ~118 registers: co-resides with the
constexpr int W_THREADS = 32 * (2 + W_EPI);          // data-parallel update CTA of csrc/adam.cu)
constexpr int W_SMEM = W_STAGES * W_STAGE_BYTES + W_EPI * 32 * W_TPAD * 4 + 2048;

struct WgradBars {
  uint64_t full[W_STAGES], empty[W_STAGES], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

struct WgradGeo {
  int B, N;
  long long K;
  int n_tiles, k_tiles, KT;      // KT = 128 or 256 columns per tile
  int accumulate;
  int bchunks, nbuf;             // MULTI: 32-row batch chunks per item; TMEM accumulators of bchunks * KT columns (1 or 2)
};

template <bool MULTI>
__global__ void __launch_bounds__(W_THREADS, 1) linear_wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dy,
                                                                       const __grid_constant__ CUtensorMap map_x,
                                                                       float* __restrict__ dw, const WgradGeo g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  float* stage_out = reinterpret_cast<float*>(smem + W_STAGES * W_STAGE_BYTES);
  WgradBars* bars = reinterpret_cast<WgradBars*>(smem + W_STAGES * W_STAGE_BYTES + W_EPI * 32 * W_TPAD * 4);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const long long items = (long long)g.n_tiles * g.k_tiles;
  const int xboxes = g.KT / 32;
  const uint32_t stage_tx = (4 + xboxes) * BOX;

  if (tid == 0) {
    for (int i = 0; i < W_STAGES; ++i) { umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 1); }
    for (int i = 0; i < 2; ++i) { umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], W_EPI); }
    umma::fence_mbar_init();
    umma::tma_prefetch_desc(&map_dy);
    umma::tma_prefetch_desc(&map_x);
  }
  if (warp == 1) umma::tmem_alloc(&bars->tmem_base, 512);
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  // item -> (n tile, k tile): consecutive items of a CTA share the n tile (its dy^T boxes stay in L2)
  if (warp == 0) {
    if (umma::elect_one()) {
      uint32_t c = 0;
      if (MULTI) {
        for (long long it = blockIdx.x; it < items; it += gridDim.x) {
          const int ni = (int)(it / g.k_tiles), ki = (int)(it % g.k_tiles);
          for (int bc = 0; bc < g.bchunks; ++bc, ++c) {                 // batch rows [32 bc, 32 bc + 32)
            const uint32_t s = c % W_STAGES;
            umma::mbar_wait(&bars->empty[s], ((c / W_STAGES) & 1) ^ 1);
            const uint32_t dst = umma::smem_u32(smem + s * W_STAGE_BYTES);
            umma::mbar_expect_tx(&bars->full[s], stage_tx);
#pragma unroll
            for (int i = 0; i < 4; ++i) umma::tma_load_2d(dst + i * BOX, &map_dy, ni * 128 + 32 * i, 32 * bc, &bars->full[s]);
            for (int j = 0; j < xboxes; ++j)
              umma::tma_load_2d(dst + (4 + j) * BOX, &map_x, ki * g.KT + 32 * j, 32 * bc, &bars->full[s]);
          }
        }
      } else {
        for (long long it = blockIdx.x; it < items; it += gridDim.x, ++c) {
          const int ni = (int)(it / g.k_tiles), ki = (int)(it % g.k_tiles);
          const uint32_t s = c % W_STAGES;
          umma::mbar_wait(&bars->empty[s], ((c / W_STAGES) & 1) ^ 1);
          const uint32_t dst = umma::smem_u32(smem + s * W_STAGE_BYTES);
          umma::mbar_expect_tx(&bars->full[s], stage_tx);
#pragma unroll
          for (int i = 0; i < 4; ++i) umma::tma_load_2d(dst + i * BOX, &map_dy, ni * 128 + 32 * i, 0, &bars->full[s]);
          for (int j = 0; j < xboxes; ++j) umma::tma_load_2d(dst + (4 + j) * BOX, &map_x, ki * g.KT + 32 * j, 0, &bars->full[s]);
        }
      }
    }
  } else if (warp == 1 && MULTI) {
    const uint32_t idesc = umma::make_idesc_tf32(128, g.KT, true, true);
    const uint32_t acc_cols = g.bchunks * g.KT;
    uint32_t c = 0, n_item = 0;
    for (long long it = blockIdx.x; it < items; it += gridDim.x, ++n_item) {
      const uint32_t a = n_item % g.nbuf, use = n_item / g.nbuf;
      umma::mbar_wait(&bars->acc_empty[a], (use & 1) ^ 1);
      for (int bc = 0; bc < g.bchunks; ++bc, ++c) {
        const uint32_t s = c % W_STAGES;
        umma::mbar_wait(&bars->full[s], (c / W_STAGES) & 1);
        umma::tc_fence_after_sync();
        const uint32_t base = umma::smem_u32(smem + s * W_STAGE_BYTES);
        if (umma::elect_one()) {
#pragma unroll
          for (int k = 0; k < NB / 8; ++k)
            umma::mma_tf32_lohi(tmem + a * acc_cols + bc * g.KT, umma::desc_lo(base + k * 1024, BOX), umma::desc_hi_sw128_base32(512),
                                umma::desc_lo(base + 4 * BOX + k * 1024, BOX), umma::desc_hi_sw128_base32(512), idesc, k > 0 ? 1u : 0u);
          umma::mma_commit(&bars->empty[s]);
          if (bc == g.bchunks - 1) umma::mma_commit(&bars->acc_full[a]);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = umma::make_idesc_tf32(128, g.KT, true, true);
    uint32_t c = 0;
    for (long long it = blockIdx.x; it < items; it += gridDim.x, ++c) {
      const uint32_t s = c % W_STAGES, a = c & 1;
      umma::mbar_wait(&bars->acc_empty[a], ((c >> 1) & 1) ^ 1);
      umma::mbar_wait(&bars->full[s], (c / W_STAGES) & 1);
      umma::tc_fence_after_sync();
      const uint32_t base = umma::smem_u32(smem + s * W_STAGE_BYTES);
      if (umma::elect_one()) {
#pragma unroll
        for (int k = 0; k < NB / 8; ++k)
          umma::mma_tf32_lohi(tmem + a * 256, umma::desc_lo(base + k * 1024, BOX), umma::desc_hi_sw128_base32(512),
                              umma::desc_lo(base + 4 * BOX + k * 1024, BOX), umma::desc_hi_sw128_base32(512), idesc, k > 0 ? 1u : 0u);
        umma::mma_commit(&bars->empty[s]);
        umma::mma_commit(&bars->acc_full[a]);
      }
      __syncwarp();
    }
  } else {
    const int quarter = warp & 3;
    uint32_t c = 0;
    for (long long it = blockIdx.x; it < items; it += gridDim.x, ++c) {
      const int ni = (int)(it / g.k_tiles), ki = (int)(it % g.k_tiles);
      const uint32_t a = MULTI ? c % g.nbuf : c & 1;
      umma::mbar_wait_sleep(&bars->acc_full[a], MULTI ? (c / g.nbuf) & 1 : (c >> 1) & 1);
      umma::tc_fence_after_sync();
      const int n0 = ni * 128 + quarter * 32;
      const long long k0 = (long long)ki * g.KT;
      float* blk = stage_out + (warp - 2) * (32 * W_TPAD);
      for (int cb = 0; cb < g.KT; cb += 32) {
        uint32_t v[32];
        if (MULTI) {
          const uint32_t col = tmem + ((uint32_t)(quarter * 32) << 16) + a * g.bchunks * g.KT + cb;
          umma::tmem_ld_32x32(col, v);
          umma::tmem_ld_wait();
          for (int bc = 1; bc < g.bchunks; ++bc) {
            uint32_t u[32];
            umma::tmem_ld_32x32(col + bc * g.KT, u);
            umma::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(u[i]) + __uint_as_float(v[i]));
          }
        } else {
          umma::tmem_ld_32x32(tmem + ((uint32_t)(quarter * 32) << 16) + a * 256 + cb, v);
          umma::tmem_ld_wait();
        }
        // lane = row n0 + lane holds 32 consecutive k: transpose through shared memory so that each store
        // instruction below writes four whole 128-byte row segments instead of 32 scattered 16-byte pieces
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<float4*>(blk + lane * W_TPAD + 4 * q) =
              make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                          __uint_as_float(v[4 * q + 3]));
        __syncwarp();
        const int cq = lane & 7;
#pragma unroll
        for (int itr = 0; itr < 8; ++itr) {
          const int r = (lane >> 3) + 4 * itr;
          const int n = n0 + r;
          const long long k = k0 + cb + 4 * cq;
          if (n < g.N && k < g.K) {                 // K % 4 == 0
            float4 o = *reinterpret_cast<const float4*>(blk + r * W_TPAD + 4 * cq);
            float4* dst = reinterpret_cast<float4*>(dw + (size_t)n * g.K + k);
            if (g.accumulate) { const float4 old = *dst; o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
            __stcs(dst, o);
          }
        }
      }
      umma::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) umma::mbar_arrive(&bars->acc_empty[a]);
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) umma::tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
// backward + Adam (world size 1): per 32 n x 128 k weight tile, ONE pass over W and its two moments
//   dgrad  dx[b][k] += sum_n dy[b][n] W[n][k]    the MMAs of MODE 1 above, same order (bit-identical dx)
//   wgrad  G^T[k][n] = sum_b x[b][k] dy[b][n]    D[128 k x 32 n]: A = x tile, B = dy chunk, both MN-major
//   Adam   W, m, v tiles updated in shared memory from G^T (TMEM), then stored by TMA in place
// The W tile is loaded once and serves as the dgrad operand and the Adam input; the weight gradient never reaches HBM:
// 24 bytes per parameter instead of 4 (dgrad) + 4 (wgrad) + 28 (Adam) + 4 (dW read back).
// Work decomposition, split plan and split partials are those of the dgrad kernel.  Warp roles (352 threads): warp 0 = TMA
// producer, warp 1 = MMA issuer + TMEM owner, warps 2..9 = epilogue (two per TMEM lane quarter, 16 n rows each), warp 10 =
// TMA stores of the updated tiles (a stage goes back to the producer as soon as its stores have read it).
// The W / m / v boxes use the SWIZZLE_128B_ATOM_32B layout of the MN-major dgrad operand for the load AND the store
// (tools/tma_store_atom32_probe.cu): element (row r, column c) of a 32 x 32 box sits in 32-byte atom (c / 8) ^ (r % 4)
// of its 128-byte row.
// ------------------------------------------------------------------------------------------------
//
// Accumulating form (ACC, dd_linear_bwd_adam_acc): the stage also carries the tile of a stored partial gradient G (the
// earlier backward passes of a gradient-accumulation window), loaded in the same boxes as W, m and v, and the epilogue
// steps with dW_chunk + G -- 28 bytes per parameter.  A fourth 16 KB tile per stage would need 250 KB at three stages, over
// the 227 KB of a block: this instantiation runs two stages (178 KB).
constexpr int BA_STAGES = 3;                          // stages of the plain form (and the size of the barrier arrays)
constexpr int BA_TILE = 4 * BOX;                      // W, m, v or G: [32 n][128 k] as 4 boxes of 32 k
constexpr int BA_EPI = 8;
constexpr int BA_THREADS = 32 * (3 + BA_EPI);
template <bool ACC> struct BaCfg {
  static constexpr int STAGES = ACC ? 2 : BA_STAGES;
  static constexpr int DY_OFF = (ACC ? 4 : 3) * BA_TILE;    // W, m, v (, G); then the dy chunk MN-major (wgrad) and K-major (dgrad)
  static constexpr int STAGE_BYTES = DY_OFF + 2 * BOX;
  static constexpr int SMEM = STAGES * STAGE_BYTES + 2 * BA_TILE + 2048;   // + x [32 b][128 k], double-buffered per item
};

struct BwdAdamBars {
  uint64_t full[BA_STAGES], empty[BA_STAGES], tile_ready[BA_STAGES], x_full[2], x_empty[2], g_full[2], g_empty[2], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
};

// shared-memory accesses by address (the tile pointer went through align1024: plain C++ would compile to generic LD / ST)
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
// Gradient norm (NORM, dd_linear_bwd_adam_sumsq): each epilogue thread adds the square of every gradient element it hands
// adam_one, in fp64, for the elements inside the [rows x g.LD] weight only (a ragged edge tile's padding is masked, not
// assumed zero); the epilogue warps fold their threads in a fixed order and dd::sumsq_fold_grid folds the CTAs into *out.
struct SumsqSink {
  dd::SumsqWorkspace* ws;
  double* out;
  int rows;                                           // N
};
// TMEM columns: [0, 64) dgrad accumulator of the item (x 2), [64, 128) G^T of the chunk (x 2)
// map_g (the stored partial gradient, ACC only) and then sink (NORM only) come last, so that the plain instantiation keeps its
// parameter layout
template <typename TOUT, bool ACC, bool NORM = false>
__global__ void __launch_bounds__(BA_THREADS, 1) linear_bwd_adam_tc_kernel(
    const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_m, const __grid_constant__ CUtensorMap map_v,
    const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_dyt, const __grid_constant__ CUtensorMap map_x,
    TOUT* __restrict__ dx, float* __restrict__ partial, StreamGeo g, const dd::AdamHyper h, const __grid_constant__ CUtensorMap map_g,
    SumsqSink sink) {
  constexpr int STAGES = BaCfg<ACC>::STAGES, STAGE_BYTES = BaCfg<ACC>::STAGE_BYTES, DY_OFF = BaCfg<ACC>::DY_OFF;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint8_t* xbuf = smem + STAGES * STAGE_BYTES;
  BwdAdamBars* bars = reinterpret_cast<BwdAdamBars*>(xbuf + 2 * BA_TILE);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int items = g.tiles * g.splits;
  const bool has_dx = dx != nullptr;

  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      umma::mbar_init(&bars->full[i], 1); umma::mbar_init(&bars->empty[i], 1); umma::mbar_init(&bars->tile_ready[i], BA_EPI);
    }
    for (int i = 0; i < 2; ++i) {
      umma::mbar_init(&bars->x_full[i], 1); umma::mbar_init(&bars->x_empty[i], 1);
      umma::mbar_init(&bars->g_full[i], 1); umma::mbar_init(&bars->g_empty[i], BA_EPI);
      umma::mbar_init(&bars->acc_full[i], 1); umma::mbar_init(&bars->acc_empty[i], BA_EPI);
    }
    umma::fence_mbar_init();
    umma::tma_prefetch_desc(&map_w); umma::tma_prefetch_desc(&map_m); umma::tma_prefetch_desc(&map_v);
    umma::tma_prefetch_desc(&map_dy); umma::tma_prefetch_desc(&map_dyt); umma::tma_prefetch_desc(&map_x);
    if (ACC) umma::tma_prefetch_desc(&map_g);
  }
  if (warp == 1) umma::tmem_alloc(&bars->tmem_base, 128);
  const uint32_t tmem = umma::tmem_publish(&bars->tmem_base);

  if (warp == 0) {
    // =========================== TMA producer ===================================================
    if (umma::elect_one()) {
      const uint32_t stage_tx = has_dx ? STAGE_BYTES : STAGE_BYTES - BOX;
      uint32_t c = 0, n_item = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x, ++n_item) {
        const int ti = it % g.tiles, si = it / g.tiles;
        const int c0 = si * g.chunks_per_split;
        const int c1 = min(c0 + g.chunks_per_split, g.chunks);
        const uint32_t xb = n_item & 1;
        umma::mbar_wait(&bars->x_empty[xb], ((n_item >> 1) & 1) ^ 1);
        umma::mbar_expect_tx(&bars->x_full[xb], BA_TILE);
#pragma unroll
        for (int i = 0; i < 4; ++i)                                                           // x[b][k tile], 4 x 32 k
          umma::tma_load_2d(umma::smem_u32(xbuf + xb * BA_TILE + i * BOX), &map_x, ti * 128 + 32 * i, 0, &bars->x_full[xb]);
        for (int ch = c0; ch < c1; ++ch, ++c) {
          const uint32_t s = c % STAGES;
          umma::mbar_wait(&bars->empty[s], ((c / STAGES) & 1) ^ 1);
          const uint32_t dst = umma::smem_u32(smem + s * STAGE_BYTES);
          umma::mbar_expect_tx(&bars->full[s], stage_tx);
#pragma unroll
          for (int i = 0; i < 4; ++i) {                                                       // [n chunk][k tile], 4 x 32 k
            umma::tma_load_2d(dst + i * BOX, &map_w, ti * 128 + 32 * i, ch * kChunk, &bars->full[s]);
            umma::tma_load_2d(dst + BA_TILE + i * BOX, &map_m, ti * 128 + 32 * i, ch * kChunk, &bars->full[s]);
            umma::tma_load_2d(dst + 2 * BA_TILE + i * BOX, &map_v, ti * 128 + 32 * i, ch * kChunk, &bars->full[s]);
            if (ACC) umma::tma_load_2d(dst + 3 * BA_TILE + i * BOX, &map_g, ti * 128 + 32 * i, ch * kChunk, &bars->full[s]);
          }
          umma::tma_load_2d(dst + DY_OFF, &map_dyt, ch * kChunk, 0, &bars->full[s]);             // dy[b][chunk], MN-major
          if (has_dx) umma::tma_load_2d(dst + DY_OFF + BOX, &map_dy, ch * kChunk, 0, &bars->full[s]);  // ... K-major
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer =======================================================
    constexpr uint32_t idesc_d = umma::make_idesc_tf32(128, NB, true, false);   // dgrad, as MODE 1
    constexpr uint32_t idesc_g = umma::make_idesc_tf32(128, NB, true, true);    // G^T = x^T dy
    uint32_t c = 0, n_item = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x, ++n_item) {
      const int si = it / g.tiles;
      const int c0 = si * g.chunks_per_split;
      const int c1 = min(c0 + g.chunks_per_split, g.chunks);
      const uint32_t a = n_item & 1;
      if (has_dx) umma::mbar_wait(&bars->acc_empty[a], ((n_item >> 1) & 1) ^ 1);
      umma::mbar_wait(&bars->x_full[a], (n_item >> 1) & 1);
      const uint32_t xbase = umma::smem_u32(xbuf + a * BA_TILE);
      for (int ch = c0; ch < c1; ++ch, ++c) {
        const uint32_t s = c % STAGES, ga = c & 1;
        umma::mbar_wait(&bars->full[s], (c / STAGES) & 1);
        umma::mbar_wait(&bars->g_empty[ga], ((c >> 1) & 1) ^ 1);
        umma::tc_fence_after_sync();
        const uint32_t base = umma::smem_u32(smem + s * STAGE_BYTES);
        if (umma::elect_one()) {
          if (has_dx) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma::mma_tf32_lohi(tmem + a * NB, umma::desc_lo(base + k * 1024, BOX), umma::desc_hi_sw128_base32(512),
                                  umma::desc_lo(base + DY_OFF + BOX + k * 32, 16), umma::desc_hi_sw128(1024), idesc_d,
                                  (ch > c0 || k > 0) ? 1u : 0u);
          }
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma::mma_tf32_lohi(tmem + 2 * NB + ga * NB, umma::desc_lo(xbase + k * 1024, BOX), umma::desc_hi_sw128_base32(512),
                                umma::desc_lo(base + DY_OFF + k * 1024, BOX), umma::desc_hi_sw128_base32(512), idesc_g,
                                k > 0 ? 1u : 0u);
          umma::mma_commit(&bars->g_full[ga]);          // also: the dgrad MMAs are done reading the old W tile
          if (ch == c1 - 1) {
            if (has_dx) umma::mma_commit(&bars->acc_full[a]);
            umma::mma_commit(&bars->x_empty[a]);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 2 + BA_EPI) {
    // =========================== TMA stores of the updated W / m / v tiles ===========================
    if (umma::elect_one()) {
      uint32_t c = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x) {
        const int ti = it % g.tiles, si = it / g.tiles;
        const int c0 = si * g.chunks_per_split;
        const int c1 = min(c0 + g.chunks_per_split, g.chunks);
        for (int ch = c0; ch < c1; ++ch, ++c) {
          const uint32_t s = c % STAGES;
          umma::mbar_wait_sleep(&bars->tile_ready[s], (c / STAGES) & 1);
          const uint32_t src = umma::smem_u32(smem + s * STAGE_BYTES);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            umma::tma_store_2d(&map_w, src + i * BOX, ti * 128 + 32 * i, ch * kChunk);
            umma::tma_store_2d(&map_m, src + BA_TILE + i * BOX, ti * 128 + 32 * i, ch * kChunk);
            umma::tma_store_2d(&map_v, src + 2 * BA_TILE + i * BOX, ti * 128 + 32 * i, ch * kChunk);
          }
          umma::bulk_commit_group();
          umma::bulk_wait_group_read<0>();
          umma::mbar_arrive(&bars->empty[s]);
        }
      }
      umma::bulk_wait_group<0>();
    }
  } else {
    // =========================== epilogue (warps 2..9) =============================================
    // thread = k lane (quarter * 32 + lane of the tile: box `quarter`, column `lane`), 16 n rows (half `sub` of the chunk)
    const int quarter = warp & 3, sub = (warp - 2) >> 2;
    uint32_t c = 0, n_item = 0;
    double nacc = 0.0;
    for (int it = blockIdx.x; it < items; it += gridDim.x, ++n_item) {
      const int ti = it % g.tiles, si = it / g.tiles;
      const int c0 = si * g.chunks_per_split;
      const int c1 = min(c0 + g.chunks_per_split, g.chunks);
      const bool k_in = ti * 128 + quarter * 32 + lane < g.LD;
      for (int ch = c0; ch < c1; ++ch, ++c) {
        const uint32_t s = c % STAGES, ga = c & 1;
        umma::mbar_wait_sleep(&bars->g_full[ga], (c >> 1) & 1);
        umma::tc_fence_after_sync();
        uint32_t gv[16];
        umma::tmem_ld_32x16(tmem + ((uint32_t)(quarter * 32) << 16) + 2 * NB + ga * NB + sub * 16, gv);
        umma::tmem_ld_wait();
        umma::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&bars->g_empty[ga]);
        const uint32_t wt = umma::smem_u32(smem + s * STAGE_BYTES + quarter * BOX);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int r = sub * 16 + j;
          const uint32_t e = wt + 4 * (r * 32 + ((((lane >> 3) ^ (r & 3)) << 3) | (lane & 7)));
          float m = lds_f32(e + BA_TILE), v = lds_f32(e + 2 * BA_TILE);
          float gr = __uint_as_float(gv[j]);
          if (ACC) gr = gr + lds_f32(e + 3 * BA_TILE);     // dd_linear_wgrad_acc's dW_chunk + G, bit for bit
          if (NORM && k_in && ch * kChunk + r < sink.rows) nacc += dd::sq(gr);
          const float p = dd::adam_one(lds_f32(e), gr, m, v, h);
          sts_f32(e, p);
          sts_f32(e + BA_TILE, m);
          sts_f32(e + 2 * BA_TILE, v);
        }
        umma::fence_proxy_async_smem();             // the writes above, then the TMA stores of warp 2 + BA_EPI
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&bars->tile_ready[s]);
        if (has_dx && ch == c1 - 1) {
          // the item's input gradient, as the dgrad kernel writes it (this warp: 16 of the 32 batch rows)
          const uint32_t a = n_item & 1;
          umma::mbar_wait_sleep(&bars->acc_full[a], (n_item >> 1) & 1);
          umma::tc_fence_after_sync();
          uint32_t v[16];
          umma::tmem_ld_32x16(tmem + ((uint32_t)(quarter * 32) << 16) + a * NB + sub * 16, v);
          umma::tmem_ld_wait();
          umma::tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) umma::mbar_arrive(&bars->acc_empty[a]);
          const int r = ti * 128 + quarter * 32 + lane;
          if (r < g.LD) {
            if (g.splits == 1) {
#pragma unroll
              for (int b = 0; b < 16; ++b)       // + 0.f as the dgrad kernel adds its (absent) bias: -0 is written as +0
                if (sub * 16 + b < g.B) dd::st<TOUT>(dx + (size_t)(sub * 16 + b) * g.LD + r, __uint_as_float(v[b]) + 0.f);
            } else {
              float* p = partial + (size_t)si * g.B * g.LD + r;
#pragma unroll
              for (int b = 0; b < 16; ++b)
                if (sub * 16 + b < g.B) p[(size_t)(sub * 16 + b) * g.LD] = __uint_as_float(v[b]);
            }
          }
        }
      }
    }
    if constexpr (NORM) {
      __shared__ double sred[BA_EPI];
      nacc = dd::warp_sum(nacc);
      if (lane == 0) sred[warp - 2] = nacc;
      asm volatile("bar.sync 1, %0;" ::"n"(32 * BA_EPI) : "memory");     // the epilogue warps only
      if (warp == 2) {
        double cta = 0.0;
        for (int w = 0; w < BA_EPI; ++w) cta += sred[w];
        dd::sumsq_fold_grid(sink.ws, cta, sink.out);
      }
    }
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) umma::tmem_dealloc(tmem, 128);
}

// split the contraction so that ~kSMs work items exist; rows = 128-row output tiles
void plan_stream(int tiles, int chunks, int& splits, int& cps) {
  splits = 1;
  if (tiles < dd::kSMs) {
    splits = dd::kSMs / tiles;
    const int maxs = (chunks + 7) / 8;            // at least 8 chunks (256 contraction elements) per split
    if (splits > maxs) splits = maxs;
    if (splits < 1) splits = 1;
  }
  cps = (chunks + splits - 1) / splits;
  splits = (chunks + cps - 1) / cps;
}

}  // namespace

namespace dd {

bool linear_tc_supported(int B, int N, long long K) {
  // TMA needs 16-byte row pitches; the streaming design pays off only for wide layers
  return B >= 1 && N % 4 == 0 && K % 4 == 0 && (long long)N * K >= (1ll << 22) && tma_available();
}

size_t linear_tc_workspace_bytes(int B, int N, long long K) {
  const int Bf = B < kLinearTcMaxRows ? B : kLinearTcMaxRows;     // forward: up to 256 rows per pass
  const int Bd = B < NB ? B : NB;                                 // input gradient: 32
  int s1, c1, s2, c2;
  plan_stream(ceil_div(N, 128), ceil_div(K, kChunk), s1, c1);      // fwd: tiles over N, contraction K
  plan_stream(ceil_div(K, 128), ceil_div(N, kChunk), s2, c2);      // dgrad: tiles over K, contraction N
  const size_t a = s1 > 1 ? (size_t)s1 * Bf * N * sizeof(float) : 0;
  const size_t b = s2 > 1 ? (size_t)s2 * Bd * K * sizeof(float) : 0;
  return (a > b ? a : b) + 256;
}

template <int NBT>
int launch_fwd(const CUtensorMap& mw, const CUtensorMap& mx, const float* bias, float* y, float* ws, const StreamGeo& g,
               cudaStream_t st) {
  auto k = linear_stream_tc_kernel<0, float, NBT>;
  if (int e = set_smem(k, SCfg<NBT>::SMEM, Carveout::kMaxShared, "linear_tc")) return e;
  const int items = g.tiles * g.splits;
  k<<<items < kSMs ? items : kSMs, THREADS, SCfg<NBT>::SMEM, st>>>(mw, mx, bias, y, ws, g);
  return check_launch("linear_fwd_tc");
}

// x fp32 [B][K] (B <= 256: one pass over the weights), W fp32 [N][K], y fp32 [B][N]
int linear_fwd_tc(const float* x, const float* w, const float* bias, float* y, void* ws, size_t ws_bytes, int B, int N,
                  long long K, cudaStream_t st) {
  if (B > kLinearTcMaxRows) return fail(DD_ERR_UNSUPPORTED, "linear_fwd_tc: %d rows per pass (max %d)", B, kLinearTcMaxRows);
  StreamGeo g;
  g.B = B; g.LD = N;
  g.tiles = ceil_div(N, 128);
  g.chunks = ceil_div(K, kChunk);
  plan_stream(g.tiles, g.chunks, g.splits, g.chunks_per_split);
  if (g.splits > 1 && ws_bytes < (size_t)g.splits * B * N * sizeof(float))
    return fail(DD_ERR_WORKSPACE, "linear_fwd_tc: workspace %zu too small for %d splits", ws_bytes, g.splits);
  const int nbt = B <= 32 ? 32 : B <= 64 ? 64 : B <= 128 ? 128 : 256;
  CUtensorMap mw, mx;
  char msg[256];
  if (tma_map_2d(&mw, w, 4, N, K, K, 32, 128, CU_TENSOR_MAP_SWIZZLE_128B, msg, sizeof msg) ||
      tma_map_2d(&mx, x, 4, B, K, K, 32, nbt, CU_TENSOR_MAP_SWIZZLE_128B, msg, sizeof msg))
    return fail(DD_ERR_UNSUPPORTED, "linear_fwd_tc: %s", msg);
  int e = nbt == 32 ? launch_fwd<32>(mw, mx, bias, y, (float*)ws, g, st)
        : nbt == 64 ? launch_fwd<64>(mw, mx, bias, y, (float*)ws, g, st)
        : nbt == 128 ? launch_fwd<128>(mw, mx, bias, y, (float*)ws, g, st)
                     : launch_fwd<256>(mw, mx, bias, y, (float*)ws, g, st);
  if (e) return e;
  if (g.splits > 1) {
    const long long n = (long long)B * N;
    split_fold_kernel<float><<<ceil_div(n, 256), 256, 0, st>>>((const float*)ws, bias, y, g.splits, n, N);
    return check_launch("linear_fwd_fold");
  }
  return 0;
}

// dy fp32 [B][N], W fp32 [N][K], dx [B][K] fp32 or bf16
int linear_dgrad_tc(const float* dy, const float* w, void* dx, int dx_dtype, void* ws, size_t ws_bytes, int B, int N,
                    long long K, cudaStream_t st) {
  StreamGeo g;
  g.B = B; g.LD = (int)K;
  g.tiles = ceil_div(K, 128);
  g.chunks = ceil_div(N, kChunk);
  plan_stream(g.tiles, g.chunks, g.splits, g.chunks_per_split);
  if (g.splits > 1 && ws_bytes < (size_t)g.splits * B * K * sizeof(float))
    return fail(DD_ERR_WORKSPACE, "linear_dgrad_tc: workspace %zu too small for %d splits", ws_bytes, g.splits);
  CUtensorMap mw, mdy;
  char msg[256];
  if (tma_map_2d(&mw, w, 4, N, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      tma_map_2d(&mdy, dy, 4, B, N, N, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B, msg, sizeof msg))
    return fail(DD_ERR_UNSUPPORTED, "linear_dgrad_tc: %s", msg);
  const int items = g.tiles * g.splits;
  const int grid = items < kSMs ? items : kSMs;
  const long long n = (long long)B * K;
  if (dx_dtype == DD_F32) {
    auto k = linear_stream_tc_kernel<1, float>;
    if (int e = set_smem(k, SCfg<NB>::SMEM, Carveout::kMaxShared, "linear_tc")) return e;
    k<<<grid, THREADS, SCfg<NB>::SMEM, st>>>(mw, mdy, nullptr, (float*)dx, (float*)ws, g);
    if (int e = check_launch("linear_dgrad_tc")) return e;
    if (g.splits > 1) split_fold_kernel<float><<<ceil_div(n, 256), 256, 0, st>>>((const float*)ws, nullptr, (float*)dx, g.splits, n, (int)K);
  } else {
    auto k = linear_stream_tc_kernel<1, __nv_bfloat16>;
    if (int e = set_smem(k, SCfg<NB>::SMEM, Carveout::kMaxShared, "linear_tc")) return e;
    k<<<grid, THREADS, SCfg<NB>::SMEM, st>>>(mw, mdy, nullptr, (__nv_bfloat16*)dx, (float*)ws, g);
    if (int e = check_launch("linear_dgrad_tc")) return e;
    if (g.splits > 1)
      split_fold_kernel<__nv_bfloat16><<<ceil_div(n, 256), 256, 0, st>>>((const float*)ws, nullptr, (__nv_bfloat16*)dx, g.splits, n, (int)K);
  }
  return g.splits > 1 ? check_launch("linear_dgrad_fold") : 0;
}

template <bool ACC, bool NORM, typename TOUT>
int launch_bwd_adam(const CUtensorMap (&maps)[7], TOUT* dx, float* ws, const StreamGeo& g, const AdamHyper& h, const SumsqSink& sink,
                    cudaStream_t st) {
  auto k = linear_bwd_adam_tc_kernel<TOUT, ACC, NORM>;
  if (int e = set_smem(k, BaCfg<ACC>::SMEM, Carveout::kMaxShared, "linear_tc")) return e;
  const int items = g.tiles * g.splits;
  k<<<items < kSMs ? items : kSMs, BA_THREADS, BaCfg<ACC>::SMEM, st>>>(maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], dx, ws,
                                                                       g, h, maps[6], sink);
  return check_launch("linear_bwd_adam_tc");
}

template <typename TOUT>
int launch_bwd_adam_any(bool acc, const CUtensorMap (&maps)[7], TOUT* dx, float* ws, const StreamGeo& g, const AdamHyper& h,
                        const SumsqSink& sink, cudaStream_t st) {
  if (sink.out)
    return acc ? launch_bwd_adam<true, true>(maps, dx, ws, g, h, sink, st) : launch_bwd_adam<false, true>(maps, dx, ws, g, h, sink, st);
  return acc ? launch_bwd_adam<true, false>(maps, dx, ws, g, h, sink, st) : launch_bwd_adam<false, false>(maps, dx, ws, g, h, sink, st);
}

// dy fp32 [B][N], x fp32 [B][K], W / m / v fp32 [N][K] updated in place; dx [B][K] fp32 or bf16 from the old W, or nullptr;
// gpart fp32 [N][K]: the stored partial gradient added to this pass's weight gradient before the step, or nullptr;
// sumsq / sumsq_ws: *sumsq = the sum of squares of the gradient the step applies (NORM), or nullptr
int linear_bwd_adam_tc(const float* dy, const float* x, float* w, float* m, float* v, const float* gpart, void* dx, int dx_dtype,
                       void* ws, size_t ws_bytes, int B, int N, long long K, const AdamHyper& h, double* sumsq,
                       SumsqWorkspace* sumsq_ws, cudaStream_t st) {
  StreamGeo g;
  g.B = B; g.LD = (int)K;
  g.tiles = ceil_div(K, 128);
  g.chunks = ceil_div(N, kChunk);
  plan_stream(g.tiles, g.chunks, g.splits, g.chunks_per_split);
  if (dx && g.splits > 1 && ws_bytes < (size_t)g.splits * B * K * sizeof(float))
    return fail(DD_ERR_WORKSPACE, "linear_bwd_adam_tc: workspace %zu too small for %d splits", ws_bytes, g.splits);
  CUtensorMap maps[7] = {};      // W, m, v, dy K-major, dy MN-major, x, G (the plain form passes an unused zero map)
  char msg[256];
  if (tma_map_2d(&maps[0], w, 4, N, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      tma_map_2d(&maps[1], m, 4, N, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      tma_map_2d(&maps[2], v, 4, N, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      tma_map_2d(&maps[3], dy, 4, B, N, N, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B, msg, sizeof msg) ||
      tma_map_2d(&maps[4], dy, 4, B, N, N, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      tma_map_2d(&maps[5], x, 4, B, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      (gpart && tma_map_2d(&maps[6], gpart, 4, N, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg)))
    return fail(DD_ERR_UNSUPPORTED, "linear_bwd_adam_tc: %s", msg);
  const long long n = (long long)B * K;
  const SumsqSink sink = {sumsq_ws, sumsq, N};
  if (dx_dtype == DD_BF16 && dx) {
    auto* d = (__nv_bfloat16*)dx;
    if (int e = launch_bwd_adam_any(gpart != nullptr, maps, d, (float*)ws, g, h, sink, st)) return e;
    if (g.splits > 1)
      split_fold_kernel<__nv_bfloat16><<<ceil_div(n, 256), 256, 0, st>>>((const float*)ws, nullptr, d, g.splits, n, (int)K);
  } else {
    auto* d = (float*)dx;
    if (int e = launch_bwd_adam_any(gpart != nullptr, maps, d, (float*)ws, g, h, sink, st)) return e;
    if (dx && g.splits > 1)
      split_fold_kernel<float><<<ceil_div(n, 256), 256, 0, st>>>((const float*)ws, nullptr, d, g.splits, n, (int)K);
  }
  return dx && g.splits > 1 ? check_launch("linear_bwd_adam_fold") : 0;
}

// dy fp32 [B][N], x fp32 [B][K] -> dW fp32 [N][K] (overwritten, or accumulated into)
int linear_wgrad_tc(const float* dy, const float* x, float* dw, int B, int N, long long K, int accumulate, cudaStream_t st) {
  WgradGeo g = {};
  g.B = B; g.N = N; g.K = K;
  g.KT = K >= 256 ? 256 : 128;
  g.n_tiles = ceil_div(N, 128);
  g.k_tiles = ceil_div(K, g.KT);
  g.accumulate = accumulate;
  CUtensorMap mdy, mx;
  char msg[256];
  if (tma_map_2d(&mdy, dy, 4, B, N, N, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      tma_map_2d(&mx, x, 4, B, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg))
    return fail(DD_ERR_UNSUPPORTED, "linear_wgrad_tc: %s", msg);
  const long long items = (long long)g.n_tiles * g.k_tiles;
  const int grid = (int)(items < kSMs ? items : kSMs);
  if (int e = set_smem(linear_wgrad_tc_kernel<false>, W_SMEM, Carveout::kMaxShared, "linear_tc")) return e;
  linear_wgrad_tc_kernel<false><<<grid, W_THREADS, W_SMEM, st>>>(mdy, mx, dw, g);
  return check_launch("linear_wgrad_tc");
}

// dy fp32 [B][N], x fp32 [B][K], 32 < B <= 128 -> dW fp32 [N][K] += the sum of the 32-row chunks' products, which are added
// up before the old value (one launch; the batch chunks of an item share its TMEM)
int linear_wgrad_acc_multi_tc(const float* dy, const float* x, float* dw, int B, int N, long long K, cudaStream_t st) {
  WgradGeo g = {};
  g.B = B; g.N = N; g.K = K;
  g.KT = K >= 256 ? 256 : 128;
  g.bchunks = ceil_div(B, NB);
  if (g.bchunks * g.KT > 512) g.KT = 128;
  if (g.bchunks * g.KT > 512)
    return fail(DD_ERR_UNSUPPORTED, "linear_wgrad_acc_tc: %d rows exceed the %d TMEM columns (at most %d)", B, 512, 4 * NB);
  g.nbuf = g.bchunks * g.KT <= 256 ? 2 : 1;
  g.n_tiles = ceil_div(N, 128);
  g.k_tiles = ceil_div(K, g.KT);
  g.accumulate = 1;
  CUtensorMap mdy, mx;
  char msg[256];
  if (tma_map_2d(&mdy, dy, 4, B, N, N, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
      tma_map_2d(&mx, x, 4, B, K, K, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg))
    return fail(DD_ERR_UNSUPPORTED, "linear_wgrad_acc_tc: %s", msg);
  const long long items = (long long)g.n_tiles * g.k_tiles;
  const int grid = (int)(items < kSMs ? items : kSMs);
  if (int e = set_smem(linear_wgrad_tc_kernel<true>, W_SMEM, Carveout::kMaxShared, "linear_tc")) return e;
  linear_wgrad_tc_kernel<true><<<grid, W_THREADS, W_SMEM, st>>>(mdy, mx, dw, g);
  return check_launch("linear_wgrad_acc_tc");
}

}  // namespace dd
