// Skinny linear layers on the CUDA cores: y[B,N] = x[B,K] W[N,K]^T + bias with a small batch
// (B <= 32 per launch; larger batches are chunked by the host wrapper below) and a very wide
// K (Encoder.fc1: K = 940,032, components.py:26,105) or a very wide N (roadmap head:
// N = 640,000, roadmap_bce_v2.py:50,75; Decoder.fc2: N = 1,253,376, components.py:69).
// fp32 weights / accumulation: this is the fp32 parity path and the on-device check for the
// tensor-core weight-streaming kernels in linear_tc.cu.  All three passes stream W exactly once
// per 32 batch rows; reductions over split K / split N go through ordered partial buffers.
#include "adam.cuh"
#include "dd_common.cuh"

namespace {

constexpr int NTHREADS = 256;

// ---------------------------------------------------------------- forward -----------------
// CTA: 8 warps x NR=2 rows each (16 rows of W), K range [k0,k1) in sub-chunks of KC floats staged
// in smem for the whole batch tile.  Lane owns float4 columns; partial sums over lanes are folded
// with a halving butterfly (31 shuffles per 32 values).
constexpr int KC = 512;
constexpr int NR = 2;

template <int BT>
__device__ __forceinline__ float butterfly_reduce(float (&v)[BT], int lane) {
  // After the loop lane l holds the full sum of element (l % BT) (BT <= 32, power of two).
#pragma unroll
  for (int half = BT / 2, step = 16; half >= 1; half >>= 1, step >>= 1) {
    const bool upper = (lane & step) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = upper ? v[i] : v[i + half];
      const float keep = upper ? v[i + half] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, step);
    }
  }
  float r = v[0];
  // BT < 32: lanes that differ only in the untouched low-order lane bits still hold partial sums
#pragma unroll
  for (int step = 16 / BT; step >= 1; step >>= 1) r += __shfl_xor_sync(0xffffffffu, r, step);
  return r;   // lane l holds element l / (32 / BT)
}

template <typename T, int BT>
__global__ void __launch_bounds__(NTHREADS) linear_fwd_simt(const T* __restrict__ x, const float* __restrict__ w,
                                                            const float* __restrict__ bias, float* __restrict__ y,
                                                            float* __restrict__ partial, int B, int N, long long K,
                                                            long long kchunk) {
  extern __shared__ __align__(16) float s_x[];   // [BT][KC]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n0 = (blockIdx.x * 8 + warp) * NR;
  const long long k0 = (long long)blockIdx.y * kchunk;
  const long long k1 = k0 + kchunk < K ? k0 + kchunk : K;
  float acc[NR][BT];
#pragma unroll
  for (int r = 0; r < NR; ++r)
#pragma unroll
    for (int b = 0; b < BT; ++b) acc[r][b] = 0.f;

  for (long long kb = k0; kb < k1; kb += KC) {
    const int kc = (int)(k1 - kb < KC ? k1 - kb : KC);   // multiple of 4
    __syncthreads();
    for (int i = tid; i < BT * (KC / 4); i += NTHREADS) {
      const int b = i / (KC / 4), q = i - b * (KC / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b < B && q * 4 < kc) {
        const T* p = x + (size_t)b * K + kb + q * 4;
        v = make_float4(dd::ld<T>(p), dd::ld<T>(p + 1), dd::ld<T>(p + 2), dd::ld<T>(p + 3));
      }
      reinterpret_cast<float4*>(s_x)[b * (KC / 4) + q] = v;
    }
    __syncthreads();
    for (int q = lane; q * 4 < kc; q += 32) {
      float4 wv[NR];
#pragma unroll
      for (int r = 0; r < NR; ++r)
        wv[r] = (n0 + r < N) ? __ldcs(reinterpret_cast<const float4*>(w + (size_t)(n0 + r) * K + kb) + q)
                             : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int b = 0; b < BT; ++b) {
        const float4 xv = reinterpret_cast<const float4*>(s_x)[b * (KC / 4) + q];
#pragma unroll
        for (int r = 0; r < NR; ++r)
          acc[r][b] = fmaf(xv.x, wv[r].x, fmaf(xv.y, wv[r].y, fmaf(xv.z, wv[r].z, fmaf(xv.w, wv[r].w, acc[r][b]))));
      }
    }
  }
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    const float tot = butterfly_reduce<BT>(acc[r], lane);
    constexpr int REP = 32 / BT;   // lanes l*REP .. l*REP+REP-1 all hold element l
    const int b = lane / REP;
    const int n = n0 + r;
    if (lane % REP == 0 && b < B && n < N) {
      if (gridDim.y == 1) y[(size_t)b * N + n] = tot + (bias ? __ldg(bias + n) : 0.f);
      else partial[((size_t)blockIdx.y * B + b) * N + n] = tot;
    }
  }
}

__global__ void splitk_reduce_kernel(const float* __restrict__ partial, const float* __restrict__ bias,
                                     float* __restrict__ y, int splits, long long bn, int N) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= bn) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += partial[(size_t)k * bn + i];
  y[i] = s + (bias ? __ldg(bias + (i % N)) : 0.f);
}

// ---------------------------------------------------------------- dgrad -------------------
// dx[b,k] = sum_n dy[b,n] W[n,k].  Thread owns a float4 of k; KT threads span k, NS = 256/KT
// n-lanes stride over the CTA's n range; dy is staged [n][b] in smem (swizzled float4 slots) and
// read as broadcasts.  NS > 1 folds the n-lanes through smem; split N goes to ordered partials.
constexpr int NCH = 128;   // n rows staged per step

template <int BT>
__device__ __forceinline__ int dy_slot(int n, int b4) { return n * BT + ((b4 ^ (n & (BT / 4 - 1))) << 2); }

template <int BT>
__device__ __forceinline__ void stage_dy(const float* __restrict__ dy, int B, int N, int nb, int nc,
                                         float* __restrict__ s_dy, int tid) {
  // s_dy[n_local][b] <- dy[b][nb + n_local]; global reads coalesced along n
  for (int i = tid; i < BT * NCH; i += NTHREADS) {
    const int b = i / NCH, nl = i - b * NCH;
    float v = 0.f;
    if (b < B && nl < nc) v = __ldg(dy + (size_t)b * N + nb + nl);
    s_dy[dy_slot<BT>(nl, b >> 2) + (b & 3)] = v;
  }
}

template <typename T, int BT, int KT>
__global__ void __launch_bounds__(NTHREADS) linear_dgrad_simt(const float* __restrict__ dy, const float* __restrict__ w,
                                                              T* __restrict__ dx, float* __restrict__ partial, int B,
                                                              int N, long long K, int nchunk) {
  constexpr int NS = NTHREADS / KT;
  extern __shared__ __align__(16) float smem[];
  float* s_dy = smem;   // [NCH][BT]; reused for the cross-lane fold when NS > 1
  const int tid = threadIdx.x;
  const int kt = tid % KT, ns = tid / KT;
  const long long kq = (long long)blockIdx.x * KT + kt;   // float4 index along K
  const bool kvalid = kq * 4 < K;
  const int nbeg = blockIdx.y * nchunk;
  const int nend = nbeg + nchunk < N ? nbeg + nchunk : N;
  float acc[BT][4];
#pragma unroll
  for (int b = 0; b < BT; ++b) acc[b][0] = acc[b][1] = acc[b][2] = acc[b][3] = 0.f;

  for (int nb = nbeg; nb < nend; nb += NCH) {
    const int nc = nend - nb < NCH ? nend - nb : NCH;
    __syncthreads();
    stage_dy<BT>(dy, B, N, nb, nc, s_dy, tid);
    __syncthreads();
    if (kvalid) {
#pragma unroll 2
      for (int nl = ns; nl < nc; nl += NS) {
        const float4 wv = __ldcs(reinterpret_cast<const float4*>(w + (size_t)(nb + nl) * K) + kq);
#pragma unroll
        for (int b4 = 0; b4 < BT / 4; ++b4) {
          const float4 d = *reinterpret_cast<const float4*>(s_dy + dy_slot<BT>(nl, b4));
          const float dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float* a = acc[b4 * 4 + e];
            a[0] = fmaf(dv[e], wv.x, a[0]);
            a[1] = fmaf(dv[e], wv.y, a[1]);
            a[2] = fmaf(dv[e], wv.z, a[2]);
            a[3] = fmaf(dv[e], wv.w, a[3]);
          }
        }
      }
    }
  }
  if (NS > 1) {
    // fold the NS n-lanes: s_red[ns][b][kt] float4  (NS*BT*KT*4 floats)
    __syncthreads();
    float4* s_red = reinterpret_cast<float4*>(smem);
#pragma unroll
    for (int b = 0; b < BT; ++b) s_red[(ns * BT + b) * KT + kt] = make_float4(acc[b][0], acc[b][1], acc[b][2], acc[b][3]);
    __syncthreads();
    if (ns == 0) {
#pragma unroll
      for (int b = 0; b < BT; ++b) {
        float4 s = s_red[b * KT + kt];
        for (int j = 1; j < NS; ++j) {
          const float4 t = s_red[(j * BT + b) * KT + kt];
          s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
        }
        acc[b][0] = s.x; acc[b][1] = s.y; acc[b][2] = s.z; acc[b][3] = s.w;
      }
    }
  }
  if (ns == 0 && kvalid) {
#pragma unroll
    for (int b = 0; b < BT; ++b) {
      if (b >= B) break;
      if (gridDim.y == 1) {
        T* o = dx + (size_t)b * K + kq * 4;
        dd::st<T>(o, acc[b][0]); dd::st<T>(o + 1, acc[b][1]); dd::st<T>(o + 2, acc[b][2]); dd::st<T>(o + 3, acc[b][3]);
      } else {
        *reinterpret_cast<float4*>(partial + ((size_t)blockIdx.y * B + b) * K + kq * 4) =
            make_float4(acc[b][0], acc[b][1], acc[b][2], acc[b][3]);
      }
    }
  }
}

template <typename T>
__global__ void splitn_reduce_kernel(const float* __restrict__ partial, T* __restrict__ dx, int splits, long long bk) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= bk) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += partial[(size_t)k * bk + i];
  dd::st<T>(dx + i, s);
}

// ---------------------------------------------------------------- wgrad -------------------
// dW[n,k] = sum_b dy[b,n] x[b,k] (+= when accumulate).  Thread keeps x[0..BT)[k..k+3] in registers
// and streams its n rows: BT*4 FMA per 16-byte store -> HBM-write-bound once B is small.
template <typename T, int BT, int KT>
__global__ void __launch_bounds__(NTHREADS) linear_wgrad_simt(const float* __restrict__ dy, const T* __restrict__ x,
                                                              float* __restrict__ dw, int B, int N, long long K,
                                                              int nchunk, int accumulate) {
  constexpr int NS = NTHREADS / KT;
  extern __shared__ __align__(16) float smem[];
  float* s_dy = smem;
  const int tid = threadIdx.x;
  const int kt = tid % KT, ns = tid / KT;
  const long long kq = (long long)blockIdx.x * KT + kt;
  const bool kvalid = kq * 4 < K;
  const int nbeg = blockIdx.y * nchunk;
  const int nend = nbeg + nchunk < N ? nbeg + nchunk : N;
  float xr[BT][4];
#pragma unroll
  for (int b = 0; b < BT; ++b) {
    if (b < B && kvalid) {
      const T* p = x + (size_t)b * K + kq * 4;
      xr[b][0] = dd::ld<T>(p); xr[b][1] = dd::ld<T>(p + 1); xr[b][2] = dd::ld<T>(p + 2); xr[b][3] = dd::ld<T>(p + 3);
    } else {
      xr[b][0] = xr[b][1] = xr[b][2] = xr[b][3] = 0.f;
    }
  }
  for (int nb = nbeg; nb < nend; nb += NCH) {
    const int nc = nend - nb < NCH ? nend - nb : NCH;
    __syncthreads();
    stage_dy<BT>(dy, B, N, nb, nc, s_dy, tid);
    __syncthreads();
    if (kvalid) {
      for (int nl = ns; nl < nc; nl += NS) {
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        float4* dst = reinterpret_cast<float4*>(dw + (size_t)(nb + nl) * K) + kq;
        if (accumulate) o = *dst;
#pragma unroll
        for (int b4 = 0; b4 < BT / 4; ++b4) {
          const float4 d = *reinterpret_cast<const float4*>(s_dy + dy_slot<BT>(nl, b4));
          const float dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float* xv = xr[b4 * 4 + e];
            o.x = fmaf(dv[e], xv[0], o.x);
            o.y = fmaf(dv[e], xv[1], o.y);
            o.z = fmaf(dv[e], xv[2], o.z);
            o.w = fmaf(dv[e], xv[3], o.w);
          }
        }
        __stcs(dst, o);
      }
    }
  }
}

// dd_linear_wgrad_acc: dW[n,k] = dW_old[n,k] + D[n,k], D bit for bit what dd_linear_wgrad writes.  D is the FMA chain of
// the chunked launches above (rows in order; each 32-row chunk padded with zero rows to its launch's BT, 8 or 32), kept in
// a register across the chunks, so that the stored gradient is added once, after the last chunk.  KT = 32 k quads x 8
// n-lanes; x [Bp][128 k] and dy [NCH n][Bp] staged in shared memory (Bp = padded rows, <= 128).
constexpr int ACC_KT = 32;
template <typename T>
__global__ void __launch_bounds__(NTHREADS) linear_wgrad_acc_simt(const float* __restrict__ dy, const T* __restrict__ x,
                                                                  float* __restrict__ dw, int B, int Bp, int N, long long K,
                                                                  int nchunk) {
  constexpr int NS = NTHREADS / ACC_KT;
  extern __shared__ __align__(16) float smem[];
  float4* s_x = reinterpret_cast<float4*>(smem);          // [Bp][ACC_KT]
  float* s_dy = smem + (size_t)Bp * ACC_KT * 4;           // [NCH][Bp]
  const int tid = threadIdx.x;
  const int kt = tid % ACC_KT, ns = tid / ACC_KT;
  const long long kq = (long long)blockIdx.x * ACC_KT + kt;
  const bool kvalid = kq * 4 < K;
  for (int i = tid; i < Bp * ACC_KT; i += NTHREADS) {
    const int b = i / ACC_KT;
    const long long k = ((long long)blockIdx.x * ACC_KT + i % ACC_KT) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b < B && k < K) {
      const T* p = x + (size_t)b * K + k;
      v = make_float4(dd::ld<T>(p), dd::ld<T>(p + 1), dd::ld<T>(p + 2), dd::ld<T>(p + 3));
    }
    s_x[i] = v;
  }
  const int nbeg = blockIdx.y * nchunk;
  const int nend = nbeg + nchunk < N ? nbeg + nchunk : N;
  for (int nb = nbeg; nb < nend; nb += NCH) {
    const int nc = nend - nb < NCH ? nend - nb : NCH;
    __syncthreads();
    for (int i = tid; i < Bp * NCH; i += NTHREADS) {
      const int b = i / NCH, nl = i - b * NCH;
      s_dy[nl * Bp + b] = (b < B && nl < nc) ? __ldg(dy + (size_t)b * N + nb + nl) : 0.f;
    }
    __syncthreads();
    if (kvalid) {
      for (int nl = ns; nl < nc; nl += NS) {
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int b4 = 0; b4 < Bp / 4; ++b4) {
          const float4 d = *reinterpret_cast<const float4*>(s_dy + nl * Bp + 4 * b4);
          const float dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float4 xv = s_x[(4 * b4 + e) * ACC_KT + kt];
            o.x = fmaf(dv[e], xv.x, o.x);
            o.y = fmaf(dv[e], xv.y, o.y);
            o.z = fmaf(dv[e], xv.z, o.z);
            o.w = fmaf(dv[e], xv.w, o.w);
          }
        }
        float4* dst = reinterpret_cast<float4*>(dw + (size_t)(nb + nl) * K) + kq;
        const float4 old = *dst;
        o.x = old.x + o.x; o.y = old.y + o.y; o.z = old.z + o.z; o.w = old.w + o.w;
        __stcs(dst, o);
      }
    }
  }
}

// db[n] = sum_b dy[b,n]
__global__ void colsum_kernel(const float* __restrict__ dy, float* __restrict__ db, int B, int N, int accumulate) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float s = accumulate ? db[n] : 0.f;
  for (int b = 0; b < B; ++b) s += dy[(size_t)b * N + n];
  db[n] = s;
}

// choose split counts so that ~4 CTAs per SM exist without oversizing the partial buffers
struct FwdPlan { int row_blocks, ksplits; long long kchunk; };
FwdPlan plan_fwd(int N, long long K) {
  FwdPlan p;
  p.row_blocks = dd::ceil_div(N, 8 * NR);
  int want = dd::ceil_div(dd::kSMs * 4, p.row_blocks);
  long long maxsplit = (K + KC - 1) / KC;
  if (want > maxsplit) want = (int)maxsplit;
  if (want < 1) want = 1;
  p.kchunk = ((K + want - 1) / want + KC - 1) / KC * KC;
  p.ksplits = dd::ceil_div(K, p.kchunk);
  return p;
}
struct DgradPlan { int kt, kblocks, nsplits, nchunk; };
DgradPlan plan_dgrad(int N, long long K) {
  DgradPlan p;
  p.kt = (K / 4 >= 256) ? 256 : 32;
  p.kblocks = dd::ceil_div(K / 4, p.kt);
  int want = dd::ceil_div(dd::kSMs * 2, p.kblocks);
  int maxsplit = dd::ceil_div(N, NCH);
  if (want > maxsplit) want = maxsplit;
  if (want < 1) want = 1;
  p.nchunk = dd::ceil_div(dd::ceil_div(N, want), NCH) * NCH;
  p.nsplits = dd::ceil_div(N, p.nchunk);
  return p;
}

template <typename T, int BT>
int fwd_launch(const T* x, const float* w, const float* bias, float* y, float* ws, int B, int N, long long K,
               cudaStream_t st) {
  const FwdPlan p = plan_fwd(N, K);
  const size_t smem = (size_t)BT * KC * sizeof(float);
  auto kern = linear_fwd_simt<T, BT>;
  if (int e = dd::set_smem(kern, smem, dd::Carveout::kDefault, "linear_fwd_simt")) return e;
  kern<<<dim3(p.row_blocks, p.ksplits), NTHREADS, smem, st>>>(x, w, bias, y, ws, B, N, K, p.kchunk);
  if (int e = dd::check_launch("linear_fwd_simt")) return e;
  if (p.ksplits > 1) {
    const long long bn = (long long)B * N;
    splitk_reduce_kernel<<<dd::ceil_div(bn, 256), 256, 0, st>>>(ws, bias, y, p.ksplits, bn, N);
    return dd::check_launch("splitk_reduce");
  }
  return 0;
}

template <typename T, int BT>
int dgrad_launch(const float* dy, const float* w, T* dx, float* ws, int B, int N, long long K, cudaStream_t st) {
  const DgradPlan p = plan_dgrad(N, K);
  dim3 grid(p.kblocks, p.nsplits);
  if (p.kt == 256) {
    const size_t smem = (size_t)NCH * BT * sizeof(float);
    linear_dgrad_simt<T, BT, 256><<<grid, NTHREADS, smem, st>>>(dy, w, dx, ws, B, N, K, p.nchunk);
  } else {
    size_t smem = (size_t)NCH * BT * sizeof(float);
    const size_t fold = (size_t)8 * BT * 32 * 4 * sizeof(float);
    if (fold > smem) smem = fold;
    auto k = linear_dgrad_simt<T, BT, 32>;
    if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "linear_dgrad_simt")) return e;
    k<<<grid, NTHREADS, smem, st>>>(dy, w, dx, ws, B, N, K, p.nchunk);
  }
  if (int e = dd::check_launch("linear_dgrad_simt")) return e;
  if (p.nsplits > 1) {
    const long long bk = (long long)B * K;
    splitn_reduce_kernel<T><<<dd::ceil_div(bk, 256), 256, 0, st>>>(ws, dx, p.nsplits, bk);
    return dd::check_launch("splitn_reduce");
  }
  return 0;
}

template <typename T, int BT>
int wgrad_launch(const float* dy, const T* x, float* dw, int B, int N, long long K, int accumulate, cudaStream_t st) {
  const int kt = (K / 4 >= 256) ? 256 : 32;
  const int kblocks = dd::ceil_div(K / 4, kt);
  int want = dd::ceil_div(dd::kSMs * 4, kblocks);
  int maxsplit = dd::ceil_div(N, NCH);
  if (want > maxsplit) want = maxsplit;
  if (want < 1) want = 1;
  const int nchunk = dd::ceil_div(dd::ceil_div(N, want), NCH) * NCH;
  dim3 grid(kblocks, dd::ceil_div(N, nchunk));
  const size_t smem = (size_t)NCH * BT * sizeof(float);
  if (kt == 256) linear_wgrad_simt<T, BT, 256><<<grid, NTHREADS, smem, st>>>(dy, x, dw, B, N, K, nchunk, accumulate);
  else linear_wgrad_simt<T, BT, 32><<<grid, NTHREADS, smem, st>>>(dy, x, dw, B, N, K, nchunk, accumulate);
  return dd::check_launch("linear_wgrad_simt");
}

template <typename T>
int wgrad_acc_launch(const float* dy, const T* x, float* dw, int B, int N, long long K, cudaStream_t st) {
  const int last = B - 32 * ((B - 1) / 32);                      // rows of the last 32-row chunk, padded as its launch pads
  const int Bp = 32 * ((B - 1) / 32) + (last <= 8 ? 8 : 32);
  const int kblocks = dd::ceil_div(K / 4, ACC_KT);
  int want = dd::ceil_div(dd::kSMs * 4, kblocks);
  int maxsplit = dd::ceil_div(N, NCH);
  if (want > maxsplit) want = maxsplit;
  if (want < 1) want = 1;
  const int nchunk = dd::ceil_div(dd::ceil_div(N, want), NCH) * NCH;
  const size_t smem = (size_t)Bp * (ACC_KT * 4 + NCH) * sizeof(float);
  auto k = linear_wgrad_acc_simt<T>;
  if (int e = dd::set_smem(k, smem, dd::Carveout::kDefault, "linear_wgrad_acc_simt")) return e;
  k<<<dim3(kblocks, dd::ceil_div(N, nchunk)), NTHREADS, smem, st>>>(dy, x, dw, B, Bp, N, K, nchunk);
  return dd::check_launch("linear_wgrad_acc_simt");
}

size_t ws_bytes_for(int B, int N, long long K) {
  const int Bc = B < 32 ? B : 32;
  const FwdPlan f = plan_fwd(N, K);
  const DgradPlan d = plan_dgrad(N, K);
  size_t a = f.ksplits > 1 ? (size_t)f.ksplits * Bc * N * sizeof(float) : 0;
  size_t b = d.nsplits > 1 ? (size_t)d.nsplits * Bc * K * sizeof(float) : 0;
  return (a > b ? a : b) + 256;
}
}  // namespace

namespace dd {
// tensor-core weight-streaming variants (linear_tc.cu): fp32 operands read as tf32, B <= 32 rows per call
bool linear_tc_supported(int B, int N, long long K);
size_t linear_tc_workspace_bytes(int B, int N, long long K);
int linear_fwd_tc(const float* x, const float* w, const float* bias, float* y, void* ws, size_t ws_bytes, int B, int N,
                  long long K, cudaStream_t st);
int linear_dgrad_tc(const float* dy, const float* w, void* dx, int dx_dtype, void* ws, size_t ws_bytes, int B, int N,
                    long long K, cudaStream_t st);
int linear_wgrad_tc(const float* dy, const float* x, float* dw, int B, int N, long long K, int accumulate, cudaStream_t st);
int linear_wgrad_acc_multi_tc(const float* dy, const float* x, float* dw, int B, int N, long long K, cudaStream_t st);
int linear_bwd_adam_tc(const float* dy, const float* x, float* w, float* m, float* v, const float* gpart, void* dx, int dx_dtype,
                       void* ws, size_t ws_bytes, int B, int N, long long K, const AdamHyper& h, double* sumsq,
                       SumsqWorkspace* sumsq_ws, cudaStream_t st);
}  // namespace dd

// tcgen05 path: only on explicit request (DD_IMPL_TCGEN05) -- fp32 callers under DD_IMPL_AUTO keep the
// 1e-5 parity kernels; tf32 operands are the bf16-mode contract (1e-2)
static bool use_tc(int impl, int B, int N, long long K) { return impl == DD_IMPL_TCGEN05 && dd::linear_tc_supported(B, N, K); }

extern "C" int dd_linear_tc_supported(int B, int N, long long K) { return dd::linear_tc_supported(B, N, K) ? 1 : 0; }

extern "C" size_t dd_linear_workspace_bytes(int B, int N, long long K) {
  if (B <= 0 || N <= 0 || K <= 0) return 256;
  const size_t a = ws_bytes_for(B, N, K), b = dd::linear_tc_supported(B, N, K) ? dd::linear_tc_workspace_bytes(B, N, K) : 0;
  return a > b ? a : b;
}

#define DD_LINEAR_COMMON(name)                                                                           \
  DD_REQUIRE(B >= 0 && N > 0 && K > 0, DD_ERR_BAD_ARG, name ": bad shape B=%d N=%d K=%lld", B, N, K);    \
  DD_REQUIRE(K % 4 == 0, DD_ERR_UNSUPPORTED, name ": K=%lld must be a multiple of 4", K);                \
  if (B == 0) return 0;

extern "C" int dd_linear_fwd(const void* x, int x_dtype, const float* w, const float* bias, float* y, void* workspace,
                             size_t ws_bytes, int B, int N, long long K, int impl, void* stream) {
  DD_REQUIRE(x && w && y, DD_ERR_BAD_ARG, "dd_linear_fwd: null pointer");
  DD_LINEAR_COMMON("dd_linear_fwd");
  DD_REQUIRE(x_dtype == DD_F32 || x_dtype == DD_BF16, DD_ERR_UNSUPPORTED, "dd_linear_fwd: dtype %d", x_dtype);
  DD_REQUIRE((uintptr_t)w % 16 == 0, DD_ERR_ALIGNMENT, "dd_linear_fwd: weight pointer must be 16-byte aligned");
  DD_REQUIRE(workspace && ws_bytes >= dd_linear_workspace_bytes(B, N, K), DD_ERR_WORKSPACE,
             "dd_linear_fwd: workspace %zu < %zu", ws_bytes, dd_linear_workspace_bytes(B, N, K));
  DD_REQUIRE(impl != DD_IMPL_TCGEN05 || (x_dtype == DD_F32 && dd::linear_tc_supported(B, N, K)), DD_ERR_UNSUPPORTED,
             "dd_linear_fwd: tcgen05 path needs fp32 x, N %% 4 == K %% 4 == 0 and N*K >= 2^22 (B=%d N=%d K=%lld)", B, N, K);
  cudaStream_t st = dd::as_stream(stream);
  const size_t esz = x_dtype == DD_F32 ? 4 : 2;
  const int rows_per_pass = use_tc(impl, B, N, K) ? 256 : 32;      // the tcgen05 forward takes up to 256 rows per weight pass
  for (int b0 = 0; b0 < B; b0 += rows_per_pass) {
    const int bc = B - b0 < rows_per_pass ? B - b0 : rows_per_pass;
    const char* xp = (const char*)x + (size_t)b0 * K * esz;
    float* yp = y + (size_t)b0 * N;
    int e;
    if (use_tc(impl, B, N, K)) {
      if ((e = dd::linear_fwd_tc((const float*)xp, w, bias, yp, workspace, ws_bytes, bc, N, K, st))) return e;
      continue;
    }
    if (x_dtype == DD_F32)
      e = bc <= 8 ? fwd_launch<float, 8>((const float*)xp, w, bias, yp, (float*)workspace, bc, N, K, st)
                  : fwd_launch<float, 32>((const float*)xp, w, bias, yp, (float*)workspace, bc, N, K, st);
    else
      e = bc <= 8 ? fwd_launch<__nv_bfloat16, 8>((const __nv_bfloat16*)xp, w, bias, yp, (float*)workspace, bc, N, K, st)
                  : fwd_launch<__nv_bfloat16, 32>((const __nv_bfloat16*)xp, w, bias, yp, (float*)workspace, bc, N, K, st);
    if (e) return e;
  }
  return 0;
}

extern "C" int dd_linear_dgrad(const float* dy, const float* w, void* dx, int dx_dtype, void* workspace,
                               size_t ws_bytes, int B, int N, long long K, int impl, void* stream) {
  DD_REQUIRE(dy && w && dx, DD_ERR_BAD_ARG, "dd_linear_dgrad: null pointer");
  DD_LINEAR_COMMON("dd_linear_dgrad");
  DD_REQUIRE(dx_dtype == DD_F32 || dx_dtype == DD_BF16, DD_ERR_UNSUPPORTED, "dd_linear_dgrad: dtype %d", dx_dtype);
  DD_REQUIRE((uintptr_t)w % 16 == 0, DD_ERR_ALIGNMENT, "dd_linear_dgrad: weight pointer must be 16-byte aligned");
  DD_REQUIRE(workspace && ws_bytes >= dd_linear_workspace_bytes(B, N, K), DD_ERR_WORKSPACE,
             "dd_linear_dgrad: workspace %zu < %zu", ws_bytes, dd_linear_workspace_bytes(B, N, K));
  DD_REQUIRE(impl != DD_IMPL_TCGEN05 || dd::linear_tc_supported(B, N, K), DD_ERR_UNSUPPORTED,
             "dd_linear_dgrad: tcgen05 path needs N %% 4 == K %% 4 == 0 and N*K >= 2^22 (B=%d N=%d K=%lld)", B, N, K);
  cudaStream_t st = dd::as_stream(stream);
  const size_t esz = dx_dtype == DD_F32 ? 4 : 2;
  for (int b0 = 0; b0 < B; b0 += 32) {
    const int bc = B - b0 < 32 ? B - b0 : 32;
    const float* dyp = dy + (size_t)b0 * N;
    char* dxp = (char*)dx + (size_t)b0 * K * esz;
    int e;
    if (use_tc(impl, B, N, K)) {
      if ((e = dd::linear_dgrad_tc(dyp, w, dxp, dx_dtype, workspace, ws_bytes, bc, N, K, st))) return e;
      continue;
    }
    if (dx_dtype == DD_F32)
      e = bc <= 8 ? dgrad_launch<float, 8>(dyp, w, (float*)dxp, (float*)workspace, bc, N, K, st)
                  : dgrad_launch<float, 32>(dyp, w, (float*)dxp, (float*)workspace, bc, N, K, st);
    else
      e = bc <= 8 ? dgrad_launch<__nv_bfloat16, 8>(dyp, w, (__nv_bfloat16*)dxp, (float*)workspace, bc, N, K, st)
                  : dgrad_launch<__nv_bfloat16, 32>(dyp, w, (__nv_bfloat16*)dxp, (float*)workspace, bc, N, K, st);
    if (e) return e;
  }
  return 0;
}

#define DD_WGRAD_COMMON(name)                                                                                          \
  DD_REQUIRE(dy && x && dw, DD_ERR_BAD_ARG, name ": null pointer");                                                    \
  DD_REQUIRE(B > 0 && N > 0 && K > 0, DD_ERR_BAD_ARG, name ": bad shape B=%d N=%d K=%lld", B, N, K);                   \
  DD_REQUIRE(K % 4 == 0, DD_ERR_UNSUPPORTED, name ": K=%lld must be a multiple of 4", K);                              \
  DD_REQUIRE(x_dtype == DD_F32 || x_dtype == DD_BF16, DD_ERR_UNSUPPORTED, name ": dtype %d", x_dtype);                 \
  DD_REQUIRE((uintptr_t)dw % 16 == 0, DD_ERR_ALIGNMENT, name ": dw pointer must be 16-byte aligned");                  \
  DD_REQUIRE(impl != DD_IMPL_TCGEN05 || (x_dtype == DD_F32 && dd::linear_tc_supported(B, N, K)), DD_ERR_UNSUPPORTED, \
             name ": tcgen05 path needs fp32 x, N %% 4 == K %% 4 == 0 and N*K >= 2^22 (B=%d N=%d K=%lld)", B, N, K);

// db[n] = sum_b dy[b,n], in the 32-row chunks of the weight-gradient launches
static int colsum_chunked(const float* dy, float* db, int B, int N, cudaStream_t st) {
  for (int b0 = 0; b0 < B; b0 += 32) {
    colsum_kernel<<<dd::ceil_div(N, 256), 256, 0, st>>>(dy + (size_t)b0 * N, db, B - b0 < 32 ? B - b0 : 32, N, b0 > 0);
    if (int e = dd::check_launch("colsum")) return e;
  }
  return 0;
}

extern "C" int dd_linear_wgrad(const float* dy, const void* x, int x_dtype, float* dw, float* db, int B, int N,
                               long long K, int impl, void* stream) {
  DD_WGRAD_COMMON("dd_linear_wgrad");
  cudaStream_t st = dd::as_stream(stream);
  const size_t esz = x_dtype == DD_F32 ? 4 : 2;
  for (int b0 = 0; b0 < B; b0 += 32) {
    const int bc = B - b0 < 32 ? B - b0 : 32;
    const float* dyp = dy + (size_t)b0 * N;
    const char* xp = (const char*)x + (size_t)b0 * K * esz;
    const int accumulate = b0 > 0;
    int e;
    if (use_tc(impl, B, N, K)) e = dd::linear_wgrad_tc(dyp, (const float*)xp, dw, bc, N, K, accumulate, st);
    else if (x_dtype == DD_F32)
      e = bc <= 8 ? wgrad_launch<float, 8>(dyp, (const float*)xp, dw, bc, N, K, accumulate, st)
                  : wgrad_launch<float, 32>(dyp, (const float*)xp, dw, bc, N, K, accumulate, st);
    else
      e = bc <= 8 ? wgrad_launch<__nv_bfloat16, 8>(dyp, (const __nv_bfloat16*)xp, dw, bc, N, K, accumulate, st)
                  : wgrad_launch<__nv_bfloat16, 32>(dyp, (const __nv_bfloat16*)xp, dw, bc, N, K, accumulate, st);
    if (e) return e;
    if (db) {
      colsum_kernel<<<dd::ceil_div(N, 256), 256, 0, st>>>(dyp, db, bc, N, accumulate);
      if (int e2 = dd::check_launch("colsum")) return e2;
    }
  }
  return 0;
}

// dd_linear_wgrad, or with accumulate: dw = dw_old + what dd_linear_wgrad writes, bit for bit (see include/dd_b200.h)
extern "C" int dd_linear_wgrad_acc(const float* dy, const void* x, int x_dtype, float* dw, float* db, int B, int N,
                                   long long K, int impl, int accumulate, void* stream) {
  if (!accumulate) return dd_linear_wgrad(dy, x, x_dtype, dw, db, B, N, K, impl, stream);
  DD_WGRAD_COMMON("dd_linear_wgrad_acc");
  DD_REQUIRE(B <= 128, DD_ERR_UNSUPPORTED, "dd_linear_wgrad_acc: accumulating takes at most 128 rows (B=%d)", B);
  cudaStream_t st = dd::as_stream(stream);
  int e;
  if (use_tc(impl, B, N, K))        // one 32-row chunk: the plain kernel's epilogue adds the old value after the MMA sum
    e = B <= 32 ? dd::linear_wgrad_tc(dy, (const float*)x, dw, B, N, K, 1, st) : dd::linear_wgrad_acc_multi_tc(dy, (const float*)x, dw, B, N, K, st);
  else if (x_dtype == DD_F32)
    e = wgrad_acc_launch<float>(dy, (const float*)x, dw, B, N, K, st);
  else
    e = wgrad_acc_launch<__nv_bfloat16>(dy, (const __nv_bfloat16*)x, dw, B, N, K, st);
  if (e) return e;
  return db ? colsum_chunked(dy, db, B, N, st) : 0;
}

// Backward pass of a wide linear layer with the Adam update of its weight folded in (world size 1): see include/dd_b200.h.
// tcgen05 path only (fp32 x, B <= 32, dd_linear_tc_supported); the bias gradient is written as by dd_linear_wgrad.
// acc: the step takes this pass's weight gradient plus grad_partial (the earlier passes of the window); sumsq: also the sum
// of squares of that gradient (nullptr: not computed).
static int bwd_adam(const char* what, bool acc, const float* dy, const float* x, float* weight, float* exp_avg, float* exp_avg_sq,
                    const float* grad_partial, void* dx, int dx_dtype, float* db, void* workspace, size_t ws_bytes, int B, int N,
                    long long K, float lr, float beta1, float beta2, float eps, float weight_decay, long long step, double* sumsq,
                    void* sumsq_ws, void* stream) {
  DD_REQUIRE(dy && x && weight && exp_avg && exp_avg_sq && (grad_partial || !acc), DD_ERR_BAD_ARG, "%s: null pointer", what);
  DD_REQUIRE(B > 0 && B <= 32 && N > 0 && K > 0 && step >= 1, DD_ERR_BAD_ARG, "%s: B=%d (<= 32) N=%d K=%lld step=%lld", what, B, N, K, step);
  DD_REQUIRE(!dx || dx_dtype == DD_F32 || dx_dtype == DD_BF16, DD_ERR_UNSUPPORTED, "%s: dtype %d", what, dx_dtype);
  DD_REQUIRE(dd::linear_tc_supported(B, N, K), DD_ERR_UNSUPPORTED, "%s: needs the tcgen05 path (N %% 4 == K %% 4 == 0, N*K >= 2^22)", what);
  DD_REQUIRE((((uintptr_t)weight | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq | (uintptr_t)grad_partial | (uintptr_t)dy | (uintptr_t)x) & 15) == 0,
             DD_ERR_ALIGNMENT, acc ? "%s: dy / x / weight / moments / grad_partial must be 16-byte aligned"
                                   : "%s: dy / x / weight / moments must be 16-byte aligned", what);
  DD_REQUIRE(!dx || (workspace && ws_bytes >= dd_linear_workspace_bytes(B, N, K)), DD_ERR_WORKSPACE,
             "%s: workspace %zu < %zu", what, ws_bytes, dd_linear_workspace_bytes(B, N, K));
  cudaStream_t st = dd::as_stream(stream);
  const dd::AdamHyper h = dd::adam_hyper(lr, beta1, beta2, eps, weight_decay, step, 1.f);
  if (int e = dd::linear_bwd_adam_tc(dy, x, weight, exp_avg, exp_avg_sq, acc ? grad_partial : nullptr, dx, dx_dtype, workspace,
                                     ws_bytes, B, N, K, h, sumsq, (dd::SumsqWorkspace*)sumsq_ws, st))
    return e;
  if (db) {
    colsum_kernel<<<dd::ceil_div(N, 256), 256, 0, st>>>(dy, db, B, N, 0);
    if (int e2 = dd::check_launch("colsum")) return e2;
  }
  return 0;
}

extern "C" int dd_linear_bwd_adam(const float* dy, const float* x, float* weight, float* exp_avg, float* exp_avg_sq, void* dx,
                                  int dx_dtype, float* db, void* workspace, size_t ws_bytes, int B, int N, long long K, float lr,
                                  float beta1, float beta2, float eps, float weight_decay, long long step, void* stream) {
  return bwd_adam("dd_linear_bwd_adam", false, dy, x, weight, exp_avg, exp_avg_sq, nullptr, dx, dx_dtype, db, workspace, ws_bytes,
                  B, N, K, lr, beta1, beta2, eps, weight_decay, step, nullptr, nullptr, stream);
}

extern "C" int dd_linear_bwd_adam_acc(const float* dy, const float* x, float* weight, float* exp_avg, float* exp_avg_sq,
                                      const float* grad_partial, void* dx, int dx_dtype, float* db, void* workspace,
                                      size_t ws_bytes, int B, int N, long long K, float lr, float beta1, float beta2, float eps,
                                      float weight_decay, long long step, void* stream) {
  return bwd_adam("dd_linear_bwd_adam_acc", true, dy, x, weight, exp_avg, exp_avg_sq, grad_partial, dx, dx_dtype, db, workspace,
                  ws_bytes, B, N, K, lr, beta1, beta2, eps, weight_decay, step, nullptr, nullptr, stream);
}

extern "C" int dd_linear_bwd_adam_sumsq(const float* dy, const float* x, float* weight, float* exp_avg, float* exp_avg_sq,
                                        const float* grad_partial, void* dx, int dx_dtype, float* db, void* workspace,
                                        size_t ws_bytes, int B, int N, long long K, float lr, float beta1, float beta2, float eps,
                                        float weight_decay, long long step, double* sumsq, void* sumsq_ws, size_t sumsq_ws_bytes,
                                        void* stream) {
  DD_REQUIRE(sumsq && sumsq_ws, DD_ERR_BAD_ARG, "dd_linear_bwd_adam_sumsq: null pointer");
  DD_REQUIRE(((uintptr_t)sumsq & 7) == 0, DD_ERR_ALIGNMENT, "dd_linear_bwd_adam_sumsq: sumsq must be 8-byte aligned");
  DD_REQUIRE(sumsq_ws_bytes >= sizeof(dd::SumsqWorkspace), DD_ERR_WORKSPACE, "dd_linear_bwd_adam_sumsq: workspace %zu < %zu",
             sumsq_ws_bytes, sizeof(dd::SumsqWorkspace));
  return bwd_adam("dd_linear_bwd_adam_sumsq", grad_partial != nullptr, dy, x, weight, exp_avg, exp_avg_sq, grad_partial, dx,
                  dx_dtype, db, workspace, ws_bytes, B, N, K, lr, beta1, beta2, eps, weight_decay, step, sumsq, sumsq_ws, stream);
}
