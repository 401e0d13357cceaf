// Fused Adam step (torch.optim.Adam at roadmap_bce_v2.py:155 / autoencoder.py:120, amsgrad off), and the
// data-parallel form that replaces "NCCL all-reduce of the gradients + N identical Adam updates" (what
// Lightning's ddp backend does for the reference) by ONE kernel over NVLink peer memory:
//
//   rank r owns elements [r*n/N, (r+1)*n/N) of every large parameter.  For its shard it
//     1. reads the N gradient replicas -- multimem.ld_reduce (the NVSwitch adds them in flight, one inbound
//        copy) when the buffers have a multicast mapping, else N-1 peer loads + 1 local load;
//     2. updates its shard of the Adam moments (m, v exist ONLY for the shard: 1/N of the optimizer state
//        and of the optimizer's HBM traffic per GPU);
//     3. writes the new weights into every replica -- multimem.st (one outbound copy, the switch
//        broadcasts) or N peer stores -- i.e. the all-gather rides in the same kernel.
//   The caller brackets the launch with cross-rank barriers (grads complete before / weights landed after).
//
// HBM-bound when local (28 B per element), NVLink-bound when sharded.
//
// Gradient clipping by the global L2 norm (torch.nn.utils.clip_grad_norm_, Lightning's gradient_clip_val) at world size 1:
// dd_grad_sumsq folds the squares of every gradient into one norm and clip coefficient on the device, and
// dd_adam_step_clipped is dd_adam_step with that coefficient read from device memory -- no host round trip, so the step
// stays free of host syncs and capturable in a CUDA graph.
#include <math.h>

#include "adam.cuh"
#include "dd_common.cuh"

namespace {

using dd::AdamHyper;
using dd::adam_one;

constexpr int kMaxRanks = 16;
constexpr int kThreads = 256;   // 256 threads x <= 96 registers: one update CTA fits on an SM beside any persistent conv CTA

struct PeerPtrs {
  const float* grad[kMaxRanks];   // every rank's gradient replica (index = rank), full length
  float* param[kMaxRanks];        // every rank's weight replica
};

__device__ __forceinline__ float4 ld_reduce_add(const float* mc) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(mc) : "memory");
  return r;
}
__device__ __forceinline__ void mc_store(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// MODE 0: local (grad / param = one pointer each).  MODE 1: peer pointers.  MODE 2: multicast pointers.
// CLIP: the gradient is multiplied by *coef (dd_grad_sumsq's clip coefficient; every thread loads it once, a cached
// broadcast, and adam_scalar_kernel<true> once per element) after grad_scale.  coef
// is the last parameter so that the instantiations without it compile to the code they had before it existed.
// UNROLL independent 16-byte granules per thread and iteration: all their loads are issued before the first use, so that
// enough bytes are in flight to cover the NVLink round trip with one resident CTA per SM.
// 80 registers: the register file is split over the SM's four sub-partitions (16 K each).  Two update warps per sub-partition
// take 2 x 2560; the input-gradient conv kernel that must run beside the update puts 4 of its 13 warps (88 registers) on one
// sub-partition, 11264 -- together exactly 16 K.  With 96 registers here that kernel queued behind the whole update
// (1.8 ms hole in the N = 2 multicast timeline, profiles/r2_step_timeline_n2_multicast_96regs.txt).
template <int MODE, int UNROLL, bool CLIP = false>
__global__ void __maxnreg__(MODE == 0 ? 96 : 80) adam_kernel(PeerPtrs pp, const float* __restrict__ mc_grad, float* __restrict__ mc_param,
                                                        float* __restrict__ m, float* __restrict__ v, long long off,
                                                        long long n, int world, int rank, AdamHyper h,
                                                        const float* __restrict__ coef_ptr = nullptr) {
  // element i of the shard is element off + i of the full tensors; n and off are multiples of 4
  const float coef = CLIP ? *coef_ptr : 1.f;
  const long long n4 = n >> 2;
  const long long stride = (long long)gridDim.x * kThreads;
  const float* __restrict__ g_own = pp.grad[MODE == 0 ? 0 : rank];
  float* __restrict__ p_own = pp.param[MODE == 0 ? 0 : rank];
  for (long long i0 = (long long)blockIdx.x * kThreads + threadIdx.x; i0 < n4; i0 += stride * UNROLL) {
    float4 g[UNROLL], p[UNROLL], mm[UNROLL], vv[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long i = i0 + u * stride;
      if (i < n4) {
        const long long e = off + 4 * i;
        g[u] = MODE == 2 ? ld_reduce_add(mc_grad + e) : *reinterpret_cast<const float4*>(g_own + e);
      }
    }
    if (MODE == 1) {
      for (int k = 1; k < world; ++k) {                // fixed summation order: rank+1, rank+2, ...
        const float* __restrict__ gk = pp.grad[(rank + k) % world];
        float4 t[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          const long long i = i0 + u * stride;
          if (i < n4) t[u] = *reinterpret_cast<const float4*>(gk + off + 4 * i);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          const long long i = i0 + u * stride;
          if (i < n4) { g[u].x += t[u].x; g[u].y += t[u].y; g[u].z += t[u].z; g[u].w += t[u].w; }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long i = i0 + u * stride;
      if (i < n4) {
        p[u] = *reinterpret_cast<const float4*>(p_own + off + 4 * i);
        mm[u] = reinterpret_cast<const float4*>(m)[i];
        vv[u] = reinterpret_cast<const float4*>(v)[i];
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long i = i0 + u * stride;
      if (i < n4) {
        const long long e = off + 4 * i;
        if (CLIP) {
          p[u].x = adam_one(p[u].x, g[u].x, mm[u].x, vv[u].x, h, coef);
          p[u].y = adam_one(p[u].y, g[u].y, mm[u].y, vv[u].y, h, coef);
          p[u].z = adam_one(p[u].z, g[u].z, mm[u].z, vv[u].z, h, coef);
          p[u].w = adam_one(p[u].w, g[u].w, mm[u].w, vv[u].w, h, coef);
        } else {
          p[u].x = adam_one(p[u].x, g[u].x, mm[u].x, vv[u].x, h);
          p[u].y = adam_one(p[u].y, g[u].y, mm[u].y, vv[u].y, h);
          p[u].z = adam_one(p[u].z, g[u].z, mm[u].z, vv[u].z, h);
          p[u].w = adam_one(p[u].w, g[u].w, mm[u].w, vv[u].w, h);
        }
        reinterpret_cast<float4*>(m)[i] = mm[u];
        reinterpret_cast<float4*>(v)[i] = vv[u];
        if (MODE == 2) {
          mc_store(mc_param + e, p[u]);
        } else if (MODE == 1) {
          for (int k = 0; k < world; ++k) *reinterpret_cast<float4*>(pp.param[(rank + k) % world] + e) = p[u];
        } else {
          *reinterpret_cast<float4*>(p_own + e) = p[u];
        }
      }
    }
  }
}

// tail (n % 4 elements) and unaligned tensors of the local form
template <bool CLIP = false>
__global__ void adam_scalar_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                   float* __restrict__ v, long long n, AdamHyper h, const float* __restrict__ coef = nullptr) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float mm = m[i], vv = v[i];
    p[i] = CLIP ? adam_one(p[i], g[i], mm, vv, h, *coef) : adam_one(p[i], g[i], mm, vv, h);
    m[i] = mm; v[i] = vv;
  }
}

int grid_for(long long n4) {
  const long long want = (n4 + kThreads - 1) / kThreads;
  const long long cap = (long long)dd::kSMs * 8;
  return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

// ---- dd_grad_sumsq -------------------------------------------------------------------------------------------------------
constexpr int kSumsqTensors = 64;              // tensors per launch; a longer list takes several launches
constexpr int kSumsqBlocks = dd::kSMs * 8;

struct TensorList {
  const float* ptr[kSumsqTensors];
  long long n[kSumsqTensors];
  int count;
};

struct SumsqWorkspace {
  double partial[kSumsqBlocks];                // CTA b's running sum over the launches of one call
  unsigned int ticket;
  unsigned int pad[3];
};

__device__ __forceinline__ double sq(float x) { return (double)x * (double)x; }   // exact: 24-bit mantissas, 48-bit product

// Grid-stride over each tensor in turn: its unaligned head (< 4 elements) and tail (< 4) by single loads, the rest as
// UNROLL independent 16-byte streaming loads per thread and iteration.  Each thread sums in fp64, each CTA folds its
// threads in a fixed order into partial[blockIdx.x] (the first launch of a call overwrites it, later ones add), and on the
// call's last launch the last CTA to finish (ticket) folds the partials in a fixed tree: the same grid gives the same bits
// on every run, and there are no float atomics.
template <int UNROLL>
__global__ void __launch_bounds__(kThreads) grad_sumsq_kernel(TensorList tl, SumsqWorkspace* __restrict__ ws, int first, int last,
                                                              float max_norm, float* __restrict__ out) {
  const long long tid = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long stride = (long long)gridDim.x * kThreads;
  double acc = 0.0;
  for (int t = 0; t < tl.count; ++t) {
    const float* __restrict__ p = tl.ptr[t];
    const long long n = tl.n[t];
    long long head = (long long)((16 - ((uintptr_t)p & 15)) & 15) >> 2;
    if (head > n) head = n;
    const long long n4 = (n - head) >> 2;
    const float4* __restrict__ p4 = reinterpret_cast<const float4*>(p + head);
    for (long long i0 = tid; i0 < n4; i0 += stride * UNROLL) {
      float4 x[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const long long i = i0 + u * stride;
        x[u] = i < n4 ? __ldcs(p4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) acc += (sq(x[u].x) + sq(x[u].y)) + (sq(x[u].z) + sq(x[u].w));
    }
    const long long tail0 = head + 4 * n4;
    if (tid < head) acc += sq(p[tid]);
    if (tid < n - tail0) acc += sq(p[tail0 + tid]);
  }
  __shared__ double sred[kThreads / 32];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  acc = dd::warp_sum(acc);
  if (lane == 0) sred[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = first ? 0.0 : ws->partial[blockIdx.x];
    double blk = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) blk += sred[w];
    ws->partial[blockIdx.x] = tot + blk;
    is_last = false;
    if (last) {
      __threadfence();
      is_last = atomicAdd(&ws->ticket, 1u) == gridDim.x - 1;
    }
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  double f = 0.0;
  for (unsigned int b = threadIdx.x; b < gridDim.x; b += kThreads) f += __ldcg(&ws->partial[b]);
  f = dd::warp_sum(f);
  __syncthreads();                              // sred is reused
  if (lane == 0) sred[warp] = f;
  __syncthreads();
  if (threadIdx.x == 0) {
    double sumsq = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) sumsq += sred[w];
    // clip_grad_norm_: total_norm in fp32; clip_coef = max_norm / (total_norm + 1e-6), which torch evaluates as
    // reciprocal(total_norm + 1e-6) * max_norm; clamp(max=1) lets NaN through
    const float norm = (float)sqrt(sumsq);
    const float c = __fmul_rn(__frcp_rn(__fadd_rn(norm, 1e-6f)), max_norm);
    out[0] = norm;
    out[1] = isnan(c) ? c : fminf(c, 1.f);
    *reinterpret_cast<double*>(out + 2) = sumsq;
    ws->ticket = 0;                             // self-reset for the next call on this stream
  }
}

}  // namespace

namespace {

// dd_adam_step and dd_adam_step_clipped: the 16-byte body and the scalar tail (or the whole of an unaligned tensor)
template <bool CLIP>
int adam_step_local(const char* what, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                    float beta1, float beta2, float eps, float weight_decay, long long step, float grad_scale, const float* coef,
                    void* stream) {
  DD_REQUIRE(param && grad && exp_avg && exp_avg_sq && (coef || !CLIP), DD_ERR_BAD_ARG, "%s: null pointer", what);
  DD_REQUIRE(n >= 0 && step >= 1, DD_ERR_BAD_ARG, "%s: n %lld step %lld", what, n, step);
  if (n == 0) return 0;
  const AdamHyper h = dd::adam_hyper(lr, beta1, beta2, eps, weight_decay, step, grad_scale);
  cudaStream_t st = dd::as_stream(stream);
  const bool aligned = ((((uintptr_t)param) | ((uintptr_t)grad) | ((uintptr_t)exp_avg) | ((uintptr_t)exp_avg_sq)) & 15) == 0;
  const long long nvec = aligned ? (n & ~3LL) : 0;
  if (nvec > 0) {
    PeerPtrs pp = {};
    pp.grad[0] = grad; pp.param[0] = param;
    adam_kernel<0, 4, CLIP><<<grid_for(nvec >> 2), kThreads, 0, st>>>(pp, nullptr, nullptr, exp_avg, exp_avg_sq, 0, nvec, 1, 0, h,
                                                                       coef);
    if (int e = dd::check_launch("adam_kernel")) return e;
  }
  if (n > nvec) {
    const long long r = n - nvec;
    adam_scalar_kernel<CLIP><<<(unsigned)((r + 255) / 256), 256, 0, st>>>(param + nvec, grad + nvec, exp_avg + nvec,
                                                                           exp_avg_sq + nvec, r, h, coef);
    if (int e = dd::check_launch("adam_scalar_kernel")) return e;
  }
  return 0;
}

}  // namespace

extern "C" int dd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                            float beta1, float beta2, float eps, float weight_decay, long long step, float grad_scale,
                            void* stream) {
  return adam_step_local<false>("dd_adam_step", param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                                step, grad_scale, nullptr, stream);
}

extern "C" int dd_adam_step_clipped(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                                    float beta1, float beta2, float eps, float weight_decay, long long step, float grad_scale,
                                    const float* coef, void* stream) {
  return adam_step_local<true>("dd_adam_step_clipped", param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                               weight_decay, step, grad_scale, coef, stream);
}

extern "C" size_t dd_grad_sumsq_workspace_bytes(void) { return sizeof(SumsqWorkspace); }

extern "C" int dd_grad_sumsq(const void* const* ptrs, const long long* numels, int count, float max_norm, float* out,
                             void* workspace, size_t ws_bytes, void* stream) {
  DD_REQUIRE(out && workspace && count >= 0 && (count == 0 || (ptrs && numels)), DD_ERR_BAD_ARG, "dd_grad_sumsq: null pointer");
  DD_REQUIRE(ws_bytes >= sizeof(SumsqWorkspace), DD_ERR_WORKSPACE, "dd_grad_sumsq: workspace %zu < %zu", ws_bytes,
             sizeof(SumsqWorkspace));
  DD_REQUIRE(isfinite(max_norm) && max_norm >= 0.f, DD_ERR_BAD_ARG, "dd_grad_sumsq: max_norm %g", (double)max_norm);
  DD_REQUIRE(((uintptr_t)out & 7) == 0, DD_ERR_ALIGNMENT, "dd_grad_sumsq: out must be 8-byte aligned");
  long long total = 0;
  for (int t = 0; t < count; ++t) {
    DD_REQUIRE(numels[t] >= 0 && (numels[t] == 0 || ptrs[t]), DD_ERR_BAD_ARG, "dd_grad_sumsq: tensor %d: null pointer or "
               "length %lld", t, numels[t]);
    DD_REQUIRE(((uintptr_t)ptrs[t] & 3) == 0, DD_ERR_ALIGNMENT, "dd_grad_sumsq: tensor %d is not 4-byte aligned", t);
    total += numels[t];
  }
  // one grid for every launch of the call (each CTA owns its partial across them), sized by the whole list
  const long long want = (total / 4 + kThreads - 1) / kThreads;
  const int grid = (int)(want < 1 ? 1 : (want < kSumsqBlocks ? want : kSumsqBlocks));
  cudaStream_t st = dd::as_stream(stream);
  SumsqWorkspace* ws = (SumsqWorkspace*)workspace;
  int t = 0;
  do {
    TensorList tl;
    tl.count = count - t < kSumsqTensors ? count - t : kSumsqTensors;
    for (int i = 0; i < tl.count; ++i) {
      tl.ptr[i] = (const float*)ptrs[t + i];
      tl.n[i] = numels[t + i];
    }
    const int first = t == 0;
    t += tl.count;
    grad_sumsq_kernel<4><<<grid, kThreads, 0, st>>>(tl, ws, first, t == count, max_norm, out);
    if (int e = dd::check_launch("grad_sumsq_kernel")) return e;
  } while (t < count);
  return 0;
}

extern "C" int dd_adam_step_sharded(const void* const* grad_replicas, void* const* param_replicas, const void* mc_grad,
                                    void* mc_param, int world, int rank, float* exp_avg_shard, float* exp_avg_sq_shard,
                                    long long shard_offset, long long shard_numel, float lr, float beta1, float beta2,
                                    float eps, float weight_decay, long long step, float grad_scale, int ctas_per_sm, void* stream) {
  DD_REQUIRE(grad_replicas && param_replicas && exp_avg_shard && exp_avg_sq_shard, DD_ERR_BAD_ARG, "dd_adam_step_sharded: null pointer");
  DD_REQUIRE(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world, DD_ERR_BAD_ARG,
             "dd_adam_step_sharded: world %d (max %d) rank %d", world, kMaxRanks, rank);
  DD_REQUIRE(shard_numel >= 0 && (shard_numel & 3) == 0 && (shard_offset & 3) == 0 && step >= 1, DD_ERR_ALIGNMENT,
             "dd_adam_step_sharded: shard offset %lld / length %lld must be multiples of 4 elements", shard_offset, shard_numel);
  if (shard_numel == 0) return 0;
  PeerPtrs pp = {};
  for (int k = 0; k < world; ++k) {
    pp.grad[k] = (const float*)grad_replicas[k];
    pp.param[k] = (float*)param_replicas[k];
    DD_REQUIRE(pp.grad[k] && pp.param[k], DD_ERR_BAD_ARG, "dd_adam_step_sharded: replica %d is null", k);
    DD_REQUIRE(((((uintptr_t)pp.grad[k]) | ((uintptr_t)pp.param[k])) & 15) == 0, DD_ERR_ALIGNMENT,
               "dd_adam_step_sharded: replica %d is not 16-byte aligned", k);
  }
  const AdamHyper h = dd::adam_hyper(lr, beta1, beta2, eps, weight_decay, step, grad_scale);
  cudaStream_t st = dd::as_stream(stream);
  // ctas_per_sm = 1 leaves room for a persistent conv CTA beside each update CTA (update overlapped with the backward pass)
  const long long want = ((shard_numel >> 2) + kThreads - 1) / kThreads;
  const long long cap = (long long)dd::kSMs * (ctas_per_sm >= 1 && ctas_per_sm <= 8 ? ctas_per_sm : 8);
  const int grid = (int)(want < cap ? want : cap);
  // An SM's L1 / shared-memory split only changes when the SM is idle: with the default carveout (all L1 for a kernel that
  // uses no shared memory) the persistent conv kernels of the backward pass (90-210 KB of shared memory per CTA) could not
  // join an SM that runs an update CTA and queued behind the whole update (1.2 ms gap seen in the step timeline).
  static const bool carveout_set = [] {
    cudaFuncSetAttribute(adam_kernel<1, 2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaFuncSetAttribute(adam_kernel<2, 4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    return true;
  }();
  (void)carveout_set;
  if (mc_grad && mc_param)
    adam_kernel<2, 4><<<grid, kThreads, 0, st>>>(pp, (const float*)mc_grad, (float*)mc_param, exp_avg_shard, exp_avg_sq_shard,
                                              shard_offset, shard_numel, world, rank, h);
  else
    adam_kernel<1, 2><<<grid, kThreads, 0, st>>>(pp, nullptr, nullptr, exp_avg_shard, exp_avg_sq_shard, shard_offset, shard_numel,
                                              world, rank, h);
  return dd::check_launch("adam_kernel(sharded)");
}
