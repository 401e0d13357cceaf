// Per-tensor gradient norms (FusedAdam's track_grad_norm, Lightning's grad_norm): one fp64 sum of squares per tensor, on the
// device and deterministic, for the gradients FusedAdam stores (world size 1 without the fused backward + Adam kernel,
// accumulation buffers, the data-parallel flat bucket).  The wide weights whose step runs inside a kernel get their sums
// from that kernel (dd_linear_bwd_adam_sumsq, dd_adam_step_sharded_sumsq).
// Its own translation unit: beside grad_sumsq_kernel in adam.cu, this kernel changed that one's register allocation.
#include <stdint.h>

#include "adam.cuh"
#include "dd_common.cuh"

namespace {

using dd::sq;

constexpr int kThreads = 256;
constexpr int kMaxRanks = 16;                  // as dd_adam_step_sharded's
constexpr int kSumsqTensors = 64;              // tensors per launch; a longer list takes several launches
constexpr int kSumsqBlocks = dd::kSumsqMaxCtas;

struct PeerPtrs {
  const float* grad[kMaxRanks];                // every rank's gradient replica (index = rank)
};

// ---- dd_grad_sumsq_each / dd_grad_sumsq_each_replicas ------------------------------------------------------------------
// One fp64 sum of squares per tensor (gradient norms per parameter).  Local form: tensor t is ptr[t][0, n[t]), any 4-byte
// alignment.  REPL form (a data-parallel flat bucket): element j of tensor t is the rank mean as the sharded update consumes
// it, (g_rank + g_rank+1 + ... + g_rank+world-1)[off[t] + j] * scale, the replicas summed in adam_kernel<1>'s order;
// off[t] is a multiple of 4 elements and the replicas are 16-byte aligned.
struct EachList {
  const float* ptr[kSumsqTensors];
  long long off[kSumsqTensors];
  long long n[kSumsqTensors];
  double* out[kSumsqTensors];
  int count;
};

struct EachWorkspace {
  double partial[kSumsqTensors][kSumsqBlocks];   // [tensor][CTA]
  unsigned int ticket;
  unsigned int pad[3];
};

template <bool REPL>
__device__ __forceinline__ float4 each_load4(const EachList& tl, const PeerPtrs& pp, int world, int rank, float scale, int t,
                                             long long e) {
  if (!REPL) return __ldcs(reinterpret_cast<const float4*>(tl.ptr[t] + e));
  float4 g = *reinterpret_cast<const float4*>(pp.grad[rank] + tl.off[t] + e);
  for (int k = 1; k < world; ++k) {
    const float4 x = *reinterpret_cast<const float4*>(pp.grad[(rank + k) % world] + tl.off[t] + e);
    g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
  }
  return make_float4(g.x * scale, g.y * scale, g.z * scale, g.w * scale);
}

template <bool REPL>
__device__ __forceinline__ float each_load1(const EachList& tl, const PeerPtrs& pp, int world, int rank, float scale, int t,
                                            long long e) {
  if (!REPL) return tl.ptr[t][e];
  float g = pp.grad[rank][tl.off[t] + e];
  for (int k = 1; k < world; ++k) g += pp.grad[(rank + k) % world][tl.off[t] + e];
  return g * scale;
}

// Grid-stride over each tensor in turn (16-byte loads, UNROLL in flight per thread), each CTA folds its threads into
// partial[t][its index]; the last CTA (ticket) folds every tensor's partials in CTA order, one warp per tensor.
template <bool REPL, int UNROLL>
__global__ void __launch_bounds__(kThreads) grad_sumsq_each_kernel(EachList tl, PeerPtrs pp, int world, int rank, float scale,
                                                                   EachWorkspace* __restrict__ ws) {
  const long long tid = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long stride = (long long)gridDim.x * kThreads;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ double sred[kThreads / 32];
  __shared__ bool is_last;
  for (int t = 0; t < tl.count; ++t) {
    const long long n = tl.n[t];
    long long head = REPL ? 0 : (long long)((16 - ((uintptr_t)tl.ptr[t] & 15)) & 15) >> 2;
    if (head > n) head = n;
    const long long n4 = (n - head) >> 2;
    double acc = 0.0;
    for (long long i0 = tid; i0 < n4; i0 += stride * UNROLL) {
      float4 x[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const long long i = i0 + u * stride;
        x[u] = i < n4 ? each_load4<REPL>(tl, pp, world, rank, scale, t, head + 4 * i) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) acc += (sq(x[u].x) + sq(x[u].y)) + (sq(x[u].z) + sq(x[u].w));
    }
    const long long tail0 = head + 4 * n4;
    if (tid < head) acc += sq(each_load1<REPL>(tl, pp, world, rank, scale, t, tid));
    if (tid < n - tail0) acc += sq(each_load1<REPL>(tl, pp, world, rank, scale, t, tail0 + tid));
    acc = dd::warp_sum(acc);
    if (lane == 0) sred[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double blk = 0.0;
      for (int w = 0; w < kThreads / 32; ++w) blk += sred[w];
      ws->partial[t][blockIdx.x] = blk;
    }
    __syncthreads();                              // sred is reused by the next tensor
  }
  if (threadIdx.x == 0) {
    __threadfence();
    is_last = atomicAdd(&ws->ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int t = warp; t < tl.count; t += kThreads / 32) {
    double f = 0.0;
    for (unsigned int b = lane; b < gridDim.x; b += 32) f += __ldcg(&ws->partial[t][b]);
    f = dd::warp_sum(f);
    if (lane == 0) *tl.out[t] = f;
  }
  if (threadIdx.x == 0) ws->ticket = 0;           // self-reset for the next launch on this stream
}

// Both forms: the tensor list in launches of kSumsqTensors, one grid sized by the whole list.
int grad_sumsq_each(const char* what, const void* const* ptrs, const long long* offs, const long long* numels, double* const* outs,
                    int count, const PeerPtrs& pp, int world, int rank, float scale, void* workspace, size_t ws_bytes,
                    void* stream) {
  DD_REQUIRE(workspace && count >= 0 && (count == 0 || (numels && outs)), DD_ERR_BAD_ARG, "%s: null pointer", what);
  DD_REQUIRE(ws_bytes >= sizeof(EachWorkspace), DD_ERR_WORKSPACE, "%s: workspace %zu < %zu", what, ws_bytes, sizeof(EachWorkspace));
  const bool repl = offs != nullptr;
  long long total = 0;
  for (int t = 0; t < count; ++t) {
    DD_REQUIRE(outs[t] && ((uintptr_t)outs[t] & 7) == 0, DD_ERR_ALIGNMENT, "%s: out %d is null or not 8-byte aligned", what, t);
    DD_REQUIRE(numels[t] >= 0, DD_ERR_BAD_ARG, "%s: tensor %d: length %lld", what, t, numels[t]);
    if (repl) {
      DD_REQUIRE(offs[t] >= 0 && (offs[t] & 3) == 0, DD_ERR_ALIGNMENT, "%s: tensor %d: offset %lld is not a multiple of 4",
                 what, t, offs[t]);
    } else {
      DD_REQUIRE(numels[t] == 0 || ptrs[t], DD_ERR_BAD_ARG, "%s: tensor %d: null pointer", what, t);
      DD_REQUIRE(((uintptr_t)ptrs[t] & 3) == 0, DD_ERR_ALIGNMENT, "%s: tensor %d is not 4-byte aligned", what, t);
    }
    total += numels[t];
  }
  if (count == 0) return 0;
  const long long want = (total / 4 + kThreads - 1) / kThreads;
  const int grid = (int)(want < 1 ? 1 : (want < kSumsqBlocks ? want : kSumsqBlocks));
  cudaStream_t st = dd::as_stream(stream);
  EachWorkspace* ws = (EachWorkspace*)workspace;
  for (int t = 0; t < count; t += kSumsqTensors) {
    EachList tl = {};
    tl.count = count - t < kSumsqTensors ? count - t : kSumsqTensors;
    for (int i = 0; i < tl.count; ++i) {
      tl.ptr[i] = repl ? nullptr : (const float*)ptrs[t + i];
      tl.off[i] = repl ? offs[t + i] : 0;
      tl.n[i] = numels[t + i];
      tl.out[i] = outs[t + i];
    }
    if (repl)
      grad_sumsq_each_kernel<true, 2><<<grid, kThreads, 0, st>>>(tl, pp, world, rank, scale, ws);
    else
      grad_sumsq_each_kernel<false, 4><<<grid, kThreads, 0, st>>>(tl, pp, world, rank, scale, ws);
    if (int e = dd::check_launch("grad_sumsq_each_kernel")) return e;
  }
  return 0;
}

}  // namespace

extern "C" size_t dd_grad_sumsq_each_workspace_bytes(void) { return sizeof(EachWorkspace); }

extern "C" int dd_grad_sumsq_each(const void* const* ptrs, const long long* numels, double* const* outs, int count,
                                  void* workspace, size_t ws_bytes, void* stream) {
  DD_REQUIRE(count == 0 || ptrs, DD_ERR_BAD_ARG, "dd_grad_sumsq_each: null pointer");
  return grad_sumsq_each("dd_grad_sumsq_each", ptrs, nullptr, numels, outs, count, PeerPtrs{}, 1, 0, 1.f, workspace, ws_bytes,
                         stream);
}

extern "C" int dd_grad_sumsq_each_replicas(const void* const* grad_replicas, int world, int rank, float grad_scale,
                                           const long long* offsets, const long long* numels, double* const* outs, int count,
                                           void* workspace, size_t ws_bytes, void* stream) {
  DD_REQUIRE(grad_replicas && (count == 0 || offsets), DD_ERR_BAD_ARG, "dd_grad_sumsq_each_replicas: null pointer");
  DD_REQUIRE(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world, DD_ERR_BAD_ARG,
             "dd_grad_sumsq_each_replicas: world %d (max %d) rank %d", world, kMaxRanks, rank);
  PeerPtrs pp = {};
  for (int k = 0; k < world; ++k) {
    pp.grad[k] = (const float*)grad_replicas[k];
    DD_REQUIRE(pp.grad[k] && ((uintptr_t)pp.grad[k] & 15) == 0, DD_ERR_ALIGNMENT,
               "dd_grad_sumsq_each_replicas: replica %d is null or not 16-byte aligned", k);
  }
  return grad_sumsq_each("dd_grad_sumsq_each_replicas", nullptr, offsets, numels, outs, count, pp, world, rank, grad_scale,
                         workspace, ws_bytes, stream);
}

