// torch.optim.Adam's update of one element (amsgrad off, L2 weight decay), shared by the Adam kernels of adam.cu and the
// fused backward + Adam kernel of linear_tc.cu: one expression, so both compile to the same arithmetic and produce the same
// bits.
#pragma once
#include <math.h>

#include "dd_common.cuh"

namespace dd {

struct AdamHyper {
  float beta1, beta2, eps, step_size, inv_sqrt_bc2, weight_decay, grad_scale;
};

// g is the gradient as the step applies it (already scaled)
__device__ __forceinline__ float adam_apply(float p, float g, float& m, float& v, const AdamHyper& h) {
  if (h.weight_decay != 0.f) g = fmaf(h.weight_decay, p, g);          // torch.optim.Adam: L2 term added to the gradient
  m = m + (1.f - h.beta1) * (g - m);                                   // lerp, as torch's fused kernel
  v = h.beta2 * v + (1.f - h.beta2) * g * g;
  const float denom = sqrtf(v) * h.inv_sqrt_bc2 + h.eps;
  return p - h.step_size * (m / denom);
}

__device__ __forceinline__ float adam_one(float p, float g, float& m, float& v, const AdamHyper& h) {
  return adam_apply(p, g * h.grad_scale, m, v, h);
}

// With clip_grad_norm_'s coefficient: the gradient is scaled, then clipped (torch multiplies .grad by the coefficient
// before Adam adds the L2 term).  coef == 1 gives adam_one's bits.
__device__ __forceinline__ float adam_one(float p, float g, float& m, float& v, const AdamHyper& h, float coef) {
  return adam_apply(p, (g * h.grad_scale) * coef, m, v, h);
}

// ---- deterministic fp64 sums of squares over a grid (gradient norms) ----------------------------------------------------
// g*g is exact in fp64 (24-bit mantissas, 48-bit product).  Each CTA folds its threads in a fixed order into partial[its
// index]; the last CTA to finish (ticket) adds the partials in a fixed order: the same grid gives the same bits on every run,
// and there are no float atomics.  The workspace is zeroed once by its owner and resets itself; launches that share one
// must be ordered.
constexpr int kSumsqMaxCtas = kSMs * 8;
struct SumsqWorkspace {
  double partial[kSumsqMaxCtas];
  unsigned int ticket;
  unsigned int pad[3];
};

__device__ __forceinline__ double sq(float x) { return (double)x * (double)x; }

// Called by one whole warp of every CTA of the grid, with the CTA's sum in lane 0; the last CTA writes the grid's sum to *out.
__device__ __forceinline__ void sumsq_fold_grid(SumsqWorkspace* ws, double cta, double* out) {
  const int lane = threadIdx.x & 31;
  unsigned int last = 0;
  if (lane == 0) {
    ws->partial[blockIdx.x] = cta;
    __threadfence();
    last = atomicAdd(&ws->ticket, 1u) == gridDim.x - 1;
  }
  if (!__shfl_sync(0xffffffffu, last, 0)) return;
  __threadfence();
  double s = 0.0;
  for (unsigned int b = lane; b < gridDim.x; b += 32) s += __ldcg(&ws->partial[b]);
  s = warp_sum(s);
  if (lane == 0) {
    *out = s;
    ws->ticket = 0;
  }
}

// bias corrections of step t >= 1, in double
inline AdamHyper adam_hyper(float lr, float beta1, float beta2, float eps, float weight_decay, long long step, float grad_scale) {
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  AdamHyper h;
  h.beta1 = beta1; h.beta2 = beta2; h.eps = eps; h.weight_decay = weight_decay; h.grad_scale = grad_scale;
  h.step_size = (float)((double)lr / bc1);
  h.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  return h;
}

}  // namespace dd
