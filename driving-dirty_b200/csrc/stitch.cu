// K1: six-view stitch.  mosaic[b,c,h,j*W+w] = views[b,order[j],c,h,w], order = {0,1,2,5,4,3}
// (reference: roadmap_bce_v2.py:53-64, autoencoder.py:53-73).  Pure data movement, HBM-bound:
// algorithmic bytes = 2 * 4 * B*18*H*W.  One CTA walks whole mosaic rows; lanes move 8-byte
// pairs (view rows are 1224 B = 8-byte aligned only, SURVEY H3), four pairs in flight per lane.
#include "dd_common.cuh"

namespace {

template <int MODE>  // 0 = plain, 1 = mask variant (x zeroed block + y)
__global__ void __launch_bounds__(256) stitch_rows_kernel(const float* __restrict__ views,
                                                          float* __restrict__ mosaic,
                                                          float* __restrict__ y, int B, int H, int W,
                                                          int slot) {
  const int rows = B * 3 * H;
  const int W2 = W >> 1;       // pairs per view row
  const int pairs = 6 * W2;    // pairs per mosaic row
  const size_t view_elems = (size_t)3 * H * W;
  for (int row = blockIdx.x; row < rows; row += gridDim.x) {
    const int h = row % H;
    const int c = (row / H) % 3;
    const int b = row / (3 * H);
    const float* vbase = views + (size_t)b * 6 * view_elems + ((size_t)c * H + h) * W;
    float2* orow = reinterpret_cast<float2*>(mosaic + (size_t)row * 6 * W);
    // four independent 8-byte pairs per lane and trip, all loads issued before the first store: 8 KB in flight per CTA
    for (int i0 = threadIdx.x; i0 < pairs; i0 += 4 * blockDim.x) {
      float2 v[4];
      int jj[4], ww[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i < pairs) {
          jj[u] = i / W2;
          ww[u] = i - jj[u] * W2;
          v[u] = __ldcs(reinterpret_cast<const float2*>(vbase + (size_t)dd::view_of_slot(jj[u]) * view_elems) + ww[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i < pairs) {
          if (MODE == 1 && jj[u] == slot) {
            reinterpret_cast<float2*>(y + (size_t)row * W)[ww[u]] = v[u];
            v[u] = make_float2(0.f, 0.f);
          }
          __stcs(orow + i, v[u]);
        }
      }
    }
  }
}

template <int MODE, typename TIN>  // generic scalar path (odd W, or u8 input)
__global__ void __launch_bounds__(256) stitch_scalar_kernel(const TIN* __restrict__ views,
                                                            float* __restrict__ mosaic,
                                                            float* __restrict__ y, int B, int H, int W,
                                                            int slot) {
  const long long total = (long long)B * 3 * H * 6 * W;
  const size_t view_elems = (size_t)3 * H * W;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int wm = (int)(idx % (6 * W));
    const long long row = idx / (6 * W);
    const int h = (int)(row % H);
    const int c = (int)((row / H) % 3);
    const int b = (int)(row / (3 * H));
    const int j = wm / W, w = wm - j * W;
    const TIN raw = views[(size_t)b * 6 * view_elems + (size_t)dd::view_of_slot(j) * view_elems +
                          ((size_t)c * H + h) * W + w];
    float v;
    if (sizeof(TIN) == 1) v = __fdiv_rn((float)raw, 255.0f);  // == ToTensor: x.float()/255
    else v = (float)raw;
    if (MODE == 1 && j == slot) {
      y[(size_t)row * W + w] = v;
      v = 0.f;
    }
    mosaic[idx] = v;
  }
}

// ToTensor as a pass of its own (data_helper.py:109-114): out[i] = float(in[i]) / 255, bit-identical (the IEEE division is
// done once per CTA for the 256 possible bytes).  16 bytes in, four 16-byte stores out per thread and iteration.
__global__ void __launch_bounds__(256) u8_to_f32_kernel(const uint8_t* __restrict__ in, float* __restrict__ out, long long n) {
  __shared__ float lut[256];
  lut[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.0f);
  __syncthreads();
  const long long n16 = n >> 4;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) {
    const uint4 raw = __ldcs(reinterpret_cast<const uint4*>(in) + i);
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      __stcs(reinterpret_cast<float4*>(out) + 4 * i + k,
             make_float4(lut[w[k] & 255u], lut[(w[k] >> 8) & 255u], lut[(w[k] >> 16) & 255u], lut[w[k] >> 24]));
  }
  for (long long i = (n16 << 4) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = lut[in[i]];
}

// Backward of the stitch (and of the mask variant, slot >= 0): dviews[b,v,c,h,w] = dmosaic[b,c,h,j*W+w] with j the slot
// showing view v (the order is its own inverse), except that the masked slot's view takes dy[b,c,h,w] (0 for dy == NULL):
// its block of x was zeroed and passes nothing back.  Thread = views element, so every element is written once.
__global__ void __launch_bounds__(256) unstitch_kernel(const float* __restrict__ dmosaic, const float* __restrict__ dy,
                                                       float* __restrict__ dviews, int B, int H, int W, int slot) {
  const long long total = (long long)B * 18 * H * W;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int w = (int)(idx % W);
    long long r = idx / W;
    const int h = (int)(r % H);
    r /= H;
    const int c = (int)(r % 3);
    r /= 3;
    const int j = dd::view_of_slot((int)(r % 6));
    const long long b = r / 6;
    const size_t row = ((size_t)b * 3 + c) * H + h;
    float g;
    if (j == slot) g = dy ? dy[row * W + w] : 0.f;
    else g = dmosaic[row * 6 * W + (size_t)j * W + w];
    dviews[idx] = g;
  }
}

int launch_stitch(const float* views, float* x, float* y, int B, int H, int W, int slot, int mode,
                  cudaStream_t st) {
  const int rows = B * 3 * H;
  const bool vec = (W % 2 == 0) && ((uintptr_t)views % 8 == 0) && ((uintptr_t)x % 8 == 0) &&
                   (mode == 0 || (uintptr_t)y % 8 == 0);
  if (vec) {
    int grid = rows < dd::kSMs * 8 ? rows : dd::kSMs * 8;
    if (mode == 0) stitch_rows_kernel<0><<<grid, 256, 0, st>>>(views, x, y, B, H, W, slot);
    else stitch_rows_kernel<1><<<grid, 256, 0, st>>>(views, x, y, B, H, W, slot);
  } else {
    long long total = (long long)rows * 6 * W;
    int grid = (int)((total + 255) / 256 < dd::kSMs * 8 ? (total + 255) / 256 : dd::kSMs * 8);
    if (mode == 0) stitch_scalar_kernel<0, float><<<grid, 256, 0, st>>>(views, x, y, B, H, W, slot);
    else stitch_scalar_kernel<1, float><<<grid, 256, 0, st>>>(views, x, y, B, H, W, slot);
  }
  return dd::check_launch("stitch");
}
}  // namespace

extern "C" int dd_stitch_f32(const float* views, float* mosaic, int B, int H, int W, void* stream) {
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_stitch_f32: bad shape B=%d H=%d W=%d", B, H, W);
  if (B == 0) return 0;   // empty batch: nothing to move (torch hands out null pointers for empty tensors)
  DD_REQUIRE(views && mosaic, DD_ERR_BAD_ARG, "dd_stitch_f32: null pointer");
  return launch_stitch(views, mosaic, nullptr, B, H, W, -1, 0, dd::as_stream(stream));
}

extern "C" int dd_stitch_mask_f32(const float* views, float* x, float* y, int B, int H, int W, int slot,
                                  void* stream) {
  DD_REQUIRE(views && x && y, DD_ERR_BAD_ARG, "dd_stitch_mask_f32: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_stitch_mask_f32: bad shape");
  DD_REQUIRE(slot >= 0 && slot < 6, DD_ERR_BAD_ARG, "dd_stitch_mask_f32: slot %d outside [0,6)", slot);
  if (B == 0) return 0;
  return launch_stitch(views, x, y, B, H, W, slot, 1, dd::as_stream(stream));
}

extern "C" int dd_unstitch_f32(const float* dmosaic, const float* dy, float* dviews, int B, int H, int W, int slot,
                               void* stream) {
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_unstitch_f32: bad shape B=%d H=%d W=%d", B, H, W);
  DD_REQUIRE(slot >= -1 && slot < 6, DD_ERR_BAD_ARG, "dd_unstitch_f32: slot %d outside [-1,6)", slot);
  if (B == 0) return 0;
  DD_REQUIRE(dmosaic && dviews, DD_ERR_BAD_ARG, "dd_unstitch_f32: null pointer");
  const long long total = (long long)B * 18 * H * W;
  const int grid = (int)((total + 255) / 256 < dd::kSMs * 8 ? (total + 255) / 256 : dd::kSMs * 8);
  unstitch_kernel<<<grid, 256, 0, dd::as_stream(stream)>>>(dmosaic, dy, dviews, B, H, W, slot);
  return dd::check_launch("unstitch");
}

extern "C" int dd_stitch_u8(const uint8_t* views, float* mosaic, int B, int H, int W, void* stream) {
  DD_REQUIRE(views && mosaic, DD_ERR_BAD_ARG, "dd_stitch_u8: null pointer");
  DD_REQUIRE(B >= 0 && H > 0 && W > 0, DD_ERR_BAD_ARG, "dd_stitch_u8: bad shape");
  if (B == 0) return 0;
  long long total = (long long)B * 3 * H * 6 * W;
  int grid = (int)((total + 255) / 256 < dd::kSMs * 8 ? (total + 255) / 256 : dd::kSMs * 8);
  stitch_scalar_kernel<0, uint8_t><<<grid, 256, 0, dd::as_stream(stream)>>>(views, mosaic, nullptr, B, H, W, -1);
  return dd::check_launch("stitch_u8");
}

extern "C" int dd_u8_to_f32(const uint8_t* in, float* out, long long n, void* stream) {
  DD_REQUIRE(n >= 0, DD_ERR_BAD_ARG, "dd_u8_to_f32: n=%lld", n);
  if (n == 0) return 0;
  DD_REQUIRE(in && out, DD_ERR_BAD_ARG, "dd_u8_to_f32: null pointer");
  DD_REQUIRE((uintptr_t)in % 16 == 0 && (uintptr_t)out % 16 == 0, DD_ERR_ALIGNMENT, "dd_u8_to_f32: pointers must be 16-byte aligned");
  const long long want = ((n >> 4) + 255) / 256;
  const int grid = (int)(want < 1 ? 1 : (want < dd::kSMs * 8 ? want : dd::kSMs * 8));
  u8_to_f32_kernel<<<grid, 256, 0, dd::as_stream(stream)>>>(in, out, n);
  return dd::check_launch("u8_to_f32");
}
