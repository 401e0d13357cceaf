// Hardware probe for the operand paths of linear_tc.cu: fp32 matrices in global memory -> TMA boxes with
// 128-byte swizzle -> tcgen05.mma kind::tf32, K-major and MN-major operands.  Integer-valued data, so
// the tf32 products are exact; prints max |D - ref| per experiment.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o tools/umma_tf32_probe tools/umma_tf32_probe.cu
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <vector>

#include "../driving-dirty_b200/csrc/tma_host.h"
#include "../driving-dirty_b200/csrc/umma.cuh"

struct Plan {
  int a_boxes, b_boxes;            // TMA boxes per stage for A / B
  int a_box_bytes, b_box_bytes;
  int a_c0[8], a_c1[8], b_c0[8], b_c1[8];   // box coordinates (stage 0); per-stage advance below
  int a_dc0, a_dc1, b_dc0, b_dc1;  // coordinate advance per stage
  int stages, mma_per_stage;
  uint32_t a_kstep, b_kstep;       // descriptor start advance per MMA (bytes)
  uint32_t a_lbo, a_sbo, b_lbo, b_sbo;
  uint32_t idesc, N;
  int a_base32, b_base32;          // operand uses SWIZZLE_128B_BASE32B (MN-major tf32)
};

__global__ void __launch_bounds__(128) probe(const __grid_constant__ CUtensorMap ta, const __grid_constant__ CUtensorMap tb,
                                             float* d, Plan p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full, done;
  __shared__ uint32_t tmem_base;
  const uint32_t a_bytes = p.a_boxes * p.a_box_bytes, b_bytes = p.b_boxes * p.b_box_bytes;
  uint8_t* sa = smem;
  uint8_t* sb = smem + ((a_bytes + 1023) / 1024) * 1024;
  if (threadIdx.x == 0) { umma::mbar_init(&full, 1); umma::mbar_init(&done, 1); umma::fence_mbar_init(); }
  if (threadIdx.x < 32) umma::tmem_alloc(&tmem_base, 256);
  umma::tc_fence_before_sync();
  __syncthreads();
  umma::tc_fence_after_sync();
  const uint32_t tbase = tmem_base;
  if (threadIdx.x == 0) {
    uint32_t acc = 0;
    for (int s = 0; s < p.stages; ++s) {
      umma::mbar_expect_tx(&full, a_bytes + b_bytes);
      for (int i = 0; i < p.a_boxes; ++i)
        umma::tma_load_2d(umma::smem_u32(sa) + i * p.a_box_bytes, &ta, p.a_c0[i] + s * p.a_dc0, p.a_c1[i] + s * p.a_dc1, &full);
      for (int i = 0; i < p.b_boxes; ++i)
        umma::tma_load_2d(umma::smem_u32(sb) + i * p.b_box_bytes, &tb, p.b_c0[i] + s * p.b_dc0, p.b_c1[i] + s * p.b_dc1, &full);
      umma::mbar_wait(&full, s & 1);
      umma::tc_fence_after_sync();
      for (int k = 0; k < p.mma_per_stage; ++k) {
        const uint32_t a_lo = umma::desc_lo(umma::smem_u32(sa) + k * p.a_kstep, p.a_lbo);
        const uint32_t b_lo = umma::desc_lo(umma::smem_u32(sb) + k * p.b_kstep, p.b_lbo);
        umma::mma_tf32_lohi(tbase, a_lo, p.a_base32 ? umma::desc_hi_sw128_base32(p.a_sbo) : umma::desc_hi_sw128(p.a_sbo), b_lo,
                            p.b_base32 ? umma::desc_hi_sw128_base32(p.b_sbo) : umma::desc_hi_sw128(p.b_sbo), p.idesc, acc);
        acc = 1;
      }
      umma::mma_commit(&done);
      umma::mbar_wait(&done, s & 1);     // smem is reused by the next stage
    }
  }
  __syncthreads();
  umma::tc_fence_after_sync();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (uint32_t c = 0; c < p.N; c += 32) {
    uint32_t r[32];
    umma::tmem_ld_32x32(tbase + ((uint32_t)(warp * 32) << 16) + c, r);
    umma::tmem_ld_wait();
    for (int j = 0; j < 32; ++j) d[(size_t)(warp * 32 + lane) * p.N + c + j] = __uint_as_float(r[j]);
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (threadIdx.x < 32) umma::tmem_dealloc(tbase, 256);
}

static float val(int i, int j, int salt) { return (float)(((i * 7 + j * 13 + salt * 5) % 9) - 4); }

static int run(const char* name, const std::vector<float>& A, int a_rows, int a_cols, const std::vector<float>& B, int b_rows,
               int b_cols, uint32_t a_box_rows, uint32_t b_box_rows, Plan p, const std::vector<float>& ref) {
  float *dA, *dB, *dD;
  cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dD, 128 * 256 * 4);
  cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
  cudaMemset(dD, 0xff, 128 * 256 * 4);
  CUtensorMap ta, tb;
  char msg[256];
  const CUtensorMapSwizzle a_sw = p.a_base32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
  const CUtensorMapSwizzle b_sw = p.b_base32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
  if (dd::tma_map_2d(&ta, dA, 4, a_rows, a_cols, a_cols, 32, a_box_rows, a_sw, msg, sizeof msg) ||
      dd::tma_map_2d(&tb, dB, 4, b_rows, b_cols, b_cols, 32, b_box_rows, b_sw, msg, sizeof msg)) {
    printf("%-52s %s\n", name, msg);
    return 1;
  }
  p.a_box_bytes = a_box_rows * 128; p.b_box_bytes = b_box_rows * 128;
  const size_t smem = 1024 + ((p.a_boxes * p.a_box_bytes + 1023) / 1024) * 1024 + p.b_boxes * p.b_box_bytes + 1024;
  cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  probe<<<1, 128, smem>>>(ta, tb, dD, p);
  cudaError_t err = cudaDeviceSynchronize();
  if (err != cudaSuccess) { printf("%-52s CUDA error: %s\n", name, cudaGetErrorString(err)); return 2; }
  std::vector<float> out((size_t)128 * p.N);
  cudaMemcpy(out.data(), dD, out.size() * 4, cudaMemcpyDeviceToHost);
  double maxerr = 0; int bad = 0;
  for (size_t i = 0; i < out.size(); ++i) { double e = fabs((double)out[i] - ref[i]); if (!(e <= 1e-3)) ++bad; if (e > maxerr || e != e) maxerr = e; }
  printf("%-52s max|err| %-10.3g mismatches %d / %zu  %s\n", name, maxerr, bad, out.size(), bad ? "FAIL" : "ok");
  cudaFree(dA); cudaFree(dB); cudaFree(dD);
  return bad ? 3 : 0;
}

int main() {
  int rc = 0;
  {  // forward: D[n=128][b=32] = sum_k W[n][k] X[b][k];  W [128][64], X [32][64]; both K-major; 2 stages x 4 MMAs (K = 8)
    const int K = 64;
    std::vector<float> W(128 * K), X(32 * K), ref(128 * 32);
    for (int n = 0; n < 128; ++n) for (int k = 0; k < K; ++k) W[n * K + k] = val(n, k, 1);
    for (int b = 0; b < 32; ++b) for (int k = 0; k < K; ++k) X[b * K + k] = val(b, k, 2);
    for (int n = 0; n < 128; ++n) for (int b = 0; b < 32; ++b) { float s = 0; for (int k = 0; k < K; ++k) s += W[n * K + k] * X[b * K + k]; ref[n * 32 + b] = s; }
    Plan p; memset(&p, 0, sizeof(p));
    p.a_boxes = 1; p.b_boxes = 1; p.a_dc0 = 32; p.b_dc0 = 32; p.stages = 2; p.mma_per_stage = 4;
    p.a_kstep = 32; p.b_kstep = 32; p.a_lbo = 16; p.b_lbo = 16; p.a_sbo = 1024; p.b_sbo = 1024;
    p.N = 32; p.idesc = umma::make_idesc_tf32(128, 32, false, false);
    rc |= run("fwd   K-major A (W) x K-major B (x), SW128, tf32", W, 128, K, X, 32, K, 128, 32, p, ref);
  }
  {  // dgrad: D[k=128][b=32] = sum_n W[n][k] dy[b][n];  W [64 n][128 k] -> A MN-major (4 boxes of 32 k x 32 n per stage);
     // dy [32 b][64 n] -> B K-major; stage = 32 n = 4 MMAs
    const int N = 64;
    std::vector<float> W(N * 128), DY(32 * N), ref(128 * 32);
    for (int n = 0; n < N; ++n) for (int k = 0; k < 128; ++k) W[n * 128 + k] = val(n, k, 3);
    for (int b = 0; b < 32; ++b) for (int n = 0; n < N; ++n) DY[b * N + n] = val(b, n, 4);
    for (int k = 0; k < 128; ++k) for (int b = 0; b < 32; ++b) { float s = 0; for (int n = 0; n < N; ++n) s += W[n * 128 + k] * DY[b * N + n]; ref[k * 32 + b] = s; }
    Plan p; memset(&p, 0, sizeof(p));
    p.a_boxes = 4; for (int i = 0; i < 4; ++i) { p.a_c0[i] = 32 * i; p.a_c1[i] = 0; }
    p.a_dc1 = 32;                          // next stage: next 32 rows (n) of W
    p.b_boxes = 1; p.b_dc0 = 32;           // next 32 n of dy
    p.stages = 2; p.mma_per_stage = 4;
    p.a_kstep = 1024; p.a_lbo = 32 * 128; p.a_sbo = 1024;      // MN-major: K step = 8 rows; LBO = next 32-k block (one box)
    p.b_kstep = 32; p.b_lbo = 16; p.b_sbo = 1024;
    p.N = 32; p.idesc = umma::make_idesc_tf32(128, 32, true, false);
    run("dgrad MN-major A (W^T) SW128 x K-major B (dy), tf32 (expected wrong)", W, N, 128, DY, 32, N, 32, 32, p, ref);
    p.a_base32 = 1; p.a_sbo = 512;
    rc |= run("dgrad MN-major A BASE32B sbo=512 kstep=1024", W, N, 128, DY, 32, N, 32, 32, p, ref);
    p.a_sbo = 1024;
    run("dgrad MN-major A BASE32B sbo=1024 kstep=1024 (expected wrong)", W, N, 128, DY, 32, N, 32, 32, p, ref);
  }
  {  // wgrad: D[n=128][k=64] = sum_b dy[b][n] x[b][k];  dy [32 b][128 n] -> A MN-major (4 boxes); x [32 b][64 k] -> B MN-major
     // (2 boxes); one stage, 4 MMAs over b
    std::vector<float> DY(32 * 128), X(32 * 64), ref(128 * 64);
    for (int b = 0; b < 32; ++b) for (int n = 0; n < 128; ++n) DY[b * 128 + n] = val(b, n, 5);
    for (int b = 0; b < 32; ++b) for (int k = 0; k < 64; ++k) X[b * 64 + k] = val(b, k, 6);
    for (int n = 0; n < 128; ++n) for (int k = 0; k < 64; ++k) { float s = 0; for (int b = 0; b < 32; ++b) s += DY[b * 128 + n] * X[b * 64 + k]; ref[n * 64 + k] = s; }
    Plan p; memset(&p, 0, sizeof(p));
    p.a_boxes = 4; for (int i = 0; i < 4; ++i) { p.a_c0[i] = 32 * i; p.a_c1[i] = 0; }
    p.b_boxes = 2; for (int i = 0; i < 2; ++i) { p.b_c0[i] = 32 * i; p.b_c1[i] = 0; }
    p.stages = 1; p.mma_per_stage = 4;
    p.a_kstep = 1024; p.a_lbo = 32 * 128; p.a_sbo = 1024;
    p.b_kstep = 1024; p.b_lbo = 32 * 128; p.b_sbo = 1024;
    p.N = 64; p.idesc = umma::make_idesc_tf32(128, 64, true, true);
    p.a_base32 = p.b_base32 = 1; p.a_sbo = p.b_sbo = 512;
    rc |= run("wgrad MN-major A (dy^T) x MN-major B (x), BASE32B sbo=512", DY, 32, 128, X, 32, 64, 32, 32, p, ref);
  }
  return rc;
}
