// Hardware probe for the fused backward + Adam kernel of linear_tc.cu: a TMA box loaded with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B
// (the MN-major tf32 operand layout) is updated in shared memory and written back by a TMA STORE through the same tensor map.
//   1. load layout: element (r, c) of a 32 x 32 fp32 box sits at float r * 32 + 8 * ((c / 8) ^ (r % 4)) + c % 8
//   2. store: the modified box lands in global memory at the box coordinates; with a ragged edge the out-of-range part is
//      clipped (the sentinels around it stay)
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o tools/tma_store_atom32_probe tools/tma_store_atom32_probe.cu -lcuda
#include <stdio.h>
#include <vector>

#include "../driving-dirty_b200/csrc/tma_host.h"
#include "../driving-dirty_b200/csrc/umma.cuh"

constexpr int R = 60, C = 60;       // global matrices [R][C] fp32; box at (32, 32) is ragged (28 x 28 in range)

__global__ void probe(const __grid_constant__ CUtensorMap tin, const __grid_constant__ CUtensorMap tout, const float* in,
                      int c0, int r0, int* layout_bad, float* dump) {
  __shared__ __align__(1024) float box[32 * 32];
  __shared__ uint64_t full;
  if (threadIdx.x == 0) { umma::mbar_init(&full, 1); umma::fence_mbar_init(); }
  __syncthreads();
  if (threadIdx.x == 0) {
    umma::mbar_expect_tx(&full, sizeof box);
    umma::tma_load_2d(umma::smem_u32(box), &tin, c0, r0, &full);
  }
  umma::mbar_wait(&full, 0);
  for (int i = threadIdx.x; i < 32 * 32; i += blockDim.x) {
    dump[i] = box[i];
    const int r = i / 32, c = i % 32;
    const float want = (r0 + r < R && c0 + c < C) ? in[(r0 + r) * C + c0 + c] : 0.f;
    if (box[r * 32 + 8 * ((c / 8) ^ (r % 4)) + c % 8] != want) atomicAdd(layout_bad, 1);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 32 * 32; i += blockDim.x) {
    const int r = i / 32, c = i % 32;
    box[r * 32 + 8 * ((c / 8) ^ (r % 4)) + c % 8] += 0.5f;
  }
  umma::fence_proxy_async_smem();
  __syncthreads();
  if (threadIdx.x == 0) {
    umma::tma_store_2d(&tout, umma::smem_u32(box), c0, r0);
    umma::bulk_commit_group();
    umma::bulk_wait_group<0>();
  }
}

int main() {
  std::vector<float> h_in(R * C), h_out(R * C), dump(32 * 32);
  for (int r = 0; r < R; ++r)
    for (int c = 0; c < C; ++c) h_in[r * C + c] = (float)(r * 1000 + c);
  float *in, *out, *d_dump;
  int* bad;
  cudaMalloc(&in, R * C * 4); cudaMalloc(&out, R * C * 4); cudaMalloc(&d_dump, 32 * 32 * 4); cudaMalloc(&bad, 4);
  cudaMemcpy(in, h_in.data(), R * C * 4, cudaMemcpyHostToDevice);
  int all_ok = 1;
  const int starts[2][2] = {{0, 0}, {32, 32}};
  for (const auto& st : starts) {
    const int c0 = st[0], r0 = st[1];
    std::vector<float> sentinel(R * C, -7.f);
    cudaMemcpy(out, sentinel.data(), R * C * 4, cudaMemcpyHostToDevice);
    cudaMemset(bad, 0, 4);
    CUtensorMap tin, tout;
    char msg[256];
    if (dd::tma_map_2d(&tin, in, 4, R, C, C, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg) ||
        dd::tma_map_2d(&tout, out, 4, R, C, C, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, msg, sizeof msg)) {
      printf("encode failed: %s\n", msg);
      return 1;
    }
    probe<<<1, 256>>>(tin, tout, in, c0, r0, bad, d_dump);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("launch failed: %s\n", cudaGetErrorString(e)); return 1; }
    int h_bad = 0;
    cudaMemcpy(&h_bad, bad, 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(h_out.data(), out, R * C * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(dump.data(), d_dump, 32 * 32 * 4, cudaMemcpyDeviceToHost);
    int store_bad = 0, stored = 0;
    for (int r = 0; r < R; ++r)
      for (int c = 0; c < C; ++c) {
        const bool in_box = r >= r0 && r < r0 + 32 && c >= c0 && c < c0 + 32;
        const float want = in_box ? h_in[r * C + c] + 0.5f : -7.f;
        stored += in_box;
        if (h_out[r * C + c] != want) ++store_bad;
      }
    printf("box at (col %d, row %d) of a %d x %d fp32 matrix, SWIZZLE_128B_ATOM_32B:\n", c0, r0, R, C);
    printf("  1. load layout r*32 + 8*((c/8) ^ (r%%4)) + c%%8: %s (%d of 1024 elements differ)\n", h_bad ? "FAIL" : "PASS", h_bad);
    printf("  2. TMA store through the same map: %s (%d of %d elements differ; %d in range, %d sentinels)\n",
           store_bad ? "FAIL" : "PASS", store_bad, R * C, stored, R * C - stored);
    if (h_bad) {
      printf("  landed rows 0..7 (value = row * 1000 + col of the source):\n");
      for (int r = 0; r < 8; ++r) {
        printf("   ");
        for (int q = 0; q < 32; q += 8) printf(" %7.0f", dump[r * 32 + q]);
        printf("\n");
      }
    }
    all_ok &= !h_bad && !store_bad;
  }
  printf("%s\n", all_ok ? "ALL PASS" : "SOME FAILED");
  return all_ok ? 0 : 1;
}
