// Host-side TMA descriptor (CUtensorMap) construction without linking libcuda: the driver entry point
// cuTensorMapEncodeTiled is fetched through the runtime (cudaGetDriverEntryPoint).  Every tensor map of the library is
// encoded here.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace dd {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn tma_encoder() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

inline bool tma_available() { return tma_encoder() != nullptr; }

// Tiled map of 2 to 4 dimensions (dims / box innermost first, strides in bytes), out-of-range elements = 0.
// Returns 0 on success, else the driver's error (-1: no encoder) and, if msg is given, a description of the map in msg.
inline int tma_encode(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims,
                      const cuuint64_t* strides, const cuuint32_t* box, const cuuint32_t* estr, CUtensorMapSwizzle swizzle,
                      char* msg, size_t msg_len) {
  int r = -1;
  if (EncodeTiledFn enc = tma_encoder()) {
    // cuTensorMapEncodeTiled is a DRIVER call: it needs a current context on the calling thread.  PyTorch's
    // autograd worker threads may not have one yet (the runtime binds it lazily; seen as error 201 =
    // CUDA_ERROR_INVALID_CONTEXT from backward passes) -- a runtime no-op binds the primary context.
    static thread_local bool ctx_bound = false;
    if (!ctx_bound) { cudaFree(nullptr); ctx_bound = true; }
    const CUresult e = enc(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    r = e == CUDA_SUCCESS ? 0 : (int)e;
  }
  if (r != 0 && msg) {
    unsigned long long d[4] = {1, 1, 1, 1};
    unsigned b[4] = {1, 1, 1, 1};
    for (int i = 0; i < rank && i < 4; ++i) { d[i] = dims[i]; b[i] = box[i]; }
    snprintf(msg, msg_len, "cuTensorMapEncodeTiled -> %d (base %p, dims %llux%llux%llux%llu, pitch %llu B, box %ux%ux%ux%u, swizzle %d)",
             r, base, d[0], d[1], d[2], d[3], (unsigned long long)strides[0], b[0], b[1], b[2], b[3], (int)swizzle);
  }
  return r;
}

// Row-major 2-D matrix [rows][cols] of 4-byte (fp32) or 2-byte (bf16) elements, row pitch in elements; box = box_cols x
// box_rows with box_cols * elem_bytes = the swizzle span: 128 B for CU_TENSOR_MAP_SWIZZLE_128B and _128B_ATOM_32B (the
// 32-byte-atom variant that MN-major tf32 operands need), 64 B for CU_TENSOR_MAP_SWIZZLE_64B.
inline int tma_map_2d(CUtensorMap* map, const void* base, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                      uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swizzle, char* msg, size_t msg_len) {
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {pitch_elems * (uint64_t)elem_bytes};
  const cuuint32_t box[2] = {box_cols, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return tma_encode(map, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims,
                    strides, box, estr, swizzle, msg, msg_len);
}

// NHWC bf16 activation [B][H][W][C] as a 4-D tensor (c, w, h, b) with a box of 32 channels x box_w SOURCE pixels of one
// row, taking every estride-th pixel (box_w <= 256; estride 2 -> ceil(box_w / 2) pixels land), 64-byte swizzle (inner
// extent = 64 bytes: a whole pixel when C = 32).  The tile that lands is at once the K-major SWIZZLE_64B operand of a
// forward conv (rows = pixels, K = channels) and the MN-major one of a weight gradient (K = pixels); a tap is a shift of
// the operand's start address by whole pixels (tools/tma_layout_probe.cu, tools/tma_sw64_mn_probe.cu).  Full 32-byte
// sectors from L2 and one request per row, against half sectors and four requests with 8-channel boxes.
inline int tma_map_nhwc_sw64(CUtensorMap* map, const void* base, uint64_t B, uint64_t H, uint64_t W, uint64_t C, uint32_t box_w,
                             uint32_t estride, char* msg, size_t msg_len) {
  const cuuint64_t dims[4] = {C, W, H, B};
  const cuuint64_t strides[3] = {C * 2, W * C * 2, H * W * C * 2};
  const cuuint32_t box[4] = {32, box_w, 1, 1};
  const cuuint32_t estr[4] = {1, estride, 1, 1};
  return tma_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_64B, msg,
                    msg_len);
}

}  // namespace dd
