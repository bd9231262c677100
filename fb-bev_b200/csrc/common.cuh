// common.cuh -- shared helpers for the sm_100a kernels behind libfbbev_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fbbev_b200.h"

#define FBBEV_API extern "C" __attribute__((visibility("default")))

namespace fbbev {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

static inline cudaStream_t as_stream(fbbev_stream_t s) {
  return reinterpret_cast<cudaStream_t>(s);
}

// Returns the pending launch error (positive cudaError_t) or 0.
static inline int launch_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? FBBEV_OK : static_cast<int>(e);
}

// Diagnostics only: cumulative number of kernel launches issued by this library
// (bench.py reports it as `gpu_launches`).  Defined in capi.cu.
void count_launch(int n = 1);

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// SM count of the current device, queried once (148, a B200's, if the query
// fails).
static inline int sm_count() {
  static int n_sm = 0;
  if (n_sm == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (n_sm <= 0) n_sm = 148;
  }
  return n_sm;
}

// Streaming (evict-first) 128-bit / 32-bit stores for write-once outputs.
__device__ __forceinline__ void st_stream(float4* p, const float4& v) {
  __stcs(p, v);
}
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }

// y = M x for a row-major 3x3 M, in the rounding order torch's broadcast
// (..,3,3) @ (..,3,1) matmul has on B200 (torch 2.11 / cuBLAS 12.8; identified
// by tools/micro/matmul_order2.py over all 18 FMA / non-FMA association orders,
// 100 % of 5.4 M points at five problem sizes):
//   y_i = fma(m_i1, x_1, m_i0 * x_0) + m_i2 * x_2            (batched 'n' kernel)
// and, when `seq` is set, the sequential FMA chain
//   y_i = fma(m_i2, x_2, fma(m_i1, x_1, m_i0 * x_0))
// which cuBLAS uses for a single column-major matrix broadcast over the batch
// (torch.inverse returns column-major; with one matrix in total the expand is a
// stride-0 view and the transposed layout reaches cuBLAS as op 't').
__device__ __forceinline__ float dot3_ref(float m0, float m1, float m2, float x,
                                          float y, float z, bool seq) {
  const float s = __fmaf_rn(m1, y, __fmul_rn(m0, x));
  return seq ? __fmaf_rn(m2, z, s) : __fadd_rn(s, __fmul_rn(m2, z));
}
__device__ __forceinline__ void mat3_apply_ref(const float* __restrict__ m,
                                               float x, float y, float z,
                                               bool seq, float& ox, float& oy,
                                               float& oz) {
  ox = dot3_ref(__ldg(m + 0), __ldg(m + 1), __ldg(m + 2), x, y, z, seq);
  oy = dot3_ref(__ldg(m + 3), __ldg(m + 4), __ldg(m + 5), x, y, z, seq);
  oz = dot3_ref(__ldg(m + 6), __ldg(m + 7), __ldg(m + 8), x, y, z, seq);
}

}  // namespace fbbev
