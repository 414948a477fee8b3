// Shared device/host helpers for libregnn_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/regnn_b200.h"

namespace regnn {

constexpr float kRelationSlope = 0.01f;  // nn.LeakyReLU() default: layer/REGraphConv.py:60
constexpr int kWarpsPerBlock = 8;        // row-parallel kernels: 256 threads, one row per (sub)warp
constexpr int kMaxPartialBlocks = 4736;  // 148 SMs x 32: cap on the grid of the kernels that emit per-block partial sums

void set_error(const char* fmt, ...);
int check_launch(const char* what);

// csr_build.cu: device-wide exclusive scan (block_sums: ceil(n / 4096) + 1 entries; in == out is allowed) and the
// source-sorted view of a destination-sorted CSR (workspace: regnn_csr_build_workspace_bytes(num_nodes, num_edges)).
void exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* block_sums, cudaStream_t stream);
void build_transposed_view(const int32_t* indices, const int32_t* row, int64_t num_nodes, int64_t num_edges,
                           int32_t* indptr_t, int32_t* indices_t, int32_t* slot_t, void* workspace,
                           cudaStream_t stream);

#define REGNN_REQUIRE(cond, code, ...)        \
  do {                                        \
    if (!(cond)) {                            \
      ::regnn::set_error(__VA_ARGS__);        \
      return (code);                          \
    }                                         \
  } while (0)

// 32-bit integer finaliser of the counter-based generators (neighbour sampling, attention dropout)
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t z) {
  z ^= z >> 16; z *= 0x7feb352du;
  z ^= z >> 15; z *= 0x846ca68bu;
  z ^= z >> 16;
  return z;
}

__device__ __forceinline__ float leaky(float x, float slope) { return x > 0.f ? x : x * slope; }
// PyTorch's leaky_relu_backward convention: the negative slope applies at x == 0.
__device__ __forceinline__ float leaky_grad(float x, float slope) { return x > 0.f ? 1.f : slope; }

__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
// Streaming 128-bit load that does not allocate in L1 (gathered rows are not reused by this SM).
__device__ __forceinline__ float4 ldg4_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// Request a line into L2 without holding a register for it: the value is loaded later, at L2 latency.
// exp(x) as one FMUL + MUFU.EX2 (ex2.approx.ftz: 2^-22 relative error like __expf, results below 2^-126 flush to 0;
// __expf without -ftz spends three more instructions per call on the subnormal range).  exp(-inf) = 0.
__device__ __forceinline__ float fast_exp(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ float dot4(float4 a, float4 b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}
__device__ __forceinline__ void fma4(float4& acc, float s, float4 v) {
  acc.x = fmaf(s, v.x, acc.x);
  acc.y = fmaf(s, v.y, acc.y);
  acc.z = fmaf(s, v.z, acc.z);
  acc.w = fmaf(s, v.w, acc.w);
}
__device__ __forceinline__ void scale4(float4& a, float s) {
  a.x *= s; a.y *= s; a.z *= s; a.w *= s;
}

// Butterfly sum over aligned groups of WIDTH lanes (WIDTH a power of two <= 32); every lane of the
// group ends with the total.  Fixed order => deterministic.
template <int WIDTH>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = WIDTH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float group_sum_rt(float v, int width) {
  for (int o = width >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_max_int(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Opts a kernel in to more than 48 KB of dynamic shared memory when needed.
template <typename K>
inline int set_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      set_error("dynamic shared memory request of %zu bytes rejected: %s", bytes, cudaGetErrorString(e));
      return REGNN_ERR_UNSUPPORTED_SHAPE;
    }
  }
  return REGNN_OK;
}

// Grid of a persistent kernel: exactly one resident wave (SMs x blocks per SM), never more than the partial slots.
template <typename K>
inline int resident_blocks(K kernel, size_t smem) {
  int dev = 0, sms = 148, per_sm = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kWarpsPerBlock * 32, smem) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  const int want = sms * per_sm;
  return want < kMaxPartialBlocks ? want : kMaxPartialBlocks;
}

inline int partial_blocks(int64_t rows) {
  int64_t b = (rows + kWarpsPerBlock - 1) / kWarpsPerBlock;
  if (b < 1) b = 1;
  return (int)(b < kMaxPartialBlocks ? b : kMaxPartialBlocks);
}

// Final fixed-order reduction of per-block double partials into a relation-gradient table:
//   d_theta[i] = alpha * LeakyReLU'(alpha*theta[i]) * sum_b partials[b*stride + i],  i < count
void launch_relation_grad_finalize(const double* partials, int num_blocks, int stride, int count,
                                   const float* theta, float alpha, float* d_theta,
                                   cudaStream_t stream);
// out[i] = sum_b partials[b*stride + offset + i]
void launch_colsum_finalize(const double* partials, int num_blocks, int stride, int offset,
                            int count, float* out, cudaStream_t stream);

}  // namespace regnn
