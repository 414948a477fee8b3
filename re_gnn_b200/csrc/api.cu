// Library-wide plumbing: version, status strings, thread-local error text, and the small fixed-order
// finalize kernels shared by every backward pass.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace regnn {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return REGNN_ERR_CUDA;
  }
  return REGNN_OK;
}

// One warp per table entry: lane l sums blocks l, l+32, ... in order, then a fixed xor-tree combines the
// 32 lane sums => the summation order is a pure function of num_blocks (deterministic).
__global__ void relation_grad_finalize_kernel(const double* __restrict__ partials, int num_blocks,
                                              int stride, int count, const float* __restrict__ theta,
                                              float alpha, float* __restrict__ d_theta) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= count) return;
  double s = 0.0;
  for (int b = lane; b < num_blocks; b += 32) s += partials[(size_t)b * stride + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) {
    const float z = theta[i] * alpha;
    d_theta[i] = (float)(s * (double)(alpha * leaky_grad(z, kRelationSlope)));
  }
}

__global__ void colsum_finalize_kernel(const double* __restrict__ partials, int num_blocks,
                                       int stride, int offset, int count, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= count) return;
  double s = 0.0;
  for (int b = lane; b < num_blocks; b += 32) s += partials[(size_t)b * stride + offset + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[i] = (float)s;
}

void launch_relation_grad_finalize(const double* partials, int num_blocks, int stride, int count,
                                   const float* theta, float alpha, float* d_theta,
                                   cudaStream_t stream) {
  const int warps = 4;
  relation_grad_finalize_kernel<<<(count + warps - 1) / warps, warps * 32, 0, stream>>>(
      partials, num_blocks, stride, count, theta, alpha, d_theta);
}

void launch_colsum_finalize(const double* partials, int num_blocks, int stride, int offset,
                            int count, float* out, cudaStream_t stream) {
  const int warps = 4;
  colsum_finalize_kernel<<<(count + warps - 1) / warps, warps * 32, 0, stream>>>(
      partials, num_blocks, stride, offset, count, out);
}

}  // namespace regnn

extern "C" {

int regnn_version(void) { return 201; }  // 2xx: round-2 ABI (regnn_spmm_bwd_fused takes Y / d_norm); 201: the attention
                                         // entry points take a regnn_attn_dropout_t next to keep

const char* regnn_status_string(int status) {
  switch (status) {
    case REGNN_OK: return "ok";
    case REGNN_ERR_INVALID_ARG: return "invalid argument";
    case REGNN_ERR_UNSUPPORTED_SHAPE: return "unsupported shape";
    case REGNN_ERR_CUDA: return "CUDA error";
    case REGNN_ERR_WORKSPACE_TOO_SMALL: return "workspace too small";
    default: return "unknown status";
  }
}

const char* regnn_last_error_string(void) { return regnn::g_err; }

int regnn_max_partial_blocks(void) { return regnn::kMaxPartialBlocks; }

}  // extern "C"
