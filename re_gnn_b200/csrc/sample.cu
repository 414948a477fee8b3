// Neighbour sampling on the device for the sampled-minibatch path (BASELINE config 5).
// Replaces the CPU `torch_sparse.sample_adj` behind PyG's NeighborSampler (mag/regnn_ns.py:206-214).
//
// Specification (shared bit-for-bit with oracle/sampler_oracle.py): for target t with in-degree deg and
// fan-out f, k = min(deg, f) in-edges are taken WITHOUT replacement: all of them if deg <= f, otherwise the
// slots indptr[t] + P(j), j = 0..f-1, where P is a pseudo-random permutation of [0, deg): a 4-round balanced
// Feistel network on b bits (2^b >= deg, b even) with cycle walking, keyed by mix(key, t).  Counter-based:
// no RNG state, any (seed, epoch, rank, batch) reproduces its sample on any device.  Integer work only.
#include "common.cuh"

namespace regnn {

__host__ __device__ __forceinline__ uint32_t feistel_perm(uint32_t x, uint32_t deg, uint32_t key) {
  int b = 2;
  while ((1u << b) < deg) b += 2;          // even number of bits, 2^b >= deg
  const int h = b >> 1;
  const uint32_t mask = (1u << h) - 1u;
  uint32_t y = x;
  do {                                      // cycle walking: stay inside [0, deg)
    uint32_t L = y >> h, R = y & mask;
#pragma unroll
    for (uint32_t r = 0; r < 4; ++r) {
      const uint32_t f = mix32(R * 0x9E3779B1u + key + r * 0x85EBCA6Bu) & mask;
      const uint32_t nl = R;
      R = L ^ f;
      L = nl;
    }
    y = (L << h) | R;
  } while (y >= deg);
  return y;
}

__global__ void sample_neighbors_kernel(const int32_t* __restrict__ indptr, const int64_t* __restrict__ targets,
                                        int64_t num_targets, int fanout, uint32_t key_lo, uint32_t key_hi,
                                        int32_t* __restrict__ out_slot) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= num_targets * fanout) return;
  const int64_t i = tid / fanout;
  const uint32_t j = (uint32_t)(tid % fanout);
  const int64_t t = targets[i];
  const int32_t s0 = indptr[t];
  const uint32_t deg = (uint32_t)(indptr[t + 1] - s0);
  int32_t slot = -1;
  if (j < deg) {
    if (deg <= (uint32_t)fanout) slot = s0 + (int32_t)j;
    else slot = s0 + (int32_t)feistel_perm(j, deg, mix32(key_lo ^ mix32((uint32_t)t + key_hi)));
  }
  out_slot[tid] = slot;
}

}  // namespace regnn

using namespace regnn;

extern "C" int regnn_sample_neighbors(const int32_t* indptr, const int64_t* targets, int64_t num_targets,
                                      int fanout, uint64_t key, int32_t* out_slot, void* stream) {
  REGNN_REQUIRE(indptr && out_slot && (num_targets == 0 || targets), REGNN_ERR_INVALID_ARG, "sample_neighbors: null pointer");
  REGNN_REQUIRE(fanout >= 1 && num_targets >= 0, REGNN_ERR_INVALID_ARG, "sample_neighbors: fanout must be >= 1");
  const int64_t total = num_targets * fanout;
  if (total == 0) return REGNN_OK;
  sample_neighbors_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      indptr, targets, num_targets, fanout, (uint32_t)(key & 0xffffffffu), (uint32_t)(key >> 32), out_slot);
  return check_launch("regnn_sample_neighbors");
}

// ---- GraphSAINT random-walk roots (mag/regnn_saint.py:185-190: GraphSAINTRandomWalkSampler) ---------------
// One thread per root: `walk_length` steps along OUT-edges (transposed view), the next hop chosen by a
// counter-based hash -- no RNG state, bit-exact with oracle/sampler_oracle.py::random_walks.  A node without
// out-edges keeps the walker in place (torch_sparse's behaviour for dangling nodes).
namespace regnn {
__global__ void random_walk_kernel(const int32_t* __restrict__ indptr_t, const int32_t* __restrict__ indices_t,
                                   int64_t num_nodes, int64_t num_roots, int walk_length, uint32_t key_lo,
                                   uint32_t key_hi, int64_t* __restrict__ walks) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num_roots) return;
  int64_t cur = (int64_t)(mix32(key_lo ^ mix32((uint32_t)i * 0x9E3779B1u + key_hi)) % (uint32_t)num_nodes);
  walks[i * (walk_length + 1)] = cur;
  for (int step = 1; step <= walk_length; ++step) {
    const int32_t t0 = indptr_t[cur];
    const uint32_t deg = (uint32_t)(indptr_t[cur + 1] - t0);
    if (deg > 0) {
      const uint32_t r = mix32(key_hi ^ mix32((uint32_t)i * 0x85EBCA6Bu + (uint32_t)step * 0xC2B2AE35u + key_lo));
      cur = indices_t[t0 + (int32_t)(r % deg)];
    }
    walks[i * (walk_length + 1) + step] = cur;
  }
}
}  // namespace regnn

extern "C" int regnn_random_walk(const int32_t* indptr_t, const int32_t* indices_t, int64_t num_nodes,
                                 int64_t num_roots, int walk_length, uint64_t key, int64_t* walks, void* stream) {
  REGNN_REQUIRE(indptr_t && walks && num_nodes > 0 && num_nodes < 0xffffffffLL, REGNN_ERR_INVALID_ARG, "random_walk: bad arguments");
  REGNN_REQUIRE(walk_length >= 0 && num_roots >= 0, REGNN_ERR_INVALID_ARG, "random_walk: negative size");
  if (num_roots == 0) return REGNN_OK;
  regnn::random_walk_kernel<<<(unsigned)((num_roots + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      indptr_t, indices_t, num_nodes, num_roots, walk_length, (uint32_t)(key & 0xffffffffu), (uint32_t)(key >> 32), walks);
  return regnn::check_launch("regnn_random_walk");
}
