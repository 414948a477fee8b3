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

// The j-th sampled in-edge slot of node t, or -1 when j >= min(in-degree, fanout).
__device__ __forceinline__ int32_t sampled_slot(const int32_t* __restrict__ indptr, int64_t t, uint32_t j, int fanout,
                                                uint32_t key_lo, uint32_t key_hi) {
  const int32_t s0 = indptr[t];
  const uint32_t deg = (uint32_t)(indptr[t + 1] - s0);
  if (j >= deg) return -1;
  if (deg <= (uint32_t)fanout) return s0 + (int32_t)j;
  return s0 + (int32_t)feistel_perm(j, deg, mix32(key_lo ^ mix32((uint32_t)t + key_hi)));
}

__global__ void sample_neighbors_kernel(const int32_t* __restrict__ indptr, const int64_t* __restrict__ targets,
                                        int64_t num_targets, int fanout, uint32_t key_lo, uint32_t key_hi,
                                        int32_t* __restrict__ out_slot) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= num_targets * fanout) return;
  const int64_t i = tid / fanout;
  out_slot[tid] = sampled_slot(indptr, targets[i], (uint32_t)(tid % fanout), fanout, key_lo, key_hi);
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

// ---- Device-built minibatch blocks -------------------------------------------------------------------------
// One sampled layer without a host round trip (regnn_sample_layer), and the CSR views of one block straight from
// it (regnn_block_csr_build).  Target i's valid slots are the first k_i = min(in-degree, fanout) of its fan-out row,
// so the sampled edges, compacted in sample order, are the block's in-CSR already: row_off = exclusive scan of k_i.
// Relabelling: targets store their position in a persistent [N] map, sampled sources that are not targets raise a
// flag, and an exclusive scan of the flags in global-id order gives every new source its position -- new sources
// in ascending global id, as torch.unique orders them.  Stores of equal values, integer counters and atomicMin
// only: the result does not depend on the order in which threads run.
namespace regnn {

constexpr int32_t kUnmapped = 0x7fffffff;   // pos_map entry of a node that is not a target of the current layer

__device__ __forceinline__ int64_t targets_of(const int32_t* num_targets, int64_t max_targets) {
  return num_targets ? (int64_t)*num_targets : max_targets;
}

// Long-row statistics of the row split of a CSR view (graph.py: _row_split): rows with more than `threshold`
// slots and the number of `threshold`-slot fragments they are cut into.
__device__ __forceinline__ void count_long_row(int64_t deg, int threshold, int32_t* stats) {
  if (deg > threshold) {
    atomicAdd(stats, 1);
    atomicAdd(stats + 1, (int32_t)((deg + threshold - 1) / threshold));
  }
}

__global__ void frontier_rows_kernel(const int32_t* __restrict__ indptr, const int64_t* __restrict__ targets,
                                     int64_t max_targets, const int32_t* __restrict__ num_targets, int fanout,
                                     int threshold, int32_t* __restrict__ pos_map, int64_t* __restrict__ new_n_id,
                                     uint32_t* __restrict__ row_off, int32_t* __restrict__ info) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > max_targets) return;
  const int64_t t = targets_of(num_targets, max_targets);
  uint32_t k = 0;
  if (i < t) {
    const int64_t v = targets[i];
    atomicMin(&pos_map[v], (int32_t)i);     // a repeated target keeps its first position
    new_n_id[i] = v;
    k = (uint32_t)min(indptr[v + 1] - indptr[v], fanout);
    if (k == 0) atomicAdd(&info[REGNN_SAMPLE_INFO_EMPTY_ROWS], 1);
    count_long_row(k, threshold, info + REGNN_SAMPLE_INFO_IN_SPLIT);
    count_long_row(k + 1, threshold, info + REGNN_SAMPLE_INFO_IN_SPLIT_LOOPS);
  }
  row_off[i] = k;     // scanned in place afterwards; entry max_targets becomes the number of sampled edges
}

__global__ void frontier_slots_kernel(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                      const int32_t* __restrict__ eid, const int64_t* __restrict__ targets,
                                      int64_t max_targets, const int32_t* __restrict__ num_targets, int fanout,
                                      uint32_t key_lo, uint32_t key_hi, const uint32_t* __restrict__ row_off,
                                      const int32_t* __restrict__ pos_map, uint32_t* __restrict__ flags,
                                      int32_t* __restrict__ src_global, int64_t* __restrict__ dst_local,
                                      int64_t* __restrict__ edge_id) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i = tid / fanout;
  if (i >= targets_of(num_targets, max_targets)) return;
  const uint32_t j = (uint32_t)(tid % fanout), e0 = row_off[i];
  if (j >= row_off[i + 1] - e0) return;
  const int32_t slot = sampled_slot(indptr, targets[i], j, fanout, key_lo, key_hi);
  const int64_t e = (int64_t)e0 + j;
  const int32_t u = indices[slot];
  src_global[e] = u;
  dst_local[e] = i;
  edge_id[e] = eid[slot];
  if (pos_map[u] == kUnmapped) flags[u] = 1u;
}

__global__ void frontier_relabel_kernel(int64_t max_targets, const int32_t* __restrict__ num_targets,
                                        const uint32_t* __restrict__ row_off, int64_t num_nodes,
                                        const int32_t* __restrict__ src_global, const int32_t* __restrict__ pos_map,
                                        const uint32_t* __restrict__ flags, const uint32_t* __restrict__ excl,
                                        int64_t* __restrict__ new_n_id, int64_t* __restrict__ src_local,
                                        int32_t* __restrict__ src_hist, int32_t* __restrict__ info) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t t = targets_of(num_targets, max_targets);
  const int64_t num_edges = row_off[max_targets];
  if (e == 0) {
    info[REGNN_SAMPLE_INFO_SOURCES] = (int32_t)(t + excl[num_nodes - 1] + flags[num_nodes - 1]);
    info[REGNN_SAMPLE_INFO_EDGES] = (int32_t)num_edges;
  }
  if (e >= num_edges) return;
  const int32_t u = src_global[e];
  int64_t p = pos_map[u];
  if (p == kUnmapped) {
    p = t + excl[u];
    new_n_id[p] = u;
  }
  src_local[e] = p;
  atomicAdd(&src_hist[p], 1);
}

// Restores pos_map / flags for the next layer and counts the long rows of the block's transposed view.
__global__ void frontier_finish_kernel(int64_t max_sources, int64_t max_targets, const int32_t* __restrict__ num_targets,
                                       const int64_t* __restrict__ new_n_id, const int32_t* __restrict__ src_hist,
                                       int threshold, int32_t* __restrict__ pos_map, uint32_t* __restrict__ flags,
                                       int32_t* __restrict__ info) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= max_sources || v >= info[REGNN_SAMPLE_INFO_SOURCES]) return;
  const int64_t t = targets_of(num_targets, max_targets);
  const int64_t u = new_n_id[v];
  if (v < t) pos_map[u] = kUnmapped;
  else flags[u] = 0u;
  const int32_t d = src_hist[v];
  count_long_row(d, threshold, info + REGNN_SAMPLE_INFO_OUT_SPLIT);
  count_long_row(d + (v < t ? 1 : 0), threshold, info + REGNN_SAMPLE_INFO_OUT_SPLIT_LOOPS);
}

__global__ void block_csr_fill_kernel(const int64_t* __restrict__ src_local, const int64_t* __restrict__ dst_local,
                                      const int64_t* __restrict__ edge_id, const uint32_t* __restrict__ row_off,
                                      const int64_t* __restrict__ targets, int64_t num_src, int64_t num_dst,
                                      int64_t num_sampled, const int64_t* __restrict__ edge_type,
                                      const int64_t* __restrict__ node_type, int num_edge_types, int loops,
                                      int64_t* __restrict__ src, int64_t* __restrict__ dst, int64_t* __restrict__ etype1,
                                      int32_t* __restrict__ indptr, int32_t* __restrict__ indices,
                                      int32_t* __restrict__ eid, int32_t* __restrict__ row,
                                      uint8_t* __restrict__ et_csr, int num_relations, int32_t* __restrict__ status) {
  const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (x <= num_src) indptr[x] = (int32_t)(x <= num_dst ? row_off[x] + loops * x : num_sampled + loops * num_dst);
  if (x >= num_sampled + loops * num_dst) return;
  int64_t u, v, s, ty;
  if (x < num_sampled) {           // sampled edge x of row v: slot x + v when every earlier row ends in its loop
    u = src_local[x];
    v = dst_local[x];
    s = x + loops * v;
    ty = edge_type[edge_id[x]];
  } else {                         // typed self loop of target v (edge id num_sampled + v): the last slot of row v
    v = x - num_sampled;
    u = v;
    s = (int64_t)row_off[v + 1] + v;
    ty = node_type[targets[v]] + num_edge_types;
  }
  src[x] = u;
  dst[x] = v;
  etype1[x] = ty + 1;
  if (ty < 0 || ty >= num_relations) {   // reported through *status; slot typed 0 so no table is indexed out of range
    *status = 1;
    ty = 0;
  }
  indices[s] = (int32_t)u;
  eid[s] = (int32_t)x;
  row[s] = (int32_t)v;
  et_csr[s] = (uint8_t)ty;
}

__global__ void etype_transpose_kernel(const uint8_t* __restrict__ et_csr, const int32_t* __restrict__ slot_t,
                                       int64_t n, uint8_t* __restrict__ et_t) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) et_t[j] = et_csr[slot_t[j]];
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
static int64_t scan_blocks(int64_t n) { return (n + 4095) / 4096 + 1; }
static unsigned grid_of(int64_t n) { return (unsigned)((n > 0 ? n + 255 : 256) / 256); }

}  // namespace regnn

extern "C" size_t regnn_sample_layer_workspace_bytes(int64_t num_nodes, int64_t max_targets, int fanout) {
  const int64_t slots = max_targets * fanout, nb = scan_blocks(num_nodes > max_targets ? num_nodes : max_targets + 1);
  return align256((size_t)(slots > 0 ? slots : 1) * 4) + align256((size_t)(num_nodes > 0 ? num_nodes : 1) * 4) +
         align256((size_t)nb * 4);
}

extern "C" int regnn_sample_layer(const int32_t* indptr, const int32_t* indices, const int32_t* eid, int64_t num_nodes,
                                  const int64_t* targets, int64_t max_targets, const int32_t* num_targets, int fanout,
                                  uint64_t key, int split_threshold, int32_t* pos_map, uint32_t* flags,
                                  int64_t* new_n_id, int64_t max_sources, int64_t* src_local, int64_t* dst_local,
                                  int64_t* edge_id, uint32_t* row_off, int32_t* src_hist, int32_t* info,
                                  void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr && indices && eid && pos_map && flags && new_n_id && src_local && dst_local && edge_id &&
                row_off && src_hist && info && workspace && (max_targets == 0 || targets),
                REGNN_ERR_INVALID_ARG, "sample_layer: null pointer");
  REGNN_REQUIRE(num_nodes >= 1 && num_nodes < ((int64_t)1 << 31) - 1 && max_targets >= 0 && fanout >= 1 &&
                split_threshold >= 1, REGNN_ERR_INVALID_ARG, "sample_layer: bad sizes");
  const int64_t slots = max_targets * fanout;
  REGNN_REQUIRE(slots < ((int64_t)1 << 31) - 1, REGNN_ERR_UNSUPPORTED_SHAPE, "sample_layer: %lld slots exceed int32",
                (long long)slots);
  REGNN_REQUIRE(max_sources >= max_targets + (slots < num_nodes ? slots : num_nodes), REGNN_ERR_INVALID_ARG,
                "sample_layer: max_sources=%lld below max_targets + min(num_nodes, max_targets * fanout)",
                (long long)max_sources);
  REGNN_REQUIRE(workspace_bytes >= regnn_sample_layer_workspace_bytes(num_nodes, max_targets, fanout),
                REGNN_ERR_WORKSPACE_TOO_SMALL, "sample_layer workspace too small");
  char* p = (char*)workspace;
  int32_t* src_global = (int32_t*)p;
  p += align256((size_t)(slots > 0 ? slots : 1) * 4);
  uint32_t* excl = (uint32_t*)p;
  p += align256((size_t)num_nodes * 4);
  uint32_t* block_sums = (uint32_t*)p;
  const uint32_t key_lo = (uint32_t)(key & 0xffffffffu), key_hi = (uint32_t)(key >> 32);

  cudaMemsetAsync(info, 0, REGNN_SAMPLE_INFO_WORDS * sizeof(int32_t), stream);
  cudaMemsetAsync(src_hist, 0, (size_t)(max_sources > 0 ? max_sources : 1) * sizeof(int32_t), stream);
  frontier_rows_kernel<<<grid_of(max_targets + 1), 256, 0, stream>>>(indptr, targets, max_targets, num_targets, fanout,
                                                                     split_threshold, pos_map, new_n_id, row_off, info);
  exclusive_scan_u32(row_off, row_off, max_targets + 1, block_sums, stream);
  frontier_slots_kernel<<<grid_of(slots), 256, 0, stream>>>(indptr, indices, eid, targets, max_targets, num_targets,
                                                            fanout, key_lo, key_hi, row_off, pos_map, flags, src_global,
                                                            dst_local, edge_id);
  exclusive_scan_u32(flags, excl, num_nodes, block_sums, stream);
  frontier_relabel_kernel<<<grid_of(slots), 256, 0, stream>>>(max_targets, num_targets, row_off, num_nodes, src_global,
                                                              pos_map, flags, excl, new_n_id, src_local, src_hist, info);
  frontier_finish_kernel<<<grid_of(max_sources), 256, 0, stream>>>(max_sources, max_targets, num_targets, new_n_id,
                                                                   src_hist, split_threshold, pos_map, flags, info);
  return check_launch("regnn_sample_layer");
}

extern "C" int regnn_block_csr_build(const int64_t* src_local, const int64_t* dst_local, const int64_t* edge_id,
                                     const uint32_t* row_off, const int64_t* targets, int64_t num_src, int64_t num_dst,
                                     int64_t num_sampled, const int64_t* edge_type, const int64_t* node_type,
                                     int num_edge_types, int self_loops, int num_relations, int64_t* src, int64_t* dst,
                                     int64_t* etype1, int32_t* indptr, int32_t* indices, int32_t* eid, int32_t* row,
                                     int32_t* indptr_t, int32_t* indices_t, int32_t* slot_t, uint8_t* et_csr,
                                     uint8_t* et_t, int32_t* counts, int32_t* status, void* workspace,
                                     size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  const int loops = self_loops ? 1 : 0;
  const int64_t num_edges = num_sampled + loops * num_dst;
  REGNN_REQUIRE(num_dst >= 0 && num_src >= num_dst && num_sampled >= 0, REGNN_ERR_INVALID_ARG,
                "block_csr_build: bad sizes");
  REGNN_REQUIRE(num_src < ((int64_t)1 << 31) - 1 && num_edges < ((int64_t)1 << 31) - 1, REGNN_ERR_UNSUPPORTED_SHAPE,
                "block_csr_build: block exceeds int32 indexing");
  REGNN_REQUIRE(num_relations >= 1 && num_relations <= REGNN_MAX_RELATIONS, REGNN_ERR_UNSUPPORTED_SHAPE,
                "num_relations=%d outside [1, %d]", num_relations, REGNN_MAX_RELATIONS);
  REGNN_REQUIRE(row_off && indptr && indptr_t && workspace && (num_sampled == 0 || (src_local && dst_local && edge_id &&
                edge_type)) && status && (num_edges == 0 || (src && dst && etype1 && indices && eid && row && indices_t &&
                slot_t && et_csr && et_t)) && (!loops || num_dst == 0 || (targets && node_type)),
                REGNN_ERR_INVALID_ARG, "block_csr_build: null pointer");
  REGNN_REQUIRE(workspace_bytes >= regnn_csr_build_workspace_bytes(num_src, num_edges), REGNN_ERR_WORKSPACE_TOO_SMALL,
                "block_csr_build workspace too small");
  block_csr_fill_kernel<<<grid_of((num_edges > num_src ? num_edges : num_src + 1)), 256, 0, stream>>>(
      src_local, dst_local, edge_id, row_off, targets, num_src, num_dst, num_sampled, edge_type, node_type,
      num_edge_types, loops, src, dst, etype1, indptr, indices, eid, row, et_csr, num_relations, status);
  build_transposed_view(indices, row, num_src, num_edges, indptr_t, indices_t, slot_t, workspace, stream);
  if (num_edges > 0) etype_transpose_kernel<<<grid_of(num_edges), 256, 0, stream>>>(et_csr, slot_t, num_edges, et_t);
  int rc = check_launch("regnn_block_csr_build");
  if (rc != REGNN_OK || counts == nullptr) return rc;
  return regnn_relation_counts(row, et_csr, num_edges, num_src, num_relations, counts, stream);
}

// ---- GraphSAINT induced subgraph (mag/regnn_saint.py:185-190: GraphSAINTRandomWalkSampler) ----------------------
// The subgraph of the walk nodes: its nodes are the distinct listed nodes in ascending global id (torch.unique's
// order), its edges every in-edge of those rows whose source is listed too, in (row, CSR slot) order -- which is the
// subgraph's in-CSR already.  Listed nodes raise a flag in a persistent [N] map; an exclusive scan of the flags over
// all N gives node v its row excl[v].  Each row's slot range is cut into fragments of at most kInducedFragSlots slots
// (MAG hub rows have 10^4-10^5 in-edges, and walks reach a row in proportion to its in-degree), one warp per
// fragment: warp ballots count the kept slots, a scan of the fragment counts gives every fragment its output offset,
// and the fill replays the ballots to write each kept slot at that offset plus its rank.  Stores of equal values,
// integer counters and scans only: the result does not depend on the order in which threads run.
namespace regnn {

constexpr int kInducedFragSlots = 256;

static int64_t induced_frag_capacity(int64_t num_edges, int64_t max_rows) {
  return max_rows + (num_edges + kInducedFragSlots - 1) / kInducedFragSlots;   // sum of max(1, ceil(deg / 256))
}

struct InducedWorkspace {
  uint32_t* excl;         // [num_nodes] exclusive scan of the flags: the row of a listed node
  uint32_t* frag_first;   // [max_rows + 1] first fragment of each row (scan of the per-row fragment counts)
  uint32_t* frag_row;     // [frag_cap] row of each fragment
  uint32_t* frag_off;     // [frag_cap + 1] output offset of each fragment (scan of the kept-slot counts)
  uint32_t* block_sums;   // scan spine
};

static size_t induced_workspace_layout(int64_t num_nodes, int64_t num_edges, int64_t max_rows, char* base,
                                       InducedWorkspace* ws) {
  const int64_t cap = induced_frag_capacity(num_edges, max_rows);
  int64_t longest = num_nodes > cap + 1 ? num_nodes : cap + 1;
  if (max_rows + 1 > longest) longest = max_rows + 1;
  const size_t sizes[5] = {align256((size_t)(num_nodes > 0 ? num_nodes : 1) * 4), align256((size_t)(max_rows + 1) * 4),
                           align256((size_t)(cap > 0 ? cap : 1) * 4), align256((size_t)(cap + 1) * 4),
                           align256((size_t)scan_blocks(longest) * 4)};
  uint32_t** parts[5] = {&ws->excl, &ws->frag_first, &ws->frag_row, &ws->frag_off, &ws->block_sums};
  size_t off = 0;
  for (int i = 0; i < 5; ++i) {
    if (base) *parts[i] = (uint32_t*)(base + off);
    off += sizes[i];
  }
  return off;
}

__global__ void induced_flag_kernel(const int64_t* __restrict__ nodes, int64_t num_listed, int64_t num_nodes,
                                    uint32_t* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num_listed) return;
  const int64_t v = nodes[i];
  if (v >= 0 && v < num_nodes) flags[v] = 1u;
}

// One thread per node: a listed node v stores itself at row excl[v] and the number of fragments of its slot range
// (at least one, so that every row owns a fragment and row_off[r] is the offset of its first one).
__global__ void induced_rows_kernel(const int32_t* __restrict__ indptr, int64_t num_nodes,
                                    const uint32_t* __restrict__ flags, const uint32_t* __restrict__ excl,
                                    int64_t* __restrict__ n_id, uint32_t* __restrict__ frag_count,
                                    int32_t* __restrict__ info) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v == 0) info[REGNN_SAMPLE_INFO_SOURCES] = (int32_t)(excl[num_nodes - 1] + flags[num_nodes - 1]);
  if (v >= num_nodes || !flags[v]) return;
  const uint32_t r = excl[v];
  const int64_t deg = indptr[v + 1] - indptr[v];
  n_id[r] = v;
  frag_count[r] = deg > kInducedFragSlots ? (uint32_t)((deg + kInducedFragSlots - 1) / kInducedFragSlots) : 1u;
}

// One warp per fragment (frag_cap + 1 warps; those past the last fragment store a zero count for the scan).
__global__ void induced_frag_count_kernel(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                          const uint32_t* __restrict__ flags, const uint32_t* __restrict__ excl,
                                          const int64_t* __restrict__ n_id, const uint32_t* __restrict__ frag_first,
                                          int64_t frag_cap, const int32_t* __restrict__ info,
                                          uint32_t* __restrict__ frag_row, uint32_t* __restrict__ frag_count,
                                          int32_t* __restrict__ src_hist) {
  const int64_t f = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (f > frag_cap) return;
  const int64_t n_sub = info[REGNN_SAMPLE_INFO_SOURCES];
  if (f >= (int64_t)frag_first[n_sub]) {
    if (lane == 0) frag_count[f] = 0u;
    return;
  }
  int64_t lo = 0, hi = n_sub;                // the row r with frag_first[r] <= f < frag_first[r + 1]
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)frag_first[mid] <= f) lo = mid;
    else hi = mid;
  }
  const int64_t v = n_id[lo];
  const int64_t s0 = indptr[v] + (f - (int64_t)frag_first[lo]) * kInducedFragSlots;
  const int64_t s1 = min(s0 + kInducedFragSlots, (int64_t)indptr[v + 1]);
  uint32_t kept = 0;
  for (int64_t base = s0; base < s1; base += 32) {
    const int64_t s = base + lane;
    bool keep = false;
    if (s < s1) {
      const int32_t u = indices[s];
      keep = flags[u] != 0u;
      if (keep) atomicAdd(&src_hist[excl[u]], 1);
    }
    kept += __popc(__ballot_sync(0xffffffffu, keep));
  }
  if (lane == 0) {
    frag_row[f] = (uint32_t)lo;
    frag_count[f] = kept;
  }
}

// One thread per row slot 0..max_rows: row_off from the fragment offsets, and the statistics of both views.
__global__ void induced_rows_finish_kernel(int64_t max_rows, const uint32_t* __restrict__ frag_first,
                                           const uint32_t* __restrict__ frag_off, const int32_t* __restrict__ src_hist,
                                           int threshold, uint32_t* __restrict__ row_off, int32_t* __restrict__ info) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > max_rows) return;
  const int64_t n_sub = info[REGNN_SAMPLE_INFO_SOURCES];
  const uint32_t e0 = frag_off[frag_first[r < n_sub ? r : n_sub]];
  row_off[r] = e0;
  if (r == n_sub) info[REGNN_SAMPLE_INFO_EDGES] = (int32_t)e0;
  if (r >= n_sub) return;
  const int64_t deg = (int64_t)frag_off[frag_first[r + 1]] - e0;
  if (deg == 0) atomicAdd(&info[REGNN_SAMPLE_INFO_EMPTY_ROWS], 1);
  count_long_row(deg, threshold, info + REGNN_SAMPLE_INFO_IN_SPLIT);
  count_long_row(src_hist[r], threshold, info + REGNN_SAMPLE_INFO_OUT_SPLIT);
}

// The count kernel's ballots again, each kept slot written at its fragment's offset plus its rank in the fragment.
__global__ void induced_fill_kernel(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                    const int32_t* __restrict__ eid, const uint32_t* __restrict__ flags,
                                    const uint32_t* __restrict__ excl, const int64_t* __restrict__ n_id,
                                    int64_t num_rows, int64_t num_sub_edges, const uint32_t* __restrict__ frag_first,
                                    const uint32_t* __restrict__ frag_row, const uint32_t* __restrict__ frag_off,
                                    int64_t* __restrict__ src_local, int64_t* __restrict__ dst_local,
                                    int64_t* __restrict__ edge_id) {
  const int64_t f = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (f >= (int64_t)frag_first[num_rows]) return;
  const uint32_t r = frag_row[f];
  const int64_t v = n_id[r];
  const int64_t s0 = indptr[v] + (f - (int64_t)frag_first[r]) * kInducedFragSlots;
  const int64_t s1 = min(s0 + kInducedFragSlots, (int64_t)indptr[v + 1]);
  int64_t out = frag_off[f];
  for (int64_t base = s0; base < s1; base += 32) {
    const int64_t s = base + lane;
    int32_t u = 0;
    bool keep = false;
    if (s < s1) {
      u = indices[s];
      keep = flags[u] != 0u;
    }
    const uint32_t ballot = __ballot_sync(0xffffffffu, keep);
    const int64_t e = out + __popc(ballot & ((1u << lane) - 1u));
    if (keep && e < num_sub_edges) {
      src_local[e] = excl[u];
      dst_local[e] = r;
      edge_id[e] = eid[s];
    }
    out += __popc(ballot);
  }
}

__global__ void induced_clear_flags_kernel(const int64_t* __restrict__ n_id, int64_t num_rows,
                                           uint32_t* __restrict__ flags) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < num_rows) flags[n_id[r]] = 0u;
}

static unsigned warp_grid_of(int64_t warps) { return grid_of(warps * 32); }

}  // namespace regnn

extern "C" size_t regnn_induced_subgraph_workspace_bytes(int64_t num_nodes, int64_t num_edges, int64_t num_listed) {
  InducedWorkspace ws;
  const int64_t max_rows = num_listed < num_nodes ? num_listed : num_nodes;
  return induced_workspace_layout(num_nodes, num_edges, max_rows < 0 ? 0 : max_rows, nullptr, &ws);
}

extern "C" int regnn_induced_subgraph_count(const int32_t* indptr, const int32_t* indices, int64_t num_nodes,
                                            int64_t num_edges, const int64_t* nodes, int64_t num_listed,
                                            int split_threshold, uint32_t* flags, int64_t* n_id, uint32_t* row_off,
                                            int32_t* src_hist, int32_t* info, void* workspace, size_t workspace_bytes,
                                            void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr && flags && n_id && row_off && src_hist && info && workspace && (num_listed == 0 || nodes) &&
                (num_edges == 0 || indices), REGNN_ERR_INVALID_ARG, "induced_subgraph_count: null pointer");
  REGNN_REQUIRE(num_nodes >= 1 && num_listed >= 0 && num_edges >= 0 && split_threshold >= 1, REGNN_ERR_INVALID_ARG,
                "induced_subgraph_count: bad sizes");
  REGNN_REQUIRE(num_nodes < ((int64_t)1 << 31) - 1 && num_edges < ((int64_t)1 << 31) - 1, REGNN_ERR_UNSUPPORTED_SHAPE,
                "induced_subgraph_count: %lld nodes / %lld edges exceed int32 indexing", (long long)num_nodes,
                (long long)num_edges);
  REGNN_REQUIRE(workspace_bytes >= regnn_induced_subgraph_workspace_bytes(num_nodes, num_edges, num_listed),
                REGNN_ERR_WORKSPACE_TOO_SMALL, "induced_subgraph workspace too small");
  const int64_t max_rows = num_listed < num_nodes ? num_listed : num_nodes;
  const int64_t cap = induced_frag_capacity(num_edges, max_rows);
  InducedWorkspace ws;
  induced_workspace_layout(num_nodes, num_edges, max_rows, (char*)workspace, &ws);

  cudaMemsetAsync(info, 0, REGNN_SAMPLE_INFO_WORDS * sizeof(int32_t), stream);
  cudaMemsetAsync(src_hist, 0, (size_t)(max_rows > 0 ? max_rows : 1) * sizeof(int32_t), stream);
  cudaMemsetAsync(ws.frag_first, 0, (size_t)(max_rows + 1) * sizeof(uint32_t), stream);
  induced_flag_kernel<<<grid_of(num_listed), 256, 0, stream>>>(nodes, num_listed, num_nodes, flags);
  exclusive_scan_u32(flags, ws.excl, num_nodes, ws.block_sums, stream);
  induced_rows_kernel<<<grid_of(num_nodes), 256, 0, stream>>>(indptr, num_nodes, flags, ws.excl, n_id, ws.frag_first,
                                                              info);
  exclusive_scan_u32(ws.frag_first, ws.frag_first, max_rows + 1, ws.block_sums, stream);
  induced_frag_count_kernel<<<warp_grid_of(cap + 1), 256, 0, stream>>>(indptr, indices, flags, ws.excl, n_id,
                                                                       ws.frag_first, cap, info, ws.frag_row,
                                                                       ws.frag_off, src_hist);
  exclusive_scan_u32(ws.frag_off, ws.frag_off, cap + 1, ws.block_sums, stream);
  induced_rows_finish_kernel<<<grid_of(max_rows + 1), 256, 0, stream>>>(max_rows, ws.frag_first, ws.frag_off, src_hist,
                                                                        split_threshold, row_off, info);
  return check_launch("regnn_induced_subgraph_count");
}

extern "C" int regnn_induced_subgraph_fill(const int32_t* indptr, const int32_t* indices, const int32_t* eid,
                                           int64_t num_nodes, int64_t num_edges, int64_t num_listed, uint32_t* flags,
                                           const int64_t* n_id, int64_t num_rows, int64_t num_sub_edges,
                                           int64_t* src_local, int64_t* dst_local, int64_t* edge_id, void* workspace,
                                           size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  const int64_t max_rows = num_listed < num_nodes ? num_listed : num_nodes;
  REGNN_REQUIRE(indptr && flags && n_id && workspace && (num_edges == 0 || (indices && eid)) &&
                (num_sub_edges == 0 || (src_local && dst_local && edge_id)), REGNN_ERR_INVALID_ARG,
                "induced_subgraph_fill: null pointer");
  REGNN_REQUIRE(num_nodes >= 1 && num_edges >= 0 && num_listed >= 0 && num_rows >= 0 && num_rows <= max_rows &&
                num_sub_edges >= 0 && num_sub_edges <= num_edges, REGNN_ERR_INVALID_ARG,
                "induced_subgraph_fill: bad sizes");
  REGNN_REQUIRE(num_nodes < ((int64_t)1 << 31) - 1 && num_edges < ((int64_t)1 << 31) - 1, REGNN_ERR_UNSUPPORTED_SHAPE,
                "induced_subgraph_fill: %lld nodes / %lld edges exceed int32 indexing", (long long)num_nodes,
                (long long)num_edges);
  REGNN_REQUIRE(workspace_bytes >= regnn_induced_subgraph_workspace_bytes(num_nodes, num_edges, num_listed),
                REGNN_ERR_WORKSPACE_TOO_SMALL, "induced_subgraph workspace too small");
  InducedWorkspace ws;
  induced_workspace_layout(num_nodes, num_edges, max_rows, (char*)workspace, &ws);
  induced_fill_kernel<<<warp_grid_of(induced_frag_capacity(num_edges, max_rows)), 256, 0, stream>>>(
      indptr, indices, eid, flags, ws.excl, n_id, num_rows, num_sub_edges, ws.frag_first, ws.frag_row, ws.frag_off,
      src_local, dst_local, edge_id);
  induced_clear_flags_kernel<<<grid_of(num_rows), 256, 0, stream>>>(n_id, num_rows, flags);
  return check_launch("regnn_induced_subgraph_fill");
}
