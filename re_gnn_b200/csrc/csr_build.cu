// Graph construction on the device: destination-sorted CSR + source-sorted (transposed) view +
// edge-type permutation.  Replaces DGL's lazy CSR builds behind run_regnn.py:84-87 /
// layer/REGraphConv.py:69.  Integer work only; results are bit-exact against oracle/csr_oracle.py.
//
// Sort: hand-written stable LSD radix sort, 8-bit digits, (key = node id, value = edge id / slot).
// Per pass: per-tile digit histogram -> exclusive scan over the digit-major (digit, tile) count
// matrix -> stable scatter (warp match_any ranks + per-warp digit counters).  HBM-bound integer
// streaming: 4 B key + 4 B value read and written once per pass (+4 B for the histogram read).
#include "common.cuh"

namespace regnn {

constexpr int kSortThreads = 256;
constexpr int kSortItems = 8;
constexpr int kSortTile = kSortThreads * kSortItems;  // 2048 keys per block
constexpr int kScanThreads = 256;
constexpr int kScanItems = 16;
constexpr int kScanTile = kScanThreads * kScanItems;  // 4096 counters per block

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// ---- exclusive scan (uint32) ---------------------------------------------------------------------
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();  // protect warp_sums reuse across calls
  if (lane == 31) warp_sums[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    uint32_t w = lane < nw ? warp_sums[lane] : 0u, winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    warp_sums[lane] = winc - w;  // exclusive prefix of warp totals
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  return warp_sums[wid] + inc - v;
}

__global__ void scan_reduce_kernel(const uint32_t* __restrict__ in, int64_t n,
                                   uint32_t* __restrict__ block_sums) {
  __shared__ uint32_t total;
  int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  uint32_t s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) s += in[base + i];
  block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// Single block: exclusive scan of block_sums in place (loops with a carry for long arrays).
__global__ void scan_spine_kernel(uint32_t* __restrict__ block_sums, int64_t nb) {
  __shared__ uint32_t total;
  uint32_t carry = 0;
  for (int64_t base = 0; base < nb; base += blockDim.x) {
    int64_t i = base + threadIdx.x;
    uint32_t v = i < nb ? block_sums[i] : 0u;
    uint32_t ex = block_exclusive_scan(v, &total);
    if (i < nb) block_sums[i] = carry + ex;
    carry += total;
    __syncthreads();
  }
}

__global__ void scan_apply_kernel(const uint32_t* __restrict__ in, int64_t n,
                                  const uint32_t* __restrict__ block_sums,
                                  uint32_t* __restrict__ out) {
  __shared__ uint32_t total;
  int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  uint32_t v[kScanItems], s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = base + i < n ? in[base + i] : 0u;
    s += v[i];
  }
  uint32_t run = block_exclusive_scan(s, &total) + block_sums[blockIdx.x];
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = run;
    run += v[i];
  }
}

void exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* block_sums,
                        cudaStream_t stream) {
  if (n <= 0) return;
  int64_t nb = (n + kScanTile - 1) / kScanTile;
  scan_reduce_kernel<<<(unsigned)nb, kScanThreads, 0, stream>>>(in, n, block_sums);
  scan_spine_kernel<<<1, 1024, 0, stream>>>(block_sums, nb);
  scan_apply_kernel<<<(unsigned)nb, kScanThreads, 0, stream>>>(in, n, block_sums, out);
}

// ---- radix sort passes ---------------------------------------------------------------------------
__global__ void init_keys_kernel(const int64_t* __restrict__ key_ids,
                                 const int64_t* __restrict__ other_ids, int64_t n_nodes, int64_t n,
                                 uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                 int* __restrict__ err) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t k = key_ids[i], o = other_ids[i];
  if (k < 0 || k >= n_nodes || o < 0 || o >= n_nodes) {
    *err = 1;  // benign race: any writer stores the same value
    k = 0;
  }
  keys[i] = (uint32_t)k;
  vals[i] = (uint32_t)i;
}

__global__ void init_keys32_kernel(const int32_t* __restrict__ key_ids, int64_t n,
                                   uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = (uint32_t)key_ids[i];
  vals[i] = (uint32_t)i;
}

__global__ void radix_hist_kernel(const uint32_t* __restrict__ keys, int64_t n, int shift,
                                  uint32_t* __restrict__ counts, int64_t num_tiles) {
  __shared__ uint32_t hist[256];
  hist[threadIdx.x] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * kSortTile;
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    int64_t i = base + r * kSortThreads + threadIdx.x;
    if (i < n) atomicAdd(&hist[(keys[i] >> shift) & 255u], 1u);  // integer counts: order-free
  }
  __syncthreads();
  counts[(int64_t)threadIdx.x * num_tiles + blockIdx.x] = hist[threadIdx.x];
}

__global__ void __launch_bounds__(kSortThreads)
radix_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                     uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int64_t n,
                     int shift, const uint32_t* __restrict__ offsets, int64_t num_tiles) {
  __shared__ uint32_t wh[kSortThreads / 32][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < (kSortThreads / 32) * 256; i += kSortThreads) (&wh[0][0])[i] = 0;
  __syncthreads();

  // Warp w owns the contiguous span [w*256, w*256+256) of the tile, visited in 8 rounds of 32.
  const int64_t base = (int64_t)blockIdx.x * kSortTile + w * (32 * kSortItems) + lane;
  uint32_t k[kSortItems], v[kSortItems], local[kSortItems];
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    int64_t i = base + r * 32;
    k[r] = i < n ? keys_in[i] : 0u;
    v[r] = i < n ? vals_in[i] : 0u;
  }
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const bool valid = base + r * 32 < n;
    const uint32_t digit = valid ? ((k[r] >> shift) & 255u) : 256u;
    const uint32_t peers = __match_any_sync(0xffffffffu, digit);
    const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
    local[r] = valid ? wh[w][digit] + rank : 0u;
    __syncwarp();
    if (valid && rank == 0) wh[w][digit] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  {  // exclusive prefix over the warps of this block, per digit (thread d owns digit d)
    uint32_t run = 0;
#pragma unroll
    for (int ww = 0; ww < kSortThreads / 32; ++ww) {
      uint32_t t = wh[ww][threadIdx.x];
      wh[ww][threadIdx.x] = run;
      run += t;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    if (base + r * 32 < n) {
      const uint32_t digit = (k[r] >> shift) & 255u;
      const uint32_t pos = offsets[(int64_t)digit * num_tiles + blockIdx.x] + wh[w][digit] + local[r];
      keys_out[pos] = k[r];
      vals_out[pos] = v[r];
    }
  }
}

struct SortBuffers {
  uint32_t *keys_a, *keys_b, *vals_a, *vals_b, *counts, *block_sums;
  int* err;
  int64_t num_tiles;
};

static int key_bits(int64_t n_nodes) {
  int bits = 1;
  while (bits < 32 && ((int64_t)1 << bits) < n_nodes) ++bits;
  return bits;
}

// Sorts (keys_a, vals_a) stably by key; returns through *keys / *vals the buffers holding the result.
static void radix_sort_pairs(SortBuffers& sb, int64_t n, int bits, uint32_t** keys, uint32_t** vals,
                             cudaStream_t stream) {
  uint32_t *kin = sb.keys_a, *kout = sb.keys_b, *vin = sb.vals_a, *vout = sb.vals_b;
  if (n > 0) {
    for (int shift = 0; shift < bits; shift += 8) {
      radix_hist_kernel<<<(unsigned)sb.num_tiles, kSortThreads, 0, stream>>>(kin, n, shift, sb.counts,
                                                                              sb.num_tiles);
      exclusive_scan_u32(sb.counts, sb.counts, 256 * sb.num_tiles, sb.block_sums, stream);
      radix_scatter_kernel<<<(unsigned)sb.num_tiles, kSortThreads, 0, stream>>>(
          kin, vin, kout, vout, n, shift, sb.counts, sb.num_tiles);
      uint32_t* t = kin; kin = kout; kout = t;
      t = vin; vin = vout; vout = t;
    }
  }
  *keys = kin;
  *vals = vin;
}

// indptr[v] = first sorted position whose key is >= v (keys sorted ascending); indptr[N] = n.
// One thread per row, binary search: no serial walk over runs of empty rows (sampled blocks have
// tens of thousands of trailing rows without in-edges).
__global__ void boundary_fill_kernel(const uint32_t* __restrict__ keys, int64_t n, int64_t n_nodes,
                                     int32_t* __restrict__ indptr) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v > n_nodes) return;
  int64_t lo = 0, hi = n;  // first index with keys[idx] >= v
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)keys[mid] < v) lo = mid + 1; else hi = mid;
  }
  indptr[v] = (int32_t)lo;
}

__global__ void finish_csr_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                  const int64_t* __restrict__ src, int64_t n,
                                  int32_t* __restrict__ indices, int32_t* __restrict__ eid,
                                  int32_t* __restrict__ row) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  uint32_t e = vals[s];
  eid[s] = (int32_t)e;
  row[s] = (int32_t)keys[s];
  indices[s] = (int32_t)src[e];
}

__global__ void finish_csc_kernel(const uint32_t* __restrict__ vals, const int32_t* __restrict__ row,
                                  int64_t n, int32_t* __restrict__ indices_t,
                                  int32_t* __restrict__ slot_t) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  uint32_t s = vals[j];
  slot_t[j] = (int32_t)s;
  indices_t[j] = row[s];
}

__global__ void etype_permute_kernel(const int64_t* __restrict__ etype, const int32_t* __restrict__ eid,
                                     const int32_t* __restrict__ slot_t, int64_t n, int num_rel,
                                     uint8_t* __restrict__ et_csr, uint8_t* __restrict__ et_t,
                                     int* __restrict__ err) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t a = etype[eid[i]];
  int64_t b = etype[eid[slot_t[i]]];
  if (a < 1 || a > num_rel || b < 1 || b > num_rel) {
    *err = 1;
    a = b = 1;
  }
  et_csr[i] = (uint8_t)(a - 1);
  et_t[i] = (uint8_t)(b - 1);
}

static SortBuffers carve(void* ws, int64_t n_edges) {
  SortBuffers sb;
  char* p = (char*)ws;
  size_t eb = align256((size_t)(n_edges > 0 ? n_edges : 1) * 4);
  sb.num_tiles = (n_edges + kSortTile - 1) / kSortTile;
  if (sb.num_tiles < 1) sb.num_tiles = 1;
  size_t cb = align256((size_t)256 * sb.num_tiles * 4);
  size_t bb = align256((size_t)((256 * sb.num_tiles + kScanTile - 1) / kScanTile + 1) * 4);
  sb.keys_a = (uint32_t*)p; p += eb;
  sb.keys_b = (uint32_t*)p; p += eb;
  sb.vals_a = (uint32_t*)p; p += eb;
  sb.vals_b = (uint32_t*)p; p += eb;
  sb.counts = (uint32_t*)p; p += cb;
  sb.block_sums = (uint32_t*)p; p += bb;
  sb.err = (int*)p;
  return sb;
}

// Source-sorted view of a destination-sorted CSR: a stable sort of the CSR slots by their source id.
void build_transposed_view(const int32_t* indices, const int32_t* row, int64_t num_nodes, int64_t num_edges,
                           int32_t* indptr_t, int32_t* indices_t, int32_t* slot_t, void* workspace,
                           cudaStream_t stream) {
  SortBuffers sb = carve(workspace, num_edges);
  const int T = 256;
  const unsigned eb = (unsigned)((num_edges + T - 1) / T), ebp = (unsigned)((num_nodes + 1 + T - 1) / T);
  uint32_t *keys, *vals;
  if (num_edges > 0) init_keys32_kernel<<<eb, T, 0, stream>>>(indices, num_edges, sb.keys_a, sb.vals_a);
  radix_sort_pairs(sb, num_edges, key_bits(num_nodes), &keys, &vals, stream);
  boundary_fill_kernel<<<ebp, T, 0, stream>>>(keys, num_edges, num_nodes, indptr_t);
  if (num_edges > 0) finish_csc_kernel<<<eb, T, 0, stream>>>(vals, row, num_edges, indices_t, slot_t);
}

}  // namespace regnn

using namespace regnn;

extern "C" size_t regnn_csr_build_workspace_bytes(int64_t num_nodes, int64_t num_edges) {
  (void)num_nodes;
  int64_t e = num_edges > 0 ? num_edges : 1;
  int64_t tiles = (e + kSortTile - 1) / kSortTile;
  return 4 * align256((size_t)e * 4) + align256((size_t)256 * tiles * 4) +
         align256((size_t)((256 * tiles + kScanTile - 1) / kScanTile + 1) * 4) + 256;
}

extern "C" int regnn_csr_build(const int64_t* src, const int64_t* dst, int64_t num_nodes,
                               int64_t num_edges, int32_t* indptr, int32_t* indices, int32_t* eid,
                               int32_t* row, int32_t* indptr_t, int32_t* indices_t, int32_t* slot_t,
                               void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(num_nodes >= 0 && num_edges >= 0, REGNN_ERR_INVALID_ARG, "negative graph size");
  REGNN_REQUIRE(num_nodes < ((int64_t)1 << 31) - 1 && num_edges < ((int64_t)1 << 31) - 1,
                REGNN_ERR_UNSUPPORTED_SHAPE, "graph exceeds int32 indexing (N=%lld, E=%lld)",
                (long long)num_nodes, (long long)num_edges);
  REGNN_REQUIRE(workspace_bytes >= regnn_csr_build_workspace_bytes(num_nodes, num_edges),
                REGNN_ERR_WORKSPACE_TOO_SMALL, "csr_build workspace too small");
  REGNN_REQUIRE(indptr && indptr_t && workspace, REGNN_ERR_INVALID_ARG, "null pointer");
  SortBuffers sb = carve(workspace, num_edges);
  const int bits = key_bits(num_nodes);
  const int T = 256;
  const unsigned eb = (unsigned)((num_edges + T - 1) / T), ebp = (unsigned)((num_nodes + 1 + T - 1) / T);
  cudaMemsetAsync(sb.err, 0, sizeof(int), stream);
  uint32_t *keys, *vals;

  // destination-sorted CSR
  if (num_edges > 0)
    init_keys_kernel<<<eb, T, 0, stream>>>(dst, src, num_nodes, num_edges, sb.keys_a, sb.vals_a, sb.err);
  radix_sort_pairs(sb, num_edges, bits, &keys, &vals, stream);
  boundary_fill_kernel<<<ebp, T, 0, stream>>>(keys, num_edges, num_nodes, indptr);
  if (num_edges > 0) finish_csr_kernel<<<eb, T, 0, stream>>>(keys, vals, src, num_edges, indices, eid, row);
  build_transposed_view(indices, row, num_nodes, num_edges, indptr_t, indices_t, slot_t, workspace, stream);

  int rc = check_launch("regnn_csr_build");
  if (rc != REGNN_OK) return rc;
  int err = 0;
  cudaMemcpyAsync(&err, sb.err, sizeof(int), cudaMemcpyDeviceToHost, stream);
  cudaError_t ce = cudaStreamSynchronize(stream);
  REGNN_REQUIRE(ce == cudaSuccess, REGNN_ERR_CUDA, "regnn_csr_build: %s", cudaGetErrorString(ce));
  REGNN_REQUIRE(err == 0, REGNN_ERR_INVALID_ARG, "edge endpoint outside [0, %lld)", (long long)num_nodes);
  return REGNN_OK;
}

extern "C" int regnn_etype_permute(const int64_t* etype_1based, const int32_t* eid,
                                   const int32_t* slot_t, int64_t num_edges, int num_relations,
                                   uint8_t* etype_csr, uint8_t* etype_t, int32_t* status_scratch,
                                   void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(num_relations >= 1 && num_relations <= REGNN_MAX_RELATIONS, REGNN_ERR_UNSUPPORTED_SHAPE,
                "num_relations=%d outside [1, %d]", num_relations, REGNN_MAX_RELATIONS);
  REGNN_REQUIRE(status_scratch, REGNN_ERR_INVALID_ARG, "null status scratch");
  if (num_edges == 0) return REGNN_OK;
  cudaMemsetAsync(status_scratch, 0, sizeof(int), stream);
  etype_permute_kernel<<<(unsigned)((num_edges + 255) / 256), 256, 0, stream>>>(
      etype_1based, eid, slot_t, num_edges, num_relations, etype_csr, etype_t, status_scratch);
  int rc = check_launch("regnn_etype_permute");
  if (rc != REGNN_OK) return rc;
  int err = 0;
  cudaMemcpyAsync(&err, status_scratch, sizeof(int), cudaMemcpyDeviceToHost, stream);
  cudaError_t ce = cudaStreamSynchronize(stream);
  REGNN_REQUIRE(ce == cudaSuccess, REGNN_ERR_CUDA, "regnn_etype_permute: %s", cudaGetErrorString(ce));
  REGNN_REQUIRE(err == 0, REGNN_ERR_INVALID_ARG, "edge type outside [1, %d]", num_relations);
  return REGNN_OK;
}
