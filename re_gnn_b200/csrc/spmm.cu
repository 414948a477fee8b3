// REGCN / REMixHop aggregation kernels: relation-weighted in-degree norm, the fused
// norm * (relation-weighted SpMM) * norm, and the deterministic backward reductions.
// Reference call sites: layer/REGraphConv.py:58-98, layer/REMixHopConv.py:50-82.
//
// All of these are gather-bound (HBM / L2 bandwidth): one source row of 4F bytes per edge.
// Three generations of the SpMM live here, newest last:
//   spmm_bwd_w_kernel                 one row per lane group in natural row order (regnn_spmm_bwd_w, F > 512);
//   spmm_stream_kernel                a warp streams the concatenated slots of 32 rows (F > 128, row sub-ranges);
//   spmm_rowgroup_kernel              lane groups over the degree-sorted row list (F <= 128, full range): the
//                                     production kernels, forward at 96 % of the measured HBM bandwidth.
// Every variant sums a row's slots in slot order: no atomics, bit-identical run to run and to each other.
#include <initializer_list>

#include "common.cuh"

namespace regnn {

struct SpmmArgs {
  const int32_t* indptr;
  const int32_t* indices;
  const uint8_t* etype;
  const float* theta;
  float alpha;
  int R;
  const float* norm_src;
  const float* norm_dst;
  const float* X;
  int64_t ldx;
  float* Y;
  int64_t ldy;
  int64_t row_begin, row_end;
  int F;
  // long-row fragments (see regnn_rowsplit_t): work items [0, nfrag) are fragments, padded to nfrag_pad
  const int32_t* frag_row;
  const int32_t* frag_begin;
  int nfrag, nfrag_pad, threshold;
  float* partial;  // [nfrag][F] un-normalised fragment sums
};

// Row-block owners of the feature-sliced multi-GPU scheme (regnn_peer_rows_t): row v of a result belongs to rank
// v / per and lives at base[v / per] + (v % per) * ld + col -- a peer-mapped (NVLink) address for remote ranks.
struct PeerRows {
  float* const* base;
  uint32_t per;
  int64_t ld, col;
  __device__ __forceinline__ float* row(int64_t v) const {
    const uint32_t q = (uint32_t)v / per;
    return base[q] + (size_t)((uint32_t)v - q * per) * ld + col;
  }
};


template <int VW> struct Vec;
template <> struct Vec<4> {
  using T = float4;
  static __device__ __forceinline__ T zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
  static __device__ __forceinline__ T load(const float* p) { return ldg4(p); }
  static __device__ __forceinline__ void store(float* p, T v) { st4(p, v); }
  static __device__ __forceinline__ void fma(T& a, float s, T v) { fma4(a, s, v); }
  static __device__ __forceinline__ float dot(T a, T b) { return dot4(a, b); }
  static __device__ __forceinline__ T scaled(T a, float s) { scale4(a, s); return a; }
};
template <> struct Vec<1> {
  using T = float;
  static __device__ __forceinline__ T zero() { return 0.f; }
  static __device__ __forceinline__ T load(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ void store(float* p, T v) { *p = v; }
  static __device__ __forceinline__ void fma(T& a, float s, T v) { a = fmaf(s, v, a); }
  static __device__ __forceinline__ float dot(T a, T b) { return a * b; }
  static __device__ __forceinline__ T scaled(T a, float s) { return a * s; }
};

template <int C> struct Unroll { static constexpr int U = C <= 1 ? 8 : (C <= 2 ? 4 : (C <= 4 ? 2 : 1)); };

// ---- long-row fragments ---------------------------------------------------------------------------
// Work items of every SpMM kernel below: fragments of long rows first (lowest block ids start first, so the
// heaviest rows never form the tail), then the ordinary rows.  A fragment writes its un-normalised partial sum
// to `partial`; spmm_frag_finalize_kernel adds the fragments of a row in fragment order.
// Y[v] = norm_dst[v] * sum over the fragments of long row v (fragment order => deterministic).
__global__ void spmm_frag_finalize_kernel(const int32_t* __restrict__ long_rows,
                                          const int32_t* __restrict__ frag_ptr, int num_long,
                                          const float* __restrict__ partial, const float* __restrict__ norm_dst,
                                          float* __restrict__ Y, int64_t ldy, int F, int64_t row_begin,
                                          int64_t row_end) {
  const int l = blockIdx.x;
  if (l >= num_long) return;
  const int64_t v = long_rows[l];
  if (v < row_begin || v >= row_end) return;
  const int f0 = frag_ptr[l], f1 = frag_ptr[l + 1];
  const float nd = norm_dst != nullptr ? norm_dst[v] : 1.f;
  for (int c = threadIdx.x; c < F; c += blockDim.x) {
    float s = 0.f;
    for (int f = f0; f < f1; ++f) s += partial[(size_t)f * F + c];
    Y[(size_t)v * ldy + c] = s * nd;
  }
}

// Scatter variant of the above for the feature-sliced scheme: the row goes to its owner rank's row block (and, when
// Ylocal != null, also to the local slab), and the row dots of the norm gradient are taken here because the finished
// row is no longer in local memory:  xdx[v] = <Xrow[v], dX[v]>  or, folded (d_norm != null),
//   d_norm[v] = ( [sides&2] <Yfwd[v], Gd[v]> + [sides&1] <Xrow[v], dX[v]> ) / norm[v]   (this rank's columns only).
struct FragPeerExtra {
  float* Ylocal; int64_t ldl;                 // forward: local copy of the finished rows
  const float* Xrow; int64_t ldr; float* xdx; // backward: <Xrow, dX>
  const float* Yfwd; int64_t ldyf; const float* Gd; int64_t ldg; const float* norm; int sides; float* d_norm;
};
__global__ void spmm_frag_finalize_peer_kernel(const int32_t* __restrict__ long_rows,
                                               const int32_t* __restrict__ frag_ptr, int num_long,
                                               const float* __restrict__ partial, const float* __restrict__ norm_dst,
                                               PeerRows peers, int F, FragPeerExtra ex) {
  __shared__ float red[4];
  const int l = blockIdx.x;
  if (l >= num_long) return;
  const int64_t v = long_rows[l];
  const int f0 = frag_ptr[l], f1 = frag_ptr[l + 1];
  const float nd = norm_dst != nullptr ? norm_dst[v] : 1.f;
  float* yrow = peers.row(v);
  const bool want_x = ex.xdx != nullptr || (ex.d_norm != nullptr && (ex.sides & 1));
  const bool want_y = ex.d_norm != nullptr && (ex.sides & 2);
  float p = 0.f;
  for (int c = threadIdx.x; c < F; c += blockDim.x) {
    float s = 0.f;
    for (int f = f0; f < f1; ++f) s += partial[(size_t)f * F + c];
    s *= nd;
    yrow[c] = s;
    if (ex.Ylocal != nullptr) ex.Ylocal[(size_t)v * ex.ldl + c] = s;
    if (want_x) p = fmaf(ex.Xrow[(size_t)v * ex.ldr + c], s, p);
    if (want_y) p = fmaf(ex.Yfwd[(size_t)v * ex.ldyf + c], ex.Gd[(size_t)v * ex.ldg + c], p);
  }
  if (want_x || want_y) {  // fixed-shape block reduction (4 warps)
    p = group_sum<32>(p);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = p;
    __syncthreads();
    if (threadIdx.x == 0) {
      const float t = (red[0] + red[1]) + (red[2] + red[3]);
      if (ex.d_norm != nullptr) ex.d_norm[v] = t / ex.norm[v];
      else ex.xdx[v] = t;
    }
  }
}

// Row block -> column slabs over peer memory (the input exchange of the feature-sliced scheme): this rank's
// rows [0, rows) x all F columns are cut into P column slices; slice q lands in rank q's slab
// [P*per, F/P] at row row_offset + i.  Per peer the destination is ONE contiguous range, written with
// coalesced 128-bit stores (full NVLink packets); the strided side is the local read.
// Peers are visited in a rank-rotated order (rank r starts with peer r, then r+1, ...): blocks are scheduled y-major, so
// without the rotation every rank would write to peer 0 first, then peer 1, ... -- P senders on one receiver's NVLink
// ingress while the other links idle (measured at 8 GPUs: 0.35 ms per 109 MB push, 311 GB/s per rank).
__global__ void rows_to_slabs_kernel(const float* __restrict__ X, int64_t ldx, int64_t rows, int Fc,
                                     int64_t row_offset, float* const* __restrict__ peer_slabs, int first_peer) {
  const int q = (int)((blockIdx.y + (unsigned)first_peer) % gridDim.y);
  const int L = Fc >> 2;  // 128-bit chunks per slab row
  const int64_t total = rows * L;
  float4* dst = reinterpret_cast<float4*>(peer_slabs[q]) + row_offset * L;
  const float* src = X + (size_t)q * Fc;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / L;
    const int c = (int)(e - i * L) << 2;
    dst[e] = ldg4_stream(src + (size_t)i * ldx + c);
  }
}

// Indexed row push of the halo exchange (destination-row blocks that exchange only the rows a peer's edges reference):
// the rows send_rows[ptr[q] .. ptr[q+1]) of this rank's block go to consecutive rows of peer q's halo buffer, from row
// recv_offset[q] on.  One group of G lanes per row (G = the row's 128-bit chunks rounded up to a power of two, at most
// 32): the row index is loaded once, then the group streams the row with 128-bit reads and one contiguous store burst.
// Peers in rank-rotated order as in rows_to_slabs_kernel.  The small per-peer tables travel as a kernel parameter.
struct HaloPeers {
  int64_t ptr[REGNN_HALO_MAX_RANKS + 1];
  int64_t recv_offset[REGNN_HALO_MAX_RANKS];
};

__global__ void halo_push_kernel(const float* __restrict__ X, int64_t ldx, int L, int G,
                                 const int32_t* __restrict__ send_rows, const __grid_constant__ HaloPeers hp,
                                 float* const* __restrict__ peer_bufs, int64_t ldb, int first_peer) {
  const int q = (int)((blockIdx.y + (unsigned)first_peer) % gridDim.y);
  const int64_t begin = hp.ptr[q];
  const int64_t cnt = hp.ptr[q + 1] - begin;
  if (cnt == 0) return;
  float* dst = peer_bufs[q] + hp.recv_offset[q] * ldb;
  const int lane = threadIdx.x % G;
  const int64_t groups = (int64_t)gridDim.x * (blockDim.x / G);
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G; i < cnt; i += groups) {
    const float* src = X + (int64_t)__ldg(send_rows + begin + i) * ldx;
    float* out = dst + i * ldb;
    for (int c = lane; c < L; c += G) st4(out + 4 * c, ldg4_stream(src + 4 * c));
  }
}

// Indexed row scatter, the reverse direction of halo_push_kernel (the per-slot logit gradients of the REGAT backward go
// back to the owners of their destination rows): the rows ptr[q] .. ptr[q+1] of this rank's buffer go to rows
// dst_rows[k] of peer q's buffer.  The rows are W = num_heads floats (1..8), not whole 128-bit chunks: one lane per
// float, so consecutive lanes read consecutive floats of the contiguous source range and store 4-byte words.  Peers in
// rank-rotated order; the per-peer offsets travel as a kernel parameter.
__global__ void halo_scatter_kernel(const float* __restrict__ X, int64_t ldx, int W,
                                    const int32_t* __restrict__ dst_rows, const __grid_constant__ HaloPeers hp,
                                    float* const* __restrict__ peer_bufs, int64_t ldb, int first_peer) {
  const int q = (int)((blockIdx.y + (unsigned)first_peer) % gridDim.y);
  const int64_t begin = hp.ptr[q];
  const int64_t total = (hp.ptr[q + 1] - begin) * W;
  if (total == 0) return;
  float* dst = peer_bufs[q];
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / W;
    const int c = (int)(e - i * W);
    dst[(int64_t)__ldg(dst_rows + begin + i) * ldb + c] = __ldg(X + (begin + i) * ldx + c);
  }
}

// Indexed per-slot push of the REGATv2 halo backward, the transpose of halo_scatter_kernel: the forward stored the logit
// and the sign mask of an edge in its destination's in-view slot, but the source-major edge pass runs on the owner of
// the source.  For k in ptr[q] .. ptr[q+1], slot s = send_slots[k] goes to row recv_offset[q] + (k - ptr[q]) of peer
// q's two buffers: logit[s, 0:H] (4-byte words) and mask[s, 0:C] (C = ceil(H*D/128) 128-bit words).  One group of G
// lanes per slot (G = H + C rounded up to a power of two, at most 32): the slot index is loaded once per group, lanes
// [0, C) move the mask words and lanes [C, C+H) the logits.  Peers in rank-rotated order as in halo_push_kernel.
__global__ void halo_push_slots_kernel(const float* __restrict__ logit, int H, const uint4* __restrict__ mask, int C,
                                       int G, const int32_t* __restrict__ send_slots, const __grid_constant__ HaloPeers hp,
                                       float* const* __restrict__ peer_logit, float* const* __restrict__ peer_mask,
                                       int first_peer) {
  const int q = (int)((blockIdx.y + (unsigned)first_peer) % gridDim.y);
  const int64_t begin = hp.ptr[q];
  const int64_t cnt = hp.ptr[q + 1] - begin;
  if (cnt == 0) return;
  float* dl = peer_logit[q] + hp.recv_offset[q] * H;
  uint4* dm = reinterpret_cast<uint4*>(peer_mask[q]) + hp.recv_offset[q] * C;
  const int lane = threadIdx.x % G, W = C + H;
  const int64_t groups = (int64_t)gridDim.x * (blockDim.x / G);
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G; i < cnt; i += groups) {
    const int64_t s = __ldg(send_slots + begin + i);
    for (int c = lane; c < W; c += G) {
      if (c < C) dm[i * C + c] = __ldg(mask + s * C + c);
      else dl[i * H + (c - C)] = __ldg(logit + s * H + (c - C));
    }
  }
}

// Column slab -> row blocks over peer memory, for the kernels that have no scatter epilogue of their own (the fused
// attention kernels: one head slice per rank): rows [q*per, (q+1)*per) of this rank's slab S [N, Fc] go to rank q's row
// block at column col_offset.  The local read is contiguous, every destination row gets one Fc*4-byte store burst
// (64..512 bytes); peers in rank-rotated order as above.
__global__ void slabs_to_rows_kernel(const float* __restrict__ S, int64_t lds, int64_t rows, int Fc, PeerRows peers,
                                     int first_peer) {
  const int q = (int)((blockIdx.y + (unsigned)first_peer) % gridDim.y);
  const int L = Fc >> 2;
  const int64_t r0 = (int64_t)q * peers.per;
  const int64_t cnt = min(rows, r0 + (int64_t)peers.per) - r0;
  if (cnt <= 0) return;
  const int64_t total = cnt * L;
  float* dst = peers.base[q] + peers.col;
  const float* src = S + (size_t)r0 * lds;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / L;
    const int c = (int)(e - i * L) << 2;
    st4(dst + (size_t)i * peers.ld + c, ldg4_stream(src + (size_t)i * lds + c));
  }
}

// ---- per-block reduction of lane-local relation bins ------------------------------------------
// bins: [warps][R][32] floats (lane-local running sums), scratch: [warps][R] doubles.
__device__ __forceinline__ void reduce_bins(const float* bins, double* scratch, int R,
                                            double* __restrict__ out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncwarp();
  for (int r = 0; r < R; ++r) {
    double t = (double)bins[((size_t)warp * R + r) * 32 + lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) scratch[warp * R + r] = t;
  }
  __syncthreads();
  for (int r = threadIdx.x; r < R; r += blockDim.x) {
    double s = 0.0;
    for (int w = 0; w < kWarpsPerBlock; ++w) s += scratch[w * R + r];
    out[r] = s;
  }
}

// ---- streaming SpMM (the production forward / backward kernel) ---------------------------------------
// One warp streams the CONCATENATED slot range of a block of RB consecutive rows: column indices, edge
// types and norm[src] are read coalesced 32 slots at a time (and prefetched one batch ahead), U source
// rows are gathered with fully coalesced 128-bit loads before any FMA, and the accumulator is flushed
// whenever the slot stream crosses a row boundary.  Short rows therefore cost no dependent-latency
// bubble of their own: the gather pipeline never drains inside a block.  Rows longer than the split
// threshold are skipped here and covered by fragment items (first in the grid).
//
// BINS variant (backward, run on the transposed view): per slot the gathered row G[dst] is also dotted
// with the row-level tile Xrow[u] (staged in shared memory by TMA bulk copies, cp.async.bulk +
// mbarrier) and added to a lane-local per-relation bin: d w[r] = sum_e norm*norm*<X[src], G[dst]> falls
// out of the same gather that produces dX -- no second pass over the edges.
template <> struct Vec<2> {
  using T = float2;
  static __device__ __forceinline__ T zero() { return make_float2(0.f, 0.f); }
  static __device__ __forceinline__ T load(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
  static __device__ __forceinline__ void store(float* p, T v) { *reinterpret_cast<float2*>(p) = v; }
  static __device__ __forceinline__ void fma(T& a, float s, T v) { a.x = fmaf(s, v.x, a.x); a.y = fmaf(s, v.y, a.y); }
  static __device__ __forceinline__ float dot(T a, T b) { return fmaf(a.x, b.x, a.y * b.y); }
  static __device__ __forceinline__ T scaled(T a, float s) { return make_float2(a.x * s, a.y * s); }
};
template <int VW> __device__ __forceinline__ typename Vec<VW>::T lds_vec(const float* p);
template <> __device__ __forceinline__ float4 lds_vec<4>(const float* p) { return *reinterpret_cast<const float4*>(p); }
template <> __device__ __forceinline__ float2 lds_vec<2>(const float* p) { return *reinterpret_cast<const float2*>(p); }
template <> __device__ __forceinline__ float lds_vec<1>(const float* p) { return *p; }

struct StreamArgs {
  SpmmArgs s;
  // BINS only
  const float* Xrow;     // row-level operand of the per-edge dot (forward input X), leading dim ldr
  int64_t ldr;
  double* partials;      // [gridDim.x][R]
  int use_tma;           // rows are 16-byte aligned multiples of 16 bytes: stage the tile with cp.async.bulk
  float* xdx;            // optional [N]: <Xrow[u], dX[u]> per row (the source-side half of d_norm), or null
  // spmm_rowgroup_kernel<BINS> only: the norm gradient folded into the same pass (d_norm != null)
  //   d_norm[u] = ( [dn_sides&2] <Yfwd[u], G[u]> + [dn_sides&1] <Xrow[u], dX[u]> ) / norm[u]
  const float* Yfwd;     // forward result rows (leading dim ldyf)
  int64_t ldyf;
  const float* norm;     // the norm vector itself (divisor)
  int dn_sides;
  float* d_norm;
  // spmm_rowgroup_kernel only
  const int32_t* order;  // rows not covered by fragments, by descending slot count
  int64_t n_order;
  PeerRows peers;        // base != null: result rows go to the row blocks of their owner ranks (peer memory)
  float* Ylocal;         // forward scatter: optional local copy of the result slab (leading dim ldl)
  int64_t ldl;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  uint32_t done = 0;
  for (int spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    if (spin > (1 << 24)) __trap();  // never hang the GPU on a lost copy
  }
}

constexpr int kRowsPerItem = 32;      // rows per warp item, plain variant
constexpr int kRowsPerItemBins = 8;   // rows per warp item, BINS variant (bounds the shared-memory tile)

template <int C, int VW, bool BINS>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, (C <= 1 ? 4 : 1))
spmm_stream_kernel(StreamArgs sa) {
  using V = Vec<VW>;
  using T = typename V::T;
  constexpr int U = C == 1 ? (BINS ? 4 : 6) : Unroll<C>::U;  // 6 gathers x 32 warps/SM beat 8 x 24 (measured)
  constexpr int RB = BINS ? kRowsPerItemBins : kRowsPerItem;
  const SpmmArgs& a = sa.s;
  __shared__ float w_s[256];
  extern __shared__ __align__(16) unsigned char dsm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Fp = (a.F + 3) & ~3;  // tile row pitch (floats), keeps rows 16-byte aligned
  // dynamic smem (BINS): [warps] mbarrier | [warps][R] double scratch | [warps][R][32] bins | [warps][RB][Fp] tile
  uint64_t* bars = reinterpret_cast<uint64_t*>(dsm);
  double* scratch = reinterpret_cast<double*>(dsm + 64);
  float* bins = reinterpret_cast<float*>(scratch + kWarpsPerBlock * a.R);
  float* tiles = bins + (size_t)kWarpsPerBlock * a.R * 32;
  float* mytile = tiles + (size_t)warp * RB * Fp;
  float* mybins = bins + (size_t)warp * a.R * 32 + lane;
  uint64_t* mybar = bars + warp;
  if (a.etype != nullptr)
    for (int i = threadIdx.x; i < a.R; i += blockDim.x) w_s[i] = leaky(a.theta[i] * a.alpha, kRelationSlope);
  if (BINS) {
    for (int r = 0; r < a.R; ++r) mybins[r * 32] = 0.f;
    if (lane == 0) mbar_init(mybar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  bool col_ok[C];
#pragma unroll
  for (int k = 0; k < C; ++k) col_ok[k] = (lane + k * 32) * VW < a.F;
  const float* xcol = a.X + (size_t)lane * VW;
  const int64_t rows = a.row_end - a.row_begin;
  const int64_t nitems = a.nfrag_pad + (rows + RB - 1) / RB;
  const int64_t stride = BINS ? (int64_t)gridDim.x * kWarpsPerBlock : nitems;  // plain: one item per warp
  uint32_t phase = 0;

  for (int64_t wi = (int64_t)blockIdx.x * kWarpsPerBlock + warp; wi < nitems; wi += stride) {
    // ---- decode the item: a fragment of a long row, or a block of RB rows
    const bool is_frag = wi < a.nfrag_pad;
    int64_t r0 = 0;
    int nrows = 0, my_begin = 0, my_end = 0;
    if (is_frag) {
      if (wi < a.nfrag) {
        const int64_t v = a.frag_row[wi];
        if (v >= a.row_begin && v < a.row_end) {
          r0 = v;
          nrows = 1;
          my_begin = a.frag_begin[wi];
          my_end = my_begin + min(a.threshold, a.indptr[v + 1] - my_begin);
        }
      }
    } else {
      r0 = a.row_begin + (wi - a.nfrag_pad) * RB;
      nrows = (int)min((int64_t)RB, a.row_end - r0);
      if (lane < nrows) {
        my_begin = a.indptr[r0 + lane];
        my_end = a.indptr[r0 + lane + 1];
      }
    }
    if (nrows <= 0) continue;  // warp-uniform
    const float my_nd = (lane < nrows && a.norm_dst != nullptr) ? a.norm_dst[r0 + lane] : 1.f;
    const unsigned longmask = is_frag ? 0u : __ballot_sync(0xffffffffu, lane < nrows && my_end - my_begin > a.threshold);
    if (BINS) {  // stage the row-level tile (rows r0 .. r0+nrows-1 of Xrow) with TMA bulk copies
      __syncwarp();  // every lane is done reading the previous tile
      if (sa.use_tma) {
        if (lane == 0) {
          const uint32_t row_bytes = (uint32_t)a.F * 4u;
          mbar_expect_tx(mybar, row_bytes * (uint32_t)nrows);
          for (int r = 0; r < nrows; ++r)
            bulk_g2s(mytile + (size_t)r * Fp, sa.Xrow + (size_t)(r0 + r) * sa.ldr, row_bytes, mybar);
        }
      } else {  // odd widths / unaligned rows: plain coalesced copy
        for (int r = 0; r < nrows; ++r)
          for (int c = lane; c < a.F; c += 32) mytile[(size_t)r * Fp + c] = sa.Xrow[(size_t)(r0 + r) * sa.ldr + c];
        __syncwarp();
      }
    }
    bool tile_ready = !BINS || !sa.use_tma;

    int cur = 0;
    while (cur < nrows) {
      if ((longmask >> cur) & 1u) {  // long row: covered by fragments
        ++cur;
        continue;
      }
      const unsigned rest = longmask >> cur;
      const int seg_end = min(nrows, rest ? cur + __ffs(rest) - 1 : nrows);
      const int s_begin = __shfl_sync(0xffffffffu, my_begin, cur);
      const int s_end = __shfl_sync(0xffffffffu, my_end, seg_end - 1);
      int row = cur;
      int row_end_slot = __shfl_sync(0xffffffffu, my_end, row);
      float nd_cur = __shfl_sync(0xffffffffu, my_nd, row);
      T acc[C], trow[C];   // trow: the row-level tile slice of the current row (BINS), kept in registers
#pragma unroll
      for (int k = 0; k < C; ++k) acc[k] = trow[k] = V::zero();
      bool trow_valid = false;
      int cur_rel = 0;      // run-length accumulation of the relation bins: one shared-memory update per run
      float racc = 0.f;

      auto load_trow = [&]() {
        const float* tp = mytile + (size_t)row * Fp + (size_t)lane * VW;
#pragma unroll
        for (int k = 0; k < C; ++k) trow[k] = col_ok[k] ? lds_vec<VW>(tp + (size_t)k * 32 * VW) : V::zero();
        trow_valid = true;
      };
      auto flush = [&]() {
        if (BINS && sa.xdx != nullptr && !is_frag) {  // <X[u], dX[u]> while dX[u] is still in registers
          if (!trow_valid) load_trow();
          float d = 0.f;
#pragma unroll
          for (int k = 0; k < C; ++k) d += V::dot(acc[k], trow[k]);
          d = group_sum<32>(d) * nd_cur;
          if (lane == 0) sa.xdx[r0 + row] = d;
        }
        trow_valid = false;
        if (is_frag) {
          float* y = a.partial + (size_t)wi * a.F + (size_t)lane * VW;
#pragma unroll
          for (int k = 0; k < C; ++k)
            if (col_ok[k]) V::store(y + (size_t)k * 32 * VW, acc[k]);
        } else {
          float* y = a.Y + (size_t)(r0 + row) * a.ldy + (size_t)lane * VW;
#pragma unroll
          for (int k = 0; k < C; ++k)
            if (col_ok[k]) V::store(y + (size_t)k * 32 * VW, V::scaled(acc[k], nd_cur));
        }
#pragma unroll
        for (int k = 0; k < C; ++k) acc[k] = V::zero();
      };

      // prefetch of the first batch
      int nidx = 0, net = 0;
      float ncoef = 0.f, nns = 0.f;
      if (s_begin + lane < s_end) {
        const int s = s_begin + lane;
        nidx = a.indices[s];
        if (a.etype != nullptr) net = a.etype[s];
        nns = a.norm_src != nullptr ? __ldg(a.norm_src + nidx) : 1.f;
        ncoef = (a.etype != nullptr ? w_s[net] : 1.f) * nns;
      }
      for (int s = s_begin; s < s_end; s += 32) {
        const int idx = nidx, et = net;
        const float coef = ncoef, ns = nns;
        nidx = net = 0;
        ncoef = nns = 0.f;
        if (s + 32 + lane < s_end) {
          const int sn = s + 32 + lane;
          nidx = a.indices[sn];
          if (a.etype != nullptr) net = a.etype[sn];
          nns = a.norm_src != nullptr ? __ldg(a.norm_src + nidx) : 1.f;
          ncoef = (a.etype != nullptr ? w_s[net] : 1.f) * nns;
        }
        const int cnt = min(32, s_end - s);
        for (int j = 0; j < cnt; j += U) {
          int sidx[U];
          T x[U][C];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int jj = min(j + u, cnt - 1);
            sidx[u] = __shfl_sync(0xffffffffu, idx, jj);
#pragma unroll
            for (int k = 0; k < C; ++k)
              x[u][k] = (j + u < cnt && col_ok[k]) ? V::load(xcol + (size_t)sidx[u] * a.ldx + (size_t)k * 32 * VW)
                                                   : V::zero();
          }
          if (BINS && !tile_ready) {  // first use of the tile: the bulk copies had the index loads to hide behind
            mbar_wait(mybar, phase);
            phase ^= 1u;
            tile_ready = true;
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (j + u < cnt) {  // warp-uniform
              const int slot = s + j + u;
              while (slot >= row_end_slot) {  // crossed a row boundary (also walks over empty rows)
                flush();
                ++row;
                row_end_slot = __shfl_sync(0xffffffffu, my_end, row);
                nd_cur = __shfl_sync(0xffffffffu, my_nd, row);
              }
              const float sc = __shfl_sync(0xffffffffu, coef, j + u);
#pragma unroll
              for (int k = 0; k < C; ++k) V::fma(acc[k], sc, x[u][k]);
              if (BINS) {
                const float sb = __shfl_sync(0xffffffffu, ns, j + u) * nd_cur;
                const int se = __shfl_sync(0xffffffffu, et, j + u);
                if (!trow_valid) load_trow();
                float d = 0.f;
#pragma unroll
                for (int k = 0; k < C; ++k) d += V::dot(x[u][k], trow[k]);
                if (se != cur_rel) {  // warp-uniform: lane-local bin, fixed order, bank-conflict free
                  mybins[cur_rel * 32] += racc;
                  racc = 0.f;
                  cur_rel = se;
                }
                racc = fmaf(sb, d, racc);
              }
            }
          }
        }
      }
      if (BINS && !tile_ready) {  // segment without slots: the flush below still needs the tile
        mbar_wait(mybar, phase);
        phase ^= 1u;
        tile_ready = true;
      }
      while (row < seg_end) {  // last row of the segment + trailing empty rows
        flush();
        ++row;
        if (row < seg_end) nd_cur = __shfl_sync(0xffffffffu, my_nd, row);
      }
      if (BINS) mybins[cur_rel * 32] += racc;
      cur = seg_end;
    }
    if (BINS && !tile_ready) {  // item without a single short-row slot: still consume the barrier phase
      mbar_wait(mybar, phase);
      phase ^= 1u;
    }
  }
  if (BINS) reduce_bins(bins, scratch, a.R, sa.partials + (size_t)blockIdx.x * a.R);
}

// ---- rows of F <= 128 floats: lane-group SpMM over degree-sorted rows -----------------------------------
// A 128-bit chunk per lane covers a row of F floats with G = 4 / 8 / 16 / 32 lanes, so a warp works on
// 32/G rows at once -- one gather instruction fetches 32/G source rows (the column slabs of the
// feature-sliced multi-GPU scheme, hidden width 64 of the HGB models, the F = 128 headline workload).  Rows come from `order` (rows not
// covered by fragments, by descending slot count, built once per graph): neighbouring lane groups get
// rows of (nearly) equal length, so the warp-uniform trip count wastes almost nothing, and each row is
// summed by ONE lane group in slot order -- bit-identical to the whole-warp kernels, no cross-lane fold, no
// row-boundary bookkeeping.  Fragments of long rows (all `threshold` slots long) are the first items.
// BINS: as in spmm_stream_kernel, but the row-level operand Xrow[u] is one 128-bit register per lane.
// Occupancy beats loads per warp here as well (measured, MAG graph, F = 64 / 32 / 16 forward): 6 blocks/SM x 2
// gathers 1.07 / 0.57 / 0.37 ms, 4 x 4: 1.21 / 0.63 / 0.38, 3 x 8: 1.53 / 0.79 / 0.47.  F = 128 (whole warp per
// row): 8 x 2 2.05 ms, 6 x 2 2.10, 4 x 4 2.35 (the streaming kernel: 2.35); fused backward 4 x 4 2.73 (streaming 2.88).
#ifndef REGNN_RG_BLOCKS
#define REGNN_RG_BLOCKS (G == 32 ? 8 : 6)
#endif
#ifndef REGNN_RG_U
#define REGNN_RG_U 2
#endif
#ifndef REGNN_RGB_BLOCKS
#define REGNN_RGB_BLOCKS 4
#endif
#ifndef REGNN_RGB_U
#define REGNN_RGB_U 4
#endif
// Tried and dropped (round 2, measured on the MAG graph): the fused backward with 16 / 8 / 4 lanes x TWO 128-bit chunks
// per lane (twice the rows in flight per warp): 2.41 vs 2.43 ms at F = 128, 1.31 vs 1.19 at F = 64, 0.86 vs 0.72 at
// F = 32 -- no gain where it is equal, slower on narrow rows; 5 / 6 resident blocks per SM by capping registers at
// 48 / 40 (2.52 / 2.56 ms) and 3 blocks x 71 registers (2.91): 4 x 4 gathers stays.
// Two gathers per lane with more resident blocks (r3e, folded norm gradient, F = 128 / 64 / 16): 4 x 2 2.99 / 1.55 / 0.64 ms,
// 5 x 2 (48 registers) 3.14 / 1.46 / 0.64, 6 x 2 (40) 2.94 / 1.61 / 0.71, 8 x 2 (32, 40 B spilled) 2.96 / 1.61 / 0.78 against
// 4 x 4: 2.63 / 1.36 / 0.62.
// Also dropped (measured, r3a): decoding the item header ahead of time in the persistent backward (row id two iterations
// ahead, row pointers one ahead, the next row's slot arrays prefetched into L2 at the end of the current row; no spills
// at 64 registers): 2.95 vs 2.70 ms at F = 128 with the folded norm gradient, 1.54 vs 1.36 at F = 64, 0.74 vs 0.61 at
// F = 16 -- the extra loads ahead of every row's gathers cost more than the shorter per-row chain saves.
// Cooperative slot loads pay off where the kernel is issue-bound (fused backward: 2.73 -> 2.44 ms at F = 128,
// 1.37 -> 1.22 at 64, 0.53 -> 0.50 at 16); the forward kernel is HBM-bound and slightly faster without (2.05 vs 2.14).
// Dropped (r5a, measured, profiles/r5a_check_l2_hot.jsonl, one B200 at 1000 W): an L2 eviction policy meant to keep the
// most-gathered rows cached.  Per slot a uint8 gather count min(255, degree of the gathered row), loaded like the edge
// type; gathers of rows below a threshold (the hot set filling a budget of 32..112 MB) loaded evict-first
// (createpolicy.fractional.L2::evict_first + ld.global.nc.L2::cache_hint, predicated against a plain load because the
// policy is a warp-uniform descriptor operand), the index / edge-type / count loads, X[u] and the result stores
// evict-first too; no L2 set-aside.  Bit-identical, but every arm lost, MAG graph, forward / fused backward (DNORM):
// F = 128 plain 1.91 / 2.69 ms, streams demoted with every gather hot 2.42 / 2.89, budgets 32..112 MB 2.31..2.36 /
// 2.81..2.84; F = 64 plain 1.09 / 1.36, streams only 1.22 / 1.47, budgets 1.15..1.17 / 1.45.  The byte model put 22..38 %
// of the gathers in the hot set at F = 128 (30..56 % at F = 64); demoting the cold gathers won back 0.05..0.1 ms against
// the streams-only arm, far less than the hinted loads cost (the extra count load per slot, two predicated gathers, and
// at <false,32> 36 bytes of spill under the 32-register cap).  Hit rates were not measured (no profiler): inferred from
// time only.  Whole-step bench: 5.04..5.07 ms against 4.77..4.78 for the plain kernels.
#ifndef REGNN_RG_COOP
#define REGNN_RG_COOP BINS
#endif
template <bool BINS, int G, bool DNORM = false>   // DNORM (BINS only): the norm gradient is produced in the same pass
__global__ void __launch_bounds__(kWarpsPerBlock * 32, BINS ? REGNN_RGB_BLOCKS : REGNN_RG_BLOCKS)
spmm_rowgroup_kernel(StreamArgs sa) {
  static_assert(BINS || !DNORM, "the folded norm gradient belongs to the backward kernel");
  static_assert(G == 4 || G == 8 || G == 16 || G == 32, "lane groups of 4, 8, 16 or 32 lanes");
  constexpr int GPW = 32 / G;                          // rows per warp
  constexpr int U = BINS ? REGNN_RGB_U : REGNN_RG_U;   // gathers in flight per lane
  constexpr bool kCoop = REGNN_RG_COOP;
  const SpmmArgs& a = sa.s;
  __shared__ float w_s[256];
  extern __shared__ __align__(16) unsigned char dsm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G;
  // dynamic smem (BINS): [warps][R] double scratch | [warps][R][32] lane-local bins
  double* scratch = reinterpret_cast<double*>(dsm);
  float* bins = reinterpret_cast<float*>(scratch + kWarpsPerBlock * a.R);
  float* mybins = bins + (size_t)warp * a.R * 32 + lane;
  const bool weighted = a.etype != nullptr;
  if (weighted)
    for (int i = threadIdx.x; i < a.R; i += blockDim.x) w_s[i] = leaky(a.theta[i] * a.alpha, kRelationSlope);
  if (BINS)
    for (int r = 0; r < a.R; ++r) mybins[r * 32] = 0.f;
  __syncthreads();

  // lanes past the last column gather column 0 (same sectors as lane 0) and are masked at the stores
  const bool col_ok = lg * 4 < a.F;
  const char* xbytes = reinterpret_cast<const char*>(a.X + (col_ok ? lg : 0) * 4);
  const uint32_t ldxb = (uint32_t)a.ldx * 4u;  // row pitch in bytes: one IMAD.WIDE per gather
  const int64_t nitems = (int64_t)a.nfrag + sa.n_order;
  const int64_t nwork = (nitems + GPW - 1) / GPW;
  const int64_t stride = BINS ? (int64_t)gridDim.x * kWarpsPerBlock : nwork;  // plain: one item per warp

  for (int64_t wi = (int64_t)blockIdx.x * kWarpsPerBlock + warp; wi < nwork; wi += stride) {
    const int64_t vi = wi * GPW + grp;
    int64_t v = -1;
    int begin = 0, len = 0;
    const bool is_frag = vi < a.nfrag;
    if (vi < nitems) {
      if (is_frag) {
        v = a.frag_row[vi];
        begin = a.frag_begin[vi];
        len = min(a.threshold, a.indptr[v + 1] - begin);
      } else {
        v = sa.order[vi - a.nfrag];
        begin = a.indptr[v];
        len = a.indptr[v + 1] - begin;
      }
    }
    const int maxlen = __reduce_max_sync(0xffffffffu, len);
    const float nd = (v >= 0 && a.norm_dst != nullptr) ? a.norm_dst[v] : 1.f;
    float4 trow = make_float4(0.f, 0.f, 0.f, 0.f);
    if (BINS && v >= 0 && col_ok) trow = ldg4(sa.Xrow + (size_t)v * sa.ldr + lg * 4);
    // norm gradient, destination-side half: <Y[u], G[u]> of the row this lane group owns.  Fragments: long_row_dnorm_kernel.
    const bool want_ydg = DNORM && (sa.dn_sides & 2) && v >= 0 && col_ok && !is_frag;
    if constexpr (DNORM) {
      if (want_ydg) {  // into L2 now (no registers held), read after the gathers
        prefetch_l2(sa.Yfwd + (size_t)v * sa.ldyf + lg * 4);
        prefetch_l2(xbytes + (uint64_t)(uint32_t)v * ldxb);
      }
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int cur_rel = 0;
    float racc = 0.f;
    const int32_t* ip = a.indices + begin;
    const uint8_t* ep = a.etype + begin;

    if constexpr (kCoop) {
      // Cooperative slot loads: lane lg of a group holds slot t0+lg of the group's row (column index, edge type,
      // norm[src], coefficient) -- one coalesced load per G slots, broadcast inside the group by shuffles --
      // instead of every lane loading every slot's scalars.  The next batch is in flight behind the gathers.
      static_assert(G % U == 0, "a round must not straddle a slot batch");
      const int gbase = lane & ~(G - 1);
      auto load_batch = [&](int t0, int& bi, int& be, float& bn) {
        const int t = t0 + lg;
        bi = -1;
        be = 0;
        bn = 0.f;
        if (t < len) {
          bi = __ldg(ip + t);
          be = weighted ? (int)__ldg(ep + t) : 0;
          bn = a.norm_src != nullptr ? __ldg(a.norm_src + bi) : 1.f;
        }
      };
      int nbi, nbe;
      float nbn;
      load_batch(0, nbi, nbe, nbn);
      for (int t0 = 0; t0 < maxlen; t0 += G) {
        const int bi = nbi, be = nbe;
        const float bn = nbn;
        const float bc = (weighted ? w_s[be] : 1.f) * bn;  // 0 for a missing slot
        if (t0 + G < maxlen) load_batch(t0 + G, nbi, nbe, nbn);
        const int cnt = min(G, maxlen - t0);
        for (int j = 0; j < cnt; j += U) {
          float4 x[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int si = __shfl_sync(0xffffffffu, bi, gbase + j + u);
            x[u] = si >= 0 ? ldg4(reinterpret_cast<const float*>(xbytes + (uint64_t)(uint32_t)si * ldxb))
                           : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int from = gbase + j + u;
            fma4(acc, __shfl_sync(0xffffffffu, bc, from), x[u]);
            if (BINS) {
              const int se = __shfl_sync(0xffffffffu, be, from);
              const float sn = __shfl_sync(0xffffffffu, bn, from);
              const float d = dot4(x[u], trow);
              if (t0 + j + u < len && se != cur_rel) {  // lane-local bin, slot order, bank-conflict free
                mybins[cur_rel * 32] += racc;
                racc = 0.f;
                cur_rel = se;
              }
              racc = fmaf(sn * nd, d, racc);
            }
          }
        }
      }
    } else {
      int nidx[U], net[U];  // next round's column indices / edge types (-1 = no slot)
#pragma unroll
      for (int u = 0; u < U; ++u) {
        nidx[u] = u < len ? __ldg(ip + u) : -1;
        net[u] = (weighted && u < len) ? (int)__ldg(ep + u) : 0;
      }
      for (int t = 0; t < maxlen; t += U) {
        int idx[U], et[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          idx[u] = nidx[u];
          et[u] = net[u];
        }
        float4 x[U];
        float ns[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          // The gather and the norm[src] load test the slot separately on purpose: with one shared flag the two loads
          // become one branch, and at the 32-register cap of <false,32> (8 blocks/SM) ptxas spilled 28 bytes inside the
          // gather loop (552 instructions; 512 and no spill this way).  MAG, F = 128: 2.05 -> 1.89 ms (profiles/r5a_*).
          x[u] = idx[u] >= 0 ? ldg4(reinterpret_cast<const float*>(xbytes + (uint64_t)(uint32_t)idx[u] * ldxb))
                             : make_float4(0.f, 0.f, 0.f, 0.f);
          ns[u] = idx[u] >= 0 ? (a.norm_src != nullptr ? __ldg(a.norm_src + idx[u]) : 1.f) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {  // indices of the next round: in flight behind this round's gathers
          const int tn = t + U + u;
          nidx[u] = tn < len ? __ldg(ip + tn) : -1;
          net[u] = (weighted && tn < len) ? (int)__ldg(ep + tn) : 0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const float coef = (weighted ? w_s[et[u]] : 1.f) * ns[u];  // 0 for a missing slot
          fma4(acc, coef, x[u]);
          if (BINS) {
            const float d = dot4(x[u], trow);
            if (idx[u] >= 0 && et[u] != cur_rel) {  // lane-local bin, slot order, bank-conflict free
              mybins[cur_rel * 32] += racc;
              racc = 0.f;
              cur_rel = et[u];
            }
            racc = fmaf(ns[u] * nd, d, racc);
          }
        }
      }
    }
    if (BINS) {
      mybins[cur_rel * 32] += racc;
      if constexpr (DNORM) {  // the whole norm gradient of row u in this pass: no separate row-dot kernel
        float p = (sa.dn_sides & 1) ? dot4(acc, trow) * nd : 0.f;   // <X[u], dX[u]> while dX[u] is in registers
        if (want_ydg)
          p += dot4(ldg4(sa.Yfwd + (size_t)v * sa.ldyf + lg * 4),
                    ldg4(reinterpret_cast<const float*>(xbytes + (uint64_t)(uint32_t)v * ldxb)));
        p = group_sum<G>(p);
        if (lg == 0 && v >= 0 && !is_frag) sa.d_norm[v] = p / sa.norm[v];
      } else if (sa.xdx != nullptr) {  // <X[u], dX[u]> only (long rows: long_row_dnorm_kernel)
        const float d = group_sum<G>(dot4(acc, trow)) * nd;
        if (lg == 0 && v >= 0 && !is_frag) sa.xdx[v] = d;
      }
    }
    if (v >= 0 && col_ok) {
      if (is_frag) {
        st4(a.partial + (size_t)vi * a.F + lg * 4, acc);
      } else {
        scale4(acc, nd);
        float* yrow = sa.peers.base != nullptr ? sa.peers.row(v) : a.Y + (size_t)v * a.ldy;
        st4(yrow + lg * 4, acc);  // 64..256 contiguous bytes per row: a full NVLink write packet when remote
        if (!BINS && sa.peers.base != nullptr && sa.Ylocal != nullptr) st4(sa.Ylocal + (size_t)v * sa.ldl + lg * 4, acc);
      }
    }
  }
  if (BINS) reduce_bins(bins, scratch, a.R, sa.partials + (size_t)blockIdx.x * a.R);
}

// d_norm[v] = ( [sides&2] <Y[v],G[v]> + [sides&1] <X[v],dX[v]> ) / norm[v]   (pure streaming, row per warp).
// xdx != null supplies <X[v],dX[v]> (produced by the fused backward), so X and dX are not read again.
constexpr int kRowdotRows = 4;  // rows per warp: 2-4 x 4 independent 128-bit loads in flight per lane
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
rowdot_norm_kernel(const float* __restrict__ norm, int sides, const float* __restrict__ X, int64_t ldx,
                   const float* __restrict__ Y, int64_t ldy, const float* __restrict__ G, int64_t ldg,
                   const float* __restrict__ dX, int64_t lddx, const float* __restrict__ xdx, int F,
                   int64_t row_begin, int64_t row_end, float* __restrict__ d_norm) {
  const int lane = threadIdx.x & 31;
  const int64_t v0 = row_begin + ((int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5)) * kRowdotRows;
  if (v0 >= row_end) return;
  const bool use_x = (sides & 1) && xdx == nullptr;
  const bool vec = (F & 3) == 0 && ((ldy | ldg) & 3) == 0 && ((((uintptr_t)Y) | ((uintptr_t)G)) & 15) == 0 &&
                   (!use_x || (((ldx | lddx) & 3) == 0 && ((((uintptr_t)X) | ((uintptr_t)dX)) & 15) == 0));
  float p[kRowdotRows];
#pragma unroll
  for (int r = 0; r < kRowdotRows; ++r) p[r] = 0.f;
  if (vec) {
    for (int c = lane * 4; c < F; c += 128) {
#pragma unroll
      for (int r = 0; r < kRowdotRows; ++r) {
        const int64_t v = v0 + r;
        if (v < row_end) {
          if (sides & 2) p[r] += dot4(ldg4(Y + (size_t)v * ldy + c), ldg4(G + (size_t)v * ldg + c));
          if (use_x) p[r] += dot4(ldg4(X + (size_t)v * ldx + c), ldg4(dX + (size_t)v * lddx + c));
        }
      }
    }
  } else {
    for (int c = lane; c < F; c += 32) {
#pragma unroll
      for (int r = 0; r < kRowdotRows; ++r) {
        const int64_t v = v0 + r;
        if (v < row_end) {
          if (sides & 2) p[r] = fmaf(__ldg(Y + (size_t)v * ldy + c), __ldg(G + (size_t)v * ldg + c), p[r]);
          if (use_x) p[r] = fmaf(__ldg(X + (size_t)v * ldx + c), __ldg(dX + (size_t)v * lddx + c), p[r]);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < kRowdotRows; ++r) {
    const int64_t v = v0 + r;
    float t = group_sum<32>(p[r]);
    if (v < row_end && lane == 0) {
      if ((sides & 1) && xdx != nullptr) t += xdx[v];
      d_norm[v] = t / norm[v];
    }
  }
}

// The long rows' share of the norm gradient (their dX is only complete after the fragment finalize):
//   xdx[v] = <X[v], dX[v]>                                                         (xdx != null)
//   d_norm[v] = ( [sides&2] <Y[v], G[v]> + [sides&1] <X[v], dX[v]> ) / norm[v]      (d_norm != null)
__global__ void long_row_dnorm_kernel(const int32_t* __restrict__ long_rows, int num_long, const float* __restrict__ X,
                                      int64_t ldx, const float* __restrict__ dX, int64_t lddx, int F, int64_t row_begin,
                                      int64_t row_end, float* __restrict__ xdx, const float* __restrict__ Y, int64_t ldy,
                                      const float* __restrict__ Gd, int64_t ldg, const float* __restrict__ norm, int sides,
                                      float* __restrict__ d_norm) {
  const int lane = threadIdx.x & 31;
  const int l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (l >= num_long) return;
  const int64_t v = long_rows[l];
  if (v < row_begin || v >= row_end) return;
  float p = 0.f, q = 0.f;
  if (xdx != nullptr || (sides & 1))
    for (int c = lane; c < F; c += 32) p = fmaf(__ldg(X + (size_t)v * ldx + c), dX[(size_t)v * lddx + c], p);
  if (d_norm != nullptr && (sides & 2))
    for (int c = lane; c < F; c += 32) q = fmaf(__ldg(Y + (size_t)v * ldy + c), __ldg(Gd + (size_t)v * ldg + c), q);
  p = group_sum<32>(p);
  q = group_sum<32>(q);
  if (lane == 0) {
    if (xdx != nullptr) xdx[v] = p;
    if (d_norm != nullptr) d_norm[v] = (((sides & 1) ? p : 0.f) + q) / norm[v];
  }
}

struct SpmmBwdArgs {
  const int32_t* indptr;
  const int32_t* indices;
  const uint8_t* etype;
  int R;
  const float* norm;
  int sides;  // bit 0: source side scaled by norm, bit 1: destination side
  const float* X;  int64_t ldx;
  const float* Y;  int64_t ldy;
  const float* G;  int64_t ldg;
  const float* dX; int64_t lddx;
  int64_t row_begin, row_end;
  int F;
  double* partials;
  float* d_norm;
  const int32_t* frag_row;
  const int32_t* frag_begin;
  int nfrag, threshold;
};

// Destination-major pass: d_norm rows and (WEIGHTED) the per-relation sums of
// norm[src]*norm[dst]*<X[src], G[dst]>.  Persistent grid; each warp walks work items (fragments of
// long rows first, then ordinary rows) in a fixed order.  The row-local d_norm is produced by the
// item that starts the row.
template <int G, int C, int VW, bool WEIGHTED>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
spmm_bwd_w_kernel(SpmmBwdArgs a) {
  using V = Vec<VW>;
  using T = typename V::T;
  constexpr int U = Unroll<C>::U;
  constexpr int GPW = 32 / G;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* scratch = reinterpret_cast<double*>(smem_raw);                      // [warps][R]
  float* bins = reinterpret_cast<float*>(scratch + kWarpsPerBlock * a.R);     // [warps][R][32]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G;
  float* mybins = bins + (size_t)warp * a.R * 32 + lane;
  if (WEIGHTED)
    for (int r = 0; r < a.R; ++r) mybins[r * 32] = 0.f;

  bool col_ok[C];
#pragma unroll
  for (int k = 0; k < C; ++k) col_ok[k] = (lg + k * G) * VW < a.F;
  const int64_t rows = a.row_end - a.row_begin;
  const int64_t nfrag_groups = (a.nfrag + GPW - 1) / GPW;
  const int64_t ngroups = nfrag_groups + (rows + GPW - 1) / GPW;

  for (int64_t rg = (int64_t)blockIdx.x * kWarpsPerBlock + warp; rg < ngroups;
       rg += (int64_t)gridDim.x * kWarpsPerBlock) {
    bool row_ok = false, first = true;
    int64_t v = 0;
    int s0 = 0, len = 0;
    if (rg < nfrag_groups) {
      const int64_t fi = rg * GPW + grp;
      if (fi < a.nfrag) {
        v = a.frag_row[fi];
        if (v >= a.row_begin && v < a.row_end) {
          s0 = a.frag_begin[fi];
          len = min(a.threshold, a.indptr[v + 1] - s0);
          first = s0 == a.indptr[v];
          row_ok = true;
        }
      }
    } else {
      v = a.row_begin + (rg - nfrag_groups) * GPW + grp;
      if (v < a.row_end) {
        s0 = a.indptr[v];
        len = a.indptr[v + 1] - s0;
        row_ok = len <= a.threshold;
        if (!row_ok) len = 0;
      }
    }
    float nv = 1.f;
    T g[C];
    float p = 0.f;
    if (row_ok) nv = a.norm != nullptr ? a.norm[v] : 1.f;
#pragma unroll
    for (int k = 0; k < C; ++k) {
      g[k] = V::zero();
      if (row_ok && col_ok[k]) {
        const size_t c = (size_t)(lg + k * G) * VW;
        g[k] = V::load(a.G + (size_t)v * a.ldg + c);
        if (first && a.d_norm != nullptr) {
          if (a.sides & 2) p += V::dot(V::load(a.Y + (size_t)v * a.ldy + c), g[k]);
          if (a.sides & 1) p += V::dot(V::load(a.X + (size_t)v * a.ldx + c), V::load(a.dX + (size_t)v * a.lddx + c));
        }
      }
    }
    p = group_sum<G>(p);
    if (row_ok && first && lg == 0 && a.d_norm != nullptr) a.d_norm[v] = p / nv;

    if (WEIGHTED) {
#pragma unroll
      for (int k = 0; k < C; ++k) g[k] = V::scaled(g[k], (a.sides & 2) ? nv : 1.f);
      const int maxlen = (G == 32) ? len : warp_max_int(len);
      const float* xcol = a.X + (size_t)lg * VW;
      const bool src_scaled = a.norm != nullptr && (a.sides & 1);
      int nidx = 0, net = 0;
      float nns = 0.f;
      if (lg < len) {
        const int s = s0 + lg;
        nidx = a.indices[s];
        net = a.etype[s];
        nns = src_scaled ? __ldg(a.norm + nidx) : 1.f;
      }
      for (int base = 0; base < maxlen; base += G) {
        const int idx = nidx, et = net;
        const float ns = nns;
        nidx = net = 0;
        nns = 0.f;
        if (base + G + lg < len) {
          const int s = s0 + base + G + lg;
          nidx = a.indices[s];
          net = a.etype[s];
          nns = src_scaled ? __ldg(a.norm + nidx) : 1.f;
        }
        const int cnt = min(G, maxlen - base);
        for (int j = 0; j < cnt; j += U) {
          int sidx[U], set[U];
          float sn[U];
          T x[U][C];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int jj = min(j + u, G - 1);
            sidx[u] = __shfl_sync(0xffffffffu, idx, jj, G);
            set[u] = __shfl_sync(0xffffffffu, et, jj, G);
            sn[u] = __shfl_sync(0xffffffffu, ns, jj, G);
            const bool valid = base + j + u < len && j + u < G;
            if (!valid) sn[u] = 0.f;
#pragma unroll
            for (int k = 0; k < C; ++k)
              x[u][k] = (valid && col_ok[k]) ? V::load(xcol + (size_t)sidx[u] * a.ldx + (size_t)k * G * VW)
                                             : V::zero();
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            float d = 0.f;
#pragma unroll
            for (int k = 0; k < C; ++k) d += V::dot(x[u][k], g[k]);
            mybins[set[u] * 32] += sn[u] * d;  // lane-local bin: fixed order, conflict-free
          }
        }
      }
    }
  }
  if (WEIGHTED) reduce_bins(bins, scratch, a.R, a.partials + (size_t)blockIdx.x * a.R);
}

// ---- relation-weighted in-degree norm ------------------------------------------------------------
// clamp_min > 0: max(deg, clamp_min)^q (REGraphConv & co. use 1).  clamp_min <= 0: deg^q with no clamp and 0 for
// deg == 0 (rows without in-edges; the mean/add aggregators of the MAG stack, mag/regnn_saint.py:254-258).
// d deg = [deg >= clamp_min] * q * max(deg, clamp_min)^(q-1) * d_norm  (clamp passes the gradient at equality:
// PyTorch semantics); without a clamp every non-empty row passes.
__device__ __forceinline__ float ddeg_from(float d, float exponent, float clamp_min, float dn) {
  if (clamp_min > 0.f) return d >= clamp_min ? exponent * powf(fmaxf(d, clamp_min), exponent - 1.f) * dn : 0.f;
  return d != 0.f ? exponent * powf(d, exponent - 1.f) * dn : 0.f;
}
__device__ __forceinline__ float norm_from_deg(float deg, float exponent, float clamp_min) {
  if (clamp_min <= 0.f && deg == 0.f) return 0.f;
  const float c = clamp_min > 0.f ? fmaxf(deg, clamp_min) : deg;
  if (exponent == -0.5f) return 1.f / sqrtf(c);
  if (exponent == -1.f) return 1.f / c;
  return powf(c, exponent);
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
wdeg_norm_fwd_kernel(const int32_t* __restrict__ indptr, const uint8_t* __restrict__ etype,
                     const float* __restrict__ theta, float alpha, int R, float exponent, float clamp_min,
                     int64_t row_begin, int64_t row_end, float* __restrict__ deg,
                     float* __restrict__ norm) {
  constexpr int G = 8;
  __shared__ float w_s[256];
  for (int i = threadIdx.x; i < R; i += blockDim.x) w_s[i] = leaky(theta[i] * alpha, kRelationSlope);
  __syncthreads();
  const int lg = threadIdx.x % G;
  const int64_t v = row_begin + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
  float acc = 0.f;
  if (v < row_end) {
    const int s1 = indptr[v + 1];
    for (int s = indptr[v] + lg; s < s1; s += G) acc += w_s[etype[s]];
  }
  acc = group_sum<G>(acc);
  if (v < row_end && lg == 0) {
    if (deg != nullptr) deg[v] = acc;
    norm[v] = norm_from_deg(acc, exponent, clamp_min);
  }
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
wdeg_norm_bwd_kernel(const int32_t* __restrict__ indptr, const uint8_t* __restrict__ etype, int R,
                     float exponent, float clamp_min, int64_t row_begin, int64_t row_end,
                     const float* __restrict__ deg, const float* __restrict__ d_norm,
                     double* __restrict__ partials) {
  constexpr int G = 8, GPW = 32 / G;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* scratch = reinterpret_cast<double*>(smem_raw);
  float* bins = reinterpret_cast<float*>(scratch + kWarpsPerBlock * R);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G;
  float* mybins = bins + (size_t)warp * R * 32 + lane;
  for (int r = 0; r < R; ++r) mybins[r * 32] = 0.f;
  const int64_t rows = row_end - row_begin;
  const int64_t ngroups = (rows + GPW - 1) / GPW;
  for (int64_t rg = (int64_t)blockIdx.x * kWarpsPerBlock + warp; rg < ngroups;
       rg += (int64_t)gridDim.x * kWarpsPerBlock) {
    const int64_t v = row_begin + rg * GPW + grp;
    if (v < row_end) {
      const float d = deg[v];
      // clamp(min=1) passes the gradient at deg == 1 (PyTorch semantics)
      const float dd = ddeg_from(d, exponent, clamp_min, d_norm[v]);
      const int s1 = indptr[v + 1];
      for (int s = indptr[v] + lg; s < s1; s += G) mybins[etype[s] * 32] += dd;
    }
  }
  reduce_bins(bins, scratch, R, partials + (size_t)blockIdx.x * R);
}

// ---- slot-parallel variants of the two norm kernels (R <= 32) ----------------------------------------
// A warp owns a block of 32 consecutive rows and strides its 32 lanes over the block's concatenated
// slot range, so a hub row with 1e4-1e5 in-edges costs the same per slot as any other row.  The row of
// a slot is found by a 5-step binary search over the block's row ends (shared memory).
// Forward: integer per-(row, relation) counts (shared-memory integer atomics: order-free and exact),
// then deg[v] = sum_r count[v][r] * w[r] in relation order.  Backward: lane-local relation bins.
constexpr int kWdegRows = 32;

__device__ __forceinline__ int row_of_slot(const int* ends, int nrows, int s) {
  int lo = 0, hi = nrows - 1;  // first row whose end is > s
#pragma unroll
  for (int it = 0; it < 5; ++it) {
    const int mid = (lo + hi) >> 1;
    if (lo < hi) {
      if (ends[mid] > s) hi = mid; else lo = mid + 1;
    }
  }
  return lo;
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
wdeg_norm_fwd_slot_kernel(const int32_t* __restrict__ indptr, const uint8_t* __restrict__ etype,
                          const float* __restrict__ theta, float alpha, int R, float exponent, float clamp_min,
                          int64_t row_begin, int64_t row_end, float* __restrict__ deg,
                          float* __restrict__ norm) {
  __shared__ float w_s[32];
  __shared__ int ends_s[kWarpsPerBlock][kWdegRows];
  __shared__ int cnt_s[kWarpsPerBlock][kWdegRows * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < R) w_s[threadIdx.x] = leaky(theta[threadIdx.x] * alpha, kRelationSlope);
  __syncthreads();
  const int64_t r0 = row_begin + ((int64_t)blockIdx.x * kWarpsPerBlock + warp) * kWdegRows;
  if (r0 >= row_end) return;
  const int nrows = (int)min((int64_t)kWdegRows, row_end - r0);
  int my_begin = 0, my_end = 0;
  if (lane < nrows) {
    my_begin = indptr[r0 + lane];
    my_end = indptr[r0 + lane + 1];
    ends_s[warp][lane] = my_end;
  }
  int* cnt = cnt_s[warp];
  for (int i = lane; i < nrows * R; i += 32) cnt[i] = 0;
  const int s_begin = __shfl_sync(0xffffffffu, my_begin, 0);
  const int s_end = __shfl_sync(0xffffffffu, my_end, nrows - 1);
  __syncwarp();
  for (int s = s_begin + lane; s < s_end; s += 32)
    atomicAdd(&cnt[row_of_slot(ends_s[warp], nrows, s) * R + etype[s]], 1);
  __syncwarp();
  if (lane < nrows) {
    float d = 0.f;
    for (int r = 0; r < R; ++r) d = fmaf((float)cnt[lane * R + r], w_s[r], d);
    if (deg != nullptr) deg[r0 + lane] = d;
    norm[r0 + lane] = norm_from_deg(d, exponent, clamp_min);
  }
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
wdeg_norm_bwd_slot_kernel(const int32_t* __restrict__ indptr, const uint8_t* __restrict__ etype, int R,
                          float exponent, float clamp_min, int64_t row_begin, int64_t row_end,
                          const float* __restrict__ deg, const float* __restrict__ d_norm,
                          double* __restrict__ partials) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* scratch = reinterpret_cast<double*>(smem_raw);
  float* bins = reinterpret_cast<float*>(scratch + kWarpsPerBlock * R);
  __shared__ int ends_s[kWarpsPerBlock][kWdegRows];
  __shared__ float dd_s[kWarpsPerBlock][kWdegRows];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* mybins = bins + (size_t)warp * R * 32 + lane;
  for (int r = 0; r < R; ++r) mybins[r * 32] = 0.f;
  const int64_t nblocks = (row_end - row_begin + kWdegRows - 1) / kWdegRows;
  for (int64_t b = (int64_t)blockIdx.x * kWarpsPerBlock + warp; b < nblocks; b += (int64_t)gridDim.x * kWarpsPerBlock) {
    const int64_t r0 = row_begin + b * kWdegRows;
    const int nrows = (int)min((int64_t)kWdegRows, row_end - r0);
    int my_begin = 0, my_end = 0;
    __syncwarp();
    if (lane < nrows) {
      my_begin = indptr[r0 + lane];
      my_end = indptr[r0 + lane + 1];
      ends_s[warp][lane] = my_end;
      const float d = deg[r0 + lane];
      // clamp(min=1) passes the gradient at deg == 1 (PyTorch semantics)
      dd_s[warp][lane] = ddeg_from(d, exponent, clamp_min, d_norm[r0 + lane]);
    }
    const int s_begin = __shfl_sync(0xffffffffu, my_begin, 0);
    const int s_end = __shfl_sync(0xffffffffu, my_end, nrows - 1);
    __syncwarp();
    for (int s = s_begin + lane; s < s_end; s += 32)
      mybins[etype[s] * 32] += dd_s[warp][row_of_slot(ends_s[warp], nrows, s)];
  }
  reduce_bins(bins, scratch, R, partials + (size_t)blockIdx.x * R);
}

// ---- count-based variants of the two norm kernels ----------------------------------------------------
// cnt[v][r] = number of in-edges of v with relation r is a property of the graph, not of the parameters:
// it is built once per (graph, e_feat) by relation_count_kernel (integer atomics: exact, order-free).
// Then deg[v] = sum_r cnt[v][r]*w[r] and d w[r] = sum_v d_deg[v]*cnt[v][r] are dense streaming passes over
// an [N,R] int32 matrix -- no per-edge work and no sensitivity to hub rows on the per-step path.
__global__ void relation_count_kernel(const int32_t* __restrict__ row, const uint8_t* __restrict__ etype,
                                      int64_t num_edges, int R, int32_t* __restrict__ cnt) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < num_edges) atomicAdd(&cnt[(size_t)row[s] * R + etype[s]], 1);
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
wdeg_norm_fwd_cnt_kernel(const int32_t* __restrict__ cnt, const float* __restrict__ theta, float alpha, int R,
                         float exponent, float clamp_min, int64_t row_begin, int64_t row_end, float* __restrict__ deg,
                         float* __restrict__ norm) {
  __shared__ float w_s[256];
  for (int i = threadIdx.x; i < R; i += blockDim.x) w_s[i] = leaky(theta[i] * alpha, kRelationSlope);
  __syncthreads();
  const int64_t v = row_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= row_end) return;
  const int32_t* c = cnt + (size_t)v * R;
  float d = 0.f;
  for (int r = 0; r < R; ++r) d = fmaf((float)__ldg(c + r), w_s[r], d);
  if (deg != nullptr) deg[v] = d;
  norm[v] = norm_from_deg(d, exponent, clamp_min);
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
wdeg_norm_bwd_cnt_kernel(const int32_t* __restrict__ cnt, int R, float exponent, float clamp_min, int64_t row_begin,
                         int64_t row_end, const float* __restrict__ deg, const float* __restrict__ d_norm,
                         double* __restrict__ partials) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* scratch = reinterpret_cast<double*>(smem_raw);
  float* bins = reinterpret_cast<float*>(scratch + kWarpsPerBlock * R);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* mybins = bins + (size_t)warp * R * 32 + lane;
  for (int r = 0; r < R; ++r) mybins[r * 32] = 0.f;
  for (int64_t v = row_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < row_end;
       v += (int64_t)gridDim.x * blockDim.x) {
    const float d = deg[v];
    // clamp(min=1) passes the gradient at deg == 1 (PyTorch semantics)
    const float dd = ddeg_from(d, exponent, clamp_min, d_norm[v]);
    const int32_t* c = cnt + (size_t)v * R;
    for (int r = 0; r < R; ++r) mybins[r * 32] = fmaf(dd, (float)__ldg(c + r), mybins[r * 32]);
  }
  reduce_bins(bins, scratch, R, partials + (size_t)blockIdx.x * R);
}

// ---- dispatch ---------------------------------------------------------------------------------------
static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

struct Shape { int G, C, VW; };

// Picks lanes-per-row G, 128-bit (or scalar) chunks per lane C.  Returns false if F is too wide.
static bool pick_shape(int F, bool vec_ok, Shape* s) {
  if (vec_ok && F % 4 == 0) {
    const int f4 = F / 4;
    int G = 32;
    if (f4 <= 4) G = 4;
    else if (f4 <= 8) G = 8;
    else if (f4 <= 16) G = 16;
    else if (f4 % 32 != 0 && f4 % 16 == 0 && f4 / 16 <= 3) G = 16;  // e.g. F=192: 16 lanes x 3
    int C = (f4 + G - 1) / G;
    if (C > 8) return false;
    if (C > 4) C = 8;
    *s = {G, C, 4};
    return true;
  }
  int G = 32;
  if (F <= 4) G = 4;
  else if (F <= 8) G = 8;
  else if (F <= 16) G = 16;
  int C = (F + G - 1) / G;
  if (C > 8) return false;
  if (C > 4) C = 8;
  *s = {G, C, 1};
  return true;
}

#define REGNN_DISPATCH_GC(G_, C_, VW_, CALL)                    \
  if (sh.G == G_ && sh.C == C_ && sh.VW == VW_) {               \
    constexpr int G = G_, C = C_, VW = VW_;                     \
    CALL;                                                       \
    launched = true;                                            \
  }
#define REGNN_DISPATCH_SHAPES(CALL)                                                            \
  REGNN_DISPATCH_GC(4, 1, 4, CALL) REGNN_DISPATCH_GC(8, 1, 4, CALL) REGNN_DISPATCH_GC(16, 1, 4, CALL) \
  REGNN_DISPATCH_GC(16, 3, 4, CALL)                                                            \
  REGNN_DISPATCH_GC(32, 1, 4, CALL) REGNN_DISPATCH_GC(32, 2, 4, CALL) REGNN_DISPATCH_GC(32, 3, 4, CALL) \
  REGNN_DISPATCH_GC(32, 4, 4, CALL) REGNN_DISPATCH_GC(32, 8, 4, CALL)                          \
  REGNN_DISPATCH_GC(4, 1, 1, CALL) REGNN_DISPATCH_GC(8, 1, 1, CALL) REGNN_DISPATCH_GC(16, 1, 1, CALL) \
  REGNN_DISPATCH_GC(32, 1, 1, CALL) REGNN_DISPATCH_GC(32, 2, 1, CALL) REGNN_DISPATCH_GC(32, 3, 1, CALL) \
  REGNN_DISPATCH_GC(32, 4, 1, CALL) REGNN_DISPATCH_GC(32, 8, 1, CALL)

}  // namespace regnn

using namespace regnn;

extern "C" int regnn_relation_counts(const int32_t* row, const uint8_t* etype_csr, int64_t num_edges,
                                     int64_t num_nodes, int num_relations, int32_t* counts, void* stream) {
  REGNN_REQUIRE(counts && (num_edges == 0 || (row && etype_csr)), REGNN_ERR_INVALID_ARG, "relation_counts: null pointer");
  REGNN_REQUIRE(num_relations >= 1 && num_relations <= REGNN_MAX_RELATIONS, REGNN_ERR_UNSUPPORTED_SHAPE,
                "num_relations=%d outside [1,%d]", num_relations, REGNN_MAX_RELATIONS);
  cudaMemsetAsync(counts, 0, (size_t)num_nodes * num_relations * sizeof(int32_t), (cudaStream_t)stream);
  if (num_edges > 0)
    relation_count_kernel<<<(unsigned)((num_edges + 255) / 256), 256, 0, (cudaStream_t)stream>>>(row, etype_csr, num_edges,
                                                                                               num_relations, counts);
  return check_launch("regnn_relation_counts");
}

extern "C" int regnn_wdeg_norm_fwd(const int32_t* indptr, const uint8_t* etype_csr, const int32_t* counts,
                                   const float* theta, float alpha, int num_relations,
                                   float exponent, float clamp_min, int64_t row_begin, int64_t row_end, float* deg,
                                   float* norm, void* stream) {
  REGNN_REQUIRE(theta && norm && (counts || (indptr && etype_csr)), REGNN_ERR_INVALID_ARG, "wdeg_norm_fwd: null pointer");
  REGNN_REQUIRE(num_relations >= 1 && num_relations <= REGNN_MAX_RELATIONS, REGNN_ERR_UNSUPPORTED_SHAPE,
                "num_relations=%d outside [1,%d]", num_relations, REGNN_MAX_RELATIONS);
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "wdeg_norm_fwd: empty/negative row range");
  if (rows == 0) return REGNN_OK;
  const int threads = kWarpsPerBlock * 32;
  if (counts != nullptr) {
    wdeg_norm_fwd_cnt_kernel<<<(unsigned)((rows + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        counts, theta, alpha, num_relations, exponent, clamp_min, row_begin, row_end, deg, norm);
  } else if (num_relations <= 32) {
    const int64_t blocks = (rows + kWarpsPerBlock * kWdegRows - 1) / (kWarpsPerBlock * kWdegRows);
    wdeg_norm_fwd_slot_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
        indptr, etype_csr, theta, alpha, num_relations, exponent, clamp_min, row_begin, row_end, deg, norm);
  } else {
    const int64_t blocks = (rows * 8 + threads - 1) / threads;
    wdeg_norm_fwd_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
        indptr, etype_csr, theta, alpha, num_relations, exponent, clamp_min, row_begin, row_end, deg, norm);
  }
  return check_launch("regnn_wdeg_norm_fwd");
}

static size_t bins_smem_bytes(int R) { return (size_t)kWarpsPerBlock * R * (sizeof(double) + 32 * sizeof(float)); }

extern "C" int regnn_wdeg_norm_bwd(const int32_t* indptr, const uint8_t* etype_csr, const int32_t* counts,
                                   const float* theta, float alpha, int num_relations,
                                   float exponent, float clamp_min, int64_t row_begin, int64_t row_end,
                                   const float* deg, const float* d_norm, double* partials,
                                   float* d_theta, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE((counts || (indptr && etype_csr)) && theta && deg && d_norm && partials && d_theta,
                REGNN_ERR_INVALID_ARG, "wdeg_norm_bwd: null pointer");
  const int R = num_relations;
  REGNN_REQUIRE(R >= 1 && R <= REGNN_MAX_RELATIONS, REGNN_ERR_UNSUPPORTED_SHAPE, "num_relations=%d outside [1,%d]", R,
                REGNN_MAX_RELATIONS);
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "wdeg_norm_bwd: negative row range");
  const int nb = partial_blocks(rows);
  const size_t smem = bins_smem_bytes(R);
  // the opt-in to > 48 KB of dynamic shared memory (R >= 46) is per kernel: set it on the one that is launched
  int rc = REGNN_OK;
  if (counts != nullptr) {
    if ((rc = set_smem(wdeg_norm_bwd_cnt_kernel, smem)) != REGNN_OK) return rc;
    wdeg_norm_bwd_cnt_kernel<<<nb, kWarpsPerBlock * 32, smem, stream>>>(counts, R, exponent, clamp_min, row_begin, row_end, deg,
                                                                         d_norm, partials);
  } else if (R <= 32) {
    if ((rc = set_smem(wdeg_norm_bwd_slot_kernel, smem)) != REGNN_OK) return rc;
    wdeg_norm_bwd_slot_kernel<<<nb, kWarpsPerBlock * 32, smem, stream>>>(indptr, etype_csr, R, exponent, clamp_min, row_begin,
                                                                          row_end, deg, d_norm, partials);
  } else {
    if ((rc = set_smem(wdeg_norm_bwd_kernel, smem)) != REGNN_OK) return rc;
    wdeg_norm_bwd_kernel<<<nb, kWarpsPerBlock * 32, smem, stream>>>(indptr, etype_csr, R, exponent, clamp_min,
                                                                     row_begin, row_end, deg, d_norm, partials);
  }
  launch_relation_grad_finalize(partials, nb, R, R, theta, alpha, d_theta, stream);
  return check_launch("regnn_wdeg_norm_bwd");
}

struct StreamShape { int C, VW; };

static bool aligned_to(const void* p, int bytes) { return ((uintptr_t)p & (bytes - 1)) == 0; }

// Vector width and 32-lane chunks per row for the streaming kernels.  `align` = largest power of two
// (<= 16 bytes) dividing every base pointer and leading dimension (in bytes).
static bool pick_stream_shape(int F, int align, StreamShape* sh) {
  int VW = 1;
  if (align >= 16 && F % 4 == 0 && F >= 96) VW = 4;
  else if (align >= 8 && F % 2 == 0 && F >= 34) VW = 2;
  int C = (F + 32 * VW - 1) / (32 * VW);
  if (C > 8) {
    if (VW == 1 && align >= 8 && F % 2 == 0) { VW = 2; C = (F + 63) / 64; }
    if (C > 8 && align >= 16 && F % 4 == 0) { VW = 4; C = (F + 127) / 128; }
    if (C > 8) return false;
  }
  if (C > 4) C = 8;
  *sh = {C, VW};
  return true;
}

static int common_align(std::initializer_list<const void*> ptrs, std::initializer_list<int64_t> lds) {
  int al = 16;
  for (const void* p : ptrs)
    while (p != nullptr && al > 4 && !aligned_to(p, al)) al >>= 1;
  for (int64_t ld : lds)
    while (al > 4 && (ld * 4) % al != 0) al >>= 1;
  return al;
}

#define REGNN_STREAM_CASE(C_, VW_, BINS_, CALL)     \
  if (sh.C == C_ && sh.VW == VW_) {                 \
    constexpr int C = C_, VW = VW_;                 \
    constexpr bool BINS = BINS_;                    \
    CALL;                                           \
    launched = true;                                \
  }
#define REGNN_STREAM_DISPATCH(BINS_, CALL)                                                          \
  REGNN_STREAM_CASE(1, 4, BINS_, CALL) REGNN_STREAM_CASE(2, 4, BINS_, CALL) REGNN_STREAM_CASE(3, 4, BINS_, CALL) \
  REGNN_STREAM_CASE(4, 4, BINS_, CALL) REGNN_STREAM_CASE(8, 4, BINS_, CALL)                          \
  REGNN_STREAM_CASE(1, 2, BINS_, CALL) REGNN_STREAM_CASE(2, 2, BINS_, CALL) REGNN_STREAM_CASE(3, 2, BINS_, CALL) \
  REGNN_STREAM_CASE(4, 2, BINS_, CALL) REGNN_STREAM_CASE(8, 2, BINS_, CALL)                          \
  REGNN_STREAM_CASE(1, 1, BINS_, CALL) REGNN_STREAM_CASE(2, 1, BINS_, CALL) REGNN_STREAM_CASE(3, 1, BINS_, CALL) \
  REGNN_STREAM_CASE(4, 1, BINS_, CALL) REGNN_STREAM_CASE(8, 1, BINS_, CALL)

// Lane-group width of spmm_rowgroup_kernel for this call, or 0 when the whole-warp kernels must run: needs the
// degree-sorted row order (which lists the rows of the FULL range), F <= 128 in whole 128-bit chunks, 16-byte rows.
#ifndef REGNN_RG_MAXF
#define REGNN_RG_MAXF 128  // one 128-bit chunk per lane: up to a whole warp per row
#endif
static int rowgroup_lanes(int F, const int32_t* order, int64_t row_begin, int align) {
  if (order == nullptr || row_begin != 0 || F > REGNN_RG_MAXF || F % 4 != 0 || align < 16) return 0;
  return F > 64 ? 32 : (F > 32 ? 16 : (F > 16 ? 8 : 4));
}
#define REGNN_ROWGROUP_CASE(G_, BINS_, CALL) \
  if (G == G_) {                             \
    constexpr int GL = G_;                   \
    constexpr bool BINS = BINS_;             \
    CALL;                                    \
    launched = true;                         \
  }
#define REGNN_ROWGROUP_DISPATCH(BINS_, CALL)                                                               \
  REGNN_ROWGROUP_CASE(32, BINS_, CALL) REGNN_ROWGROUP_CASE(16, BINS_, CALL) REGNN_ROWGROUP_CASE(8, BINS_, CALL) \
  REGNN_ROWGROUP_CASE(4, BINS_, CALL)


static int fill_split(SpmmArgs& a, const regnn_rowsplit_t* split, float* ws, const char* who) {
  a.frag_row = a.frag_begin = nullptr;
  a.nfrag = a.nfrag_pad = 0;
  a.threshold = 0x7fffffff;
  a.partial = ws;
  if (split == nullptr || split->num_frags <= 0) return REGNN_OK;
  REGNN_REQUIRE(ws && split->long_rows && split->frag_ptr && split->frag_row && split->frag_begin && split->threshold > 0,
                REGNN_ERR_INVALID_ARG, "%s: incomplete row split", who);
  a.frag_row = split->frag_row;
  a.frag_begin = split->frag_begin;
  a.nfrag = split->num_frags;
  a.nfrag_pad = (a.nfrag + kWarpsPerBlock - 1) / kWarpsPerBlock * kWarpsPerBlock;
  a.threshold = split->threshold;
  return REGNN_OK;
}

// Validates a regnn_peer_rows_t and turns it into the device-side struct (base == null: no scatter).
static int fill_peers(PeerRows* out, const regnn_peer_rows_t* peers, int feat, int64_t rows, const char* who) {
  *out = PeerRows{nullptr, 1u, 0, 0};
  if (peers == nullptr) return REGNN_OK;
  REGNN_REQUIRE(peers->base != nullptr && peers->num_ranks >= 1 && peers->rows_per_rank >= 1 &&
                    peers->rows_per_rank < (1ll << 31) && rows <= peers->rows_per_rank * peers->num_ranks &&
                    peers->col_offset >= 0 && peers->col_offset % 4 == 0 && peers->ld % 4 == 0 &&
                    peers->ld >= peers->col_offset + feat,
                REGNN_ERR_INVALID_ARG, "%s: bad peer row-block table", who);
  *out = PeerRows{peers->base, (uint32_t)peers->rows_per_rank, peers->ld, peers->col_offset};
  return REGNN_OK;
}

static int spmm_fwd_impl(const int32_t* indptr, const int32_t* indices, const uint8_t* etype,
                         const float* theta, float alpha, int num_relations,
                         const float* norm_src, const float* norm_dst, const float* X,
                         int64_t ldx, float* Y, int64_t ldy, int64_t row_begin,
                         int64_t row_end, int feat, const regnn_rowsplit_t* split,
                         float* split_workspace, const int32_t* row_order, const regnn_peer_rows_t* peers,
                         float* y_local, int64_t ldl, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (peers != nullptr) { Y = const_cast<float*>(X); ldy = feat; }  // Y is unused: keep the checks below simple
  REGNN_REQUIRE(y_local == nullptr || (peers != nullptr && ldl >= feat && ldl % 4 == 0 && aligned_to(y_local, 16)),
                REGNN_ERR_INVALID_ARG, "spmm_fwd: bad local result slab");
  REGNN_REQUIRE(indptr && X && Y,  /* per-edge arrays may be NULL when E == 0 */ REGNN_ERR_INVALID_ARG, "spmm_fwd: null pointer");
  REGNN_REQUIRE(etype == nullptr || theta != nullptr, REGNN_ERR_INVALID_ARG, "spmm_fwd: etype without theta");
  REGNN_REQUIRE(etype == nullptr || (num_relations >= 1 && num_relations <= REGNN_MAX_RELATIONS),
                REGNN_ERR_UNSUPPORTED_SHAPE, "num_relations=%d outside [1,%d]", num_relations, REGNN_MAX_RELATIONS);
  REGNN_REQUIRE(feat >= 1 && ldx >= feat && ldy >= feat, REGNN_ERR_INVALID_ARG, "spmm_fwd: bad feature width / leading dimension");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "spmm_fwd: negative row range");
  if (rows == 0) return REGNN_OK;
  StreamShape sh;
  REGNN_REQUIRE(pick_stream_shape(feat, common_align({X, Y, split_workspace}, {ldx, ldy, (int64_t)feat}), &sh),
                REGNN_ERR_UNSUPPORTED_SHAPE, "spmm_fwd: feature width %d too wide (max 1024 with 16-byte, 512 with 8-byte, 256 with 4-byte "
                "aligned operands)", feat);
  StreamArgs sa{};
  sa.s = SpmmArgs{indptr, indices, etype, theta, alpha, num_relations, norm_src, norm_dst, X, ldx, Y, ldy,
                  row_begin, row_end, feat, nullptr, nullptr, 0, 0, 0x7fffffff, nullptr};
  int rc = fill_split(sa.s, split, split_workspace, "spmm_fwd");
  if (rc != REGNN_OK) return rc;
  bool launched = false;
  const int G = rowgroup_lanes(feat, row_order, row_begin, common_align({X, Y, split_workspace}, {ldx, ldy, (int64_t)feat}));
  rc = fill_peers(&sa.peers, peers, feat, rows, "spmm_fwd");
  if (rc != REGNN_OK) return rc;
  sa.Ylocal = y_local;
  sa.ldl = ldl;
  REGNN_REQUIRE(peers == nullptr || G != 0, REGNN_ERR_UNSUPPORTED_SHAPE,
                "spmm_fwd: the peer scatter needs the lane-group kernel (row_order, full range, F <= 128, F %% 4 == 0)");
  if (G != 0) {  // narrow rows over the degree-sorted row order
    REGNN_REQUIRE(ldx < (1ll << 30), REGNN_ERR_UNSUPPORTED_SHAPE, "spmm_fwd: leading dimension too large");
    sa.order = row_order;
    sa.n_order = rows - (sa.s.nfrag > 0 ? split->num_long : 0);
    const int64_t nwork = (sa.s.nfrag + sa.n_order + 32 / G - 1) / (32 / G);
    const unsigned blocks = (unsigned)((nwork + kWarpsPerBlock - 1) / kWarpsPerBlock);
    REGNN_ROWGROUP_DISPATCH(false, (spmm_rowgroup_kernel<BINS, GL><<<blocks, kWarpsPerBlock * 32, 0, stream>>>(sa)))
  } else {
    const int64_t nitems = sa.s.nfrag_pad + (rows + kRowsPerItem - 1) / kRowsPerItem;
    const unsigned blocks = (unsigned)((nitems + kWarpsPerBlock - 1) / kWarpsPerBlock);
    REGNN_STREAM_DISPATCH(false, (spmm_stream_kernel<C, VW, BINS><<<blocks, kWarpsPerBlock * 32, 0, stream>>>(sa)))
  }
  REGNN_REQUIRE(launched, REGNN_ERR_UNSUPPORTED_SHAPE, "spmm_fwd: no kernel for C=%d VW=%d", sh.C, sh.VW);
  if (sa.s.nfrag > 0 && peers != nullptr)
    spmm_frag_finalize_peer_kernel<<<split->num_long, 128, 0, stream>>>(
        split->long_rows, split->frag_ptr, split->num_long, split_workspace, norm_dst, sa.peers, feat,
        FragPeerExtra{y_local, ldl, nullptr, 0, nullptr, nullptr, 0, nullptr, 0, nullptr, 0, nullptr});
  else if (sa.s.nfrag > 0)
    spmm_frag_finalize_kernel<<<split->num_long, 128, 0, stream>>>(split->long_rows, split->frag_ptr, split->num_long,
                                                                   split_workspace, norm_dst, Y, ldy, feat, row_begin, row_end);
  return check_launch("regnn_spmm_fwd");
}

extern "C" int regnn_spmm_fwd(const int32_t* indptr, const int32_t* indices, const uint8_t* etype,
                              const float* theta, float alpha, int num_relations,
                              const float* norm_src, const float* norm_dst, const float* X,
                              int64_t ldx, float* Y, int64_t ldy, int64_t row_begin,
                              int64_t row_end, int feat, const regnn_rowsplit_t* split,
                              float* split_workspace, const int32_t* row_order, void* stream) {
  return spmm_fwd_impl(indptr, indices, etype, theta, alpha, num_relations, norm_src, norm_dst, X, ldx, Y, ldy,
                       row_begin, row_end, feat, split, split_workspace, row_order, nullptr, nullptr, 0, stream);
}

extern "C" int regnn_spmm_fwd_scatter(const int32_t* indptr, const int32_t* indices, const uint8_t* etype,
                                      const float* theta, float alpha, int num_relations,
                                      const float* norm_src, const float* norm_dst, const float* X,
                                      int64_t ldx, int64_t num_rows, int feat, const regnn_rowsplit_t* split,
                                      float* split_workspace, const int32_t* row_order,
                                      const regnn_peer_rows_t* peers, float* y_local, int64_t ldl, void* stream) {
  REGNN_REQUIRE(peers != nullptr, REGNN_ERR_INVALID_ARG, "spmm_fwd_scatter: null peer table");
  return spmm_fwd_impl(indptr, indices, etype, theta, alpha, num_relations, norm_src, norm_dst, X, ldx, nullptr, 0,
                       0, num_rows, feat, split, split_workspace, row_order, peers, y_local, ldl, stream);
}

extern "C" int regnn_rows_to_slabs(const float* X, int64_t ldx, int64_t num_rows, int feat, int num_ranks,
                                   int64_t row_offset, float* const* peer_slabs, void* stream) {
  REGNN_REQUIRE(X && peer_slabs && num_ranks >= 1 && num_rows >= 0 && row_offset >= 0, REGNN_ERR_INVALID_ARG,
                "rows_to_slabs: bad argument");
  REGNN_REQUIRE(feat % (4 * num_ranks) == 0 && ldx % 4 == 0 && aligned_to(X, 16), REGNN_ERR_UNSUPPORTED_SHAPE,
                "rows_to_slabs: F=%d must split into whole 128-bit chunks over %d ranks (16-byte aligned rows)", feat,
                num_ranks);
  if (num_rows == 0) return REGNN_OK;
  const int Fc = feat / num_ranks;
  const int64_t total = num_rows * (Fc / 4);
  const int64_t want = (total + 255) / 256;
  const unsigned bx = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  // this rank's index = row_offset / rows-per-rank; any rotation that differs per rank spreads the traffic, so the row
  // offset itself (taken modulo the rank count of a block-sized stride) is enough when num_rows > 0
  const int first_peer = (int)((row_offset / (num_rows > 0 ? num_rows : 1)) % num_ranks);
  rows_to_slabs_kernel<<<dim3(bx, (unsigned)num_ranks), 256, 0, (cudaStream_t)stream>>>(X, ldx, num_rows, Fc, row_offset,
                                                                                     peer_slabs, first_peer);
  return check_launch("regnn_rows_to_slabs");
}

extern "C" int regnn_halo_push(const float* X, int64_t ldx, int feat, const int32_t* send_rows, const int64_t* send_ptr,
                               const int64_t* recv_offset, float* const* peer_bufs, int64_t ldb, int num_ranks, int rank,
                               void* stream) {
  REGNN_REQUIRE(X && send_ptr && recv_offset && peer_bufs && num_ranks >= 1 && rank >= 0 && rank < num_ranks,
                REGNN_ERR_INVALID_ARG, "halo_push: bad argument");
  REGNN_REQUIRE(num_ranks <= REGNN_HALO_MAX_RANKS, REGNN_ERR_UNSUPPORTED_SHAPE, "halo_push: %d ranks (max %d)", num_ranks,
                REGNN_HALO_MAX_RANKS);
  REGNN_REQUIRE(feat >= 4 && feat % 4 == 0 && ldx >= feat && ldb >= feat && ldx % 4 == 0 && ldb % 4 == 0 &&
                    aligned_to(X, 16),
                REGNN_ERR_UNSUPPORTED_SHAPE, "halo_push: F=%d must be whole 128-bit chunks in 16-byte aligned rows", feat);
  HaloPeers hp;
  int64_t most = 0;
  hp.ptr[0] = send_ptr[0];
  REGNN_REQUIRE(send_ptr[0] >= 0, REGNN_ERR_INVALID_ARG, "halo_push: negative send offset");
  for (int q = 0; q < num_ranks; ++q) {
    const int64_t cnt = send_ptr[q + 1] - send_ptr[q];
    REGNN_REQUIRE(cnt >= 0 && recv_offset[q] >= 0, REGNN_ERR_INVALID_ARG,
                  "halo_push: peer %d has a negative row count or receive offset", q);
    hp.ptr[q + 1] = send_ptr[q + 1];
    hp.recv_offset[q] = recv_offset[q];
    most = cnt > most ? cnt : most;
  }
  if (most == 0) return REGNN_OK;
  REGNN_REQUIRE(send_rows != nullptr, REGNN_ERR_INVALID_ARG, "halo_push: null send list");
  const int L = feat / 4;
  int G = 1;
  while (G < L && G < 32) G <<= 1;
  const int64_t want = (most * G + 255) / 256;
  const unsigned bx = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  halo_push_kernel<<<dim3(bx, (unsigned)num_ranks), 256, 0, (cudaStream_t)stream>>>(X, ldx, L, G, send_rows, hp,
                                                                                  peer_bufs, ldb, rank);
  return check_launch("regnn_halo_push");
}

extern "C" int regnn_halo_scatter(const float* X, int64_t ldx, int width, const int64_t* send_ptr, const int32_t* dst_rows,
                                  float* const* peer_bufs, int64_t ldb, int num_ranks, int rank, void* stream) {
  REGNN_REQUIRE(X && send_ptr && peer_bufs && num_ranks >= 1 && rank >= 0 && rank < num_ranks, REGNN_ERR_INVALID_ARG,
                "halo_scatter: bad argument");
  REGNN_REQUIRE(num_ranks <= REGNN_HALO_MAX_RANKS, REGNN_ERR_UNSUPPORTED_SHAPE, "halo_scatter: %d ranks (max %d)",
                num_ranks, REGNN_HALO_MAX_RANKS);
  REGNN_REQUIRE(width >= 1 && ldx >= width && ldb >= width, REGNN_ERR_INVALID_ARG,
                "halo_scatter: W=%d with leading dimensions %lld / %lld", width, (long long)ldx, (long long)ldb);
  REGNN_REQUIRE(send_ptr[0] >= 0, REGNN_ERR_INVALID_ARG, "halo_scatter: negative send offset");
  HaloPeers hp;
  int64_t most = 0;
  hp.ptr[0] = send_ptr[0];
  for (int q = 0; q < num_ranks; ++q) {
    const int64_t cnt = send_ptr[q + 1] - send_ptr[q];
    REGNN_REQUIRE(cnt >= 0, REGNN_ERR_INVALID_ARG, "halo_scatter: peer %d has a negative row count", q);
    hp.ptr[q + 1] = send_ptr[q + 1];
    hp.recv_offset[q] = 0;
    most = cnt > most ? cnt : most;
  }
  if (most == 0) return REGNN_OK;
  REGNN_REQUIRE(dst_rows != nullptr, REGNN_ERR_INVALID_ARG, "halo_scatter: null destination rows");
  const int64_t want = (most * width + 255) / 256;
  const unsigned bx = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  halo_scatter_kernel<<<dim3(bx, (unsigned)num_ranks), 256, 0, (cudaStream_t)stream>>>(X, ldx, width, dst_rows, hp,
                                                                                     peer_bufs, ldb, rank);
  return check_launch("regnn_halo_scatter");
}

extern "C" int regnn_halo_push_slots(const float* logit, int num_heads, const uint32_t* qmask, int num_chunks,
                                     const int32_t* send_slots, const int64_t* send_ptr, const int64_t* recv_offset,
                                     float* const* peer_logit, float* const* peer_mask, int num_ranks, int rank,
                                     void* stream) {
  REGNN_REQUIRE(logit && qmask && send_ptr && recv_offset && peer_logit && peer_mask && num_heads >= 1 &&
                    num_chunks >= 1 && num_ranks >= 1 && rank >= 0 && rank < num_ranks,
                REGNN_ERR_INVALID_ARG, "halo_push_slots: bad argument");
  REGNN_REQUIRE(num_ranks <= REGNN_HALO_MAX_RANKS, REGNN_ERR_UNSUPPORTED_SHAPE, "halo_push_slots: %d ranks (max %d)",
                num_ranks, REGNN_HALO_MAX_RANKS);
  REGNN_REQUIRE(aligned_to(qmask, 16), REGNN_ERR_UNSUPPORTED_SHAPE,
                "halo_push_slots: the mask rows must be 16-byte aligned 128-bit words");
  REGNN_REQUIRE(send_ptr[0] >= 0, REGNN_ERR_INVALID_ARG, "halo_push_slots: negative send offset");
  HaloPeers hp;
  int64_t most = 0;
  hp.ptr[0] = send_ptr[0];
  for (int q = 0; q < num_ranks; ++q) {
    const int64_t cnt = send_ptr[q + 1] - send_ptr[q];
    REGNN_REQUIRE(cnt >= 0 && recv_offset[q] >= 0, REGNN_ERR_INVALID_ARG,
                  "halo_push_slots: peer %d has a negative slot count or receive offset", q);
    hp.ptr[q + 1] = send_ptr[q + 1];
    hp.recv_offset[q] = recv_offset[q];
    most = cnt > most ? cnt : most;
  }
  if (most == 0) return REGNN_OK;
  REGNN_REQUIRE(send_slots != nullptr, REGNN_ERR_INVALID_ARG, "halo_push_slots: null send list");
  int G = 1;
  while (G < num_heads + num_chunks && G < 32) G <<= 1;
  const int64_t want = (most * G + 255) / 256;
  const unsigned bx = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  halo_push_slots_kernel<<<dim3(bx, (unsigned)num_ranks), 256, 0, (cudaStream_t)stream>>>(
      logit, num_heads, reinterpret_cast<const uint4*>(qmask), num_chunks, G, send_slots, hp, peer_logit, peer_mask, rank);
  return check_launch("regnn_halo_push_slots");
}

extern "C" int regnn_slabs_to_rows(const float* S, int64_t lds, int64_t num_rows, int feat,
                                   const regnn_peer_rows_t* peers, void* stream) {
  REGNN_REQUIRE(S && peers && num_rows >= 0 && feat >= 4 && feat % 4 == 0 && lds % 4 == 0 && aligned_to(S, 16),
                REGNN_ERR_INVALID_ARG, "slabs_to_rows: bad argument (16-byte aligned rows of whole 128-bit chunks)");
  PeerRows pr;
  int rc = fill_peers(&pr, peers, feat, num_rows, "slabs_to_rows");
  if (rc != REGNN_OK) return rc;
  if (num_rows == 0) return REGNN_OK;
  const int64_t total = (int64_t)pr.per * (feat / 4);
  const int64_t want = (total + 255) / 256;
  const unsigned bx = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  const int first_peer = (int)((peers->col_offset / feat) % peers->num_ranks);   // this rank's index: rotated peer order
  slabs_to_rows_kernel<<<dim3(bx, (unsigned)peers->num_ranks), 256, 0, (cudaStream_t)stream>>>(S, lds, num_rows, feat, pr,
                                                                                              first_peer);
  return check_launch("regnn_slabs_to_rows");
}

static int spmm_bwd_fused_impl(const int32_t* indptr_t, const int32_t* indices_t,
                               const uint8_t* etype_t, const float* theta, float alpha,
                               int num_relations, const float* norm, int norm_sides, const float* X,
                               int64_t ldx, const float* Gd, int64_t ldg, float* dX, int64_t lddx,
                               int64_t row_begin, int64_t row_end, int feat, double* partials,
                               float* d_theta, float* xdx, const float* Yfwd, int64_t ldyf, float* d_norm,
                               const regnn_rowsplit_t* split_t,
                               float* split_workspace, const int32_t* row_order_t, const regnn_peer_rows_t* peers,
                               void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (peers != nullptr) { dX = const_cast<float*>(X); lddx = ldx; }  // dX is unused: keep the checks below simple
  REGNN_REQUIRE(indptr_t && theta && X && Gd && dX && partials && d_theta,
                REGNN_ERR_INVALID_ARG, "spmm_bwd_fused: null pointer");
  const int R = num_relations;
  REGNN_REQUIRE(R >= 1 && R <= REGNN_MAX_RELATIONS, REGNN_ERR_UNSUPPORTED_SHAPE, "num_relations=%d outside [1,%d]", R,
                REGNN_MAX_RELATIONS);  // the shared-memory budget (bins + tile) is checked by set_smem below
  REGNN_REQUIRE(feat >= 1 && ldx >= feat && ldg >= feat && lddx >= feat, REGNN_ERR_INVALID_ARG,
                "spmm_bwd_fused: bad feature width / leading dimension");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "spmm_bwd_fused: negative row range");
  StreamShape sh;
  REGNN_REQUIRE(pick_stream_shape(feat, common_align({X, Gd, dX, split_workspace}, {ldx, ldg, lddx, (int64_t)feat}), &sh),
                REGNN_ERR_UNSUPPORTED_SHAPE, "spmm_bwd_fused: feature width %d too wide", feat);
  const int sides = norm != nullptr ? (norm_sides & 3) : 0;
  StreamArgs sa{};
  // transposed view: gathered rows are destinations (scaled when the forward scaled its destination side)
  sa.s = SpmmArgs{indptr_t, indices_t, etype_t, theta, alpha, R, (sides & 2) ? norm : nullptr, (sides & 1) ? norm : nullptr,
                  Gd, ldg, dX, lddx, row_begin, row_end, feat, nullptr, nullptr, 0, 0, 0x7fffffff, nullptr};
  int rc = fill_split(sa.s, split_t, split_workspace, "spmm_bwd_fused");
  if (rc != REGNN_OK) return rc;
  sa.Xrow = X;
  sa.ldr = ldx;
  sa.partials = partials;
  sa.use_tma = (feat % 4 == 0 && aligned_to(X, 16) && ldx % 4 == 0) ? 1 : 0;
  sa.xdx = xdx;
  const int Fp = (feat + 3) & ~3;
  if (d_norm != nullptr) {  // folded norm gradient: lane-group kernel only (the caller falls back to regnn_rowdot_norm_bwd)
    REGNN_REQUIRE(norm != nullptr && (!(sides & 2) || (Yfwd != nullptr && ldyf >= feat)),
                  REGNN_ERR_INVALID_ARG, "spmm_bwd_fused: d_norm needs norm and (destination side scaled) Y");
    REGNN_REQUIRE(!(sides & 2) || (aligned_to(Yfwd, 16) && ldyf % 4 == 0), REGNN_ERR_INVALID_ARG,
                  "spmm_bwd_fused: Y rows must be 16-byte aligned");
    sa.Yfwd = Yfwd; sa.ldyf = ldyf; sa.norm = norm; sa.dn_sides = sides; sa.d_norm = d_norm;
  }
  const size_t smem = 64 + (size_t)kWarpsPerBlock * R * (sizeof(double) + 32 * sizeof(float)) +
                      (size_t)kWarpsPerBlock * kRowsPerItemBins * Fp * sizeof(float);
  int nb = partial_blocks(rows / kRowsPerItemBins + sa.s.nfrag + 1);
  bool launched = false;
  const int G = rowgroup_lanes(feat, row_order_t, row_begin,
                               common_align({X, Gd, dX, split_workspace}, {ldx, ldg, lddx, (int64_t)feat}));
  rc = fill_peers(&sa.peers, peers, feat, rows, "spmm_bwd_fused");
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(peers == nullptr || G != 0, REGNN_ERR_UNSUPPORTED_SHAPE,
                "spmm_bwd_fused: the peer scatter needs the lane-group kernel (row_order_t, full range, F <= 128, F %% 4 == 0)");
  REGNN_REQUIRE(d_norm == nullptr || G != 0, REGNN_ERR_UNSUPPORTED_SHAPE,
                "spmm_bwd_fused: the folded norm gradient needs the lane-group kernel (row_order_t, full range, F <= 128, "
                "F %% 4 == 0); use regnn_rowdot_norm_bwd otherwise");
  // persistent kernels: exactly one resident wave (148 SMs x blocks per SM), never more than the partial slots
  if (G != 0) {
    REGNN_REQUIRE(ldg < (1ll << 30), REGNN_ERR_UNSUPPORTED_SHAPE, "spmm_bwd_fused: leading dimension too large");
    sa.order = row_order_t;
    sa.n_order = rows - (sa.s.nfrag > 0 ? split_t->num_long : 0);
    const size_t gsmem = (size_t)kWarpsPerBlock * R * (sizeof(double) + 32 * sizeof(float));
    if (d_norm != nullptr) {
      REGNN_ROWGROUP_DISPATCH(true, (rc = set_smem(spmm_rowgroup_kernel<BINS, GL, true>, gsmem),
                                     nb = min(nb, resident_blocks(spmm_rowgroup_kernel<BINS, GL, true>, gsmem)),
                                     spmm_rowgroup_kernel<BINS, GL, true><<<nb, kWarpsPerBlock * 32, gsmem, stream>>>(sa)))
    } else {
      REGNN_ROWGROUP_DISPATCH(true, (rc = set_smem(spmm_rowgroup_kernel<BINS, GL>, gsmem),
                                     nb = min(nb, resident_blocks(spmm_rowgroup_kernel<BINS, GL>, gsmem)),
                                     spmm_rowgroup_kernel<BINS, GL><<<nb, kWarpsPerBlock * 32, gsmem, stream>>>(sa)))
    }
  } else {
    REGNN_STREAM_DISPATCH(true, (rc = set_smem(spmm_stream_kernel<C, VW, BINS>, smem),
                                 nb = min(nb, resident_blocks(spmm_stream_kernel<C, VW, BINS>, smem)),
                                 spmm_stream_kernel<C, VW, BINS><<<nb, kWarpsPerBlock * 32, smem, stream>>>(sa)))
  }
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(launched, REGNN_ERR_UNSUPPORTED_SHAPE, "spmm_bwd_fused: no kernel for C=%d VW=%d", sh.C, sh.VW);
  if (sa.s.nfrag > 0 && peers != nullptr)
    spmm_frag_finalize_peer_kernel<<<split_t->num_long, 128, 0, stream>>>(
        split_t->long_rows, split_t->frag_ptr, split_t->num_long, split_workspace, sa.s.norm_dst, sa.peers, feat,
        FragPeerExtra{nullptr, 0, X, ldx, xdx, Yfwd, ldyf, Gd, ldg, norm, sides, d_norm});
  else if (sa.s.nfrag > 0)
    spmm_frag_finalize_kernel<<<split_t->num_long, 128, 0, stream>>>(split_t->long_rows, split_t->frag_ptr,
                                                                     split_t->num_long, split_workspace, sa.s.norm_dst, dX,
                                                                     lddx, feat, row_begin, row_end);
  if (sa.s.nfrag > 0 && (xdx != nullptr || d_norm != nullptr) && peers == nullptr)
    long_row_dnorm_kernel<<<(split_t->num_long + 3) / 4, 128, 0, stream>>>(split_t->long_rows, split_t->num_long, X, ldx, dX,
                                                                           lddx, feat, row_begin, row_end, xdx, Yfwd, ldyf, Gd,
                                                                           ldg, norm, sides, d_norm);
  launch_relation_grad_finalize(partials, nb, R, R, theta, alpha, d_theta, stream);
  return check_launch("regnn_spmm_bwd_fused");
}

extern "C" int regnn_spmm_bwd_fused(const int32_t* indptr_t, const int32_t* indices_t,
                                    const uint8_t* etype_t, const float* theta, float alpha,
                                    int num_relations, const float* norm, int norm_sides, const float* X,
                                    int64_t ldx, const float* Gd, int64_t ldg, float* dX, int64_t lddx,
                                    int64_t row_begin, int64_t row_end, int feat, double* partials,
                                    float* d_theta, float* xdx, const float* Y, int64_t ldy, float* d_norm,
                                    const regnn_rowsplit_t* split_t,
                                    float* split_workspace, const int32_t* row_order_t, void* stream) {
  return spmm_bwd_fused_impl(indptr_t, indices_t, etype_t, theta, alpha, num_relations, norm, norm_sides, X, ldx, Gd, ldg,
                             dX, lddx, row_begin, row_end, feat, partials, d_theta, xdx, Y, ldy, d_norm, split_t,
                             split_workspace, row_order_t, nullptr, stream);
}

extern "C" int regnn_spmm_bwd_fused_scatter(const int32_t* indptr_t, const int32_t* indices_t,
                                            const uint8_t* etype_t, const float* theta, float alpha,
                                            int num_relations, const float* norm, int norm_sides, const float* X,
                                            int64_t ldx, const float* Gd, int64_t ldg, int64_t num_rows, int feat,
                                            double* partials, float* d_theta, float* xdx, const float* Y, int64_t ldy,
                                            float* d_norm, const regnn_rowsplit_t* split_t, float* split_workspace,
                                            const int32_t* row_order_t, const regnn_peer_rows_t* peers, void* stream) {
  REGNN_REQUIRE(peers != nullptr, REGNN_ERR_INVALID_ARG, "spmm_bwd_fused_scatter: null peer table");
  return spmm_bwd_fused_impl(indptr_t, indices_t, etype_t, theta, alpha, num_relations, norm, norm_sides, X, ldx, Gd, ldg,
                             nullptr, 0, 0, num_rows, feat, partials, d_theta, xdx, Y, ldy, d_norm, split_t,
                             split_workspace, row_order_t, peers, stream);
}

extern "C" int regnn_rowdot_norm_bwd(const float* norm, int norm_sides, const float* X, int64_t ldx,
                                     const float* Y, int64_t ldy, const float* Gd, int64_t ldg,
                                     const float* dX, int64_t lddx, const float* xdx, int64_t row_begin,
                                     int64_t row_end, int feat, float* d_norm, void* stream) {
  REGNN_REQUIRE(norm && Y && Gd && d_norm && (xdx || (X && dX)), REGNN_ERR_INVALID_ARG, "rowdot_norm_bwd: null pointer");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0 && feat >= 1, REGNN_ERR_INVALID_ARG, "rowdot_norm_bwd: bad range / width");
  if (rows == 0) return REGNN_OK;
  const int64_t rows_per_block = (int64_t)kWarpsPerBlock * kRowdotRows;
  rowdot_norm_kernel<<<(unsigned)((rows + rows_per_block - 1) / rows_per_block), kWarpsPerBlock * 32, 0,
                       (cudaStream_t)stream>>>(norm, norm_sides & 3, X, ldx, Y, ldy, Gd, ldg, dX, lddx, xdx, feat,
                                               row_begin, row_end, d_norm);
  return check_launch("regnn_rowdot_norm_bwd");
}

extern "C" int regnn_spmm_bwd_w(const int32_t* indptr, const int32_t* indices, const uint8_t* etype,
                                const float* theta, float alpha, int num_relations,
                                const float* norm, int norm_sides, const float* X, int64_t ldx, const float* Y,
                                int64_t ldy, const float* Gd, int64_t ldg, const float* dX,
                                int64_t lddx, int64_t row_begin, int64_t row_end, int feat,
                                double* partials, float* d_theta, float* d_norm,
                                const regnn_rowsplit_t* split, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr && X && Y && Gd && dX, REGNN_ERR_INVALID_ARG, "spmm_bwd_w: null pointer");
  const bool weighted = etype != nullptr;
  const int R = weighted ? num_relations : 1;
  REGNN_REQUIRE(!weighted || (theta && partials && d_theta), REGNN_ERR_INVALID_ARG, "spmm_bwd_w: null relation buffers");
  REGNN_REQUIRE(R >= 1 && R <= REGNN_MAX_RELATIONS, REGNN_ERR_UNSUPPORTED_SHAPE, "num_relations=%d outside [1,%d]", R,
                REGNN_MAX_RELATIONS);
  REGNN_REQUIRE(feat >= 1 && ldx >= feat && ldy >= feat && ldg >= feat && lddx >= feat, REGNN_ERR_INVALID_ARG,
                "spmm_bwd_w: bad feature width / leading dimension");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "spmm_bwd_w: negative row range");
  const bool vec_ok = aligned16(X) && aligned16(Y) && aligned16(Gd) && aligned16(dX) && ldx % 4 == 0 &&
                      ldy % 4 == 0 && ldg % 4 == 0 && lddx % 4 == 0;
  Shape sh;
  REGNN_REQUIRE(pick_shape(feat, vec_ok, &sh), REGNN_ERR_UNSUPPORTED_SHAPE,
                "spmm_bwd_w: feature width %d too wide", feat);
  const bool use_split = split != nullptr && split->num_frags > 0;
  REGNN_REQUIRE(!use_split || (split->frag_row && split->frag_begin && split->threshold > 0), REGNN_ERR_INVALID_ARG,
                "spmm_bwd_w: incomplete row split");
  SpmmBwdArgs a{indptr, indices, etype, R, norm, norm != nullptr ? (norm_sides & 3) : 0, X, ldx, Y, ldy, Gd, ldg, dX, lddx, row_begin, row_end,
                feat, partials, d_norm, use_split ? split->frag_row : nullptr, use_split ? split->frag_begin : nullptr,
                use_split ? split->num_frags : 0, use_split ? split->threshold : 0x7fffffff};
  const int nb = partial_blocks(rows);
  const size_t smem = weighted ? bins_smem_bytes(R) : 16;
  bool launched = false;
  int rc = REGNN_OK;
  if (weighted) {
    REGNN_DISPATCH_SHAPES((rc = set_smem(spmm_bwd_w_kernel<G, C, VW, true>, smem),
                           spmm_bwd_w_kernel<G, C, VW, true><<<nb, kWarpsPerBlock * 32, smem, stream>>>(a)))
  } else {
    REGNN_DISPATCH_SHAPES((spmm_bwd_w_kernel<G, C, VW, false><<<nb, kWarpsPerBlock * 32, smem, stream>>>(a)))
  }
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(launched, REGNN_ERR_UNSUPPORTED_SHAPE, "spmm_bwd_w: no kernel for G=%d C=%d VW=%d", sh.G, sh.C, sh.VW);
  if (weighted) launch_relation_grad_finalize(partials, nb, R, R, theta, alpha, d_theta, stream);
  return check_launch("regnn_spmm_bwd_w");
}
