// Fused REGAT / REGATv2 kernels: edge logits + LeakyReLU + per-destination online softmax + weighted aggregation in
// ONE pass over the in-edges of each destination row, and a deterministic backward that gathers every edge's row ONCE
// (source-major over the transposed view, per-destination statistics from a streaming pre-pass) followed by streaming
// reductions over per-slot scalars.
// Reference call sites: layer/REGATConv.py:71-92, layer/REGATv2Conv.py:133-152 (DGL: gsddmm(add), 4-kernel
// edge_softmax, broadcast gspmm; autograd: gspmm on the reverse graph + gsddmm(dot)).
//
// Mapping (all hot kernels): a row of H*D floats is cut into slices of min(H*D, 128) floats; G = 4 / 8 / 16 / 32 lanes
// own one (row, slice) item with a 128-bit chunk each, so a warp works on 32/G rows and every gathered row is read with
// coalesced LDG.128; heads of D <= 128 never straddle a slice, per-head dot products are compile-time butterflies over
// the D/4 lanes of a head.  A wide head (D = 256 / 512) is one warp item whose lanes hold CPL = D/128 chunks each, the
// dot product being the lane's CPL partial dots + the 32-lane butterfly (kernels that reduce over a head take CPL; the
// others work per slice and take wide heads as they are).  Rows come from the degree-sorted row list, long rows are cut
// into fragments (merged by finalize kernels).
#include <type_traits>

#include "common.cuh"

namespace regnn {

struct AttnArgs {
  const int32_t* indptr;   // CSR (dst-major) or transposed (src-major) row pointers
  const int32_t* indices;
  const int32_t* eid;      // slot -> edge id (dst-major)  |  slot_t (src-major)
  const uint8_t* etype;
  const float* theta;      // [R,H]
  float alpha;
  int R;
  const float* feat;       // GAT: feat [N,H,D]   GATv2: fs
  const float* fd;         // GATv2 only
  const float* el;         // GAT: el [N,H]       GATv2: attn [H,D]
  const float* er;         // GAT: er [N,H]
  float slope;
  const float* keep;       // [E,H] edge-id order or null
  const float* G;
  int H, D;
  int d_shift;             // log2(D) when D is a power of two (the common case), else -1: avoids integer divisions
  int hg_count;            // ceil(H*D / 128)
  int64_t row_begin, row_end;
  float* o0;               // fwd: out      gather pass: d_feat / d_fs
  float* o1;               // fwd: rowmax   gather pass: d_el
  float* o2;               // fwd: rowsum   gather pass: dpre / dl per slot    streaming passes: d_er / d_fd
  float* o3;               // fwd: attn_out
  double* partials;
  const float* a_csr;      // REGATv2 backward: the saved logits (gather pass)
  const float* d_csr;      // per-slot dpre / dl (streaming passes)
  // long-row fragments (regnn_rowsplit_t): items [0, nfrag) are fragments (padded to nfrag_pad in the
  // grid-mapped kernels); their partial results go to p0/p1/p2 and are merged by the finalize kernels
  const int32_t* frag_row;
  const int32_t* frag_begin;
  int nfrag, nfrag_pad, threshold;
  float* p0;               // [nfrag][H*D]  partial rows (fwd: un-normalised acc; bwd: d_feat / d_fd / d_fs)
  float* p1;               // [nfrag][H]    fwd: fragment max      bwd: d_er / d_el partial
  float* p2;               // [nfrag][H]    fwd: fragment sum
  // row-group REGAT kernels: rows of the view that are not cut into fragments, by descending slot count (null:
  // natural order over [row_begin, row_end), rows longer than the threshold skipped)
  const int32_t* order;
  int64_t n_order;
  // gat_bwd_src epilogue (optional): d_feat[u,h,:] += d_el[u,h]*attn_l[h,:] + d_er[u,h]*attn_r[h,:]
  const float* attn_l;
  const int32_t* a_csr_eid;  // gat_bwd_edges with a dropout mask: CSR slot -> edge id
  // counter-based attention dropout (regnn_attn_dropout_t), read by the HASH instantiations only
  uint32_t drop_key_lo, drop_key_hi, drop_threshold;
  float drop_scale;
  int drop_head_offset, drop_heads_total;
};

// Keep factor of edge id e, head h of the call under regnn_attn_dropout_t (the counter hash stated in
// include/regnn_b200.h): a few integer instructions from the edge id the kernel has already loaded, in place of a
// 4-byte load from an [E,H] mask.
__device__ __forceinline__ float hashed_keep(const AttnArgs& a, int e, int h) {
  const uint64_t c = (uint64_t)(uint32_t)e * (uint32_t)a.drop_heads_total + (uint32_t)(a.drop_head_offset + h);
  uint32_t x = mix32((uint32_t)c ^ a.drop_key_lo);
  x = mix32(x + (uint32_t)(c >> 32) * 0x9E3779B1u + a.drop_key_hi);
  return x >= a.drop_threshold ? a.drop_scale : 0.f;
}

__device__ __forceinline__ void load_rel_table(float* w_s, const AttnArgs& a) {
  if (a.etype != nullptr) {
    const int n = a.R * a.H;
    for (int i = threadIdx.x; i < n; i += blockDim.x) w_s[i] = leaky(a.theta[i] * a.alpha, kRelationSlope);
  }
  __syncthreads();
}

__device__ __forceinline__ float4 add4(float4 a, float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 leaky4(float4 q, float s) {
  return make_float4(leaky(q.x, s), leaky(q.y, s), leaky(q.z, s), leaky(q.w, s));
}
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }

// Head-group mapping: a row of H*D floats is cut into 128-float slices ("head groups"); ONE WARP owns
// one (row | fragment, head group) item, lane l holding the 128-bit slice [128*hg + 4*l, +4).  Heads are
// independent in both layers, so the HG = ceil(H*D/128) warps of a row never have to talk to each other,
// every gathered source slice is one fully coalesced 512-byte request, and each lane needs a single
// float4 per edge -- which leaves registers for kUA rows in flight per lane.
struct Group {
  int hg, col, hl, h_lo, nh, lph;
  bool ok, leader;
};
__device__ __forceinline__ int div_d(const AttnArgs& a, int x) { return a.d_shift >= 0 ? (x >> a.d_shift) : x / a.D; }
__device__ __forceinline__ Group make_group(const AttnArgs& a, int hg, int lane) {
  Group g;
  const int HD = a.H * a.D;
  g.hg = hg;
  g.col = hg * 128 + lane * 4;
  g.ok = g.col < HD;
  g.h_lo = div_d(a, hg * 128);
  const int h_hi = min(a.H - 1, div_d(a, hg * 128 + 127));
  g.nh = h_hi - g.h_lo + 1;
  g.hl = g.ok ? div_d(a, g.col) : g.h_lo;
  const int lanes_per_head = a.D >> 2;
  g.lph = min(32, lanes_per_head);
  g.leader = g.ok && (g.col - g.hl * a.D == 0);   // first lane of its head
  return g;
}
__device__ __forceinline__ int num_groups(const AttnArgs& a) { return a.hg_count; }
// (item index, head group) of warp item wi; 32-bit arithmetic whenever the item count allows it
__device__ __forceinline__ void split_item(int64_t wi, int HG, int64_t* ri, int* hg) {
  if (wi < 0x7fffffffLL) {
    const unsigned w = (unsigned)wi;
    *ri = w / (unsigned)HG;
    *hg = (int)(w % (unsigned)HG);
  } else {
    *ri = wi / HG;
    *hg = (int)(wi % HG);
  }
}

// =================================================================================================
// Row-group REGAT kernels (forward, destination-major backward, source-major backward).
//
// Mapping (as spmm_rowgroup_kernel): a 128-bit chunk per lane covers a slice of min(H*D, 128) floats of a row with
// G = 4 / 8 / 16 / 32 lanes, so a warp works on 32/G rows at once and one gather instruction fetches 32/G source rows;
// rows wider than 128 floats are cut into H*D/128 slices that are independent items (heads never mix).  Rows come
// from the degree-sorted row list of the view, fragments of long rows first.
// Every lane evaluates the logit of ITS OWN head for the edge at hand (one 4-byte load of el[src,h], served by the
// same sector for all lanes of the group, + er[v,h] from a register + the relation table in shared memory), so the
// edge softmax needs no cross-lane max / sum and no shared-memory staging: the lanes of a head carry identical
// running (max, sum) pairs.  Online softmax per batch of U edges: one rescale exp per batch + one exp per edge.
// Column indices / edge types are loaded cooperatively (lane l of a group loads slot t0+l) and broadcast by shuffles.
struct RowItem {
  int64_t v, fi;
  int begin, len, hg;
  bool frag;
};

// CPL > 1 (wide heads, G = 32): an item is a (row, head) pair and it.hg is the head; see kernels taking CPL below
template <int G, int CPL = 1>
__device__ __forceinline__ RowItem rg_item(const AttnArgs& a, int64_t wi, int grp) {
  constexpr int GPW = 32 / G;
  RowItem it{-1, 0, 0, 0, 0, false};
  const int64_t nrows = a.order != nullptr ? a.n_order : (a.row_end - a.row_begin);
  const int64_t nitems = (a.nfrag + nrows) * (a.hg_count / CPL);
  const int64_t vi = wi * GPW + grp;
  if (vi >= nitems) return it;
  int64_t ri = vi;
  if (a.hg_count / CPL > 1) split_item(vi, a.hg_count / CPL, &ri, &it.hg);
  if (ri < a.nfrag) {
    it.frag = true;
    it.fi = ri;
    const int64_t v = a.frag_row[ri];
    if (v >= a.row_begin && v < a.row_end) {
      it.v = v;
      it.begin = a.frag_begin[ri];
      it.len = min(a.threshold, a.indptr[v + 1] - it.begin);
    }
  } else {
    const int64_t v = a.order != nullptr ? (int64_t)a.order[ri - a.nfrag] : a.row_begin + (ri - a.nfrag);
    const int b = a.indptr[v];
    const int l = a.indptr[v + 1] - b;
    if (l <= a.threshold) {  // longer rows are covered by fragments
      it.v = v;
      it.begin = b;
      it.len = l;
    }
  }
  return it;
}
__device__ __forceinline__ int64_t rg_num_work(const AttnArgs& a, int G, int CPL = 1) {
  const int64_t nrows = a.order != nullptr ? a.n_order : (a.row_end - a.row_begin);
  const int GPW = 32 / G;
  return ((a.nfrag + nrows) * (a.hg_count / CPL) + GPW - 1) / GPW;
}

#ifndef REGNN_FWD_PF
#define REGNN_FWD_PF 0
#endif
#ifndef REGNN_PF_BYTES
#define REGNN_PF_BYTES 128
#endif
constexpr int kUG = 4;  // edges per online-softmax batch (= gathers in flight per lane)

// EXTRA: attention dropout mask and / or attention output (both need edge ids); HASH (implies EXTRA): the dropout
// factor comes from hashed_keep instead of a.keep
// The HASH instantiations keep their explicit-mask siblings' blocks per SM: one block less removes most of their spills
// but was slower on the MAG graph (B200, forward + backward of the core: REGAT H8 D16 11.8 ms instead of 10.5)
template <int G, bool EXTRA, bool HASH = false>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, (EXTRA || G < 32) ? 4 : 5)   // 48 registers spill for G < 32
gat_fwd_rg_kernel(AttnArgs a) {
  static_assert(EXTRA || !HASH, "the hashed dropout factor needs the edge ids");
  constexpr int U = kUG;
  static_assert(G % U == 0, "a batch must not straddle a cooperative slot load");
  extern __shared__ __align__(16) float smem[];
  float* w_s = smem;
  load_rel_table(w_s, a);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G, gbase = lane & ~(G - 1);
  const int H = a.H, HD = H * a.D;
  const int64_t wi = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  if (wi >= rg_num_work(a, G)) return;  // warp-uniform
  const RowItem it = rg_item<G>(a, wi, grp);
  const int col = it.hg * 128 + lg * 4;
  const bool col_ok = col < HD;
  const int h = col_ok ? (col >> a.d_shift) : 0;
  const bool act = it.v >= 0 && col_ok;
  const bool leader = act && (col & (a.D - 1)) == 0;
  const int len = it.v >= 0 ? it.len : 0;
  const int maxlen = __reduce_max_sync(0xffffffffu, len);
  const bool has_rel = a.etype != nullptr;
  constexpr bool need_eid = EXTRA;
  const float er_v = act ? __ldg(a.er + (size_t)it.v * H + h) : 0.f;
  const float* fcol = a.feat + (col_ok ? col : 0);
  const float* elh = a.el + h;
  const int32_t* ip = a.indices + it.begin;
  const uint8_t* ep = a.etype + it.begin;
  const int32_t* eidp = a.eid + it.begin;
  float4 acc = zero4();
  float m = -INFINITY, s = 0.f;

  for (int t0 = 0; t0 < maxlen; t0 += G) {
    int bi = -1, be = 0, beid = 0;
    {
      const int t = t0 + lg;
      if (t < len) {
        bi = __ldg(ip + t);
        if (has_rel) be = __ldg(ep + t);
        if (need_eid) beid = __ldg(eidp + t);
#if REGNN_FWD_PF
        {
          const char* fr = reinterpret_cast<const char*>(a.feat + it.hg * 128) + (uint64_t)(uint32_t)bi * ((uint32_t)HD * 4u);
          const int nl = (min(128, HD - it.hg * 128) * 4 + REGNN_PF_BYTES - 1) / REGNN_PF_BYTES;
          for (int k = 0; k < nl; ++k) prefetch_l2(fr + k * REGNN_PF_BYTES);
          prefetch_l2(a.el + (uint64_t)(uint32_t)bi * (uint32_t)H);
        }
#endif
      }
    }
    const int cnt = min(G, maxlen - t0);
    for (int j = 0; j < cnt; j += U) {
      float4 x[U];
      float l[U];
      int si[U], seid[EXTRA ? U : 1];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        si[u] = __shfl_sync(0xffffffffu, bi, gbase + j + u);
        const bool ok = si[u] >= 0 && col_ok;
        x[u] = ok ? ldg4(fcol + (size_t)si[u] * HD) : zero4();
        l[u] = ok ? __ldg(elh + (size_t)si[u] * H) : 0.f;
      }
      float bm = -INFINITY;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float pre = l[u] + er_v;
        if (has_rel) pre += w_s[__shfl_sync(0xffffffffu, be, gbase + j + u) * H + h];
        if (EXTRA) seid[u] = __shfl_sync(0xffffffffu, beid, gbase + j + u);
        l[u] = si[u] >= 0 ? leaky(pre, a.slope) : -INFINITY;
        bm = fmaxf(bm, l[u]);
      }
      if (bm > -INFINITY) {  // uniform within a lane group
        const float m_new = fmaxf(m, bm);
        const float sc = fast_exp(m - m_new);  // first batch: exp(-inf) = 0
        m = m_new;
        s *= sc;
        scale4(acc, sc);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          float p = fast_exp(l[u] - m_new);  // 0 for a missing slot
          s += p;
          if (EXTRA && si[u] >= 0 && act) {
            const size_t o = (size_t)seid[u] * H + h;
            if (a.o3 != nullptr && leader) a.o3[o] = l[u];  // raw logit; normalised after the row
            if (HASH) p *= hashed_keep(a, seid[u], h);
            else if (a.keep != nullptr) p *= __ldg(a.keep + o);
          }
          fma4(acc, p, x[u]);
        }
      }
    }
  }

  if (it.frag) {  // un-normalised partial + fragment statistics; attn_frag_finalize_kernel merges them
    if (act) st4(a.p0 + (size_t)it.fi * HD + col, acc);
    if (leader) {
      a.p1[(size_t)it.fi * H + h] = m;
      a.p2[(size_t)it.fi * H + h] = s;
    }
    return;
  }
  const float inv = s > 0.f ? 1.f / s : 0.f;
  const float mm = len > 0 ? m : 0.f;
  if (act) {
    scale4(acc, inv);
    st4(a.o0 + (size_t)it.v * HD + col, acc);
    if (leader) {
      a.o1[(size_t)it.v * H + h] = mm;
      a.o2[(size_t)it.v * H + h] = s;
    }
  }
  if (EXTRA && a.o3 != nullptr) {  // get_attention: stored logits -> a*keep, edge-id order; the lanes of a head share its slots
    __syncwarp();
    const int lph = min(G, a.D >> 2);
    if (act && ((it.hg << 7) & (a.D - 1)) == 0)   // D > 128: only the warp of a head's first slice, which stored its logits
      for (int t = lg & (lph - 1); t < len; t += lph) {
        const size_t o = (size_t)eidp[t] * H + h;
        float av = __expf(a.o3[o] - mm) * inv;
        if (HASH) av *= hashed_keep(a, eidp[t], h);
        else if (a.keep != nullptr) av *= a.keep[o];
        a.o3[o] = av;
      }
  }
}

// =================================================================================================
// REGAT backward as ONE gather pass.  The softmax backward of an edge e = (u -> v) needs
//   da_e = <feat[u,h,:], G[v,h,:]>,   a_e = exp(l_e - m_v) / s_v,   S_v = sum_e' a_e' da_e' = <out[v,h,:], G[v,h,:]>
// and the source-major pass that produces d_feat[u] = sum_e a_e G[v] gathers G[v] anyway while feat[u] is the row
// the lane group owns: with the per-destination statistics (er, m, 1/s, S) packed as one float4 per (node, head) by
// a streaming pre-pass, every per-edge quantity is available in that ONE pass -- the destination-major pass over
// feat[src] of round 1 (a second 4HD-byte gather per edge) and the [E,H] attention tensor between the passes are gone.
//   gat_bwd_stats_kernel    stats[v,h] = (er, rowmax, 1/rowsum, <out,G>)                      streaming, 2 N H D reads
//   gat_bwd_edges_kernel    d_feat[u], d_el[u], dpre[slot,h]  (source-major, row groups)      the gather pass
//   gat_bwd_der_kernel      d_er[v,h] = sum_{slots of v} dpre[slot,h]                         streaming over [E,H]
//   gat_bwd_bins_kernel     relation bins of dpre (lane-local, per-block double partials)     streaming over [E,H]
// CPL > 1 (D = 128 * CPL, G = 32): an item is a (node, head) pair, lane l reading columns h*D + 128*c + 4*l, c < CPL;
// HG is then the number of heads
template <int G, int CPL = 1>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
gat_bwd_stats_kernel(const float* __restrict__ out, const float* __restrict__ Gd, const float* __restrict__ er,
                     const float* __restrict__ rowmax, const float* __restrict__ rowsum, int64_t n, int H, int D,
                     int d_shift, int HG, float4* __restrict__ stats) {
  constexpr int GPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int lg = lane % G, grp = lane / G;
  const int HD = H * D, lph = min(G, D >> 2);
  const int64_t items = n * HG;
  for (int64_t wi = ((int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5)) * GPW; wi < items;
       wi += (int64_t)gridDim.x * kWarpsPerBlock * GPW) {
    const int64_t vi = wi + grp;
    const int64_t v = vi / HG;
    const int col = (int)(vi % HG) * (128 * CPL) + lg * 4;
    const bool act = vi < items && col < HD;
    float p = 0.f;
#pragma unroll
    for (int c = 0; c < CPL; ++c)
      if (act) {
        const float q = dot4(ldg4(out + (size_t)v * HD + col + 128 * c), ldg4(Gd + (size_t)v * HD + col + 128 * c));
        p = c == 0 ? q : p + q;
      }
    p = group_sum_rt(p, lph);
    if (act && (col & (D - 1)) == 0) {
      const size_t vh = (size_t)v * H + (col >> d_shift);
      const float sm = rowsum[vh];
      stats[vh] = make_float4(er != nullptr ? er[vh] : 0.f, rowmax[vh], sm > 0.f ? 1.f / sm : 0.f, p);
    }
  }
}

// Source-major gather pass (transposed view; AttnArgs: indptr/indices/eid = indptr_t/indices_t/slot_t, etype = etype_t,
// fd = stats as float4[N*H], G = dL/d out, a_csr = slot -> edge id when keep != null).
// The gather pass is latency-bound at HBM scale (short rows, two gathers + two statistics loads per round): resident
// warps win -- MAG graph, H8 D16: 4 blocks/SM 4.00 ms, 5: 3.66, 6 (40 registers, 24 bytes of spill): 3.49; L2-resident
// ACM H8 D64: 0.226 / 0.244 / 0.250 ms.  Tried and dropped: staging the per-destination statistics of a whole slot batch in
// shared memory (every lane fetches the nh heads of its slot, broadcast LDS.128 later) so that 4 rows of G fit in flight:
// 5.5 ms instead of 3.5 -- the extra serial load / store / __syncwarp phase costs more than the halved round trips save.
#ifndef REGNN_GATB_BLOCKS
#define REGNN_GATB_BLOCKS 6
#endif
#ifndef REGNN_GATB_PF
#define REGNN_GATB_PF 0
#endif
#ifndef REGNN_PF_BYTES
#define REGNN_PF_BYTES 128
#endif
#ifndef REGNN_GATB_U
#define REGNN_GATB_U 2
#endif
// LPH = min(G, D/4): lanes per head (compile-time butterfly); KEEP: attention dropout, its factor from a.keep or -- HASH --
// from hashed_keep.  CPL: 128-bit chunks per lane -- 1: the item is a (row | fragment, 128-float slice) pair; 2 / 4 (wide
// heads, D = 128 * CPL, G = LPH = 32): the item is a (row | fragment, head) pair, lane l holding the columns
// h*D + 128*c + 4*l, c < CPL (CPL coalesced 512-byte requests per gathered row), and a head's dot product is the sum of
// the lane's CPL partial dots followed by the 32-lane butterfly.
#define REGNN_WIDE_BLOCKS(CPL_, NARROW_) ((CPL_) == 1 ? (NARROW_) : ((CPL_) == 2 ? 4 : 2))
template <int G, int LPH, bool KEEP, bool HASH = false, int CPL = 1>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, REGNN_WIDE_BLOCKS(CPL, REGNN_GATB_BLOCKS))
gat_bwd_edges_kernel(AttnArgs a) {
  static_assert(KEEP || !HASH, "HASH is a dropout mode");
  constexpr int U = REGNN_GATB_U;  // rows of G (and statistics vectors) in flight per lane
  static_assert(G % U == 0, "a round must not straddle a slot batch");
  extern __shared__ __align__(16) float smem[];
  float* w_s = smem;
  load_rel_table(w_s, a);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G, gbase = lane & ~(G - 1);
  const int H = a.H, HD = H * a.D;
  const int64_t wi = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  if (wi >= rg_num_work(a, G, CPL)) return;
  const RowItem it = rg_item<G, CPL>(a, wi, grp);
  const int col = it.hg * (128 * CPL) + lg * 4;
  const bool col_ok = col < HD;
  const int h = col_ok ? (col >> a.d_shift) : 0;
  const bool act = it.v >= 0 && col_ok;
  const bool leader = act && (col & (a.D - 1)) == 0;
  const int len = it.v >= 0 ? it.len : 0;
  const int maxlen = __reduce_max_sync(0xffffffffu, len);
  const bool has_rel = a.etype != nullptr;
  float4 fu[CPL];
  float el_u = 0.f;
#pragma unroll
  for (int c = 0; c < CPL; ++c) fu[c] = zero4();
  if (act) {
#pragma unroll
    for (int c = 0; c < CPL; ++c) fu[c] = ldg4(a.feat + (size_t)it.v * HD + col + 128 * c);
    el_u = __ldg(a.el + (size_t)it.v * H + h);
  }
  // one IMAD.WIDE.U32 per gathered address: 32-bit index x 32-bit pitch (bytes) added to a 64-bit base
  const char* gbytes = reinterpret_cast<const char*>(a.G + (col_ok ? col : 0));
  const char* sbytes = reinterpret_cast<const char*>(a.fd) + (size_t)h * 16;
  const uint32_t gpitch = (uint32_t)HD * 4u, spitch = (uint32_t)H * 16u;
  float* dpre_h = a.o2 + h;
  const float* w_h = w_s + h;
  const int32_t* ip = a.indices + it.begin;
  const int32_t* sp = a.eid + it.begin;
  const uint8_t* ep = a.etype + it.begin;
  float4 acc[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) acc[c] = zero4();
  float del = 0.f;
#if REGNN_GATB_PF
  // the G row slice and the statistics this lane's own slot will need, into L2 while the first rounds run
  const char* pf_g = reinterpret_cast<const char*>(a.G + it.hg * 128 * CPL);
  const int pf_lines = (min(128 * CPL, HD - it.hg * 128 * CPL) * 4 + REGNN_PF_BYTES - 1) / REGNN_PF_BYTES;
  const char* pf_s = reinterpret_cast<const char*>(a.fd) + (size_t)((it.hg * 128 * CPL) >> a.d_shift) * 16;
#endif

  for (int t0 = 0; t0 < maxlen; t0 += G) {
    int bi = -1, bs = 0, be = 0;
    {
      const int t = t0 + lg;
      if (t < len) {
        bi = __ldg(ip + t);
        bs = __ldg(sp + t);
        if (has_rel) be = __ldg(ep + t);
#if REGNN_GATB_PF
        const char* gr = pf_g + (uint64_t)(uint32_t)bi * gpitch;
        for (int k = 0; k < pf_lines; ++k) prefetch_l2(gr + k * REGNN_PF_BYTES);
        prefetch_l2(pf_s + (uint64_t)(uint32_t)bi * spitch);
#endif
      }
    }
    const int cnt = min(G, maxlen - t0);
    for (int j = 0; j < cnt; j += U) {
      float4 x[U][CPL], st[U];
      int sd[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        sd[u] = __shfl_sync(0xffffffffu, bi, gbase + j + u);
        const bool ok = sd[u] >= 0 && col_ok;
#pragma unroll
        for (int c = 0; c < CPL; ++c)
          x[u][c] = ok ? ldg4(reinterpret_cast<const float*>(gbytes + (uint64_t)(uint32_t)sd[u] * gpitch + 512 * c)) : zero4();
        // missing slot: rowmax = +inf makes exp(. - rowmax) = 0, so a = dpre = 0 without per-edge masks
        st[u] = ok ? __ldg(reinterpret_cast<const float4*>(sbytes + (uint64_t)(uint32_t)sd[u] * spitch))
                   : make_float4(0.f, INFINITY, 0.f, 0.f);
      }
      float da[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float p = dot4(fu[0], x[u][0]);
#pragma unroll
        for (int c = 1; c < CPL; ++c) p += dot4(fu[c], x[u][c]);
        da[u] = group_sum<LPH>(p);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int ss = __shfl_sync(0xffffffffu, bs, gbase + j + u);
        const int se = has_rel ? __shfl_sync(0xffffffffu, be, gbase + j + u) : 0;
        float pre = el_u + st[u].x;
        if (has_rel) pre += w_h[se * H];
        const float aa = __expf(leaky(pre, a.slope) - st[u].y) * st[u].z;
        float at = aa;
        if (KEEP) {
          if (sd[u] >= 0 && act) {
            const int e = __ldg(a.a_csr_eid + ss);
            at *= HASH ? hashed_keep(a, e, h) : __ldg(a.keep + (size_t)e * H + h);
          }
        }
        const float dp = (at * da[u] - aa * st[u].w) * leaky_grad(pre, a.slope);
#pragma unroll
        for (int c = 0; c < CPL; ++c) fma4(acc[c], at, x[u][c]);
        del += dp;
        if (leader && sd[u] >= 0) dpre_h[(uint64_t)(uint32_t)ss * (uint32_t)H] = dp;   // dpre per CSR slot
      }
    }
  }
  if (!act) return;
  if (it.frag) {
#pragma unroll
    for (int c = 0; c < CPL; ++c) st4(a.p0 + (size_t)it.fi * HD + col + 128 * c, acc[c]);
    if (leader) a.p1[(size_t)it.fi * H + h] = del;
    return;
  }
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    if (a.attn_l != nullptr) fma4(acc[c], del, ldg4(a.attn_l + col + 128 * c));   // gradient through el = <feat, attn_l>
    st4(a.o0 + (size_t)it.v * HD + col + 128 * c, acc[c]);
  }
  if (leader) a.o1[(size_t)it.v * H + h] = del;
}

// d_feat[v,h,:] += d_el[v,h] * attn_l[h,:] for the long rows (their sums are only complete after frag_rowsum_kernel)
__global__ void gat_fold_long_rows_kernel(const int32_t* __restrict__ long_rows, int num_long, int H, int D,
                                          const float* __restrict__ attn_l, const float* __restrict__ d_el,
                                          float* __restrict__ d_feat, int64_t row_begin, int64_t row_end) {
  const int l = blockIdx.x;
  if (l >= num_long) return;
  const int64_t v = long_rows[l];
  if (v < row_begin || v >= row_end) return;
  const int HD = H * D;
  for (int c = threadIdx.x; c < HD; c += blockDim.x)
    d_feat[(size_t)v * HD + c] += d_el[(size_t)v * H + c / D] * attn_l[c];
}

// d_er[v,h] = sum over the CSR slots of row v of dpre[slot,h]: HP = next power of two >= H lanes per item (lane = head),
// 32/HP items per warp (fragments of long rows first, then the rows), each lane adds its head in slot order
// (deterministic), 4 loads in flight.  AttnArgs: indptr, d_csr = dpre, o2 = d_er, p1 = fragment partials.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
gat_bwd_der_kernel(AttnArgs a, int HP) {
  const int lane = threadIdx.x & 31;
  const int H = a.H, hh = lane % HP, per = 32 / HP;
  const int64_t vi = ((int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5)) * per + lane / HP;
  const int64_t rows = a.row_end - a.row_begin;
  if (vi >= a.nfrag + rows || hh >= H) return;
  int s0, s1;
  float* dst;
  if (vi < a.nfrag) {
    const int64_t v = a.frag_row[vi];
    if (v < a.row_begin || v >= a.row_end) return;
    s0 = a.frag_begin[vi];
    s1 = s0 + min(a.threshold, a.indptr[v + 1] - s0);
    dst = a.p1 + (size_t)vi * H + hh;
  } else {
    const int64_t v = a.row_begin + (vi - a.nfrag);
    s0 = a.indptr[v];
    s1 = a.indptr[v + 1];
    if (s1 - s0 > a.threshold) return;  // covered by fragments
    dst = a.o2 + (size_t)v * H + hh;
  }
  const float* p = a.d_csr + (size_t)s0 * H + hh;
  float acc = 0.f;
  int s = s0;
  for (; s + 4 <= s1; s += 4, p += 4 * H) {
    const float a0 = __ldg(p), a1 = __ldg(p + H), a2 = __ldg(p + 2 * H), a3 = __ldg(p + 3 * H);
    acc = (((acc + a0) + a1) + a2) + a3;
  }
  for (; s < s1; ++s, p += H) acc += __ldg(p);
  *dst = acc;
}

// The two reductions above and below in ONE streaming pass over dpre (used when the layer has relation embeddings):
// row sums d_er[v,h] as gat_bwd_der_kernel, and the relation bins of the same values, lane-local in shared memory
// (lane = (item-in-warp, head): conflict-free), per-block double partials.  Persistent grid-stride loop over the items.
// AttnArgs as gat_bwd_der_kernel + etype (CSR order), R, partials [gridDim.x][R*H].  Dynamic smem: [warps][R][32] floats
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
gat_bwd_der_bins_kernel(AttnArgs a, int HP) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int H = a.H, R = a.R, hh = lane % HP, per = 32 / HP;
  float* mybins = smem + (size_t)warp * R * 32 + lane;
  for (int r = 0; r < R; ++r) mybins[r * 32] = 0.f;
  const int64_t rows = a.row_end - a.row_begin;
  const int64_t nitems = a.nfrag + rows;
  for (int64_t it = (int64_t)blockIdx.x * kWarpsPerBlock + warp; it * per < nitems; it += (int64_t)gridDim.x * kWarpsPerBlock) {
    const int64_t vi = it * per + lane / HP;
    if (vi >= nitems || hh >= H) continue;
    int s0, s1;
    float* dst;
    if (vi < a.nfrag) {
      const int64_t v = a.frag_row[vi];
      if (v < a.row_begin || v >= a.row_end) continue;
      s0 = a.frag_begin[vi];
      s1 = s0 + min(a.threshold, a.indptr[v + 1] - s0);
      dst = a.p1 + (size_t)vi * H + hh;
    } else {
      const int64_t v = a.row_begin + (vi - a.nfrag);
      s0 = a.indptr[v];
      s1 = a.indptr[v + 1];
      if (s1 - s0 > a.threshold) continue;  // covered by fragments
      dst = a.o2 + (size_t)v * H + hh;
    }
    const float* p = a.d_csr + (size_t)s0 * H + hh;
    const uint8_t* tp = a.etype + s0;
    float acc = 0.f;
    int s = s0;
    for (; s + 4 <= s1; s += 4, p += 4 * H, tp += 4) {
      const float a0 = __ldg(p), a1 = __ldg(p + H), a2 = __ldg(p + 2 * H), a3 = __ldg(p + 3 * H);
      const int t0 = __ldg(tp), t1 = __ldg(tp + 1), t2 = __ldg(tp + 2), t3 = __ldg(tp + 3);
      acc = (((acc + a0) + a1) + a2) + a3;
      mybins[t0 * 32] += a0;
      mybins[t1 * 32] += a1;
      mybins[t2 * 32] += a2;
      mybins[t3 * 32] += a3;
    }
    for (; s < s1; ++s, p += H, ++tp) {
      const float a0 = __ldg(p);
      acc += a0;
      mybins[(int)__ldg(tp) * 32] += a0;
    }
    *dst = acc;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < R * H; i += blockDim.x) {
    const int r = i / H, h2 = i % H;
    double sum = 0.0;
    for (int w = 0; w < kWarpsPerBlock; ++w)
      for (int q = h2; q < 32; q += HP) sum += (double)smem[((size_t)w * R + r) * 32 + q];
    a.partials[(size_t)blockIdx.x * R * H + i] = sum;
  }
}

// Relation bins of dpre (rows of `pitch` floats, the first H used): pure streaming over [E,H] (+ the uint8 edge types), lane-local bins, per-block double partials.
// A warp reads 32/HP slots x HP heads per load; 8 loads are issued before the (loop-carried) shared-memory updates.
// Dynamic smem: [warps][R][32] floats
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
gat_bwd_bins_kernel(const uint8_t* __restrict__ etype, const float* __restrict__ dpre, int pitch,
                    const int32_t* __restrict__ indptr, int64_t row_begin, int64_t row_end, int R, int H, int HP,
                    double* __restrict__ partials) {
  constexpr int UB = 8;
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t s_begin = indptr[row_begin], s_end = indptr[row_end];
  float* mybins = smem + (size_t)warp * R * 32 + lane;
  for (int r = 0; r < R; ++r) mybins[r * 32] = 0.f;
  const int hh = lane % HP, per = 32 / HP;
  if (hh < H) {
    const int64_t tile = (int64_t)per * UB;   // slots per warp iteration
    for (int64_t s0 = s_begin + ((int64_t)blockIdx.x * kWarpsPerBlock + warp) * tile + lane / HP; s0 < s_end;
         s0 += (int64_t)gridDim.x * kWarpsPerBlock * tile) {
      float v[UB];
      int t[UB];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const int64_t s = s0 + (int64_t)u * per;
        const bool ok = s < s_end;
        t[u] = ok ? (int)__ldg(etype + s) : 0;
        v[u] = ok ? __ldg(dpre + (size_t)s * pitch + hh) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < UB; ++u) mybins[t[u] * 32] += v[u];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < R * H; i += blockDim.x) {
    const int r = i / H, h2 = i % H;
    double sum = 0.0;
    for (int w = 0; w < kWarpsPerBlock; ++w)
      for (int q = h2; q < 32; q += HP) sum += (double)smem[((size_t)w * R + r) * 32 + q];
    partials[(size_t)blockIdx.x * R * H + i] = sum;
  }
}

// Projection scores of REGAT (layer/REGATConv.py:68-69): el[n,h] = <feat[n,h,:], attn_l[h,:]>, er likewise -- one
// streaming pass over feat instead of two eager mul + sum pairs.  Same lane-group mapping as above (CPL as
// gat_bwd_stats_kernel).
template <int G, int CPL = 1>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
attn_scores_fwd_kernel(const float* __restrict__ feat, const float* __restrict__ attn_l, const float* __restrict__ attn_r,
                       int64_t n, int H, int D, int d_shift, int HG, float* __restrict__ el, float* __restrict__ er) {
  constexpr int GPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int lg = lane % G, grp = lane / G;
  const int HD = H * D, lph = min(G, D >> 2);
  const int64_t items = n * HG;
  for (int64_t wi = ((int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5)) * GPW; wi < items;
       wi += (int64_t)gridDim.x * kWarpsPerBlock * GPW) {
    const int64_t vi = wi + grp;
    const int64_t v = vi / HG;
    const int col = (int)(vi % HG) * (128 * CPL) + lg * 4;
    const bool act = vi < items && col < HD;
    float pl = 0.f, pr = 0.f;
    if (act) {
#pragma unroll
      for (int c = 0; c < CPL; ++c) {
        const float4 f = ldg4(feat + (size_t)v * HD + col + 128 * c);
        const float ql = dot4(f, ldg4(attn_l + col + 128 * c)), qr = dot4(f, ldg4(attn_r + col + 128 * c));
        pl = c == 0 ? ql : pl + ql;
        pr = c == 0 ? qr : pr + qr;
      }
    }
    pl = group_sum_rt(pl, lph);
    pr = group_sum_rt(pr, lph);
    if (act && (col & (D - 1)) == 0) {
      el[(size_t)v * H + (col >> d_shift)] = pl;
      er[(size_t)v * H + (col >> d_shift)] = pr;
    }
  }
}

// d_attn_l[h,d] = sum_n d_el[n,h] * feat[n,h,d], d_attn_r likewise: lane-local float4 accumulators over a persistent
// grid (warp w keeps slice w % HG for all its rows), per-block double partials [2*H*D], fixed-order finalize.
// d_feat != null: the same pass also finishes the feature gradient, d_feat[n,h,:] += d_er[n,h] * attn_r[h,:] (the
// destination-side score gradient, only complete after gat_bwd_der_kernel).
// Dynamic smem: [warps][2][128] floats
template <int G>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
attn_scores_bwd_kernel(const float* __restrict__ feat, const float* __restrict__ d_el, const float* __restrict__ d_er,
                       int64_t n, int H, int D, int d_shift, int HG, double* __restrict__ partials,
                       float* __restrict__ d_feat, const float* __restrict__ attn_r) {
  constexpr int GPW = 32 / G;
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G;
  const int HD = H * D;
  const int64_t nW = (int64_t)gridDim.x * kWarpsPerBlock, usable = nW - nW % HG;
  const int64_t wg = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  const int hg = (int)(wg % HG);
  const int col = hg * 128 + lg * 4;
  const bool col_ok = col < HD;
  const int h = col_ok ? (col >> d_shift) : 0;
  float4 al = zero4(), ar = zero4();
  if (wg < usable && col_ok) {
    const float4 arv = d_feat != nullptr ? ldg4(attn_r + col) : zero4();
    for (int64_t v = (wg / HG) * GPW + grp; v < n; v += (usable / HG) * GPW) {
      const float4 f = ldg4(feat + (size_t)v * HD + col);
      const float de = __ldg(d_er + (size_t)v * H + h);
      fma4(al, __ldg(d_el + (size_t)v * H + h), f);
      fma4(ar, de, f);
      if (d_feat != nullptr) {
        float4 x = *reinterpret_cast<const float4*>(d_feat + (size_t)v * HD + col);
        fma4(x, de, arv);
        st4(d_feat + (size_t)v * HD + col, x);
      }
    }
  }
  // fold the lane groups of the warp (same columns), then the warps of the block that own the same slice
#pragma unroll
  for (int o = G; o < 32; o <<= 1) {
    al.x += __shfl_xor_sync(0xffffffffu, al.x, o); al.y += __shfl_xor_sync(0xffffffffu, al.y, o);
    al.z += __shfl_xor_sync(0xffffffffu, al.z, o); al.w += __shfl_xor_sync(0xffffffffu, al.w, o);
    ar.x += __shfl_xor_sync(0xffffffffu, ar.x, o); ar.y += __shfl_xor_sync(0xffffffffu, ar.y, o);
    ar.z += __shfl_xor_sync(0xffffffffu, ar.z, o); ar.w += __shfl_xor_sync(0xffffffffu, ar.w, o);
  }
  float* mine = smem + (size_t)warp * 256;
  if (lane < G) {
    st4(mine + lg * 4, al);
    st4(mine + 128 + lg * 4, ar);
  }
  __syncthreads();
  double* outp = partials + (size_t)blockIdx.x * 2 * HD;
  for (int i = threadIdx.x; i < 2 * HD; i += blockDim.x) {
    const int c = i % HD, which = i / HD;
    double sum = 0.0;
    for (int w = 0; w < kWarpsPerBlock; ++w)  // warps of this block that own slice c/128, in warp order
      if (((int64_t)blockIdx.x * kWarpsPerBlock + w) % HG == c / 128 && (c & 127) < G * 4)
        sum += (double)smem[(size_t)w * 256 + which * 128 + (c & 127)];
    outp[i] = sum;
  }
}

// =================================================================================================
// REGATv2 forward, row-group mapping (as gat_fwd_rg_kernel): the gathered fs[src] slice feeds both the logit
// (sum_d attn*LeakyReLU(fs+fd), reduced by a compile-time butterfly over the LPH = min(G, D/4) lanes of a head) and the
// aggregation; online softmax per batch of U edges.  Nothing [E,H,D]-sized is ever written.
// Dynamic smem: w_s[R*H]
// Training (lcsr / qmask != null): the raw logit of every (CSR slot, head) and the sign of every component of
// q = fs[u] + fd[v] (LeakyReLU' is ONE BIT per feature: four warp ballots -> a 128-bit mask per (slot, 128-float slice))
// are stored for the backward, 4H + 16*ceil(HD/128) bytes per edge -- the only place where fs[u] and fd[v] meet without
// an extra gather is this pass.
#ifndef REGNN_V2F_BLOCKS
#define REGNN_V2F_BLOCKS 4
#endif
// CPL as gat_bwd_edges_kernel; a wide head still stores one 128-bit mask per (slot, 128-float slice), one per chunk
template <int G, int LPH, bool EXTRA, bool HASH = false, int CPL = 1>   // EXTRA / HASH as gat_fwd_rg_kernel
__global__ void __launch_bounds__(kWarpsPerBlock * 32, REGNN_WIDE_BLOCKS(CPL, REGNN_V2F_BLOCKS))
gatv2_fwd_rg_kernel(AttnArgs a, float* __restrict__ lcsr, uint32_t* __restrict__ qmask) {
  static_assert(EXTRA || !HASH, "the hashed dropout factor needs the edge ids");
  constexpr int U = CPL == 1 ? kUG : 2;   // a wide head holds U * CPL gathered float4 per lane
  static_assert(G % U == 0, "a batch must not straddle a cooperative slot load");
  extern __shared__ __align__(16) float smem[];
  float* w_s = smem;
  load_rel_table(w_s, a);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G, gbase = lane & ~(G - 1);
  const int H = a.H, HD = H * a.D;
  const int64_t wi = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  if (wi >= rg_num_work(a, G, CPL)) return;  // warp-uniform
  const RowItem it = rg_item<G, CPL>(a, wi, grp);
  const int col = it.hg * (128 * CPL) + lg * 4;
  const bool col_ok = col < HD;
  const int h = col_ok ? (col >> a.d_shift) : 0;
  const bool act = it.v >= 0 && col_ok;
  const bool leader = act && (col & (a.D - 1)) == 0;
  const int len = it.v >= 0 ? it.len : 0;
  const int maxlen = __reduce_max_sync(0xffffffffu, len);
  const bool has_rel = a.etype != nullptr;
  float4 fdv[CPL], at[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    fdv[c] = zero4();
    at[c] = zero4();
    if (act) fdv[c] = ldg4(a.fd + (size_t)it.v * HD + col + 128 * c);
    if (col_ok) at[c] = ldg4(a.el + col + 128 * c);
  }
  const char* fbytes = reinterpret_cast<const char*>(a.feat + (col_ok ? col : 0));
  const uint32_t fpitch = (uint32_t)HD * 4u;
  const float* w_h = w_s + h;
  const int32_t* ip = a.indices + it.begin;
  const uint8_t* ep = a.etype + it.begin;
  const int32_t* eidp = a.eid + it.begin;
  // saved outputs: 32-bit element offsets from the kernel-parameter bases (E * max(H, HG) < 2^32, checked by the caller)
  const uint32_t moff = (uint32_t)it.begin * (uint32_t)a.hg_count + (uint32_t)(it.hg * CPL);
  const uint32_t loff = (uint32_t)it.begin * (uint32_t)H + (uint32_t)h;
  float4 acc[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) acc[c] = zero4();
  float m = -INFINITY, s = 0.f;

  for (int t0 = 0; t0 < maxlen; t0 += G) {
    int bi = -1, be = 0, beid = 0;
    {
      const int t = t0 + lg;
      if (t < len) {
        bi = __ldg(ip + t);
        if (has_rel) be = __ldg(ep + t);
        if (EXTRA) beid = __ldg(eidp + t);
#if REGNN_FWD_PF
        {
          const char* fr = reinterpret_cast<const char*>(a.feat + it.hg * 128 * CPL) + (uint64_t)(uint32_t)bi * fpitch;
          const int nl = (min(128 * CPL, HD - it.hg * 128 * CPL) * 4 + REGNN_PF_BYTES - 1) / REGNN_PF_BYTES;
          for (int k = 0; k < nl; ++k) prefetch_l2(fr + k * REGNN_PF_BYTES);
        }
#endif
      }
    }
    const int cnt = min(G, maxlen - t0);
    for (int j = 0; j < cnt; j += U) {
      float4 x[U][CPL];
      float l[U];
      int si[U], seid[EXTRA ? U : 1];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        si[u] = __shfl_sync(0xffffffffu, bi, gbase + j + u);
#pragma unroll
        for (int c = 0; c < CPL; ++c)
          x[u][c] = (si[u] >= 0 && col_ok)
                        ? ldg4(reinterpret_cast<const float*>(fbytes + (uint64_t)(uint32_t)si[u] * fpitch + 512 * c))
                        : zero4();
      }
      float bm = -INFINITY;
#pragma unroll
      for (int u = 0; u < U; ++u) {   // U independent head reductions
        float4 q[CPL];
#pragma unroll
        for (int c = 0; c < CPL; ++c) q[c] = add4(x[u][c], fdv[c]);
        float lu = dot4(at[0], leaky4(q[0], a.slope));
#pragma unroll
        for (int c = 1; c < CPL; ++c) lu += dot4(at[c], leaky4(q[c], a.slope));
        lu = group_sum<LPH>(lu);
        if (has_rel) lu += w_h[__shfl_sync(0xffffffffu, be, gbase + j + u) * H];
        if (EXTRA) seid[u] = __shfl_sync(0xffffffffu, beid, gbase + j + u);
        l[u] = si[u] >= 0 ? lu : -INFINITY;
        bm = fmaxf(bm, l[u]);
        if (qmask != nullptr) {   // warp-uniform
#pragma unroll
          for (int c = 0; c < CPL; ++c) {
            uint4 b;
            b.x = __ballot_sync(0xffffffffu, q[c].x > 0.f); b.y = __ballot_sync(0xffffffffu, q[c].y > 0.f);
            b.z = __ballot_sync(0xffffffffu, q[c].z > 0.f); b.w = __ballot_sync(0xffffffffu, q[c].w > 0.f);
            if (G < 32) {
              constexpr uint32_t gm = G < 32 ? (1u << G) - 1u : 0xffffffffu;
              b.x = (b.x >> gbase) & gm; b.y = (b.y >> gbase) & gm; b.z = (b.z >> gbase) & gm; b.w = (b.w >> gbase) & gm;
            }
            const uint32_t t = (uint32_t)(t0 + j + u);
            if (si[u] >= 0 && lg == 0)   // 16 bytes per (slot, slice)
              reinterpret_cast<uint4*>(qmask)[moff + t * (uint32_t)a.hg_count + c] = b;
            if (c == CPL - 1 && si[u] >= 0 && leader) lcsr[loff + t * (uint32_t)H] = lu;
          }
        }
      }
      if (bm > -INFINITY) {  // uniform within a lane group
        const float m_new = fmaxf(m, bm);
        const float sc = fast_exp(m - m_new);
        m = m_new;
        s *= sc;
#pragma unroll
        for (int c = 0; c < CPL; ++c) scale4(acc[c], sc);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          float p = fast_exp(l[u] - m_new);  // 0 for a missing slot
          s += p;
          if (EXTRA && si[u] >= 0 && act) {
            const size_t o = (size_t)seid[u] * H + h;
            if (a.o3 != nullptr && leader) a.o3[o] = l[u];
            if (HASH) p *= hashed_keep(a, seid[u], h);
            else if (a.keep != nullptr) p *= __ldg(a.keep + o);
          }
#pragma unroll
          for (int c = 0; c < CPL; ++c) fma4(acc[c], p, x[u][c]);
        }
      }
    }
  }

  if (it.frag) {
#pragma unroll
    for (int c = 0; c < CPL; ++c)
      if (act) st4(a.p0 + (size_t)it.fi * HD + col + 128 * c, acc[c]);
    if (leader) {
      a.p1[(size_t)it.fi * H + h] = m;
      a.p2[(size_t)it.fi * H + h] = s;
    }
    return;
  }
  const float inv = s > 0.f ? 1.f / s : 0.f;
  const float mm = len > 0 ? m : 0.f;
  if (act) {
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      scale4(acc[c], inv);
      st4(a.o0 + (size_t)it.v * HD + col + 128 * c, acc[c]);
    }
    if (leader) {
      a.o1[(size_t)it.v * H + h] = mm;
      a.o2[(size_t)it.v * H + h] = s;
    }
  }
  if (EXTRA && a.o3 != nullptr) {
    __syncwarp();
    if (act)
      for (int t = lg & (LPH - 1); t < len; t += LPH) {
        const size_t o = (size_t)eidp[t] * H + h;
        float av = __expf(a.o3[o] - mm) * inv;
        if (HASH) av *= hashed_keep(a, eidp[t], h);
        else if (a.keep != nullptr) av *= a.keep[o];
        a.o3[o] = av;
      }
  }
}

// =================================================================================================
// REGATv2 backward as ONE gather pass + one streaming pass.  For an edge e = (u -> v), head h:
//   a_e = exp(l_e - m_v) / s_v,  da_e = <fs[u], G[v]>,  dl_e = a_e keep_e da_e - a_e S_v,  S_v = <out[v], G[v]>
//   d_fs[u] = sum_{Out(u)} a_e keep_e G[v] + attn (.) T_src[u],    T_src[u] = sum_{Out(u)} dl_e phi_e
//   d_fd[v] = attn (.) T_dst[v],                                    T_dst[v] = sum_{In(v)}  dl_e phi_e
//   d_attn  = sum_e dl_e LeakyReLU(fs[u]+fd[v]) = sum_u fs[u] (.) T_src[u] + sum_v fd[v] (.) T_dst[v]
// with phi_e = LeakyReLU'(fs[u]+fd[v]) in {1, slope}^D, one bit per feature.  The forward stored l_e per (slot, head)
// and the bits of phi_e per (slot, 128-float slice); with the per-destination statistics (m, 1/s, S) of
// gat_bwd_stats_kernel every quantity of the source-major pass is local to the lane that owns fs[u] -- the
// destination-major GATHER pass of round 1 / the first half of round 2 (one more 4HD-byte row per edge) is gone:
//   gatv2_bwd_edges_kernel      source-major, gathers G[v]: d_fs rows, dl per slot, block partials of fs (.) T_src
//   gatv2_bwd_dst_stream_kernel destination-major, NO gather: streams dl + sign masks in slot order -> d_fd, fd (.) T_dst
//   gat_bwd_bins_kernel         relation bins of dl (streaming)
// Measured on the MAG graph (H8 D16, 5.0 - 5.3 ms, 22 GB of DRAM traffic at 4.3 TB/s) and dropped: L2 prefetch of
// everything a slot will need (G row, statistics, logit, mask) issued with the cooperative index load: no change; one
// record per slot (logits and masks adjacent, dl written in place over the logit): 6.1 ms (the in-place store orders the
// loads of the next round behind it); statistics packed to (rowmax + log rowsum, S) float2, half the bytes: 5.8 ms, and
// ex2.approx instead of __expf: +0.4 ms -- ptxas then issues the loads of the second edge of a round after the math of
// the first (one edge in flight instead of two); 4 or 6 blocks per SM instead of 5: 6.1 / 5.5 ms.
#define REGNN_V2_STAGE_CHUNKS 592   // first-stage blocks of the d_attn column sum (4 per SM)
#ifndef REGNN_V2D_UD
#define REGNN_V2D_UD 4   // slots in flight per lane in the streaming pass
#endif
#ifndef REGNN_V2E_BLOCKS
#define REGNN_V2E_BLOCKS 5
#endif
// sum_e dl_e * phi_e with phi in {1, slope}:  slope * sum_e dl_e + (1 - slope) * sum_{e: bit set} dl_e -- one predicated add
// per component and edge (lanebit = 1 << lane-in-group).
struct PhiAcc {
  float4 p;   // sum over the edges whose bit is set
  float d;    // sum over all edges
};
__device__ __forceinline__ void phi_add(PhiAcc& t, float dl, uint4 mb, uint32_t lanebit) {
  t.d += dl;
  if (mb.x & lanebit) t.p.x += dl;
  if (mb.y & lanebit) t.p.y += dl;
  if (mb.z & lanebit) t.p.z += dl;
  if (mb.w & lanebit) t.p.w += dl;
}
__device__ __forceinline__ float4 phi_total(const PhiAcc& t, float slope) {
  const float b = slope * t.d, k = 1.f - slope;
  return make_float4(fmaf(k, t.p.x, b), fmaf(k, t.p.y, b), fmaf(k, t.p.z, b), fmaf(k, t.p.w, b));
}
__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }

// AttnArgs: indptr/indices/eid = indptr_t/indices_t/slot_t, feat = fs, fd = stats (float4[N*H]), el = attn, a_csr = the
// stored logits, a_csr_eid = slot -> edge id (keep / dropout only), o0 = d_fs, o2 = dl per slot.  dat_part: [gridDim.x][H*D].
// CPL as gat_bwd_edges_kernel: warp w of a block keeps the CPL slices of item group (block * warps + w) % (HG / CPL)
template <int G, int LPH, bool KEEP, bool HASH = false, int CPL = 1>   // KEEP / HASH as gat_bwd_edges_kernel
__global__ void __launch_bounds__(kWarpsPerBlock * 32, REGNN_WIDE_BLOCKS(CPL, REGNN_V2E_BLOCKS))
gatv2_bwd_edges_kernel(AttnArgs a, const uint32_t* __restrict__ qmask, float* __restrict__ dat_part) {
  static_assert(KEEP || !HASH, "HASH is a dropout mode");
  constexpr int U = 2;
  static_assert(G % U == 0, "a round must not straddle a slot batch");
  __shared__ __align__(16) float dat_s[kWarpsPerBlock * 128 * CPL];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G, gbase = lane & ~(G - 1);
  const int H = a.H, HD = H * a.D, HG = a.hg_count;
  const int64_t wi = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  RowItem it{-1, 0, 0, 0, 0, false};
  if (wi < rg_num_work(a, G, CPL)) it = rg_item<G, CPL>(a, wi, grp);
  const int col = it.hg * (128 * CPL) + lg * 4;
  const bool col_ok = col < HD;
  const int h = col_ok ? (col >> a.d_shift) : 0;
  const bool act = it.v >= 0 && col_ok;
  const bool leader = act && (col & (a.D - 1)) == 0;
  const int len = it.v >= 0 ? it.len : 0;
  const int maxlen = __reduce_max_sync(0xffffffffu, len);
  float4 fu[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) fu[c] = act ? ldg4(a.feat + (size_t)it.v * HD + col + 128 * c) : zero4();
  const char* gbytes = reinterpret_cast<const char*>(a.G + (col_ok ? col : 0));
  const char* sbytes = reinterpret_cast<const char*>(a.fd) + (size_t)h * 16;
  const uint32_t gpitch = (uint32_t)HD * 4u, spitch = (uint32_t)H * 16u;
  const float* lh = a.a_csr + h;
  float* dlh = a.o2 + h;
  const uint4* mk = reinterpret_cast<const uint4*>(qmask) + it.hg * CPL;
  const int32_t* ip = a.indices + it.begin;
  const int32_t* sp = a.eid + it.begin;
  float4 acc[CPL];
  PhiAcc ta[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    acc[c] = zero4();
    ta[c] = PhiAcc{zero4(), 0.f};
  }
  const uint32_t lanebit = 1u << lg;

  for (int t0 = 0; t0 < maxlen; t0 += G) {
    int bi = -1, bs = 0;
    {
      const int t = t0 + lg;
      if (t < len) {
        bi = __ldg(ip + t);
        bs = __ldg(sp + t);
      }
    }
    const int cnt = min(G, maxlen - t0);
    for (int j = 0; j < cnt; j += U) {
      float4 x[U][CPL];
      float4 st[U];
      uint4 mb[U][CPL];
      float lv[U];
      int sd[U], ss[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        sd[u] = __shfl_sync(0xffffffffu, bi, gbase + j + u);
        ss[u] = __shfl_sync(0xffffffffu, bs, gbase + j + u);
        const bool ok = sd[u] >= 0 && col_ok;
#pragma unroll
        for (int c = 0; c < CPL; ++c)
          x[u][c] = ok ? ldg4(reinterpret_cast<const float*>(gbytes + (uint64_t)(uint32_t)sd[u] * gpitch + 512 * c)) : zero4();
        // missing slot: rowmax = +inf makes exp(. - rowmax) = 0, so a = dl = 0 without per-edge masks
        st[u] = ok ? __ldg(reinterpret_cast<const float4*>(sbytes + (uint64_t)(uint32_t)sd[u] * spitch))
                   : make_float4(0.f, INFINITY, 0.f, 0.f);
        lv[u] = ok ? __ldg(lh + (uint64_t)(uint32_t)ss[u] * (uint32_t)H) : 0.f;
#pragma unroll
        for (int c = 0; c < CPL; ++c)
          mb[u][c] = ok ? __ldg(mk + (uint64_t)(uint32_t)ss[u] * (uint32_t)HG + c) : make_uint4(0u, 0u, 0u, 0u);
      }
      float da[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float p = dot4(fu[0], x[u][0]);
#pragma unroll
        for (int c = 1; c < CPL; ++c) p += dot4(fu[c], x[u][c]);
        da[u] = group_sum<LPH>(p);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float aa = __expf(lv[u] - st[u].y) * st[u].z;
        float at = aa;
        if (KEEP) {
          if (sd[u] >= 0 && act) {
            const int e = __ldg(a.a_csr_eid + ss[u]);
            at *= HASH ? hashed_keep(a, e, h) : __ldg(a.keep + (size_t)e * H + h);
          }
        }
        const float dl = at * da[u] - aa * st[u].w;
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
          fma4(acc[c], at, x[u][c]);
          phi_add(ta[c], dl, mb[u][c], lanebit);
        }
        if (leader && sd[u] >= 0) dlh[(uint64_t)(uint32_t)ss[u] * (uint32_t)H] = dl;
      }
    }
  }
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
    float4 c = zero4();
    const float4 T = phi_total(ta[k], a.slope);
    if (act) {
      const float4 at4 = ldg4(a.el + col + 128 * k);
      acc[k].x = fmaf(at4.x, T.x, acc[k].x); acc[k].y = fmaf(at4.y, T.y, acc[k].y);
      acc[k].z = fmaf(at4.z, T.z, acc[k].z); acc[k].w = fmaf(at4.w, T.w, acc[k].w);
      st4((it.frag ? a.p0 + (size_t)it.fi * HD : a.o0 + (size_t)it.v * HD) + col + 128 * k, acc[k]);
      c = mul4(fu[k], T);
    }
    // d_attn share of this block: fold the lane groups of the warp (same columns, different rows), then the warps that
    // own the same 128-float slice, in warp order
#pragma unroll
    for (int o = G; o < 32; o <<= 1) {
      c.x += __shfl_xor_sync(0xffffffffu, c.x, o); c.y += __shfl_xor_sync(0xffffffffu, c.y, o);
      c.z += __shfl_xor_sync(0xffffffffu, c.z, o); c.w += __shfl_xor_sync(0xffffffffu, c.w, o);
    }
    if (lane < G) st4(dat_s + (warp * CPL + k) * 128 + lg * 4, c);
  }
  __syncthreads();
  float* outp = dat_part + (size_t)blockIdx.x * HD;
  const int NI = HG / CPL;   // item groups: slices (CPL = 1) or heads
  for (int i = threadIdx.x; i < HD; i += blockDim.x) {
    float sum = 0.f;
    const int sl = i / 128;
    if ((i & 127) < G * 4)
      for (int w = 0; w < kWarpsPerBlock; ++w)
        if (NI == 1 || (int)(((int64_t)blockIdx.x * kWarpsPerBlock + w) % NI) == sl / CPL)
          sum += dat_s[(w * CPL + sl % CPL) * 128 + (i & 127)];
    outp[i] = sum;
  }
}

// First stage of the column sum of the [nb][W] float block partials above: block c sums rows [c*per, (c+1)*per) in row
// order into doubles (threads over columns; W < 256: 256/W row phases, folded in phase order).  out: [gridDim.x][W].
__global__ void __launch_bounds__(256)
colsum_stage_kernel(const float* __restrict__ part, int64_t nb, int W, int64_t per, double* __restrict__ out) {
  __shared__ double fold[256];
  const int nr = W < 256 ? 256 / W : 1;
  const int64_t b0 = (int64_t)blockIdx.x * per, b1 = min(nb, b0 + per);
  for (int c0 = 0; c0 < W; c0 += 256) {
    const int t = threadIdx.x;
    const int c = c0 + (nr > 1 ? t % W : t), r0 = nr > 1 ? t / W : 0;
    const bool on = c < W && r0 < nr;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (on) {
      int64_t b = b0 + r0;
      const int64_t step = nr;
      for (; b + 3 * step < b1; b += 4 * step) {
        const float v0 = __ldg(part + (size_t)b * W + c), v1 = __ldg(part + (size_t)(b + step) * W + c);
        const float v2 = __ldg(part + (size_t)(b + 2 * step) * W + c), v3 = __ldg(part + (size_t)(b + 3 * step) * W + c);
        s0 += v0; s1 += v1; s2 += v2; s3 += v3;
      }
      for (; b < b1; b += step) s0 += __ldg(part + (size_t)b * W + c);
    }
    const double s = (s0 + s1) + (s2 + s3);
    if (nr > 1) {
      fold[t] = on ? s : 0.0;
      __syncthreads();
      if (t < W) {
        double tot = 0.0;
        for (int r = 0; r < nr; ++r) tot += fold[r * W + t];
        out[(size_t)blockIdx.x * W + t] = tot;
      }
      __syncthreads();
    } else if (on) {
      out[(size_t)blockIdx.x * W + c] = s;
    }
  }
}

// Destination-major streaming pass (no gather): T_dst[v] = sum over the CSR slots of v of dl[slot,h] * phi[slot] from
// the per-slot dl and sign masks (consecutive slots = consecutive addresses, every lane of a group reads the same 16-byte
// mask and its head's dl), d_fd[v] = attn (.) T_dst[v], and the lane-local d_attn share fd[v] (.) T_dst[v] of a
// persistent grid (a warp keeps ONE 128-float slice for all its rows).  Fragments of long rows first (partial rows to
// p0; the d_attn share is linear in T, so fragments contribute directly).
// AttnArgs: indptr (CSR), fd, el = attn, d_csr = dl, o2 = d_fd, partials [gridDim.x][H*D].
#ifndef REGNN_V2DS_BLOCKS
#define REGNN_V2DS_BLOCKS 5
#endif
template <int G>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, REGNN_V2DS_BLOCKS)
gatv2_bwd_dst_stream_kernel(AttnArgs a, const uint32_t* __restrict__ qmask) {
  constexpr int GPW = 32 / G, UD = REGNN_V2D_UD;
  __shared__ __align__(16) float dat_s[kWarpsPerBlock * 128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G;
  const int H = a.H, HD = H * a.D, HG = a.hg_count;
  const int64_t nW = (int64_t)gridDim.x * kWarpsPerBlock, usable = nW - nW % HG;
  const int64_t wg = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  const int hg = (int)(wg % HG);
  const int col = hg * 128 + lg * 4;
  const bool col_ok = col < HD;
  const int h = col_ok ? (col >> a.d_shift) : 0;
  const int64_t nrows = a.row_end - a.row_begin;
  const int64_t nitems = a.nfrag + nrows;
  const uint4* mk = reinterpret_cast<const uint4*>(qmask) + hg;
  const float* dh = a.d_csr + h;
  float4 dat = zero4();

  const uint32_t lanebit = 1u << lg;
  for (int64_t rgi = wg / HG; wg < usable && rgi * GPW < nitems; rgi += usable / HG) {
    const int64_t ri = rgi * GPW + grp;
    int64_t v = -1, fi = 0;
    int begin = 0, len = 0;
    bool frag = false;
    if (ri < nitems) {
      if (ri < a.nfrag) {
        frag = true;
        fi = ri;
        const int64_t r = a.frag_row[ri];
        if (r >= a.row_begin && r < a.row_end) {
          v = r;
          begin = a.frag_begin[ri];
          len = min(a.threshold, a.indptr[r + 1] - begin);
        }
      } else {
        const int64_t r = a.row_begin + (ri - a.nfrag);
        const int b = a.indptr[r], l = a.indptr[r + 1] - b;
        if (l <= a.threshold) {
          v = r;
          begin = b;
          len = l;
        }
      }
    }
    if (v < 0 || !col_ok) continue;   // no warp-level primitives below
    prefetch_l2(a.fd + (size_t)v * HD + col);   // read after the slots (registers for loads in flight instead)
    PhiAcc ta{zero4(), 0.f};
    // running pointers, 32-bit strides: the loop body is the two loads + 9 arithmetic instructions per slot
    const float* dp = dh + (size_t)begin * H;
    const uint4* mp = mk + (size_t)begin * HG;
    const uint32_t dstep = (uint32_t)H, mstep = (uint32_t)HG;
    int left = len;
    for (; left >= UD; left -= UD, dp += UD * dstep, mp += UD * mstep) {   // full batches: no predicates
      float dl[UD];
      uint4 mb[UD];
#pragma unroll
      for (int u = 0; u < UD; ++u) {
        dl[u] = __ldg(dp + u * dstep);
        mb[u] = __ldg(mp + u * mstep);
      }
#pragma unroll
      for (int u = 0; u < UD; ++u) phi_add(ta, dl[u], mb[u], lanebit);
    }
    if (left > 0) {
      float dl[UD - 1];
      uint4 mb[UD - 1];
#pragma unroll
      for (int u = 0; u < UD - 1; ++u) {
        const bool ok = u < left;
        dl[u] = ok ? __ldg(dp + u * dstep) : 0.f;
        mb[u] = ok ? __ldg(mp + u * mstep) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < UD - 1; ++u) phi_add(ta, dl[u], mb[u], lanebit);
    }
    const float4 T = phi_total(ta, a.slope);
    const float4 fdv = ldg4(a.fd + (size_t)v * HD + col);
    st4((frag ? a.p0 + (size_t)fi * HD : a.o2 + (size_t)v * HD) + col, mul4(ldg4(a.el + col), T));
    dat.x = fmaf(fdv.x, T.x, dat.x); dat.y = fmaf(fdv.y, T.y, dat.y);
    dat.z = fmaf(fdv.z, T.z, dat.z); dat.w = fmaf(fdv.w, T.w, dat.w);
  }
#pragma unroll
  for (int o = G; o < 32; o <<= 1) {
    dat.x += __shfl_xor_sync(0xffffffffu, dat.x, o); dat.y += __shfl_xor_sync(0xffffffffu, dat.y, o);
    dat.z += __shfl_xor_sync(0xffffffffu, dat.z, o); dat.w += __shfl_xor_sync(0xffffffffu, dat.w, o);
  }
  if (lane < G) st4(dat_s + warp * 128 + lg * 4, dat);
  __syncthreads();
  double* outp = a.partials + (size_t)blockIdx.x * HD;
  for (int i = threadIdx.x; i < HD; i += blockDim.x) {
    double sum = 0.0;
    if ((i & 127) < G * 4)
      for (int w = 0; w < kWarpsPerBlock; ++w)  // warps of this block that own slice i/128, in warp order
        if (((int64_t)blockIdx.x * kWarpsPerBlock + w) % HG == i / 128) sum += (double)dat_s[w * 128 + (i & 127)];
    outp[i] = sum;
  }
}

// =================================================================================================
// Merges the fragments of every long row of a forward pass (online-softmax combine in fragment order):
//   M = max_f m_f;  S = sum_f s_f*exp(m_f-M);  out = sum_f acc_f*exp(m_f-M) / S
// and, for get_attention, normalises the row's stored logits.  One warp per (long row, head group).  HASH: the dropout
// factor of get_attention from hashed_keep.
template <bool HASH>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
attn_frag_finalize_kernel(AttnArgs a, const int32_t* __restrict__ long_rows,
                          const int32_t* __restrict__ frag_ptr, int num_long) {
  const int H = a.H, HD = H * a.D;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int HG = num_groups(a);
  const int64_t wi = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
  const int l = (int)(wi / HG);
  if (l >= num_long) return;
  const int64_t v = long_rows[l];
  if (v < a.row_begin || v >= a.row_end) return;
  const Group g = make_group(a, (int)(wi % HG), lane);
  const int f0 = frag_ptr[l], f1 = frag_ptr[l + 1];
  const size_t hh = g.hl;  // every lane tracks the statistics of its own head (redundant within a head)
  float M = -INFINITY;
  for (int f = f0; f < f1; ++f) M = fmaxf(M, a.p1[(size_t)f * H + hh]);
  float S = 0.f;
  float4 acc = zero4();
  for (int f = f0; f < f1; ++f) {
    const float sc = expf(a.p1[(size_t)f * H + hh] - M);
    S += a.p2[(size_t)f * H + hh] * sc;
    if (g.ok) fma4(acc, sc, ldg4(a.p0 + (size_t)f * HD + g.col));
  }
  const float inv = S > 0.f ? 1.f / S : 0.f;
  if (g.ok) {
    scale4(acc, inv);
    st4(a.o0 + (size_t)v * HD + g.col, acc);
    if (g.leader) {
      a.o1[(size_t)v * H + hh] = M;
      a.o2[(size_t)v * H + hh] = S;
    }
  }
  if (a.o3 != nullptr && ((g.hg << 7) & (a.D - 1)) == 0) {   // D > 128: only the warp of a head's first slice
    __syncwarp();
    const int s0 = a.indptr[v], len = a.indptr[v + 1] - s0;
    for (int i = lane; i < len * g.nh; i += 32) {
      const int h = g.h_lo + i % g.nh;
      const int e = a.eid[s0 + i / g.nh];
      const size_t o = (size_t)e * H + h;
      const float s = a.o2[(size_t)v * H + h];
      float av = expf(a.o3[o] - a.o1[(size_t)v * H + h]) * (s > 0.f ? 1.f / s : 0.f);
      if (HASH) av *= hashed_keep(a, e, h);
      else if (a.keep != nullptr) av *= a.keep[o];
      a.o3[o] = av;
    }
  }
}

// out[v][c] = sum over the fragments of long row v of partial[f][c]  (fragment order; block per row)
__global__ void frag_rowsum_kernel(const int32_t* __restrict__ long_rows, const int32_t* __restrict__ frag_ptr,
                                   int num_long, const float* __restrict__ partial, int W,
                                   float* __restrict__ out, int64_t row_begin, int64_t row_end) {
  const int l = blockIdx.x;
  if (l >= num_long) return;
  const int64_t v = long_rows[l];
  if (v < row_begin || v >= row_end) return;
  const int f0 = frag_ptr[l], f1 = frag_ptr[l + 1];
  for (int c = threadIdx.x; c < W; c += blockDim.x) {
    float s = 0.f;
    for (int f = f0; f < f1; ++f) s += partial[(size_t)f * W + c];
    out[(size_t)v * W + c] = s;
  }
}

// ---- dispatch ---------------------------------------------------------------------------------------
static bool aligned16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

static int pick_c(int HD) {
  const int c = (HD / 4 + 31) / 32;
  if (c <= 1) return 1;
  if (c <= 2) return 2;
  if (c <= 4) return 4;
  if (c <= 8) return 8;
  return 0;
}

// Fills the fragment fields of `a` from the caller's row split; returns false if it is incomplete.
static bool apply_split(AttnArgs& a, const regnn_rowsplit_t* split, float* ws) {
  a.hg_count = (a.H * a.D + 127) / 128;
  a.d_shift = -1;
  for (int b = 2; b <= 10; ++b)
    if ((1 << b) == a.D) a.d_shift = b;
  a.nfrag = a.nfrag_pad = 0;
  a.threshold = 0x7fffffff;
  if (split == nullptr || split->num_frags <= 0) return true;
  if (!ws || !split->long_rows || !split->frag_ptr || !split->frag_row || !split->frag_begin || split->threshold <= 0)
    return false;
  a.frag_row = split->frag_row;
  a.frag_begin = split->frag_begin;
  a.nfrag = split->num_frags;
  a.nfrag_pad = a.nfrag;
  a.threshold = split->threshold;
  const size_t HD = (size_t)a.H * a.D;
  a.p0 = ws;
  a.p1 = ws + (size_t)a.nfrag * HD;
  a.p2 = a.p1 + (size_t)a.nfrag * a.H;
  return true;
}

static void launch_rowsum(const regnn_rowsplit_t* split, const float* partial, int W, float* out, int64_t rb,
                          int64_t re, cudaStream_t stream) {
  frag_rowsum_kernel<<<split->num_long, 128, 0, stream>>>(split->long_rows, split->frag_ptr, split->num_long, partial,
                                                          W, out, rb, re);
}

static int check_shape(const char* who, int H, int D, int R, bool has_rel, bool needs_dot) {
  REGNN_REQUIRE(H >= 1 && H <= REGNN_MAX_HEADS, REGNN_ERR_UNSUPPORTED_SHAPE, "%s: num_heads=%d outside [1,%d]", who, H, REGNN_MAX_HEADS);
  REGNN_REQUIRE(D >= 4 && D % 4 == 0, REGNN_ERR_UNSUPPORTED_SHAPE, "%s: head_dim=%d must be a positive multiple of 4", who, D);
  REGNN_REQUIRE(pick_c(H * D) != 0, REGNN_ERR_UNSUPPORTED_SHAPE, "%s: H*D=%d exceeds 1024", who, H * D);
  if (needs_dot) {
    // a wide head (D > 128) keeps D/128 float4 accumulators per lane: D = 1024 would need 32 floats of each
    REGNN_REQUIRE(D <= 512, REGNN_ERR_UNSUPPORTED_SHAPE, "%s: head_dim=%d exceeds 512 (the widest head of the attention kernels)",
                  who, D);
    REGNN_REQUIRE((D & (D - 1)) == 0, REGNN_ERR_UNSUPPORTED_SHAPE, "%s: head_dim=%d must be a power of two in [4,512]", who, D);
  }
  if (has_rel)
    REGNN_REQUIRE(R >= 1 && R <= REGNN_MAX_RELATIONS && R * H <= 4096, REGNN_ERR_UNSUPPORTED_SHAPE,
                  "%s: num_relations=%d (x %d heads) unsupported", who, R, H);
  return REGNN_OK;
}

#define REGNN_DISPATCH_C(KERNEL, GRID, SMEM)                                  \
  do {                                                                        \
    int rc_ = set_smem(KERNEL, SMEM);                                         \
    if (rc_ != REGNN_OK) return rc_;                                          \
    KERNEL<<<GRID, kWarpsPerBlock * 32, SMEM, stream>>>(a);                   \
  } while (0)

#define REGNN_DISPATCH_FINALIZE(GRID, HASH_)                                                                           \
  attn_frag_finalize_kernel<HASH_><<<GRID, kWarpsPerBlock * 32, 0, stream>>>(a, split->long_rows, split->frag_ptr,      \
                                                                             split->num_long)

static int head_groups(int H, int D) { return (H * D + 127) / 128; }
// 128-bit chunks per lane (CPL) of the kernels that reduce over a head: 1, or D/128 for a wide head (one warp per head)
static int head_chunks(int D) { return D > 128 ? D / 128 : 1; }

// lanes per row slice of the row-group REGAT kernels: min(H*D, 128) floats in 128-bit chunks, rounded up to 4/8/16/32
static int rg_lanes(int HD) { return HD > 64 ? 32 : (HD > 32 ? 16 : (HD > 16 ? 8 : 4)); }
// work items (warps) of a row-group kernel over `rows` rows, cpl chunks per lane (items per row: hg_count / cpl)
static int64_t rg_work(const AttnArgs& a, int64_t rows, int cpl = 1) {
  const int gpw = 32 / rg_lanes(a.H * a.D);
  const int64_t nrows = a.order != nullptr ? a.n_order : rows;
  return ((a.nfrag + nrows) * (a.hg_count / cpl) + gpw - 1) / gpw;
}
// row_order lists the rows of the FULL range that are not long: only usable when the call covers [0, N)
static void apply_order(AttnArgs& a, const int32_t* row_order, const regnn_rowsplit_t* split, int64_t rows) {
  a.order = nullptr;
  a.n_order = 0;
  if (row_order != nullptr && a.row_begin == 0) {
    a.order = row_order;
    a.n_order = rows - (a.nfrag > 0 ? split->num_long : 0);
  }
}

// Fills the dropout fields of `a` (dropout != NULL); returns false if the struct is inconsistent with the call's heads.
static bool apply_dropout(AttnArgs& a, const regnn_attn_dropout_t* dropout) {
  if (dropout == nullptr) return true;
  if (dropout->head_offset < 0 || dropout->num_heads_total < dropout->head_offset + a.H) return false;
  if (!(dropout->scale >= 0.f) || dropout->scale == INFINITY) return false;
  a.drop_key_lo = (uint32_t)dropout->key;
  a.drop_key_hi = (uint32_t)(dropout->key >> 32);
  a.drop_threshold = dropout->threshold;
  a.drop_scale = dropout->scale;
  a.drop_head_offset = dropout->head_offset;
  a.drop_heads_total = dropout->num_heads_total;
  return true;
}

}  // namespace regnn

using namespace regnn;

extern "C" int regnn_gat_fwd(const int32_t* indptr, const int32_t* indices, const int32_t* eid,
                             const uint8_t* etype_csr, const float* theta, float alpha,
                             int num_relations, const float* feat, const float* el, const float* er,
                             float negative_slope, const float* keep, const regnn_attn_dropout_t* dropout,
                             int num_heads, int head_dim, int64_t row_begin, int64_t row_end, float* out, float* rowmax,
                             float* rowsum, float* attn_out, const regnn_rowsplit_t* split, float* split_workspace,
                             const int32_t* row_order, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr && feat && el && er && out && rowmax && rowsum, REGNN_ERR_INVALID_ARG, "gat_fwd: null pointer");
  REGNN_REQUIRE(keep == nullptr || dropout == nullptr, REGNN_ERR_INVALID_ARG, "gat_fwd: keep and dropout are exclusive");
  REGNN_REQUIRE((keep == nullptr && dropout == nullptr && attn_out == nullptr) || eid != nullptr, REGNN_ERR_INVALID_ARG,
                "gat_fwd: keep/dropout/attn_out need eid");
  REGNN_REQUIRE(etype_csr == nullptr || theta != nullptr, REGNN_ERR_INVALID_ARG, "gat_fwd: etype without theta");
  int rc = check_shape("gat_fwd", num_heads, head_dim, num_relations, etype_csr != nullptr, true);  // as the backward: fail early
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(aligned16(feat) && aligned16(out), REGNN_ERR_INVALID_ARG, "gat_fwd: feat/out must be 16-byte aligned");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "gat_fwd: negative row range");
  if (rows == 0) return REGNN_OK;
  AttnArgs a{};
  a.indptr = indptr; a.indices = indices; a.eid = eid; a.etype = etype_csr; a.theta = theta; a.alpha = alpha;
  a.R = etype_csr ? num_relations : 0; a.feat = feat; a.el = el; a.er = er; a.slope = negative_slope; a.keep = keep;
  a.H = num_heads; a.D = head_dim; a.row_begin = row_begin; a.row_end = row_end;
  a.o0 = out; a.o1 = rowmax; a.o2 = rowsum; a.o3 = attn_out;
  REGNN_REQUIRE(apply_split(a, split, split_workspace), REGNN_ERR_INVALID_ARG, "gat_fwd: incomplete row split");
  REGNN_REQUIRE(apply_dropout(a, dropout), REGNN_ERR_INVALID_ARG, "gat_fwd: dropout heads / scale inconsistent");
  apply_order(a, row_order, split, rows);
  const size_t smem = sizeof(float) * ((size_t)a.R * num_heads) + 16;
  const unsigned grid = (unsigned)((rg_work(a, rows) + kWarpsPerBlock - 1) / kWarpsPerBlock);
  if (dropout != nullptr) {
    switch (rg_lanes(a.H * a.D)) {
      case 4: REGNN_DISPATCH_C((gat_fwd_rg_kernel<4, true, true>), grid, smem); break;
      case 8: REGNN_DISPATCH_C((gat_fwd_rg_kernel<8, true, true>), grid, smem); break;
      case 16: REGNN_DISPATCH_C((gat_fwd_rg_kernel<16, true, true>), grid, smem); break;
      default: REGNN_DISPATCH_C((gat_fwd_rg_kernel<32, true, true>), grid, smem); break;
    }
  } else if (keep != nullptr || attn_out != nullptr) {
    switch (rg_lanes(a.H * a.D)) {
      case 4: REGNN_DISPATCH_C((gat_fwd_rg_kernel<4, true>), grid, smem); break;
      case 8: REGNN_DISPATCH_C((gat_fwd_rg_kernel<8, true>), grid, smem); break;
      case 16: REGNN_DISPATCH_C((gat_fwd_rg_kernel<16, true>), grid, smem); break;
      default: REGNN_DISPATCH_C((gat_fwd_rg_kernel<32, true>), grid, smem); break;
    }
  } else {
    switch (rg_lanes(a.H * a.D)) {
      case 4: REGNN_DISPATCH_C((gat_fwd_rg_kernel<4, false>), grid, smem); break;
      case 8: REGNN_DISPATCH_C((gat_fwd_rg_kernel<8, false>), grid, smem); break;
      case 16: REGNN_DISPATCH_C((gat_fwd_rg_kernel<16, false>), grid, smem); break;
      default: REGNN_DISPATCH_C((gat_fwd_rg_kernel<32, false>), grid, smem); break;
    }
  }
  if (a.nfrag > 0) {
    const unsigned fgrid = (unsigned)(((int64_t)split->num_long * head_groups(a.H, a.D) + kWarpsPerBlock - 1) / kWarpsPerBlock);
    if (dropout != nullptr) REGNN_DISPATCH_FINALIZE(fgrid, true);
    else REGNN_DISPATCH_FINALIZE(fgrid, false);
  }
  return check_launch("regnn_gat_fwd");
}

extern "C" int regnn_gat_bwd_stats(const float* out, const float* Gd, const float* er, const float* rowmax,
                                   const float* rowsum, int64_t num_nodes, int num_heads, int head_dim, float* stats,
                                   void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(out && Gd && rowmax && rowsum && stats && num_nodes >= 0, REGNN_ERR_INVALID_ARG,   /* er == NULL (REGATv2): stats.x = 0 */
                "gat_bwd_stats: bad argument");
  int rc = check_shape("gat_bwd_stats", num_heads, head_dim, 0, false, true);
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(aligned16(out) && aligned16(Gd) && aligned16(stats), REGNN_ERR_INVALID_ARG,
                "gat_bwd_stats: 16-byte alignment required");
  if (num_nodes == 0) return REGNN_OK;
  AttnArgs a{};
  a.H = num_heads; a.D = head_dim;
  apply_split(a, nullptr, nullptr);
  const int G = rg_lanes(num_heads * head_dim), cpl = head_chunks(head_dim), ni = a.hg_count / cpl;
  const int64_t work = (num_nodes * ni + 32 / G - 1) / (32 / G);
  const int64_t want = (work + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const unsigned grid = (unsigned)(want < 148 * 16 ? want : 148 * 16);
#define REGNN_STATS(G_, C_)                                                                                              \
  gat_bwd_stats_kernel<G_, C_><<<grid, kWarpsPerBlock * 32, 0, stream>>>(out, Gd, er, rowmax, rowsum, num_nodes,       \
                                                                        num_heads, head_dim, a.d_shift, ni,           \
                                                                        reinterpret_cast<float4*>(stats))
  switch (G * cpl) {
    case 4: REGNN_STATS(4, 1); break;
    case 8: REGNN_STATS(8, 1); break;
    case 16: REGNN_STATS(16, 1); break;
    case 64: REGNN_STATS(32, 2); break;
    case 128: REGNN_STATS(32, 4); break;
    default: REGNN_STATS(32, 1); break;
  }
#undef REGNN_STATS
  return check_launch("regnn_gat_bwd_stats");
}

extern "C" int regnn_gat_bwd_edges(const int32_t* indptr_t, const int32_t* indices_t, const int32_t* slot_t,
                                   const uint8_t* etype_t, const int32_t* eid, const float* theta, float alpha,
                                   int num_relations, const float* feat, const float* el, const float* stats,
                                   float negative_slope, const float* keep, const regnn_attn_dropout_t* dropout,
                                   const float* Gd, int num_heads,
                                   int head_dim, int64_t row_begin, int64_t row_end, float* d_feat, float* d_el,
                                   float* dpre_csr, const float* attn_l, const regnn_rowsplit_t* split_t,
                                   float* split_workspace, const int32_t* row_order_t, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr_t && feat && el && stats && Gd && d_feat && d_el, /* per-edge arrays may be NULL when E == 0 */
                REGNN_ERR_INVALID_ARG, "gat_bwd_edges: null pointer");
  REGNN_REQUIRE(keep == nullptr || dropout == nullptr, REGNN_ERR_INVALID_ARG, "gat_bwd_edges: keep and dropout are exclusive");
  REGNN_REQUIRE((keep == nullptr && dropout == nullptr) || eid != nullptr, REGNN_ERR_INVALID_ARG,
                "gat_bwd_edges: keep/dropout need eid");
  REGNN_REQUIRE(etype_t == nullptr || theta != nullptr, REGNN_ERR_INVALID_ARG, "gat_bwd_edges: etype without theta");
  int rc = check_shape("gat_bwd_edges", num_heads, head_dim, num_relations, etype_t != nullptr, true);
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(aligned16(feat) && aligned16(Gd) && aligned16(d_feat) && aligned16(stats) && aligned16(attn_l),
                REGNN_ERR_INVALID_ARG, "gat_bwd_edges: 16-byte alignment required");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "gat_bwd_edges: negative row range");
  if (rows == 0) return REGNN_OK;
  AttnArgs a{};
  a.indptr = indptr_t; a.indices = indices_t; a.eid = slot_t; a.etype = etype_t; a.theta = theta; a.alpha = alpha;
  a.R = etype_t ? num_relations : 0; a.feat = feat; a.el = el; a.fd = stats; a.slope = negative_slope; a.keep = keep;
  a.a_csr_eid = eid; a.G = Gd; a.H = num_heads; a.D = head_dim; a.row_begin = row_begin; a.row_end = row_end;
  a.o0 = d_feat; a.o1 = d_el; a.o2 = dpre_csr; a.attn_l = attn_l;
  REGNN_REQUIRE(apply_split(a, split_t, split_workspace), REGNN_ERR_INVALID_ARG, "gat_bwd_edges: incomplete row split");
  REGNN_REQUIRE(apply_dropout(a, dropout), REGNN_ERR_INVALID_ARG, "gat_bwd_edges: dropout heads / scale inconsistent");
  apply_order(a, row_order_t, split_t, rows);
  const size_t smem = sizeof(float) * ((size_t)a.R * num_heads) + 16;
  const int cpl = head_chunks(head_dim);
  const unsigned grid = (unsigned)((rg_work(a, rows, cpl) + kWarpsPerBlock - 1) / kWarpsPerBlock);
  {
    const int G = rg_lanes(a.H * a.D), lph = min(G, head_dim / 4);
    bool launched = false;
#define REGNN_EDGES_CASE(G_, L_, C_)                                                                             \
  if (G == G_ && lph == L_ && cpl == C_) {                                                                       \
    if (dropout != nullptr) REGNN_DISPATCH_C((gat_bwd_edges_kernel<G_, L_, true, true, C_>), grid, smem);        \
    else if (keep != nullptr) REGNN_DISPATCH_C((gat_bwd_edges_kernel<G_, L_, true, false, C_>), grid, smem);     \
    else REGNN_DISPATCH_C((gat_bwd_edges_kernel<G_, L_, false, false, C_>), grid, smem);                         \
    launched = true;                                                                                             \
  }
    REGNN_EDGES_CASE(4, 1, 1) REGNN_EDGES_CASE(4, 2, 1) REGNN_EDGES_CASE(4, 4, 1)
    REGNN_EDGES_CASE(8, 1, 1) REGNN_EDGES_CASE(8, 2, 1) REGNN_EDGES_CASE(8, 4, 1) REGNN_EDGES_CASE(8, 8, 1)
    REGNN_EDGES_CASE(16, 1, 1) REGNN_EDGES_CASE(16, 2, 1) REGNN_EDGES_CASE(16, 4, 1) REGNN_EDGES_CASE(16, 8, 1)
    REGNN_EDGES_CASE(16, 16, 1)
    REGNN_EDGES_CASE(32, 1, 1) REGNN_EDGES_CASE(32, 2, 1) REGNN_EDGES_CASE(32, 4, 1) REGNN_EDGES_CASE(32, 8, 1)
    REGNN_EDGES_CASE(32, 16, 1) REGNN_EDGES_CASE(32, 32, 1) REGNN_EDGES_CASE(32, 32, 2) REGNN_EDGES_CASE(32, 32, 4)
#undef REGNN_EDGES_CASE
    REGNN_REQUIRE(launched, REGNN_ERR_UNSUPPORTED_SHAPE, "gat_bwd_edges: no kernel for H=%d D=%d", num_heads, head_dim);
  }
  if (a.nfrag > 0) {
    launch_rowsum(split_t, a.p0, num_heads * head_dim, d_feat, row_begin, row_end, stream);
    launch_rowsum(split_t, a.p1, num_heads, d_el, row_begin, row_end, stream);
    if (attn_l != nullptr)
      gat_fold_long_rows_kernel<<<split_t->num_long, 128, 0, stream>>>(split_t->long_rows, split_t->num_long, num_heads,
                                                                       head_dim, attn_l, d_el, d_feat, row_begin, row_end);
  }
  return check_launch("regnn_gat_bwd_edges");
}

extern "C" int regnn_gat_bwd_reduce(const int32_t* indptr, const uint8_t* etype_csr, const float* theta, float alpha,
                                    int num_relations, const float* dpre_csr, int num_heads, int64_t row_begin,
                                    int64_t row_end, float* d_er, double* partials, float* d_theta,
                                    const regnn_rowsplit_t* split, float* split_workspace, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr && d_er, REGNN_ERR_INVALID_ARG, "gat_bwd_reduce: null pointer");
  REGNN_REQUIRE(etype_csr == nullptr || (theta && partials && d_theta), REGNN_ERR_INVALID_ARG,
                "gat_bwd_reduce: null relation buffers");
  REGNN_REQUIRE(num_heads >= 1 && num_heads <= REGNN_MAX_HEADS, REGNN_ERR_UNSUPPORTED_SHAPE, "gat_bwd_reduce: num_heads=%d", num_heads);
  const int R = etype_csr ? num_relations : 0;
  REGNN_REQUIRE(etype_csr == nullptr || (R >= 1 && R <= REGNN_MAX_RELATIONS), REGNN_ERR_UNSUPPORTED_SHAPE,
                "gat_bwd_reduce: num_relations=%d", R);
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "gat_bwd_reduce: negative row range");
  if (rows == 0) return REGNN_OK;
  int HP = 1;
  while (HP < num_heads) HP <<= 1;
  AttnArgs a{};
  a.indptr = indptr; a.H = num_heads; a.D = 4; a.row_begin = row_begin; a.row_end = row_end; a.d_csr = dpre_csr; a.o2 = d_er;
  REGNN_REQUIRE(apply_split(a, split, split_workspace), REGNN_ERR_INVALID_ARG, "gat_bwd_reduce: incomplete row split");
  a.p1 = split_workspace;   // [nfrag][H] fragment partials
  const int per = 32 / HP;
  const int64_t items = a.nfrag + rows;
  const unsigned grid = (unsigned)((items + (int64_t)per * kWarpsPerBlock - 1) / ((int64_t)per * kWarpsPerBlock));
#ifndef REGNN_GAT_REDUCE_FUSED
#define REGNN_GAT_REDUCE_FUSED 1
#endif
  // d_er and the relation bins in one pass over dpre: 0.39 instead of 0.51 ms on the MAG graph (H8); on L2-resident
  // graphs the two specialised kernels are a few microseconds faster (ACM H8 D64: 49 vs 58 us)
  if (REGNN_GAT_REDUCE_FUSED && etype_csr != nullptr && rows >= 65536) {
    const size_t smem = sizeof(float) * (size_t)kWarpsPerBlock * R * 32;
    int rc = set_smem(gat_bwd_der_bins_kernel, smem);
    if (rc != REGNN_OK) return rc;
    a.etype = etype_csr; a.R = R; a.partials = partials;
    const int nb = (int)min((int64_t)grid, (int64_t)148 * 16);
    gat_bwd_der_bins_kernel<<<nb, kWarpsPerBlock * 32, smem, stream>>>(a, HP);
    if (a.nfrag > 0) launch_rowsum(split, a.p1, num_heads, d_er, row_begin, row_end, stream);
    launch_relation_grad_finalize(partials, nb, R * num_heads, R * num_heads, theta, alpha, d_theta, stream);
    return check_launch("regnn_gat_bwd_reduce");
  }
  gat_bwd_der_kernel<<<grid, kWarpsPerBlock * 32, 0, stream>>>(a, HP);
  if (a.nfrag > 0) launch_rowsum(split, a.p1, num_heads, d_er, row_begin, row_end, stream);
  if (etype_csr != nullptr) {
    // the slot range of the row range (host-side values are not available without a sync: pass the pointers)
    const size_t smem = sizeof(float) * (size_t)kWarpsPerBlock * R * 32;
    int rc = set_smem(gat_bwd_bins_kernel, smem);
    if (rc != REGNN_OK) return rc;
    const int nb = min(partial_blocks(rows), 148 * 4);
    gat_bwd_bins_kernel<<<nb, kWarpsPerBlock * 32, smem, stream>>>(etype_csr, dpre_csr, num_heads, indptr, row_begin, row_end,
                                                                  R, num_heads, HP, partials);
    launch_relation_grad_finalize(partials, nb, R * num_heads, R * num_heads, theta, alpha, d_theta, stream);
  }
  return check_launch("regnn_gat_bwd_reduce");
}

extern "C" int regnn_attn_scores_fwd(const float* feat, const float* attn_l, const float* attn_r, int64_t num_nodes,
                                     int num_heads, int head_dim, float* el, float* er, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(feat && attn_l && attn_r && el && er && num_nodes >= 0, REGNN_ERR_INVALID_ARG, "attn_scores_fwd: bad argument");
  int rc = check_shape("attn_scores_fwd", num_heads, head_dim, 0, false, true);
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(aligned16(feat) && aligned16(attn_l) && aligned16(attn_r), REGNN_ERR_INVALID_ARG,
                "attn_scores_fwd: 16-byte alignment required");
  if (num_nodes == 0) return REGNN_OK;
  AttnArgs a{};
  a.H = num_heads; a.D = head_dim;
  apply_split(a, nullptr, nullptr);
  const int G = rg_lanes(num_heads * head_dim), cpl = head_chunks(head_dim), ni = a.hg_count / cpl;
  const int64_t work = (num_nodes * ni + 32 / G - 1) / (32 / G);
  const int64_t want = (work + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const unsigned grid = (unsigned)(want < 148 * 16 ? want : 148 * 16);
#define REGNN_SCORES_FWD(G_, C_)                                                                                      \
  attn_scores_fwd_kernel<G_, C_><<<grid, kWarpsPerBlock * 32, 0, stream>>>(feat, attn_l, attn_r, num_nodes, num_heads, \
                                                                          head_dim, a.d_shift, ni, el, er)
  switch (G * cpl) {
    case 4: REGNN_SCORES_FWD(4, 1); break;
    case 8: REGNN_SCORES_FWD(8, 1); break;
    case 16: REGNN_SCORES_FWD(16, 1); break;
    case 64: REGNN_SCORES_FWD(32, 2); break;
    case 128: REGNN_SCORES_FWD(32, 4); break;
    default: REGNN_SCORES_FWD(32, 1); break;
  }
#undef REGNN_SCORES_FWD
  return check_launch("regnn_attn_scores_fwd");
}

extern "C" int regnn_attn_scores_bwd(const float* feat, const float* d_el, const float* d_er, int64_t num_nodes,
                                     int num_heads, int head_dim, double* partials, float* d_attn_l, float* d_attn_r,
                                     float* d_feat, const float* attn_r, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(feat && d_el && d_er && partials && d_attn_l && d_attn_r && num_nodes >= 0, REGNN_ERR_INVALID_ARG,
                "attn_scores_bwd: bad argument");
  REGNN_REQUIRE(d_feat == nullptr || attn_r != nullptr, REGNN_ERR_INVALID_ARG, "attn_scores_bwd: d_feat without attn_r");
  int rc = check_shape("attn_scores_bwd", num_heads, head_dim, 0, false, true);
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(aligned16(feat) && aligned16(d_feat) && aligned16(attn_r), REGNN_ERR_INVALID_ARG,
                "attn_scores_bwd: 16-byte alignment required");
  AttnArgs a{};
  a.H = num_heads; a.D = head_dim;
  apply_split(a, nullptr, nullptr);
  const int G = rg_lanes(num_heads * head_dim), HD = num_heads * head_dim;
  const int64_t want = (num_nodes * a.hg_count / (32 / G) + kWarpsPerBlock) / kWarpsPerBlock + 1;
  int nb = (int)(want < 148 * 8 ? want : 148 * 8);
  if (nb * kWarpsPerBlock < a.hg_count) nb = (a.hg_count + kWarpsPerBlock - 1) / kWarpsPerBlock;
  const size_t smem = sizeof(float) * kWarpsPerBlock * 256;
#define REGNN_SCORES_BWD(G_)                                                                                      \
  attn_scores_bwd_kernel<G_><<<nb, kWarpsPerBlock * 32, smem, stream>>>(feat, d_el, d_er, num_nodes, num_heads, head_dim, \
                                                                       a.d_shift, a.hg_count, partials, d_feat, attn_r)
  switch (G) {
    case 4: REGNN_SCORES_BWD(4); break;
    case 8: REGNN_SCORES_BWD(8); break;
    case 16: REGNN_SCORES_BWD(16); break;
    default: REGNN_SCORES_BWD(32); break;
  }
#undef REGNN_SCORES_BWD
  launch_colsum_finalize(partials, nb, 2 * HD, 0, HD, d_attn_l, stream);
  launch_colsum_finalize(partials, nb, 2 * HD, HD, HD, d_attn_r, stream);
  return check_launch("regnn_attn_scores_bwd");
}

extern "C" int regnn_gatv2_fwd(const int32_t* indptr, const int32_t* indices, const int32_t* eid,
                               const uint8_t* etype_csr, const float* theta, float alpha,
                               int num_relations, const float* fs, const float* fd,
                               const float* attn, float negative_slope, const float* keep,
                               const regnn_attn_dropout_t* dropout, int num_heads, int head_dim, int64_t row_begin,
                               int64_t row_end,
                               float* out, float* rowmax, float* rowsum, float* attn_out, float* logit_csr,
                               uint32_t* qmask, const regnn_rowsplit_t* split, float* split_workspace,
                               const int32_t* row_order, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr && fs && fd && attn && out && rowmax && rowsum, REGNN_ERR_INVALID_ARG, "gatv2_fwd: null pointer");
  REGNN_REQUIRE(keep == nullptr || dropout == nullptr, REGNN_ERR_INVALID_ARG, "gatv2_fwd: keep and dropout are exclusive");
  REGNN_REQUIRE((keep == nullptr && dropout == nullptr && attn_out == nullptr) || eid != nullptr, REGNN_ERR_INVALID_ARG,
                "gatv2_fwd: keep/dropout/attn_out need eid");
  REGNN_REQUIRE(etype_csr == nullptr || theta != nullptr, REGNN_ERR_INVALID_ARG, "gatv2_fwd: etype without theta");
  int rc = check_shape("gatv2_fwd", num_heads, head_dim, num_relations, etype_csr != nullptr, true);
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE((logit_csr == nullptr) == (qmask == nullptr), REGNN_ERR_INVALID_ARG, "gatv2_fwd: logit_csr and qmask go together");
  REGNN_REQUIRE(aligned16(fs) && aligned16(fd) && aligned16(attn) && aligned16(out) && aligned16(qmask), REGNN_ERR_INVALID_ARG,
                "gatv2_fwd: 16-byte alignment required");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "gatv2_fwd: negative row range");
  if (rows == 0) return REGNN_OK;
  AttnArgs a{};
  a.indptr = indptr; a.indices = indices; a.eid = eid; a.etype = etype_csr; a.theta = theta; a.alpha = alpha;
  a.R = etype_csr ? num_relations : 0; a.feat = fs; a.fd = fd; a.el = attn; a.slope = negative_slope; a.keep = keep;
  a.H = num_heads; a.D = head_dim; a.row_begin = row_begin; a.row_end = row_end;
  a.o0 = out; a.o1 = rowmax; a.o2 = rowsum; a.o3 = attn_out;
  REGNN_REQUIRE(apply_split(a, split, split_workspace), REGNN_ERR_INVALID_ARG, "gatv2_fwd: incomplete row split");
  REGNN_REQUIRE(apply_dropout(a, dropout), REGNN_ERR_INVALID_ARG, "gatv2_fwd: dropout heads / scale inconsistent");
  apply_order(a, row_order, split, rows);
  const size_t smem = sizeof(float) * ((size_t)a.R * num_heads) + 16;
  const int cpl = head_chunks(head_dim);
  const unsigned grid = (unsigned)((rg_work(a, rows, cpl) + kWarpsPerBlock - 1) / kWarpsPerBlock);
  {
    const int G = rg_lanes(a.H * a.D), lph = min(G, head_dim / 4);
    const bool hash = dropout != nullptr;
    const bool extra = keep != nullptr || attn_out != nullptr;
    bool launched = false;
#define REGNN_V2F_CASE(G_, L_, C_)                                                                                     \
  if (G == G_ && lph == L_ && cpl == C_) {                                                                             \
    rc = set_smem(hash ? gatv2_fwd_rg_kernel<G_, L_, true, true, C_>                                                   \
                       : (extra ? gatv2_fwd_rg_kernel<G_, L_, true, false, C_>                                         \
                                : gatv2_fwd_rg_kernel<G_, L_, false, false, C_>), smem);                               \
    if (rc != REGNN_OK) return rc;                                                                                     \
    if (hash)                                                                                                          \
      gatv2_fwd_rg_kernel<G_, L_, true, true, C_><<<grid, kWarpsPerBlock * 32, smem, stream>>>(a, logit_csr, qmask);   \
    else if (extra)                                                                                                    \
      gatv2_fwd_rg_kernel<G_, L_, true, false, C_><<<grid, kWarpsPerBlock * 32, smem, stream>>>(a, logit_csr, qmask);  \
    else                                                                                                               \
      gatv2_fwd_rg_kernel<G_, L_, false, false, C_><<<grid, kWarpsPerBlock * 32, smem, stream>>>(a, logit_csr, qmask); \
    launched = true;                                                                                                   \
  }
    REGNN_V2F_CASE(4, 1, 1) REGNN_V2F_CASE(4, 2, 1) REGNN_V2F_CASE(4, 4, 1)
    REGNN_V2F_CASE(8, 1, 1) REGNN_V2F_CASE(8, 2, 1) REGNN_V2F_CASE(8, 4, 1) REGNN_V2F_CASE(8, 8, 1)
    REGNN_V2F_CASE(16, 1, 1) REGNN_V2F_CASE(16, 2, 1) REGNN_V2F_CASE(16, 4, 1) REGNN_V2F_CASE(16, 8, 1)
    REGNN_V2F_CASE(16, 16, 1)
    REGNN_V2F_CASE(32, 1, 1) REGNN_V2F_CASE(32, 2, 1) REGNN_V2F_CASE(32, 4, 1) REGNN_V2F_CASE(32, 8, 1)
    REGNN_V2F_CASE(32, 16, 1) REGNN_V2F_CASE(32, 32, 1) REGNN_V2F_CASE(32, 32, 2) REGNN_V2F_CASE(32, 32, 4)
#undef REGNN_V2F_CASE
    REGNN_REQUIRE(launched, REGNN_ERR_UNSUPPORTED_SHAPE, "gatv2_fwd: no kernel for H=%d D=%d", num_heads, head_dim);
  }
  if (a.nfrag > 0) {
    const unsigned fgrid = (unsigned)(((int64_t)split->num_long * head_groups(a.H, a.D) + kWarpsPerBlock - 1) / kWarpsPerBlock);
    if (dropout != nullptr) REGNN_DISPATCH_FINALIZE(fgrid, true);
    else REGNN_DISPATCH_FINALIZE(fgrid, false);
  }
  return check_launch("regnn_gatv2_fwd");
}

extern "C" int64_t regnn_gatv2_bwd_edges_blocks(int64_t num_rows, int num_frags, int num_long, int num_heads,
                                                int head_dim, int ordered) {
  if (num_rows < 0 || num_heads < 1 || head_dim < 4) return 0;
  const int HD = num_heads * head_dim, gpw = 32 / rg_lanes(HD);
  const int64_t nrows = ordered ? num_rows - num_long : num_rows;
  const int64_t work = ((num_frags + nrows) * (head_groups(num_heads, head_dim) / head_chunks(head_dim)) + gpw - 1) / gpw;
  return (work + kWarpsPerBlock - 1) / kWarpsPerBlock;
}

extern "C" int regnn_gatv2_bwd_edges(const int32_t* indptr_t, const int32_t* indices_t, const int32_t* slot_t,
                                     const int32_t* eid, const float* fs, const float* stats, const float* logit_csr,
                                     const uint32_t* qmask, const float* attn, float negative_slope, const float* keep,
                                     const regnn_attn_dropout_t* dropout, const float* Gd, int num_heads, int head_dim,
                                     int64_t row_begin, int64_t row_end,
                                     float* d_fs, float* dl_csr, float* d_attn_src, float* block_partials,
                                     double* partials, const regnn_rowsplit_t* split_t, float* split_workspace,
                                     const int32_t* row_order_t, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr_t && fs && stats && attn && Gd && d_fs && d_attn_src && block_partials && partials,
                REGNN_ERR_INVALID_ARG, "gatv2_bwd_edges: null pointer");  /* per-edge arrays may be NULL when E == 0 */
  REGNN_REQUIRE(keep == nullptr || dropout == nullptr, REGNN_ERR_INVALID_ARG, "gatv2_bwd_edges: keep and dropout are exclusive");
  REGNN_REQUIRE((keep == nullptr && dropout == nullptr) || eid != nullptr, REGNN_ERR_INVALID_ARG,
                "gatv2_bwd_edges: keep/dropout need eid");
  int rc = check_shape("gatv2_bwd_edges", num_heads, head_dim, 0, false, true);
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(aligned16(fs) && aligned16(stats) && aligned16(attn) && aligned16(Gd) && aligned16(d_fs) && aligned16(qmask),
                REGNN_ERR_INVALID_ARG, "gatv2_bwd_edges: 16-byte alignment required");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "gatv2_bwd_edges: negative row range");
  const int HD = num_heads * head_dim;
  if (rows == 0) {
    cudaMemsetAsync(d_attn_src, 0, sizeof(float) * HD, stream);
    return check_launch("regnn_gatv2_bwd_edges");
  }
  AttnArgs a{};
  a.indptr = indptr_t; a.indices = indices_t; a.eid = slot_t; a.a_csr_eid = eid; a.feat = fs; a.fd = stats;
  a.a_csr = logit_csr; a.el = attn; a.slope = negative_slope; a.keep = keep; a.G = Gd; a.H = num_heads; a.D = head_dim;
  a.row_begin = row_begin; a.row_end = row_end; a.o0 = d_fs; a.o2 = dl_csr;
  REGNN_REQUIRE(apply_split(a, split_t, split_workspace), REGNN_ERR_INVALID_ARG, "gatv2_bwd_edges: incomplete row split");
  REGNN_REQUIRE(apply_dropout(a, dropout), REGNN_ERR_INVALID_ARG, "gatv2_bwd_edges: dropout heads / scale inconsistent");
  apply_order(a, row_order_t, split_t, rows);
  const int cpl = head_chunks(head_dim);
  const int64_t nb = (rg_work(a, rows, cpl) + kWarpsPerBlock - 1) / kWarpsPerBlock;
  {
    const int G = rg_lanes(HD), lph = min(G, head_dim / 4);
    bool launched = false;
#define REGNN_V2E_CASE(G_, L_, C_)                                                                                     \
  if (G == G_ && lph == L_ && cpl == C_) {                                                                             \
    if (dropout != nullptr)                                                                                            \
      gatv2_bwd_edges_kernel<G_, L_, true, true, C_><<<(unsigned)nb, kWarpsPerBlock * 32, 0, stream>>>(a, qmask,       \
                                                                                                      block_partials); \
    else if (keep != nullptr)                                                                                          \
      gatv2_bwd_edges_kernel<G_, L_, true, false, C_><<<(unsigned)nb, kWarpsPerBlock * 32, 0, stream>>>(a, qmask,      \
                                                                                                       block_partials);\
    else                                                                                                               \
      gatv2_bwd_edges_kernel<G_, L_, false, false, C_><<<(unsigned)nb, kWarpsPerBlock * 32, 0, stream>>>(a, qmask,     \
                                                                                                        block_partials);\
    launched = true;                                                                                                   \
  }
    REGNN_V2E_CASE(4, 1, 1) REGNN_V2E_CASE(4, 2, 1) REGNN_V2E_CASE(4, 4, 1)
    REGNN_V2E_CASE(8, 1, 1) REGNN_V2E_CASE(8, 2, 1) REGNN_V2E_CASE(8, 4, 1) REGNN_V2E_CASE(8, 8, 1)
    REGNN_V2E_CASE(16, 1, 1) REGNN_V2E_CASE(16, 2, 1) REGNN_V2E_CASE(16, 4, 1) REGNN_V2E_CASE(16, 8, 1)
    REGNN_V2E_CASE(16, 16, 1)
    REGNN_V2E_CASE(32, 1, 1) REGNN_V2E_CASE(32, 2, 1) REGNN_V2E_CASE(32, 4, 1) REGNN_V2E_CASE(32, 8, 1)
    REGNN_V2E_CASE(32, 16, 1) REGNN_V2E_CASE(32, 32, 1) REGNN_V2E_CASE(32, 32, 2) REGNN_V2E_CASE(32, 32, 4)
#undef REGNN_V2E_CASE
    REGNN_REQUIRE(launched, REGNN_ERR_UNSUPPORTED_SHAPE, "gatv2_bwd_edges: no kernel for H=%d D=%d", num_heads, head_dim);
  }
  if (a.nfrag > 0) launch_rowsum(split_t, a.p0, HD, d_fs, row_begin, row_end, stream);
  // d_attn share of the source side: [nb][HD] float block partials -> [chunks][HD] doubles -> [HD]
  const int chunks = (int)(nb < REGNN_V2_STAGE_CHUNKS ? nb : REGNN_V2_STAGE_CHUNKS);
  const int64_t per = (nb + chunks - 1) / chunks;
  colsum_stage_kernel<<<chunks, 256, 0, stream>>>(block_partials, nb, HD, per, partials);
  launch_colsum_finalize(partials, chunks, HD, 0, HD, d_attn_src, stream);
  return check_launch("regnn_gatv2_bwd_edges");
}

extern "C" int regnn_gatv2_bwd_dst(const int32_t* indptr, const uint8_t* etype_csr, const float* theta, float alpha,
                                   int num_relations, const float* fd, const float* dl_csr, const uint32_t* qmask,
                                   const float* attn, float negative_slope, int num_heads, int head_dim,
                                   int64_t row_begin, int64_t row_end, float* d_fd, float* d_attn_dst, double* partials,
                                   float* d_theta, const regnn_rowsplit_t* split, float* split_workspace, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  REGNN_REQUIRE(indptr && fd && attn && d_fd && d_attn_dst && partials, REGNN_ERR_INVALID_ARG, "gatv2_bwd_dst: null pointer");
  REGNN_REQUIRE(etype_csr == nullptr || (theta && d_theta), REGNN_ERR_INVALID_ARG, "gatv2_bwd_dst: null relation buffers");
  int rc = check_shape("gatv2_bwd_dst", num_heads, head_dim, num_relations, etype_csr != nullptr, true);
  if (rc != REGNN_OK) return rc;
  REGNN_REQUIRE(aligned16(fd) && aligned16(attn) && aligned16(d_fd) && aligned16(qmask), REGNN_ERR_INVALID_ARG,
                "gatv2_bwd_dst: 16-byte alignment required");
  const int64_t rows = row_end - row_begin;
  REGNN_REQUIRE(rows >= 0, REGNN_ERR_INVALID_ARG, "gatv2_bwd_dst: negative row range");
  AttnArgs a{};
  a.indptr = indptr; a.fd = fd; a.el = attn; a.d_csr = dl_csr; a.slope = negative_slope; a.H = num_heads; a.D = head_dim;
  a.row_begin = row_begin; a.row_end = row_end; a.o2 = d_fd; a.partials = partials;
  const int R = etype_csr ? num_relations : 0, HD = num_heads * head_dim;
  REGNN_REQUIRE(apply_split(a, split, split_workspace), REGNN_ERR_INVALID_ARG, "gatv2_bwd_dst: incomplete row split");
  const int G = rg_lanes(HD), gpw = 32 / G;
  const int64_t work = ((a.nfrag + rows) * a.hg_count + gpw - 1) / gpw;
  int nb = partial_blocks(work);
  if (nb * kWarpsPerBlock < a.hg_count) nb = (a.hg_count + kWarpsPerBlock - 1) / kWarpsPerBlock;
  switch (G) {
    case 4: gatv2_bwd_dst_stream_kernel<4><<<nb, kWarpsPerBlock * 32, 0, stream>>>(a, qmask); break;
    case 8: gatv2_bwd_dst_stream_kernel<8><<<nb, kWarpsPerBlock * 32, 0, stream>>>(a, qmask); break;
    case 16: gatv2_bwd_dst_stream_kernel<16><<<nb, kWarpsPerBlock * 32, 0, stream>>>(a, qmask); break;
    default: gatv2_bwd_dst_stream_kernel<32><<<nb, kWarpsPerBlock * 32, 0, stream>>>(a, qmask); break;
  }
  if (a.nfrag > 0) launch_rowsum(split, a.p0, HD, d_fd, row_begin, row_end, stream);
  launch_colsum_finalize(partials, nb, HD, 0, HD, d_attn_dst, stream);
  if (etype_csr != nullptr && rows > 0) {   // relation bins of dl: streaming (the partials buffer is free again)
    int HP = 1;
    while (HP < num_heads) HP <<= 1;
    const size_t smem = sizeof(float) * (size_t)kWarpsPerBlock * R * 32;
    rc = set_smem(gat_bwd_bins_kernel, smem);
    if (rc != REGNN_OK) return rc;
    const int nbb = min(partial_blocks(rows), 148 * 4);
    gat_bwd_bins_kernel<<<nbb, kWarpsPerBlock * 32, smem, stream>>>(etype_csr, dl_csr, num_heads, indptr, row_begin, row_end, R,
                                                                   num_heads, HP, partials);
    launch_relation_grad_finalize(partials, nbb, R * num_heads, R * num_heads, theta, alpha, d_theta, stream);
  }
  return check_launch("regnn_gatv2_bwd_dst");
}
