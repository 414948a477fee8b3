"""Raw operator wrappers: one Python function per C-ABI entry point of ``libregnn_b200.so``.

Each wrapper allocates its outputs with the PyTorch caching allocator, passes raw device pointers
and the current CUDA stream, and raises on any error.  No arithmetic happens here and there is no
CPU branch: tensors must live on a CUDA device.
"""
import ctypes
import os

import torch

from . import _lib


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError('re_gnn_b200 operators need CUDA tensors (got %s); there is no CPU path' % t.device)
    return t.detach().to(torch.float32).contiguous()


def _rows(rows, n):
    return (0, n) if rows is None else (int(rows[0]), int(rows[1]))


def wdeg_norm_fwd(csr, et_csr, theta, alpha, exponent, rows=None, counts=None, clamp_min=1.0):
    """deg[v] = sum_in w[etype], norm = max(deg,1)^exponent -> (deg[N], norm[N]).
    ``counts``: the per-(row, relation) in-edge counts of this e_feat (Graph.etype_views()[2]); with counts, ``csr``
    may be None (the table's rows are the rows)."""
    theta = _f32(theta).view(-1)
    n = csr['indptr'].numel() - 1 if csr is not None else counts.numel() // theta.numel()
    rb, re = _rows(rows, n)
    deg = torch.empty(n, dtype=torch.float32, device=theta.device)
    norm = torch.empty(n, dtype=torch.float32, device=theta.device)
    with torch.cuda.device(theta.device):
        _lib.call('regnn_wdeg_norm_fwd', _ptr(csr['indptr'] if csr is not None else None), _ptr(et_csr), _ptr(counts),
                  _ptr(theta), float(alpha), theta.numel(), float(exponent), float(clamp_min), rb, re, _ptr(deg),
                  _ptr(norm), _stream())
        _lib.count_launches(1)
    return deg, norm


def wdeg_norm_bwd(csr, et_csr, theta, alpha, exponent, deg, d_norm, rows=None, counts=None, clamp_min=1.0):
    theta = _f32(theta).view(-1)
    d_norm = _f32(d_norm)
    r = theta.numel()
    n = csr['indptr'].numel() - 1 if csr is not None else counts.numel() // r
    rb, re = _rows(rows, n)
    partials = torch.empty(_lib.partial_blocks(re - rb) * r, dtype=torch.float64, device=theta.device)
    d_theta = torch.empty(r, dtype=torch.float32, device=theta.device)
    with torch.cuda.device(theta.device):
        _lib.call('regnn_wdeg_norm_bwd', _ptr(csr['indptr'] if csr is not None else None), _ptr(et_csr), _ptr(counts),
                  _ptr(theta), float(alpha), r, float(exponent), float(clamp_min), rb, re, _ptr(deg), _ptr(d_norm),
                  _ptr(partials), _ptr(d_theta), _stream())
        _lib.count_launches(2)
    return d_theta


def _split_args(split, feat, device):
    if split is None:
        return None, None, 0
    ws = torch.empty(split['struct'].num_frags * feat, dtype=torch.float32, device=device)
    return ctypes.byref(split['struct']), ws, 1


# widths up to this run the lane-group kernel when the degree-sorted row order is supplied
NARROW_FEAT = int(os.environ.get('REGNN_NARROW_FEAT', '128'))


def row_order(csr, transposed=False):
    """Rows of one CSR view that are not cut into fragments, by descending slot count (stable): the work list of
    the narrow-row SpMM kernels (``row_order`` of regnn_spmm_fwd / regnn_spmm_bwd_fused).  Index bookkeeping with
    torch ops on the device, built on first use and cached in the csr dict."""
    key = 'order_t' if transposed else 'order'
    if key not in csr:
        indptr = csr['indptr_t' if transposed else 'indptr']
        split = csr.get('split_t' if transposed else 'split')
        deg = indptr[1:] - indptr[:-1]
        order = torch.sort(deg, descending=True, stable=True).indices
        # long rows (more slots than the split threshold) sort first: drop them
        csr[key] = order[(split['struct'].num_long if split is not None else 0):].to(torch.int32).contiguous()
    return csr[key]


def spmm(indptr, indices, etype, theta, alpha, norm_src, norm_dst, x, rows=None, out=None, split=None, order=None):
    """Y[v] = norm_dst[v] * sum_s w[etype[s]] * norm_src[indices[s]] * X[indices[s]] over rows.
    ``split``: the long-row decomposition of this CSR view (Graph.csr()['split' | 'split_t']);
    ``order``: ``row_order`` of the same view (used for widths <= NARROW_FEAT on the full row range)."""
    x = _f32(x)
    n = indptr.numel() - 1
    rb, re = _rows(rows, n)
    f = x.shape[1]
    theta = _f32(theta).view(-1) if theta is not None else None
    if out is None:
        out = torch.empty((n, f), dtype=torch.float32, device=x.device)
        if (rb, re) != (0, n):
            out.zero_()
    sp, ws, extra = _split_args(split, f, x.device)
    with torch.cuda.device(x.device):
        _lib.call('regnn_spmm_fwd', _ptr(indptr), _ptr(indices), _ptr(etype) if theta is not None else None,
                  _ptr(theta), float(alpha), theta.numel() if theta is not None else 0, _ptr(norm_src),
                  _ptr(norm_dst), _ptr(x), x.stride(0), _ptr(out), out.stride(0), rb, re, f, sp, _ptr(ws),
                  _ptr(order) if (order is not None and f <= NARROW_FEAT and (rb, re) == (0, n)) else None, _stream())
        _lib.count_launches(1 + extra)
    return out


def spmm_bwd_w(csr, et_csr, theta, alpha, norm, x, y, g, dx, rows=None, sides=3, split=None):
    """-> (d_theta[R] or None, d_norm[N] or None).  sides: bit0 source side scaled, bit1 destination."""
    x, y, g, dx = _f32(x), _f32(y), _f32(g), _f32(dx)
    n = csr['indptr'].numel() - 1
    rb, re = _rows(rows, n)
    weighted = theta is not None
    theta = _f32(theta).view(-1) if weighted else None
    r = theta.numel() if weighted else 0
    partials = torch.empty(max(_lib.partial_blocks(re - rb) * r, 1), dtype=torch.float64, device=x.device)
    d_theta = torch.empty(r, dtype=torch.float32, device=x.device) if weighted else None
    d_norm = torch.zeros(n, dtype=torch.float32, device=x.device) if norm is not None else None
    with torch.cuda.device(x.device):
        _lib.call('regnn_spmm_bwd_w', _ptr(csr['indptr']), _ptr(csr['indices']), _ptr(et_csr) if weighted else None,
                  _ptr(theta), float(alpha), r, _ptr(norm), int(sides), _ptr(x), x.stride(0), _ptr(y), y.stride(0),
                  _ptr(g), g.stride(0), _ptr(dx), dx.stride(0), rb, re, x.shape[1], _ptr(partials),
                  _ptr(d_theta), _ptr(d_norm), ctypes.byref(split['struct']) if split is not None else None, _stream())
        _lib.count_launches(2 if weighted else 1)
    return d_theta, d_norm


def spmm_bwd_fused(csr, et_t, theta, alpha, norm, x, g, rows=None, sides=3, out=None, want_xdx=False, y=None,
                   want_dnorm=False):
    """One gather pass over the transposed view -> (dX[N,F], d_theta[R], xdx[N] | d_norm[N] | None).
    ``want_dnorm`` (needs ``y`` = the forward result when the destination side is scaled, and a shape the lane-group
    kernel covers: ``fused_dnorm_fits``): the third result is the whole norm gradient, no row-dot pass needed;
    ``want_xdx``: it is <X[u],dX[u]> only (input of ``rowdot_norm_bwd``).  See regnn_spmm_bwd_fused."""
    x, g = _f32(x), _f32(g)
    theta = _f32(theta).view(-1)
    n = csr['indptr_t'].numel() - 1
    rb, re = _rows(rows, n)
    f, r = x.shape[1], theta.numel()
    if out is None:
        out = torch.empty((n, f), dtype=torch.float32, device=x.device)
        if (rb, re) != (0, n):
            out.zero_()
    partials = torch.empty(_lib.partial_blocks(re - rb) * r, dtype=torch.float64, device=x.device)
    d_theta = torch.empty(r, dtype=torch.float32, device=x.device)
    sp, ws, extra = _split_args(csr.get('split_t'), f, x.device)
    order = row_order(csr, True) if (f <= NARROW_FEAT and (rb, re) == (0, n)) else None
    d_norm = xdx = None
    if want_dnorm:
        if order is None or norm is None:
            raise RuntimeError('the folded norm gradient needs the lane-group kernel (F <= %d, full row range)' % NARROW_FEAT)
        y = _f32(y)
        d_norm = torch.empty(n, dtype=torch.float32, device=x.device)
    elif want_xdx:
        xdx = torch.zeros(n, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.call('regnn_spmm_bwd_fused', _ptr(csr['indptr_t']), _ptr(csr['indices_t']), _ptr(et_t), _ptr(theta),
                  float(alpha), r, _ptr(norm), int(sides), _ptr(x), x.stride(0), _ptr(g), g.stride(0), _ptr(out),
                  out.stride(0), rb, re, f, _ptr(partials), _ptr(d_theta), _ptr(xdx), _ptr(y) if want_dnorm else None,
                  y.stride(0) if (want_dnorm and y is not None) else 0, _ptr(d_norm), sp, _ptr(ws), _ptr(order), _stream())
        _lib.count_launches(2 + extra * (2 if (want_xdx or want_dnorm) else 1))
    return out, d_theta, (d_norm if want_dnorm else xdx)


def fused_dnorm_fits(feat, rows_full=True):
    """True when regnn_spmm_bwd_fused can also produce d_norm (lane-group kernel: F <= NARROW_FEAT, F % 4 == 0)."""
    return rows_full and feat <= NARROW_FEAT and feat % 4 == 0


SMEM_BUDGET = 227 * 1024   # dynamic shared memory one block can opt in to on sm_100a


def fused_bwd_fits(feat, num_relations):
    """True when regnn_spmm_bwd_fused has a kernel for this shape: the lane-local relation bins (1088 bytes per
    relation) and -- for the whole-warp kernel, F > NARROW_FEAT -- the 8 x 8-row X tile must fit in shared memory.
    Otherwise the caller takes the two-pass backward (transposed regnn_spmm_fwd + regnn_spmm_bwd_w)."""
    bins = 1088 * int(num_relations)
    tile = 0 if feat <= NARROW_FEAT and feat % 4 == 0 else 64 + 256 * ((int(feat) + 3) & ~3)
    return feat <= 1024 and bins + tile <= SMEM_BUDGET


def rowdot_norm_bwd(norm, x, y, g, dx, rows=None, sides=3, xdx=None):
    """d_norm[v] = ([sides&2]<Y,G> + [sides&1]<X,dX>) / norm, rows outside the range are zero."""
    x, y, g, dx = _f32(x), _f32(y), _f32(g), _f32(dx)
    n = norm.numel()
    rb, re = _rows(rows, n)
    d_norm = torch.empty(n, dtype=torch.float32, device=x.device) if (rb, re) == (0, n) else \
        torch.zeros(n, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.call('regnn_rowdot_norm_bwd', _ptr(norm), int(sides), _ptr(x), x.stride(0), _ptr(y), y.stride(0),
                  _ptr(g), g.stride(0), _ptr(dx), dx.stride(0), _ptr(xdx), rb, re, x.shape[1], _ptr(d_norm), _stream())
        _lib.count_launches(1)
    return d_norm


def rows_to_slabs(x_own, num_ranks, row_offset, peer_slab_ptrs):
    """Pushes this rank's row block ``x_own`` [rows, F] into every rank's column slab (regnn_rows_to_slabs).
    ``peer_slab_ptrs``: int64 device tensor [P] of peer-mapped slab base addresses."""
    x_own = _f32(x_own)
    with torch.cuda.device(x_own.device):
        _lib.call('regnn_rows_to_slabs', _ptr(x_own), x_own.stride(0), x_own.shape[0], x_own.shape[1], int(num_ranks),
                  int(row_offset), _ptr(peer_slab_ptrs), _stream())
        _lib.count_launches(1)


def halo_push(x_own, send_rows, send_ptr, recv_offset, peer_buf_ptrs, ldb, rank):
    """Stores rows ``x_own[send_rows[send_ptr[q]:send_ptr[q+1]]]`` to rows ``recv_offset[q], ...`` of peer q's halo buffer
    (regnn_halo_push).  ``send_rows``: int32 device tensor of local row ids; ``send_ptr`` [P+1] / ``recv_offset`` [P]:
    host sequences of ints; ``peer_buf_ptrs``: int64 device tensor [P] of buffer base addresses (leading dimension
    ``ldb`` floats)."""
    x_own = _f32(x_own)
    p = len(recv_offset)
    with torch.cuda.device(x_own.device):
        _lib.call('regnn_halo_push', _ptr(x_own), x_own.stride(0), x_own.shape[1], _ptr(send_rows),
                  (ctypes.c_int64 * (p + 1))(*send_ptr), (ctypes.c_int64 * p)(*recv_offset), _ptr(peer_buf_ptrs),
                  int(ldb), p, int(rank), _stream())
        _lib.count_launches(1 if send_ptr[-1] > send_ptr[0] else 0)


def halo_scatter(x, send_ptr, dst_rows, peer_buf_ptrs, ldb, rank):
    """Stores rows ``x[send_ptr[q]:send_ptr[q+1]]`` to rows ``dst_rows[send_ptr[q]:send_ptr[q+1]]`` of peer q's buffer
    (regnn_halo_scatter; any row width).  ``send_ptr`` [P+1]: host sequence of ints; ``dst_rows``: int32 device tensor
    indexed like the rows of ``x``; ``peer_buf_ptrs``: int64 device tensor [P] of buffer base addresses (leading
    dimension ``ldb`` floats)."""
    x = _f32(x)
    p = len(send_ptr) - 1
    with torch.cuda.device(x.device):
        _lib.call('regnn_halo_scatter', _ptr(x), x.stride(0), x.shape[1], (ctypes.c_int64 * (p + 1))(*send_ptr),
                  _ptr(dst_rows), _ptr(peer_buf_ptrs), int(ldb), p, int(rank), _stream())
        _lib.count_launches(1 if send_ptr[-1] > send_ptr[0] else 0)


def halo_push_slots(logit, qmask, send_slots, send_ptr, recv_offset, peer_logit_ptrs, peer_mask_ptrs, rank):
    """Stores the per-slot records ``logit[s]`` ([E, H] fp32) and ``qmask[s]`` ([E, C, 4] int32, the sign masks of
    ``gatv2_fwd(save=True)``) of the slots ``s = send_slots[send_ptr[q]:send_ptr[q+1]]`` to rows ``recv_offset[q], ...``
    of peer q's logit and mask buffers (regnn_halo_push_slots).  ``send_slots``: int32 device tensor; ``send_ptr``
    [P+1] / ``recv_offset`` [P]: host sequences of ints; ``peer_*_ptrs``: int64 device tensors [P] of buffer base
    addresses (rows of H floats and of C 128-bit words)."""
    logit = _f32(logit)
    p = len(recv_offset)
    with torch.cuda.device(logit.device):
        _lib.call('regnn_halo_push_slots', _ptr(logit), logit.shape[1], _ptr(qmask), qmask.shape[1], _ptr(send_slots),
                  (ctypes.c_int64 * (p + 1))(*send_ptr), (ctypes.c_int64 * p)(*recv_offset), _ptr(peer_logit_ptrs),
                  _ptr(peer_mask_ptrs), p, int(rank), _stream())
        _lib.count_launches(1 if send_ptr[-1] > send_ptr[0] else 0)


def slabs_to_rows(slab, num_rows, peers):
    """Pushes rows [0, num_rows) of this rank's column slab ``slab`` [>= num_rows, F/P] to their owner ranks' row blocks
    (regnn_slabs_to_rows; ``peers``: a ``_lib.PeerRows``)."""
    slab = _f32(slab)
    with torch.cuda.device(slab.device):
        _lib.call('regnn_slabs_to_rows', _ptr(slab), slab.stride(0), int(num_rows), slab.shape[1], ctypes.byref(peers),
                  _stream())
        _lib.count_launches(1)


def spmm_scatter(csr, etype, theta, alpha, norm_src, norm_dst, x_cols, peers, y_local=None, transposed=False):
    """regnn_spmm_fwd_scatter: forward SpMM of a column slab, result rows stored to their owner ranks (``peers``: a
    ``_lib.PeerRows``) and, with ``y_local`` ([rows >= N, F/P] fp32), also kept as a local slab.  ``transposed``: over
    the transposed view (the backward of the un-weighted propagation; ``etype`` is then the transposed-order array)."""
    x_cols = _f32(x_cols)
    sfx = '_t' if transposed else ''
    n = csr['indptr' + sfx].numel() - 1
    f = x_cols.shape[1]
    theta = _f32(theta).view(-1) if theta is not None else None
    sp, ws, extra = _split_args(csr.get('split' + sfx), f, x_cols.device)
    with torch.cuda.device(x_cols.device):
        _lib.call('regnn_spmm_fwd_scatter', _ptr(csr['indptr' + sfx]), _ptr(csr['indices' + sfx]),
                  _ptr(etype) if theta is not None else None, _ptr(theta), float(alpha),
                  theta.numel() if theta is not None else 0, _ptr(norm_src), _ptr(norm_dst), _ptr(x_cols),
                  x_cols.stride(0), n, f, sp, _ptr(ws), _ptr(row_order(csr, transposed)), ctypes.byref(peers), _ptr(y_local),
                  y_local.stride(0) if y_local is not None else 0, _stream())
        _lib.count_launches(1 + extra)


def spmm_bwd_fused_scatter(csr, et_t, theta, alpha, norm, x_cols, g_cols, peers, sides=3, y_cols=None):
    """regnn_spmm_bwd_fused_scatter -> (d_theta[R], d_norm[N] | None), both for this rank's columns only; the dX rows go
    to their owner ranks.  ``y_cols`` (the local result slab of ``spmm_scatter``) switches the folded norm gradient on."""
    x_cols, g_cols = _f32(x_cols), _f32(g_cols)
    theta = _f32(theta).view(-1)
    n = csr['indptr_t'].numel() - 1
    f, r = x_cols.shape[1], theta.numel()
    partials = torch.empty(_lib.partial_blocks(n) * r, dtype=torch.float64, device=x_cols.device)
    d_theta = torch.empty(r, dtype=torch.float32, device=x_cols.device)
    d_norm = torch.empty(n, dtype=torch.float32, device=x_cols.device) if (y_cols is not None and norm is not None) else None
    sp, ws, extra = _split_args(csr.get('split_t'), f, x_cols.device)
    with torch.cuda.device(x_cols.device):
        _lib.call('regnn_spmm_bwd_fused_scatter', _ptr(csr['indptr_t']), _ptr(csr['indices_t']), _ptr(et_t), _ptr(theta),
                  float(alpha), r, _ptr(norm), int(sides), _ptr(x_cols), x_cols.stride(0), _ptr(g_cols),
                  g_cols.stride(0), n, f, _ptr(partials), _ptr(d_theta), None,
                  _ptr(y_cols) if d_norm is not None else None, y_cols.stride(0) if d_norm is not None else 0,
                  _ptr(d_norm), sp, _ptr(ws), _ptr(row_order(csr, True)), ctypes.byref(peers), _stream())
        _lib.count_launches(2 + extra)
    return d_theta, d_norm


def _attn_split(split, h, d, device):
    """(byref(struct) | None, workspace | None, extra finalize launches flag) for the attention kernels."""
    if split is None:
        return None, None
    ws = torch.empty(split['struct'].num_frags * (h * d + 2 * h), dtype=torch.float32, device=device)
    return ctypes.byref(split['struct']), ws


def _rel(theta, et_csr):
    if theta is None or et_csr is None:
        return None, None, 0
    theta = _f32(theta)
    return theta, et_csr, theta.shape[0]


def _full(rb, re, n):
    return (rb, re) == (0, n)


def _drop(dropout, heads):
    """byref(regnn_attn_dropout_t) of a ``dropout.HashedDropout`` for a call over ``heads`` heads, or None."""
    return ctypes.byref(dropout.struct(heads)) if dropout is not None else None


def dropout_kw(dropout):
    """``{'dropout': dropout}``, or no keyword at all without dropout: callers that compose the stage wrappers pass it
    this way, so that stand-ins of the stages written before the keyword existed keep working."""
    return {} if dropout is None else {'dropout': dropout}


def gat_fwd(csr, et_csr, theta, alpha, feat, el, er, slope, keep=None, want_attn=False, rows=None, dropout=None,
            eid=None):
    """-> (out, rowmax, rowsum, attention | None) for the rows of ``csr``.  ``feat`` / ``el`` are indexed by the column
    ids of ``csr`` and may have more rows than the CSR (a halo of remote sources after the own rows).
    ``dropout``: a ``HashedDropout`` (counter-based attention dropout, exclusive with ``keep``); ``eid``: the global edge
    id of every slot when it is not ``csr['eid']`` (the in-view of a halo partition)."""
    feat, el, er, keep = _f32(feat), _f32(el), _f32(er), _f32(keep)
    eid = csr.get('eid') if eid is None else eid
    _, h, d = feat.shape
    n = csr['indptr'].numel() - 1
    rb, re = _rows(rows, n)
    theta, et_csr, r = _rel(theta, et_csr)
    dev = feat.device
    out = torch.empty((n, h, d), dtype=torch.float32, device=dev)
    if not _full(rb, re, n):
        out.zero_()
    rowmax = torch.zeros((n, h), dtype=torch.float32, device=dev)
    rowsum = torch.zeros((n, h), dtype=torch.float32, device=dev)
    e = csr['indices'].numel()
    attn = torch.zeros((max(e, 1), h), dtype=torch.float32, device=dev)[:e] if want_attn else None
    sp, ws = _attn_split(csr.get('split'), h, d, dev)
    order = row_order(csr) if _full(rb, re, n) else None
    with torch.cuda.device(dev):
        _lib.call('regnn_gat_fwd', _ptr(csr['indptr']), _ptr(csr['indices']), _ptr(eid), _ptr(et_csr),
                  _ptr(theta), float(alpha), r, _ptr(feat), _ptr(el), _ptr(er), float(slope), _ptr(keep),
                  _drop(dropout, h), h, d,
                  rb, re, _ptr(out), _ptr(rowmax), _ptr(rowsum), _ptr(attn), sp, _ptr(ws), _ptr(order), _stream())
        _lib.count_launches(1 + (sp is not None))
    return out, rowmax, rowsum, attn


def gat_bwd(csr, et_csr, et_t, theta, alpha, feat, el, er, slope, keep, out, rowmax, rowsum, g, attn_l=None,
            attn_r=None, dropout=None):
    """Backward of ``gat_fwd`` as one gather pass (``gat_bwd_stats`` -> ``gat_bwd_edges`` -> ``gat_bwd_reduce``)
    -> (d_feat, d_el, d_er, d_theta | None, d_attn_l | None, d_attn_r | None).
    With ``attn_l`` / ``attn_r`` ([H*D], the projection-score vectors of layer/REGATConv.py:68-69, el = <feat, attn_l>,
    er = <feat, attn_r>) the gradients through the scores are folded in: ``d_feat`` is the total feature gradient and
    the two parameter gradients are returned (``attn_scores_bwd``).  ``dropout``: the ``HashedDropout`` of the forward."""
    stats = gat_bwd_stats(out, g, er, rowmax, rowsum)
    e = csr['indices'].numel()
    dpre = torch.empty((max(e, 1), stats.shape[1]), dtype=torch.float32, device=stats.device)[:e]   # never a NULL pointer
    d_feat, d_el = gat_bwd_edges(csr, et_t, theta, alpha, feat, el, stats, slope, g, dpre, attn_l=attn_l, keep=keep,
                                 **dropout_kw(dropout))
    d_er, d_theta = gat_bwd_reduce(csr, et_csr, theta, alpha, dpre)
    d_al = d_ar = None
    if attn_l is not None:
        d_al, d_ar = attn_scores_bwd(feat, d_el, d_er, attn_r=attn_r, d_feat=d_feat)
    return d_feat, d_el, d_er, d_theta, d_al, d_ar


# The stages of ``gat_bwd``, which is built from them.  partition.halo_gat calls them one at a time, to exchange the
# statistics before the edge pass and the per-slot logit gradients between the edge pass and the reduction.  Full row
# ranges.

def gat_bwd_stats(out, g, er, rowmax, rowsum):
    """-> stats [N, H, 4] = (er, rowmax, 1/rowsum, <out, G>) per (row, head) (regnn_gat_bwd_stats)."""
    out, g, er = _f32(out), _f32(g), _f32(er)
    n, h, d = out.shape
    stats = torch.empty((n, h, 4), dtype=torch.float32, device=out.device)
    with torch.cuda.device(out.device):
        _lib.call('regnn_gat_bwd_stats', _ptr(out), _ptr(g), _ptr(er), _ptr(rowmax), _ptr(rowsum), n, h, d, _ptr(stats),
                  _stream())
        _lib.count_launches(1)
    return stats


def gat_bwd_edges(csr, et_t, theta, alpha, feat, el, stats, slope, g, dpre, attn_l=None, keep=None, dropout=None,
                  eid=None):
    """Source-major pass over the rows of the transposed view ``csr['indptr_t']`` -> (d_feat, d_el) of those rows; the
    logit gradient of every entry j is written to ``dpre[csr['slot_t'][j]]`` ([slots, H]).  ``feat`` / ``el``: the rows'
    own values; ``g`` / ``stats``: indexed by the column ids of the view.  ``attn_l`` folds the gradient through el into
    d_feat; ``keep``: the attention-dropout mask of ``gat_fwd``, in edge-id order through ``csr['eid']``;
    ``dropout``: the ``HashedDropout`` of ``gat_fwd`` instead; ``eid``: the edge id of every slot ``csr['slot_t']``
    points at when that is not ``csr['eid']`` (the extended slots of a halo partition) (regnn_gat_bwd_edges)."""
    feat, el, g, keep = _f32(feat), _f32(el), _f32(g), _f32(keep)
    eid = (csr['eid'] if eid is None else eid) if (keep is not None or dropout is not None) else None
    theta, et_t, r = _rel(theta, et_t)
    n = csr['indptr_t'].numel() - 1
    _, h, d = feat.shape
    dev = feat.device
    d_feat = torch.empty((n, h, d), dtype=torch.float32, device=dev)
    d_el = torch.zeros((n, h), dtype=torch.float32, device=dev)
    attn_l = _f32(attn_l).view(-1) if attn_l is not None else None
    sp_t, ws_t = _attn_split(csr.get('split_t'), h, d, dev)
    with torch.cuda.device(dev):
        _lib.call('regnn_gat_bwd_edges', _ptr(csr['indptr_t']), _ptr(csr['indices_t']), _ptr(csr['slot_t']),
                  _ptr(et_t) if r else None, _ptr(eid), _ptr(theta), float(alpha),
                  r, _ptr(feat), _ptr(el), _ptr(stats), float(slope), _ptr(keep), _drop(dropout, h), _ptr(g), h, d, 0,
                  n, _ptr(d_feat),
                  _ptr(d_el), _ptr(dpre), _ptr(attn_l), sp_t, _ptr(ws_t), _ptr(row_order(csr, True)), _stream())
        _lib.count_launches(1 + (3 if sp_t is not None else 0))
    return d_feat, d_el


def gat_bwd_reduce(csr, et_csr, theta, alpha, dpre):
    """Destination-side reductions of ``dpre`` over the rows of ``csr['indptr']`` -> (d_er [N, H], d_theta [R, H] | None)
    (regnn_gat_bwd_reduce)."""
    theta, et_csr, r = _rel(theta, et_csr)
    n = csr['indptr'].numel() - 1
    h = dpre.shape[1]
    dev = dpre.device
    d_er = torch.zeros((n, h), dtype=torch.float32, device=dev)
    partials = torch.empty(max(_lib.partial_blocks(n) * r * h, 1), dtype=torch.float64, device=dev)
    d_theta = torch.zeros((r, h), dtype=torch.float32, device=dev) if r else None
    sp, ws = _attn_split(csr.get('split'), h, 0, dev)
    with torch.cuda.device(dev):
        _lib.call('regnn_gat_bwd_reduce', _ptr(csr['indptr']), _ptr(et_csr) if r else None, _ptr(theta), float(alpha), r,
                  _ptr(dpre), h, 0, n, _ptr(d_er), _ptr(partials), _ptr(d_theta), sp, _ptr(ws), _stream())
        _lib.count_launches(((1 if n >= 65536 else 2) if r else 0) + 1 + (sp is not None))
    return d_er, d_theta


def attn_scores_bwd(feat, d_el, d_er, attn_r=None, d_feat=None):
    """-> (d_attn_l [H*D], d_attn_r [H*D]) of the projection scores; with ``d_feat`` and ``attn_r`` also
    d_feat += d_er * attn_r in place (regnn_attn_scores_bwd)."""
    feat = _f32(feat)
    n, h, d = feat.shape
    dev = feat.device
    attn_r = _f32(attn_r).view(-1) if attn_r is not None else None
    partials = torch.empty(max(_lib.partial_blocks(n) * 2 * h * d, 1), dtype=torch.float64, device=dev)
    d_al = torch.empty(h * d, dtype=torch.float32, device=dev)
    d_ar = torch.empty(h * d, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.call('regnn_attn_scores_bwd', _ptr(feat), _ptr(d_el), _ptr(d_er), n, h, d, _ptr(partials), _ptr(d_al),
                  _ptr(d_ar), _ptr(d_feat), _ptr(attn_r), _stream())
        _lib.count_launches(3)
    return d_al, d_ar


def attn_scores_fwd(feat, attn_l, attn_r):
    """el[n,h] = <feat[n,h,:], attn_l[h,:]>, er likewise (regnn_attn_scores_fwd)."""
    feat = _f32(feat)
    n, h, d = feat.shape
    attn_l, attn_r = _f32(attn_l).view(-1), _f32(attn_r).view(-1)
    el = torch.empty((n, h), dtype=torch.float32, device=feat.device)
    er = torch.empty((n, h), dtype=torch.float32, device=feat.device)
    with torch.cuda.device(feat.device):
        _lib.call('regnn_attn_scores_fwd', _ptr(feat), _ptr(attn_l), _ptr(attn_r), n, h, d, _ptr(el), _ptr(er), _stream())
        _lib.count_launches(1)
    return el, er


def gatv2_fwd(csr, et_csr, theta, alpha, fs, fd, attn, slope, keep=None, want_attn=False, rows=None, save=False,
              saved=None, dropout=None, eid=None):
    """-> (out, rowmax, rowsum, attention | None, saved | None).  ``save``: also store what the backward needs, the raw
    logit of every (CSR slot, head) and the 128-bit sign mask of fs[src]+fd[dst] per (slot, 128-float slice):
    ``saved = (logit_csr [E,H], qmask [E, ceil(H*D/128), 4] int32)``.  ``saved`` given (implies ``save``): the caller's
    buffers of that layout with at least E rows, written in place (partition.halo_gatv2 passes the head of its
    per-slot exchange buffers).  ``fs`` is indexed by the column ids of ``csr`` and may have more rows than the CSR (a
    halo of remote sources after the own rows); ``fd`` has one row per CSR row.  ``csr['eid']`` is only needed with
    ``keep``, ``dropout`` or ``want_attn``.  ``dropout`` / ``eid``: as ``gat_fwd``."""
    fs, fd, keep = _f32(fs), _f32(fd), _f32(keep)
    eid = csr.get('eid') if eid is None else eid
    attn = _f32(attn).view(-1)
    n, h, d = fd.shape
    rb, re = _rows(rows, n)
    theta, et_csr, r = _rel(theta, et_csr)
    dev = fs.device
    out = torch.empty_like(fd) if (rb, re) == (0, n) else torch.zeros_like(fd)
    rowmax = torch.zeros((n, h), dtype=torch.float32, device=dev)
    rowsum = torch.zeros((n, h), dtype=torch.float32, device=dev)
    e = csr['indices'].numel()
    att = torch.zeros((max(e, 1), h), dtype=torch.float32, device=dev)[:e] if want_attn else None
    save = save or saved is not None
    if save and e * max(h, (h * d + 127) // 128) >= 2 ** 32:
        raise ValueError('gatv2_fwd(save=True): E * max(H, ceil(H*D/128)) = %d exceeds the 32-bit slot offsets of the kernel'
                         % (e * max(h, (h * d + 127) // 128)))
    if saved is not None:
        if not (saved[0].dtype == torch.float32 and saved[1].dtype == torch.int32 and saved[0].is_contiguous()
                and saved[1].is_contiguous() and tuple(saved[0].shape[1:]) == (h,)
                and tuple(saved[1].shape[1:]) == ((h * d + 127) // 128, 4) and min(saved[0].shape[0], saved[1].shape[0]) >= e):
            raise ValueError('gatv2_fwd: saved must be contiguous fp32 [>=E, H] and int32 [>=E, ceil(H*D/128), 4] buffers')
    elif save:
        saved = (torch.empty((max(e, 1), h), dtype=torch.float32, device=dev),    # max(E, 1): never a NULL pointer
                 torch.empty((max(e, 1), (h * d + 127) // 128, 4), dtype=torch.int32, device=dev))
    sp, ws = _attn_split(csr.get('split'), h, d, dev)
    order = row_order(csr) if _full(rb, re, n) else None
    with torch.cuda.device(dev):
        _lib.call('regnn_gatv2_fwd', _ptr(csr['indptr']), _ptr(csr['indices']), _ptr(eid), _ptr(et_csr),
                  _ptr(theta), float(alpha), r, _ptr(fs), _ptr(fd), _ptr(attn), float(slope), _ptr(keep),
                  _drop(dropout, h), h, d,
                  rb, re, _ptr(out), _ptr(rowmax), _ptr(rowsum), _ptr(att), _ptr(saved[0]) if save else None,
                  _ptr(saved[1]) if save else None, sp, _ptr(ws), _ptr(order), _stream())
        _lib.count_launches(1 + (sp is not None))
    return out, rowmax, rowsum, att, saved


V2_STAGE_CHUNKS = 592   # REGNN_V2_STAGE_CHUNKS (csrc/gat.cu)


def gatv2_bwd(csr, et_csr, theta, alpha, fs, fd, attn, slope, keep, out, rowmax, rowsum, saved, g, dropout=None):
    """Backward of ``gatv2_fwd(..., save=True)``: ``gat_bwd_stats`` -> ``gatv2_bwd_edges`` (the one gather pass) ->
    ``gatv2_bwd_dst`` (streaming) -> (d_fs, d_fd, d_attn [H*D], d_theta | None).  ``dropout``: the ``HashedDropout`` of
    the forward."""
    logit_csr, qmask = saved
    stats = gat_bwd_stats(out, g, None, rowmax, rowsum)
    e = csr['indices'].numel()
    dl_csr = stats.new_empty((max(e, 1), stats.shape[1]))   # never a NULL pointer
    d_fs, d_attn_src = gatv2_bwd_edges(csr, fs, stats, logit_csr, qmask, attn, slope, g, dl_csr, keep=keep,
                                       **dropout_kw(dropout))
    d_fd, d_attn_dst, d_theta = gatv2_bwd_dst(csr, et_csr, theta, alpha, fd, dl_csr, qmask, attn, slope)
    return d_fs, d_fd, d_attn_src + d_attn_dst, d_theta


# The stages of ``gatv2_bwd``.  partition.halo_gatv2 calls them one at a time, to bring the stored logits and sign masks
# of cut edges to the source's owner before the edge pass and to return the per-slot dl between the two passes.  Full
# row ranges.

def gatv2_bwd_edges(csr, fs, stats, logit_csr, qmask, attn, slope, g, dl, keep=None, dropout=None, eid=None):
    """Source-major pass over the rows of the transposed view ``csr['indptr_t']`` -> (d_fs of those rows, their share
    d_attn_src [H*D] of d_attn); the logit and the sign mask of every entry j are read from, and its dl is written to,
    slot ``csr['slot_t'][j]`` of ``logit_csr`` / ``qmask`` / ``dl`` ([slots, H], [slots, C, 4], [slots, H]).  ``fs``: the
    rows' own values; ``g`` / ``stats`` (``gat_bwd_stats`` with er=None): indexed by the column ids of the view.
    ``keep``: the attention-dropout mask of ``gatv2_fwd``, in edge-id order through ``csr['eid']``; ``dropout`` /
    ``eid``: as ``gat_bwd_edges`` (regnn_gatv2_bwd_edges)."""
    fs, keep, g = _f32(fs), _f32(keep), _f32(g)
    eid = (csr['eid'] if eid is None else eid) if (keep is not None or dropout is not None) else None
    attn = _f32(attn).view(-1)
    n = csr['indptr_t'].numel() - 1
    _, h, d = fs.shape
    dev = fs.device
    d_fs = torch.empty((n, h, d), dtype=torch.float32, device=dev)
    d_attn_src = torch.empty(h * d, dtype=torch.float32, device=dev)
    split_t = csr.get('split_t')
    sp_t, ws_t = _attn_split(split_t, h, d, dev)
    nblocks = _lib.load().regnn_gatv2_bwd_edges_blocks(n, split_t['struct'].num_frags if split_t else 0,
                                                       split_t['struct'].num_long if split_t else 0, h, d, 1)
    block_partials = torch.empty(max(nblocks, 1) * h * d, dtype=torch.float32, device=dev)
    partials = torch.empty(V2_STAGE_CHUNKS * h * d, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.call('regnn_gatv2_bwd_edges', _ptr(csr['indptr_t']), _ptr(csr['indices_t']), _ptr(csr['slot_t']),
                  _ptr(eid), _ptr(fs), _ptr(stats), _ptr(logit_csr), _ptr(qmask),
                  _ptr(attn), float(slope), _ptr(keep), _drop(dropout, h), _ptr(g), h, d, 0, n, _ptr(d_fs), _ptr(dl),
                  _ptr(d_attn_src),
                  _ptr(block_partials), _ptr(partials), sp_t, _ptr(ws_t), _ptr(row_order(csr, True)), _stream())
        _lib.count_launches(3 + (sp_t is not None))
    return d_fs, d_attn_src


def gatv2_bwd_dst(csr, et_csr, theta, alpha, fd, dl, qmask, attn, slope):
    """Destination-side streaming pass over the rows of ``csr['indptr']``, reading ``dl`` and ``qmask`` in slot order
    -> (d_fd of those rows, their share d_attn_dst [H*D] of d_attn, d_theta [R, H] | None) (regnn_gatv2_bwd_dst)."""
    fd = _f32(fd)
    attn = _f32(attn).view(-1)
    theta, et_csr, r = _rel(theta, et_csr)
    n = csr['indptr'].numel() - 1
    _, h, d = fd.shape
    dev = fd.device
    d_fd = torch.empty((n, h, d), dtype=torch.float32, device=dev)
    d_attn_dst = torch.empty(h * d, dtype=torch.float32, device=dev)
    d_theta = torch.zeros((r, h), dtype=torch.float32, device=dev) if r else None   # stays 0 when the graph has no edges
    sp, ws = _attn_split(csr.get('split'), h, d, dev)
    partials = torch.empty(max(_lib.partial_blocks() * h * d, V2_STAGE_CHUNKS * r * h), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.call('regnn_gatv2_bwd_dst', _ptr(csr['indptr']), _ptr(et_csr) if r else None, _ptr(theta), float(alpha), r,
                  _ptr(fd), _ptr(dl), _ptr(qmask), _ptr(attn), float(slope), h, d, 0, n, _ptr(d_fd),
                  _ptr(d_attn_dst), _ptr(partials), _ptr(d_theta), sp, _ptr(ws), _stream())
        _lib.count_launches(2 + (2 if r else 0) + (sp is not None))
    return d_fd, d_attn_dst, d_theta


# ---- grouped per-node-type input projection ---------------------------------------------------------------------
GROUPED_BWD_SPLITS = 8


def _host_ptrs(tensors):
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr() if t is not None else None
    return arr


def _grouped_common(tables):
    t = len(tables)
    ldx = (ctypes.c_int64 * t)(*[x.stride(0) for x in tables])
    k = (ctypes.c_int * t)(*[x.shape[1] for x in tables])
    return ldx, k


def grouped_linear_fwd(tables, weights, biases, seg_ptr, perm, local_idx, num_rows):
    """out[i] = W[t(i)] x_{t(i)}[row(i)] + b[t(i)] for all node types in one launch (regnn_grouped_linear_fwd).
    ``tables`` / ``weights`` / ``biases``: per-type lists ([n_t, K_t] fp32; nn.Linear [n_out, K_t]; [n_out] or None);
    ``seg_ptr`` int32 [T+1] on the device; ``perm`` / ``local_idx`` int64 device tensors or None."""
    tables = [_f32(x) for x in tables]
    weights = [_f32(w) for w in weights]
    biases = [_f32(b) if b is not None else None for b in biases]
    n_out = weights[0].shape[0]
    dev = tables[0].device
    out = torch.empty((num_rows, n_out), dtype=torch.float32, device=dev)
    ldx, k = _grouped_common(tables)
    with torch.cuda.device(dev):
        _lib.call('regnn_grouped_linear_fwd', len(tables), _host_ptrs(tables), ldx, k, _host_ptrs(weights),
                  _host_ptrs(biases), n_out, int(num_rows), _ptr(seg_ptr), _ptr(perm), _ptr(local_idx), _ptr(out),
                  out.stride(0), _stream())
        _lib.count_launches(1)
    return out


def grouped_linear_bwd(tables, n_out, seg_ptr, perm, local_idx, dout, want_bias):
    """-> (per-type weight gradients [n_out, K_t], per-type bias gradients [n_out] | None): regnn_grouped_linear_bwd
    writes ``GROUPED_BWD_SPLITS`` deterministic partials per type, added here in split order."""
    tables = [_f32(x) for x in tables]
    dout = _f32(dout)
    dev = dout.device
    s = GROUPED_BWD_SPLITS
    dwp = [torch.empty((s, n_out, x.shape[1]), dtype=torch.float32, device=dev) for x in tables]
    dbp = [torch.empty((s, n_out), dtype=torch.float32, device=dev) for _ in tables] if want_bias else None
    ldx, k = _grouped_common(tables)
    with torch.cuda.device(dev):
        _lib.call('regnn_grouped_linear_bwd', len(tables), _host_ptrs(tables), ldx, k, n_out, dout.shape[0], _ptr(seg_ptr),
                  _ptr(perm), _ptr(local_idx), _ptr(dout), dout.stride(0), s, _host_ptrs(dwp),
                  _host_ptrs(dbp) if want_bias else None, _stream())
        _lib.count_launches(1)
    return [p.sum(dim=0) for p in dwp], ([p.sum(dim=0) for p in dbp] if want_bias else None)
