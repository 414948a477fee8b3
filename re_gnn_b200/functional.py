"""``torch.autograd.Function`` wrappers that stitch the CUDA operators into autograd.

The backward formulas are those of SURVEY.md Appendix A (derived from the reference's layer code:
layer/REGraphConv.py:52-106, REGATConv.py:64-100, REGATv2Conv.py:103-164, REMixHopConv.py:48-94);
all reductions are executed by the deterministic kernels in ``re_gnn_b200/csrc``.
"""
import torch

from . import ops
from .dropout import HashedDropout, attn_dropout_key  # noqa: F401  (public: the dropout= argument of the attention cores)


def _check_dropout(keep, dropout, name):
    if keep is not None and dropout is not None:
        raise ValueError('%s: pass either keep (an explicit [E, H] mask) or dropout (HashedDropout), not both' % name)
    if dropout is not None and not isinstance(dropout, HashedDropout):
        raise TypeError('%s: dropout must be a HashedDropout, got %s' % (name, type(dropout).__name__))


class _WDegNorm(torch.autograd.Function):
    """norm = max(sum_in LeakyReLU_0.01(alpha*theta)[etype], 1) ** exponent."""

    @staticmethod
    def forward(ctx, graph, etv, theta, alpha, exponent, clamp_min):
        csr = graph.csr()
        deg, norm = ops.wdeg_norm_fwd(csr, etv[0], theta, alpha, exponent, counts=etv[2] if len(etv) > 2 else None,
                                      clamp_min=clamp_min)
        ctx.graph, ctx.etv, ctx.alpha, ctx.exponent, ctx.clamp_min = graph, etv, alpha, exponent, clamp_min
        ctx.save_for_backward(theta, deg)
        return norm

    @staticmethod
    def backward(ctx, d_norm):
        theta, deg = ctx.saved_tensors
        d_theta = ops.wdeg_norm_bwd(ctx.graph.csr(), ctx.etv[0], theta, ctx.alpha, ctx.exponent, deg,
                                    d_norm.contiguous(), counts=ctx.etv[2] if len(ctx.etv) > 2 else None,
                                    clamp_min=ctx.clamp_min)
        return None, None, d_theta.view_as(theta), None, None, None


def weighted_degree_norm(graph, etv, theta, alpha, exponent=-0.5, clamp_min=1.0):
    """norm = max(deg, clamp_min) ** exponent; ``clamp_min <= 0`` = no clamp (0 for rows without in-edges)."""
    return _WDegNorm.apply(graph, etv, theta, alpha, exponent, clamp_min)


class _Propagate(torch.autograd.Function):
    """Y = norm (.) A_w (norm (.) X);  theta=None -> un-weighted (A_w = A);  norm=None -> no scaling.
    ``sides``: bit 0 scales the source side, bit 1 the destination side (3 = both, the REGCN case)."""

    @staticmethod
    def forward(ctx, graph, etv, x, theta, alpha, norm, sides):
        csr = graph.csr()
        weighted = theta is not None
        ns = norm if sides & 1 else None
        nd = norm if sides & 2 else None
        y = ops.spmm(csr['indptr'], csr['indices'], etv[0] if weighted else None, theta, alpha, ns, nd, x,
                     split=csr.get('split'), order=ops.row_order(csr) if x.shape[1] <= ops.NARROW_FEAT else None)
        ctx.graph, ctx.etv, ctx.alpha, ctx.weighted, ctx.has_norm = graph, etv, alpha, weighted, norm is not None
        ctx.sides = sides
        ctx.save_for_backward(x, y, theta if weighted else None, norm)
        return y

    @staticmethod
    def backward(ctx, g):
        x, y, theta, norm = ctx.saved_tensors
        csr = ctx.graph.csr()
        g = g.contiguous()
        need_x = ctx.needs_input_grad[2]
        need_theta = ctx.weighted and ctx.needs_input_grad[3]
        need_norm = ctx.has_norm and ctx.needs_input_grad[5]
        dx = d_theta = d_norm = xdx = None
        if need_theta and ops.fused_bwd_fits(x.shape[1], theta.numel()):
            # one gather pass over the transposed view: dX, the relation gradient and the norm gradient together
            fold = need_norm and ops.fused_dnorm_fits(x.shape[1], x, g, y)
            dx, d_theta, extra = ops.spmm_bwd_fused(csr, ctx.etv[1], theta, ctx.alpha, norm, x, g, sides=ctx.sides,
                                                    want_xdx=need_norm and not fold and bool(ctx.sides & 1),
                                                    y=y if fold else None, want_dnorm=fold)
            d_theta = d_theta.view_as(theta)
            if fold:
                d_norm = extra
            else:
                xdx = extra
        else:
            if need_x or need_norm or need_theta:
                # transposed SpMM: dX[u] = ns(u) * sum_{e in Out(u)} w_e * nd(dst) * G[dst]
                # (on the transposed view the roles of the two sides swap)
                ns = norm if ctx.sides & 2 else None
                nd = norm if ctx.sides & 1 else None
                dx = ops.spmm(csr['indptr_t'], csr['indices_t'], ctx.etv[1] if ctx.weighted else None, theta,
                              ctx.alpha, ns, nd, g, split=csr.get('split_t'),
                              order=ops.row_order(csr, True) if g.shape[1] <= ops.NARROW_FEAT else None)
            if need_theta:
                d_theta, _ = ops.spmm_bwd_w(csr, ctx.etv[0], theta, ctx.alpha, norm, x, y, g, dx, sides=ctx.sides,
                                            split=csr.get('split'))
                d_theta = d_theta.view_as(theta)
        if need_norm and d_norm is None:
            d_norm = ops.rowdot_norm_bwd(norm, x, y, g, dx, sides=ctx.sides, xdx=xdx)
        return None, None, (dx if need_x else None), d_theta, None, (d_norm if need_norm else None), None


def propagate(graph, etv, x, theta, alpha, norm, sides=3):
    return _Propagate.apply(graph, etv, x, theta, alpha, norm, sides if norm is not None else 0)


def _global_max_eps(csr, out, rowmax, rowsum, attn, eps):
    """The MAG stack's softmax (mag/utils.py:28-57) subtracts the GLOBAL maximum M of all logits and adds ``eps`` to
    every denominator: a_e = exp(l_e - M) / (sum exp(l - M) + eps).  In terms of the row statistics the fused kernels
    keep (row maximum m_v, s_v = sum exp(l - m_v)) that is exp(l_e - m_v) / (s_v + eps * exp(M - m_v)): the kernel result
    is rescaled by s_v / (s_v + eps_v) and the corrected denominator is what the backward kernels then see -- their
    formula dl = a (da - sum a da) holds unchanged for the un-normalised a.  (The derivative through M itself -- one
    logit, weight sum_v (1 - s_v / (s_v + eps_v)) <out_v, G_v> -- is dropped; it vanishes unless a row's logits sit
    ~20 below the global maximum.)  In place; returns the corrected row sums."""
    indptr = csr['indptr']
    has = (indptr[1:] > indptr[:-1]).unsqueeze(1)
    m_glob = torch.where(has, rowmax, torch.full_like(rowmax, float('-inf'))).max()
    corr = eps * torch.exp(m_glob - rowmax)
    new_sum = rowsum + corr
    factor = torch.where(rowsum > 0, rowsum / new_sum, torch.zeros_like(rowsum))
    out.mul_(factor.unsqueeze(-1))
    if attn is not None and attn.numel():
        dst_of_slot = csr['row'].long()
        eid = csr['eid'].long()
        attn[eid] = attn[eid] * factor[dst_of_slot]
    return torch.where(rowsum > 0, new_sum, rowsum)


class _GatAggregate(torch.autograd.Function):
    """Fused logits + edge softmax + aggregation with el / er supplied by the caller (bipartite blocks of the MAG stack:
    the scores come from different node sets)."""

    @staticmethod
    def forward(ctx, graph, etv, feat, el, er, theta, alpha, slope, keep, want_attn, softmax_eps, dropout):
        csr = graph.csr()
        et = etv[0] if etv is not None else None
        out, rowmax, rowsum, attn = ops.gat_fwd(csr, et, theta if et is not None else None, alpha, feat, el, er,
                                                slope, keep, want_attn, **ops.dropout_kw(dropout))
        if softmax_eps:
            rowsum = _global_max_eps(csr, out, rowmax, rowsum, attn, softmax_eps)
        ctx.graph, ctx.et, ctx.alpha, ctx.slope, ctx.dropout = graph, et, alpha, slope, dropout
        ctx.et_t = etv[1] if etv is not None else None
        ctx.save_for_backward(feat, el, er, theta if et is not None else None, keep, out, rowmax, rowsum)
        if want_attn:
            ctx.mark_non_differentiable(attn)
            return out, attn
        return out, None

    @staticmethod
    def backward(ctx, g, _g_attn=None):
        feat, el, er, theta, keep, out, rowmax, rowsum = ctx.saved_tensors
        csr = ctx.graph.csr()
        d_feat, d_el, d_er, d_theta, _, _ = ops.gat_bwd(csr, ctx.et, ctx.et_t, theta, ctx.alpha, feat, el, er, ctx.slope,
                                                        keep, out, rowmax, rowsum, g.contiguous(),
                                                        **ops.dropout_kw(ctx.dropout))
        return (None, None, d_feat, d_el, d_er, d_theta.view_as(theta) if d_theta is not None else None,
                None, None, None, None, None, None)


def gat_aggregate(graph, etv, feat, el, er, theta, alpha, slope, keep=None, want_attn=False, softmax_eps=0.0,
                  dropout=None):
    """``softmax_eps`` > 0: the MAG stack's global-max softmax with ``+ eps`` in the denominator (``_global_max_eps``).
    Attention dropout: ``keep`` (an [E, H] mask in edge-id order) or ``dropout`` (a ``HashedDropout``: the kernels
    compute the mask from the edge ids, nothing is drawn or stored)."""
    _check_dropout(keep, dropout, 'gat_aggregate')
    return _GatAggregate.apply(graph, etv, feat, el, er, theta, alpha, slope, keep, want_attn, softmax_eps, dropout)


class _GatLayer(torch.autograd.Function):
    """The whole REGAT core of layer/REGATConv.py:68-92 as ONE autograd node: projection scores el / er (one streaming
    kernel instead of two eager mul + sum pairs), fused logits + edge softmax + aggregation, and a one-gather-pass
    backward with the gradients through el / er folded into its kernels (no [N,H,D] temporaries from autograd)."""

    @staticmethod
    def forward(ctx, graph, etv, feat, attn_l, attn_r, theta, alpha, slope, keep, want_attn, dropout):
        csr = graph.csr()
        et = etv[0] if etv is not None else None
        feat = feat.contiguous()
        el, er = ops.attn_scores_fwd(feat, attn_l, attn_r)
        out, rowmax, rowsum, attn = ops.gat_fwd(csr, et, theta if et is not None else None, alpha, feat, el, er,
                                                slope, keep, want_attn, **ops.dropout_kw(dropout))
        ctx.graph, ctx.et, ctx.alpha, ctx.slope, ctx.dropout = graph, et, alpha, slope, dropout
        ctx.et_t = etv[1] if etv is not None else None
        ctx.save_for_backward(feat, el, er, attn_l, attn_r, theta if et is not None else None, keep, out, rowmax, rowsum)
        if want_attn:
            ctx.mark_non_differentiable(attn)
            return out, attn
        return out, None

    @staticmethod
    def backward(ctx, g, _g_attn=None):
        feat, el, er, attn_l, attn_r, theta, keep, out, rowmax, rowsum = ctx.saved_tensors
        csr = ctx.graph.csr()
        d_feat, _, _, d_theta, d_al, d_ar = ops.gat_bwd(csr, ctx.et, ctx.et_t, theta, ctx.alpha, feat, el, er, ctx.slope,
                                                        keep, out, rowmax, rowsum, g.contiguous(), attn_l=attn_l,
                                                        attn_r=attn_r, **ops.dropout_kw(ctx.dropout))
        return (None, None, d_feat, d_al.view_as(attn_l), d_ar.view_as(attn_r),
                d_theta.view_as(theta) if d_theta is not None else None, None, None, None, None, None)


def gat_layer(graph, etv, feat, attn_l, attn_r, theta, alpha, slope, keep=None, want_attn=False, dropout=None):
    """feat [N,H,D] (source and destination side are the same nodes) -> (out [N,H,D], attention | None).
    Attention dropout: ``keep`` or ``dropout`` (a ``HashedDropout``), as ``gat_aggregate``."""
    _check_dropout(keep, dropout, 'gat_layer')
    return _GatLayer.apply(graph, etv, feat, attn_l, attn_r, theta, alpha, slope, keep, want_attn, dropout)


class _GatV2Aggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, graph, etv, fs, fd, attn, theta, alpha, slope, keep, want_attn, softmax_eps, dropout):
        csr = graph.csr()
        et = etv[0] if etv is not None else None
        train = any(ctx.needs_input_grad)
        out, rowmax, rowsum, a, saved = ops.gatv2_fwd(csr, et, theta if et is not None else None, alpha, fs, fd, attn,
                                                      slope, keep, want_attn, save=train, **ops.dropout_kw(dropout))
        if softmax_eps:
            rowsum = _global_max_eps(csr, out, rowmax, rowsum, a, softmax_eps)
        ctx.graph, ctx.et, ctx.alpha, ctx.slope, ctx.dropout = graph, et, alpha, slope, dropout
        ctx.save_for_backward(fs, fd, attn, theta if et is not None else None, keep, out, rowmax, rowsum,
                              *(saved if train else ()))
        if want_attn:
            ctx.mark_non_differentiable(a)
            return out, a
        return out, None

    @staticmethod
    def backward(ctx, g, _g_attn=None):
        fs, fd, attn, theta, keep, out, rowmax, rowsum, logit_csr, qmask = ctx.saved_tensors
        csr = ctx.graph.csr()
        d_fs, d_fd, d_attn, d_theta = ops.gatv2_bwd(csr, ctx.et, theta, ctx.alpha, fs, fd, attn, ctx.slope, keep, out,
                                                    rowmax, rowsum, (logit_csr, qmask), g.contiguous(),
                                                    **ops.dropout_kw(ctx.dropout))
        return (None, None, d_fs, d_fd, d_attn.view_as(attn),
                d_theta.view_as(theta) if d_theta is not None else None, None, None, None, None, None, None)


def gatv2_aggregate(graph, etv, fs, fd, attn, theta, alpha, slope, keep=None, want_attn=False, softmax_eps=0.0,
                    dropout=None):
    """Attention dropout: ``keep`` or ``dropout`` (a ``HashedDropout``), as ``gat_aggregate``."""
    _check_dropout(keep, dropout, 'gatv2_aggregate')
    return _GatV2Aggregate.apply(graph, etv, fs, fd, attn, theta, alpha, slope, keep, want_attn, softmax_eps, dropout)


class _GroupedLinear(torch.autograd.Function):
    """All per-node-type input projections in one launch (model/REGCN.py:36-39 ``fc_list`` + cat,
    mag/regnn_ns.py:300-326 ``group_input``).  Differentiable w.r.t. the weights and biases; the feature tables are
    inputs of the model (no gradient)."""

    @staticmethod
    def forward(ctx, seg_ptr, perm, local_idx, num_rows, num_types, *tensors):
        tables = tensors[:num_types]
        weights = tensors[num_types:2 * num_types]
        biases = tensors[2 * num_types:3 * num_types]
        if any(x.requires_grad for x in tables):
            raise NotImplementedError('grouped_linear: gradients w.r.t. the feature tables are not built '
                                      '(the reference feeds fixed input features here)')
        out = ops.grouped_linear_fwd(tables, weights, biases, seg_ptr, perm, local_idx, num_rows)
        ctx.meta = (seg_ptr, perm, local_idx, num_types, weights[0].shape[0], [b is not None for b in biases])
        ctx.save_for_backward(*tables)
        return out

    @staticmethod
    def backward(ctx, dout):
        seg_ptr, perm, local_idx, num_types, n_out, has_bias = ctx.meta
        dws, dbs = ops.grouped_linear_bwd(ctx.saved_tensors, n_out, seg_ptr, perm, local_idx, dout.contiguous(), any(has_bias))
        dbs = [d if h else None for d, h in zip(dbs, has_bias)] if dbs is not None else [None] * num_types
        return (None, None, None, None, None) + (None,) * num_types + tuple(dws) + tuple(dbs)


_SEG_PTR_CACHE = {}


def grouped_linear(tables, weights, biases, node_type=None, local_idx=None):
    """``tables[t]``: [n_t, K_t] features of node type t; ``weights[t]`` / ``biases[t]``: its nn.Linear parameters.
    ``node_type`` / ``local_idx`` ([M] int64): the type of output row i and its row in that type's table
    (mag/regnn_ns.py:300-326).  Both None: the output is the concatenation of all tables' projections in type order
    (model/REGCN.py:36-39).  -> [M, n_out].  No host synchronisation either way."""
    t = len(tables)
    dev = tables[0].device
    if node_type is None:
        sizes = tuple(int(x.shape[0]) for x in tables)
        key = (sizes, str(dev))
        if key not in _SEG_PTR_CACHE:    # one host -> device copy per distinct shape (keeps the call graph-capturable)
            _SEG_PTR_CACHE[key] = torch.tensor((0,) + sizes, dtype=torch.int64).cumsum(0).to(device=dev, dtype=torch.int32)
        seg_ptr = _SEG_PTR_CACHE[key]
        perm, num_rows = None, sum(sizes)
    else:
        perm = torch.sort(node_type, stable=True).indices
        counts = torch.bincount(node_type, minlength=t)[:t]
        seg_ptr = torch.cat([counts.new_zeros(1), counts.cumsum(0)]).to(torch.int32)
        num_rows = int(node_type.numel())
        local_idx = local_idx.to(torch.int64).contiguous()
    bs = [b if b is not None else None for b in biases]
    # autograd.Function cannot take None tensors positionally in *args for differentiable slots: pass them through as is
    return _GroupedLinear.apply(seg_ptr, perm, local_idx, num_rows, t, *tables, *weights, *bs)
