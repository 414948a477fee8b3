"""The four relation-embedded convolution modules, re-built on the fused CUDA operators.

Constructor signatures, parameter / sub-module names (checkpoint compatible), initialisation and
``forward`` call conventions follow the reference:
  REGraphConv   layer/REGraphConv.py:7-106        REGATConv     layer/REGATConv.py:10-100
  REGATv2Conv   layer/REGATv2Conv.py:12-164       REMixHopConv  layer/REMixHopConv.py:7-94
What differs is underneath: no DGL frames and no per-edge tensors -- each forward is a handful of
dense projections (cuBLAS through torch) around one fused message-passing kernel.
"""
import torch
from torch import nn

from .. import functional as RF
from ..graph import ZeroInDegreeError


class _RelationEmbedded(nn.Module):
    """Shared piece: the per-relation embedding ``edge_weight`` ([R, width], init 1/alpha) and the
    lookup of the graph's cached uint8 edge-type views for a given 1-based ``e_feat`` tensor."""

    def _init_relation(self, num_etypes, scaling_factor, width):
        self.alpha = scaling_factor
        self.edge_weight = nn.Parameter(torch.empty(num_etypes, width))

    def _reset_relation(self):
        nn.init.constant_(self.edge_weight, 1.0 / self.alpha)

    def _views(self, graph, e_feat):
        return graph.etype_views(e_feat, self.edge_weight.shape[0])


class REGraphConv(_RelationEmbedded):
    def __init__(self, num_etypes, scaling_factor, in_feats, out_feats, norm=True, bias=True,
                 activation=None, weight=True, dropout=0.):
        super().__init__()
        self.in_feats, self.out_feats = in_feats, out_feats
        self.norm, self.dropout, self.activation = norm, dropout, activation
        self._init_relation(num_etypes, scaling_factor, 1)
        if weight:
            self.weight = nn.Parameter(torch.empty(in_feats, out_feats))
        else:
            self.register_parameter('weight', None)
        if bias:
            self.bias = nn.Parameter(torch.empty(out_feats))
        else:
            self.register_parameter('bias', None)
        self.feat_dropout = nn.Dropout(p=dropout)
        self.reset_parameters()

    def reset_parameters(self):
        if self.weight is not None:
            nn.init.xavier_uniform_(self.weight)
        if self.bias is not None:
            nn.init.zeros_(self.bias)
        self._reset_relation()

    def forward(self, graph, feat, e_feat, return_embedding=False):
        h = self.feat_dropout(feat)
        etv = self._views(graph, e_feat)
        nrm = RF.weighted_degree_norm(graph, etv, self.edge_weight, self.alpha, -0.5) if self.norm else None
        project_first = self.in_feats > self.out_feats and self.weight is not None
        if project_first:  # row scaling commutes with the projection, so the norm stays fused below
            h = h @ self.weight
        rst = RF.propagate(graph, etv, h, self.edge_weight, self.alpha, nrm)
        if not project_first and self.weight is not None:
            rst = rst @ self.weight
        if self.bias is not None:
            rst = rst + self.bias
        if self.activation is not None:
            rst = self.activation(rst)
        return rst


class REMixHopConv(_RelationEmbedded):
    def __init__(self, num_etypes, scaling_factor, in_feats, out_feats, p=[0, 1, 2], dropout=0,
                 activation=None, batchnorm=False):
        super().__init__()
        self.in_dim, self.out_dim, self.p = in_feats, out_feats, p
        self.activation, self.batchnorm = activation, batchnorm
        self.dropout = nn.Dropout(dropout)
        self._init_relation(num_etypes, scaling_factor, 1)
        if batchnorm:
            self.bn = nn.BatchNorm1d(out_feats * len(p))
        self.weights = nn.ModuleDict({str(j): nn.Linear(in_feats, out_feats, bias=False) for j in p})
        self.reset_parameters()

    def reset_parameters(self):
        if self.batchnorm:
            self.bn.reset_parameters()
        for lin in self.weights.values():
            lin.reset_parameters()
        self._reset_relation()

    def forward(self, graph, feats, e_feat):
        etv = self._views(graph, e_feat)
        nrm = RF.weighted_degree_norm(graph, etv, self.edge_weight, self.alpha, -0.5)
        top = max(self.p)
        outputs = []
        for j in range(top + 1):
            if j in self.p:
                outputs.append(self.weights[str(j)](feats))
            if j < top:  # the reference's extra hop after the highest power is dead code (Q5)
                feats = RF.propagate(graph, etv, feats, None, self.alpha, nrm)
        final = torch.cat(outputs, dim=1)
        if self.batchnorm:
            final = self.bn(final)
        if self.activation is not None:
            final = self.activation(final)
        return self.dropout(final)


def _kernel_head_dim(d):
    """Head width the attention kernels run at: the next power of two >= max(4, d), at most 512 (they reduce over a
    head with butterfly shuffles, a head wider than 128 floats held as D/128 chunks per lane).  Other widths -- e.g.
    ``out_feats = num_classes`` -- are zero-padded by the layer: zero columns add nothing to any logit and their
    outputs / gradients are sliced away."""
    p = 4
    while p < d:
        p *= 2
    if p > 512:
        raise ValueError('head width %d is not supported (at most 512 per head)' % d)
    return p


def _pad_last(t, width):
    return t if t.shape[-1] == width else torch.nn.functional.pad(t, (0, width - t.shape[-1]))


def _keep_mask(drop, num_edges, num_heads, like):
    """Attention-dropout scale per (edge, head) in edge-id order, drawn like the reference does
    (``attn_drop`` applied to the [E,H,1] attention tensor)."""
    if not drop.training or drop.p == 0.0:
        return None
    return drop(torch.ones(num_edges, num_heads, 1, dtype=like.dtype, device=like.device)).view(num_edges, num_heads)


class REGATConv(_RelationEmbedded):
    def __init__(self, num_etypes, scaling_factor, in_feats, out_feats, num_heads, feat_drop=0.,
                 attn_drop=0., negative_slope=0.2, residual=False, activation=None, use_weight=True):
        super().__init__()
        self.num_etypes, self.num_heads = num_etypes, num_heads
        self.in_feats, self.out_feats, self.use_weight = in_feats, out_feats, use_weight
        self.fc = nn.Linear(in_feats, out_feats * num_heads, bias=False) if use_weight else nn.Identity()
        self.attn_l = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.attn_r = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.feat_drop, self.attn_drop = nn.Dropout(feat_drop), nn.Dropout(attn_drop)
        self.negative_slope = negative_slope
        self.leaky_relu = nn.LeakyReLU(negative_slope)
        self._init_relation(num_etypes, scaling_factor, num_heads)
        if residual:
            self.res_fc = (nn.Linear(in_feats, num_heads * out_feats, bias=False)
                           if in_feats != out_feats else nn.Identity())
        else:
            self.register_buffer('res_fc', None)
        self.activation = activation
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain('relu')
        if self.use_weight:
            nn.init.xavier_normal_(self.fc.weight, gain=gain)
        nn.init.xavier_normal_(self.attn_l, gain=gain)
        nn.init.xavier_normal_(self.attn_r, gain=gain)
        if isinstance(self.res_fc, nn.Linear):
            nn.init.xavier_normal_(self.res_fc.weight, gain=gain)
        self._reset_relation()

    def forward(self, graph, feat, edge_feats=None):
        h = self.feat_drop(feat)
        f = self.fc(h).view(-1, self.num_heads, self.out_feats)
        etv = self._views(graph, edge_feats) if edge_feats is not None else None
        keep = _keep_mask(self.attn_drop, graph.number_of_edges(), self.num_heads, f)
        dk = _kernel_head_dim(self.out_feats)
        # el / er (:68-69), logits, edge softmax and aggregation (:71-92) are one autograd node on fused kernels
        rst, _ = RF.gat_layer(graph, etv, _pad_last(f, dk), _pad_last(self.attn_l, dk), _pad_last(self.attn_r, dk),
                              self.edge_weight, self.alpha, self.negative_slope, keep)
        rst = rst[..., :self.out_feats]
        if self.res_fc is not None:
            rst = rst + self.res_fc(h).view(h.shape[0], -1, self.out_feats)
        if self.activation:
            rst = self.activation(rst)
        return rst


class REGATv2Conv(_RelationEmbedded):
    def __init__(self, num_etypes, scaling_factor, in_feats, out_feats, num_heads, feat_drop=0.,
                 attn_drop=0., negative_slope=0.2, residual=False, activation=None,
                 allow_zero_in_degree=False, bias=True, share_weights=False, use_weight=True):
        super().__init__()
        self.num_etypes, self._num_heads, self._out_feats = num_etypes, num_heads, out_feats
        self._in_src_feats, self._in_dst_feats = in_feats if isinstance(in_feats, tuple) else (in_feats, in_feats)
        self._allow_zero_in_degree = allow_zero_in_degree
        self.use_weight, self.share_weights, self.bias = use_weight, share_weights, bias
        if use_weight:
            self.fc_src = nn.Linear(self._in_src_feats, out_feats * num_heads, bias=bias)
            if isinstance(in_feats, tuple):
                self.fc_dst = nn.Linear(self._in_dst_feats, out_feats * num_heads, bias=bias)
            elif share_weights:
                self.fc_dst = self.fc_src
            else:
                self.fc_dst = nn.Linear(self._in_src_feats, out_feats * num_heads, bias=bias)
        else:
            self.fc_src, self.fc_dst = nn.Identity(), nn.Identity()
        self.attn = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.feat_drop, self.attn_drop = nn.Dropout(feat_drop), nn.Dropout(attn_drop)
        self.negative_slope = negative_slope
        self.leaky_relu = nn.LeakyReLU(negative_slope)
        self._init_relation(num_etypes, scaling_factor, num_heads)
        if residual:
            self.res_fc = (nn.Linear(self._in_dst_feats, num_heads * out_feats, bias=bias)
                           if self._in_dst_feats != out_feats else nn.Identity())
        else:
            self.register_buffer('res_fc', None)
        self.activation = activation
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain('relu')
        def init_linear(lin):
            nn.init.xavier_normal_(lin.weight, gain=gain)
            if self.bias:
                nn.init.constant_(lin.bias, 0)

        # same draw order as the reference (fc_src, fc_dst, attn, res_fc) so equal seeds give equal weights
        if self.use_weight:
            init_linear(self.fc_src)
            if not self.share_weights:
                init_linear(self.fc_dst)
        nn.init.xavier_normal_(self.attn, gain=gain)
        if isinstance(self.res_fc, nn.Linear):
            init_linear(self.res_fc)
        self._reset_relation()

    def set_allow_zero_in_degree(self, set_value):
        self._allow_zero_in_degree = set_value

    def forward(self, graph, feat, edge_feats=None, get_attention=False):
        if not self._allow_zero_in_degree and graph.has_zero_in_degree():
            raise ZeroInDegreeError(
                'There are 0-in-degree nodes in the graph, output for those nodes will be invalid. '
                'This is harmful for some applications, causing silent performance regression. '
                'Adding self-loop on the input graph by calling `g = g.add_self_loop()` will resolve '
                'the issue. Setting ``allow_zero_in_degree`` to be `True` when constructing this module '
                'will suppress the check and let the code run.')
        H, D = self._num_heads, self._out_feats
        if isinstance(feat, tuple):
            h_src, h_dst = self.feat_drop(feat[0]), self.feat_drop(feat[1])
            fs = self.fc_src(h_src).view(-1, H, D)
            fd = self.fc_dst(h_dst).view(-1, H, D)
        else:
            h_src = h_dst = self.feat_drop(feat)
            fs = self.fc_src(h_src).view(-1, H, D)
            fd = fs if self.share_weights else self.fc_dst(h_src).view(-1, H, D)
        etv = self._views(graph, edge_feats) if edge_feats is not None else None
        keep = _keep_mask(self.attn_drop, graph.number_of_edges(), H, fs)
        dk = _kernel_head_dim(D)
        rst, att = RF.gatv2_aggregate(graph, etv, _pad_last(fs, dk), _pad_last(fd, dk), _pad_last(self.attn, dk),
                                      self.edge_weight, self.alpha, self.negative_slope, keep, get_attention)
        rst = rst[..., :D]
        if self.res_fc is not None:
            rst = rst + self.res_fc(h_dst).view(h_dst.shape[0], -1, D)
        if self.activation:
            rst = self.activation(rst)
        if get_attention:
            return rst, att.unsqueeze(-1)
        return rst


class RESAGEConv(_RelationEmbedded):
    """layer/RESAGEConv.py:8-114: source-side norm with exponent -1, no destination-side norm,
    plus the (projected) root feature.  ``weight_root`` exists only for checkpoint compatibility:
    the reference allocates it and never reads it (it multiplies the root by ``weight``, :60-61)."""

    def __init__(self, num_etypes, scaling_factor, in_feats, out_feats, norm=True, bias=True,
                 activation=None, weight=True, dropout=0.):
        super().__init__()
        self.in_feats, self.out_feats = in_feats, out_feats
        self.norm, self.dropout, self.activation = norm, dropout, activation
        self._init_relation(num_etypes, scaling_factor, 1)
        if weight:
            self.weight_root = nn.Parameter(torch.zeros(in_feats, out_feats))
            self.weight = nn.Parameter(torch.empty(in_feats, out_feats))
        else:
            self.register_parameter('weight_root', None)
            self.register_parameter('weight', None)
        if bias:
            self.bias = nn.Parameter(torch.empty(out_feats))
        else:
            self.register_parameter('bias', None)
        self.feat_dropout = nn.Dropout(p=dropout)
        self.reset_parameters()

    def reset_parameters(self):
        if self.weight is not None:
            nn.init.xavier_uniform_(self.weight)
        if self.bias is not None:
            nn.init.zeros_(self.bias)
        self._reset_relation()

    def forward(self, graph, feat, e_feat):
        h = self.feat_dropout(feat)
        root = h @ self.weight if self.weight_root is not None else h
        etv = self._views(graph, e_feat)
        nrm = RF.weighted_degree_norm(graph, etv, self.edge_weight, self.alpha, -1.0) if self.norm else None
        project_first = self.in_feats > self.out_feats and self.weight is not None
        if project_first:
            h = h @ self.weight
        rst = RF.propagate(graph, etv, h, self.edge_weight, self.alpha, nrm, sides=1)
        if not project_first and self.weight is not None:
            rst = rst @ self.weight
        rst = rst + root
        if self.bias is not None:
            rst = rst + self.bias
        if self.activation is not None:
            rst = self.activation(rst)
        return rst


class REGINConv(_RelationEmbedded):
    """layer/REGINConv.py:7-66: relation-weighted sum scaled on the destination side by
    ``max(deg,1)^-1``, then ``apply_func`` and the activation (``eps`` is carried but unused there)."""

    def __init__(self, num_etypes, scaling_factor, apply_func=None, aggregator_type='sum', init_eps=0,
                 learn_eps=False, activation=None):
        super().__init__()
        if aggregator_type not in ('sum', 'max', 'mean'):
            raise KeyError('Aggregator type {} not recognized.'.format(aggregator_type))
        self.apply_func, self._aggregator_type, self.activation = apply_func, aggregator_type, activation
        if learn_eps:
            self.eps = nn.Parameter(torch.FloatTensor([init_eps]))
        else:
            self.register_buffer('eps', torch.FloatTensor([init_eps]))
        self._init_relation(num_etypes, scaling_factor, 1)
        self.reset_parameters()

    def reset_parameters(self):
        if self.apply_func is not None:
            self.apply_func.reset_parameters()
        self._reset_relation()

    def forward(self, graph, feat, e_feat):
        etv = self._views(graph, e_feat)
        nrm = RF.weighted_degree_norm(graph, etv, self.edge_weight, self.alpha, -1.0)
        rst = RF.propagate(graph, etv, feat, self.edge_weight, self.alpha, nrm, sides=2)
        if self.apply_func is not None:
            rst = self.apply_func(rst)
        if self.activation is not None:
            rst = self.activation(rst)
        return rst
