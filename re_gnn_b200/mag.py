"""MAG-stack (PyG-API) RE-GCN / RE-GAT / RE-GATv2 layers and model on the fused CUDA operators -- the
sampled-minibatch path of BASELINE config 5 ("next" row f-1 of SURVEY.md section 8).

Mirrors the constructor arguments, parameter names and forward conventions of
``REGCNConv`` / ``REGATConv`` / ``REGATv2Conv`` (mag/regnn_layers.py:24-433) and ``REGNN`` (mag/regnn_ns.py:216-346): bipartite
``(x_src, x_target)`` inputs with the targets first, ``edge_index`` [2,E] of local ids, 0-based ``edge_type``,
``self_loop_type == 2`` appending one typed self loop per target, ``aggr='mean'`` over the UN-normalised
relation weights (the ``ew`` the reference computes is returned but never used for aggregation, :119-129).
PyG / torch_scatter are not involved: the aggregation is ``regnn_spmm_fwd`` on a per-block CSR.
"""
import torch
import torch.nn.functional as F
from torch import nn

from . import functional as RF
from .graph import Graph


import os as _os

# REGNN_GROUPED_INPUT=0: the reference's per-type loop (mask / gather / Linear / scatter) instead of the grouped launch
USE_GROUPED_INPUT = _os.environ.get('REGNN_GROUPED_INPUT', '1') != '0'


def _grouped_input(lins, x_dict, node_type, local_node_idx):
    """Per-type input projection of a batch of nodes: types must be the keys 0 .. T-1 of ``x_dict`` (as in ogbn-mag's
    ``group_hetero_graph`` numbering)."""
    if not USE_GROUPED_INPUT or not node_type.is_cuda:
        width = next(iter(lins.values())).out_features
        h = torch.zeros((node_type.size(0), width), device=node_type.device, dtype=next(iter(lins.values())).weight.dtype)
        for key, x in x_dict.items():
            mask = node_type == key
            h[mask] = lins[str(key)](x[local_node_idx[mask]])
        return h
    keys = sorted(x_dict.keys())
    if keys != list(range(len(keys))):
        raise ValueError('node types must be numbered 0 .. T-1')
    tables = [x_dict[k] for k in keys]
    weights = [lins[str(k)].weight for k in keys]
    biases = [lins[str(k)].bias for k in keys]
    return RF.grouped_linear(tables, weights, biases, node_type, local_node_idx)


def _reference_edge_weights(edge_weight, col, num_targets, use_softmax):
    """``ew`` of mag/regnn_layers.py:113-124 / mag/regnn_saint.py:248-256: the relation weights of the edges normalised
    per destination -- by the weighted in-degree, or by mag/utils.py's global-max softmax with ``+ 1e-16``."""
    if use_softmax:
        ex = torch.exp(edge_weight - edge_weight.max()) if edge_weight.numel() else edge_weight
        den = torch.zeros(num_targets, dtype=ex.dtype, device=ex.device).index_add_(0, col, ex)
        return ex / (den[col] + 1e-16)
    deg = torch.zeros(num_targets, dtype=edge_weight.dtype, device=edge_weight.device).index_add_(0, col, edge_weight)
    return edge_weight * deg.pow(-1.0)[col]


class REGCNConv(nn.Module):
    def __init__(self, in_channels, out_channels, num_node_types, num_edge_types, scaling_factor=100., dropout=0.,
                 use_softmax=False, residual=False, use_norm=None, self_loop_type=1, no_re=False):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.num_node_types, self.num_edge_types = num_node_types, num_edge_types
        self.use_softmax, self.dropout, self.residual = use_softmax, dropout, residual
        self.use_norm, self.self_loop_type, self.scaling_factor = use_norm, self_loop_type, scaling_factor
        self.weight = nn.Parameter(torch.empty(in_channels, out_channels))
        if residual:
            self.weight_root = self.weight   # the reference aliases the two (:50)
        self.bias = nn.Parameter(torch.empty(out_channels))
        rw_dim = num_edge_types if self_loop_type in (1, 3) else num_edge_types + num_node_types
        self.relation_weight = nn.Parameter(torch.empty(rw_dim), requires_grad=not no_re)
        if use_norm == 'bn':
            self.norm = nn.BatchNorm1d(out_channels)
        elif use_norm == 'ln':
            self.norm = nn.LayerNorm(out_channels)
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.xavier_uniform_(self.weight)
        nn.init.zeros_(self.bias)
        nn.init.constant_(self.relation_weight, 1.0 / self.scaling_factor)
        if self.use_norm in ('bn', 'ln'):
            self.norm.reset_parameters()

    def build_block(self, edge_index, edge_type, target_node_type, n_src, n_dst):
        """Graph + 1-based edge types of one message-passing block, with the typed self loops of
        ``self_loop_type == 2`` appended (:90-96).  Reusable across calls on the same block (inference)."""
        src, dst = edge_index[0], edge_index[1]
        if self.self_loop_type == 2:
            loop = torch.arange(n_dst, dtype=src.dtype, device=src.device)
            src, dst = torch.cat([src, loop]), torch.cat([dst, loop])
            edge_type = torch.cat([edge_type, target_node_type + self.num_edge_types])
        return Graph(src, dst, n_src), (edge_type + 1).contiguous()

    def forward(self, x, edge_index, edge_type, target_node_type, return_weights=False, block=None):
        x_src, x_target = x
        n_src, n_dst = x_src.shape[0], x_target.shape[0]
        graph, etype1 = block if block is not None else self.build_block(edge_index, edge_type, target_node_type,
                                                                         n_src, n_dst)
        etv = graph.etype_views(etype1, self.relation_weight.numel())
        xs = x_src @ self.weight
        # aggr='mean': divide by the NUMBER of in-edges (incl. the appended loops); rows without edges give 0
        inv_cnt = 1.0 / graph.in_degrees().clamp(min=1).to(xs.dtype)
        out = RF.propagate(graph, etv, xs, self.relation_weight.view(-1, 1), self.scaling_factor, inv_cnt, sides=2)
        out = out[:n_dst] + self.bias
        if self.residual:
            out = out + x_target @ self.weight_root
        if self.use_norm in ('bn', 'ln'):
            out = self.norm(out)
        if return_weights:
            # the normalised per-edge weights the reference computes and returns but never aggregates with (:113-126),
            # in the order of the (self-loop-extended) edge list; a diagnostic path: plain torch ops
            w = F.leaky_relu(self.relation_weight * self.scaling_factor)
            src, dst = graph.edges()
            edge_weight = w[etype1 - 1]
            ew = _reference_edge_weights(edge_weight, dst, n_dst, self.use_softmax)
            return out, ew, w
        return out


class _MagAttentionBase(nn.Module):
    """Shared part of the MAG-stack ``REGATConv`` / ``REGATv2Conv`` (mag/regnn_layers.py:153-296, :298-433): one
    ``lin_src`` projection shared by both sides (``lin_dst`` aliases it, :188 / :333), relation embeddings
    ``[R, heads]``, typed self loops for ``self_loop_type == 2``, concat or mean over heads, bias, residual, norm.

    Softmax: the reference stabilises with the GLOBAL maximum of all logits and adds 1e-16 to every denominator
    (mag/utils.py:28-57); the fused kernels keep per-row statistics, from which the same values follow exactly
    (``functional._global_max_eps``: per-row factor s_v / (s_v + 1e-16 * exp(M - m_v)), carried into the backward)."""

    SOFTMAX_EPS = 1e-16

    def __init__(self, in_channels, out_channels, num_node_types, num_edge_types, heads=1, scaling_factor=100.,
                 concat=True, negative_slope=0.2, dropout=0.0, residual=False, use_norm=None, self_loop_type=1,
                 no_re=False):
        super().__init__()
        self.in_channels, self.out_channels, self.heads, self.concat = in_channels, out_channels, heads, concat
        self.negative_slope, self.dropout = negative_slope, dropout
        self.num_node_types, self.num_edge_types = num_node_types, num_edge_types
        self.residual, self.use_norm, self.self_loop_type = residual, use_norm, self_loop_type
        self.scaling_factor = scaling_factor
        self.out_dim = heads * out_channels if concat else out_channels
        self.lin_src = nn.Linear(in_channels, heads * out_channels, bias=False)
        self.lin_dst = self.lin_src
        self.bias = nn.Parameter(torch.empty(self.out_dim))
        rw_dim = num_edge_types if self_loop_type in (1, 3) else num_edge_types + num_node_types
        self.relation_weight = nn.Parameter(torch.empty(rw_dim, heads), requires_grad=not no_re)
        self._make_attention_parameters()
        if use_norm == 'bn':
            self.norm = nn.BatchNorm1d(self.out_dim)
        elif use_norm == 'ln':
            self.norm = nn.LayerNorm(self.out_dim)
        self.reset_parameters()

    def reset_parameters(self):
        self.lin_src.reset_parameters()
        self._reset_attention_parameters()
        nn.init.zeros_(self.bias)
        nn.init.constant_(self.relation_weight, 1.0 / self.scaling_factor)
        if self.use_norm in ('bn', 'ln'):
            self.norm.reset_parameters()

    build_block = REGCNConv.build_block

    def forward(self, x, edge_index, edge_type, target_node_type, return_weights=False, block=None):
        h, c = self.heads, self.out_channels
        if isinstance(x, torch.Tensor):
            xs = xd = self.lin_src(x).view(-1, h, c)
        else:
            xs = self.lin_src(x[0]).view(-1, h, c)
            xd = self.lin_dst(x[1]).view(-1, h, c)
        n_src, n_dst = xs.shape[0], xd.shape[0]
        graph, etype1 = block if block is not None else self.build_block(edge_index, edge_type, target_node_type,
                                                                         n_src, n_dst)
        etv = graph.etype_views(etype1, self.relation_weight.shape[0])
        out, attn = self._aggregate(graph, etv, xs, xd, n_src, return_weights)
        out = out[:n_dst]
        out = out.reshape(-1, h * c) if self.concat else out.mean(dim=1)
        out = out + self.bias
        if self.residual:
            out = out + xd.reshape(-1, h * c)
        if self.use_norm in ('bn', 'ln'):
            out = self.norm(out)
        return (out, attn) if return_weights else out

    @staticmethod
    def _pad_rows(t, n):
        """Destination-side tensors are indexed by graph row id; rows past the targets have no in-edges."""
        return t if t.shape[0] == n else torch.cat([t, t.new_zeros((n - t.shape[0],) + tuple(t.shape[1:]))])


class REGATConv(_MagAttentionBase):
    """mag/regnn_layers.py:153-296 on ``regnn_gat_fwd / _bwd_dst / _bwd_src``:
    ``logit = LeakyReLU_slope(w[etype] + <x_src, att_src>[src] + <x_dst, att_dst>[dst])``."""

    def _make_attention_parameters(self):
        self.att_src = nn.Parameter(torch.empty(1, self.heads, self.out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, self.heads, self.out_channels))

    def _reset_attention_parameters(self):
        nn.init.xavier_uniform_(self.att_src)
        nn.init.xavier_uniform_(self.att_dst)

    def _aggregate(self, graph, etv, xs, xd, n_src, want_attn):
        el = (xs * self.att_src).sum(-1)
        er = self._pad_rows((xd * self.att_dst).sum(-1), n_src)
        return RF.gat_aggregate(graph, etv, xs, el, er, self.relation_weight, self.scaling_factor, self.negative_slope,
                                None, want_attn, softmax_eps=self.SOFTMAX_EPS)


class REGATv2Conv(_MagAttentionBase):
    """mag/regnn_layers.py:298-433 on ``regnn_gatv2_fwd / _bwd_dst / _bwd_src``:
    ``logit = <att, LeakyReLU_slope(x_src[src] + x_dst[dst])> + w[etype]`` (relation term outside the activation)."""

    def _make_attention_parameters(self):
        self.att = nn.Parameter(torch.empty(1, self.heads, self.out_channels))

    def _reset_attention_parameters(self):
        nn.init.xavier_uniform_(self.att)

    def _aggregate(self, graph, etv, xs, xd, n_src, want_attn):
        return RF.gatv2_aggregate(graph, etv, xs, self._pad_rows(xd, n_src), self.att, self.relation_weight,
                                  self.scaling_factor, self.negative_slope, None, want_attn, softmax_eps=self.SOFTMAX_EPS)


class REGNN(nn.Module):
    """mag/regnn_ns.py:216-346 with per-type feature projections (``args.feats_type != 2``); the module-level
    ``args`` the reference reads (``args.model`` in {'regcn', 'regat', 'regatv2'}, ``args.self_loop_type``) become
    constructor keywords."""

    def __init__(self, in_channels, hidden_channels, out_channels, heads, num_layers, scaling_factor, dropout,
                 num_feature_dict, num_edge_types, residual, no_re, use_norm=None, self_loop_type=2, model='regcn'):
        super().__init__()
        self.in_channels, self.hidden_channels, self.out_channels = in_channels, hidden_channels, out_channels
        self.heads, self.num_layers, self.dropout = heads, num_layers, dropout
        self.residual, self.use_norm = residual, use_norm
        self.num_node_types, self.num_edge_types = len(num_feature_dict), num_edge_types
        self.model = model
        self.hidden_dim = hidden_channels if model == 'regcn' else hidden_channels * heads      # :236-239
        self.lins = nn.ModuleDict({str(k): nn.Linear(d, self.hidden_dim) for k, d in num_feature_dict.items()})
        kw = dict(dropout=dropout, residual=residual, use_norm=use_norm, self_loop_type=self_loop_type, no_re=no_re)
        if model == 'regcn':                                                                   # :254-273
            convs = [REGCNConv(hidden_channels, hidden_channels, self.num_node_types, num_edge_types, scaling_factor, **kw)
                     for _ in range(num_layers)]
        elif model in ('regat', 'regatv2'):
            cls = REGATConv if model == 'regat' else REGATv2Conv
            convs = [cls(self.hidden_dim, hidden_channels, self.num_node_types, num_edge_types, heads, scaling_factor, **kw)
                     for _ in range(num_layers)]
        else:
            raise NotImplementedError(model)
        self.convs = nn.ModuleList(convs)
        self.out_lin = nn.Linear(self.hidden_dim, out_channels)
        # model-level norm of the reference (mag/regnn_ns.py:274-277): registered and reset but never used in its
        # forward -- kept so that a reference checkpoint with use_norm set loads strictly
        if use_norm == 'bn':
            self.norm = nn.BatchNorm1d(self.hidden_dim)
        elif use_norm == 'ln':
            self.norm = nn.LayerNorm(self.hidden_dim)

    def group_input(self, x_dict, node_type, local_node_idx, n_id=None):
        """mag/regnn_ns.py:300-326: every node's features projected by the Linear of its type.  The reference loops over
        the types with a boolean mask, a CPU-side gather and a masked scatter each; here all types run in ONE grouped
        GEMM launch with the gather / scatter folded in (``functional.grouped_linear``), no host synchronisation."""
        if n_id is not None:
            node_type, local_node_idx = node_type[n_id], local_node_idx[n_id]
        return _grouped_input(self.lins, x_dict, node_type, local_node_idx)

    def prebuilt_blocks(self, blocks, edge_type, node_type):
        """The ``(Graph, etype1)`` of every device-sampled block (``sampling.Block.prebuilt``) for these convolutions,
        for ``forward(..., blocks=...)``."""
        conv = self.convs[0]
        return [b.prebuilt(edge_type, node_type, self.num_edge_types, conv.self_loop_type, conv.relation_weight.shape[0])
                for b in blocks]

    def forward(self, n_id, x_dict, adjs, edge_type, node_type, local_node_idx, blocks=None):
        """``blocks``: optional ``prebuilt_blocks`` of the batch, passed to the convolutions instead of building each
        block's graph from ``adjs``."""
        x = self.group_input(x_dict, node_type, local_node_idx, n_id)
        node_type = node_type[n_id]
        for i, (edge_index, e_id, size) in enumerate(adjs):
            x_target, node_type = x[:size[1]], node_type[:size[1]]
            if blocks is None:
                x = self.convs[i]((x, x_target), edge_index, edge_type[e_id], node_type)
            else:
                x = self.convs[i]((x, x_target), edge_index, None, node_type, block=blocks[i])
            x = F.dropout(F.relu(x), p=self.dropout, training=self.training)
        return self.out_lin(x).log_softmax(dim=-1)


@torch.no_grad()
def full_graph_inference(model, x_dict, edge_index, edge_type, node_type, local_node_idx):
    """Layer-wise full-neighbour inference (mag/regnn_ns.py:348-369) without leaving the device: the reference
    walks ``NeighborSampler(sizes=[-1])`` batches and bounces activations through host memory per layer; with
    every node as a target and all its in-edges, that is one full-graph convolution per layer.  The CSR (with
    the typed self loops) is built once and shared by all layers."""
    n = node_type.numel()
    x = model.group_input(x_dict, node_type, local_node_idx)
    block = model.convs[0].build_block(edge_index, edge_type, node_type, n, n)
    for conv in model.convs:
        x = F.relu(conv((x, x), edge_index, edge_type, node_type, block=block))
    return model.out_lin(x)


def allreduce_gradients(params, world_size, group=None):
    """Data-parallel gradient averaging: ONE all-reduce of the flattened gradients per step."""
    import torch.distributed as dist
    grads = [p.grad for p in params if p.grad is not None]
    if not grads or world_size == 1:
        return 0
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat /= world_size
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()
    return flat.numel()


def train_step(model, optimizer, sampler, seeds, labels, x_dict, edge_type, node_type, local_node_idx, epoch, batch,
               world_size=1):
    """One sampled-minibatch training step (mag/regnn_ns.py:399-407 + gradient all-reduce).  A batch sampled on a
    CUDA device reaches the convolutions with its graphs prebuilt from the sample.
    Returns (loss tensor, number of sampled edges)."""
    n_id, blocks = sampler.sample(seeds, epoch=epoch, batch=batch)
    adjs = [(b.edge_index, b.eid, b.size) for b in blocks]
    prebuilt = model.prebuilt_blocks(blocks, edge_type, node_type) if n_id.is_cuda else None
    optimizer.zero_grad(set_to_none=True)
    out = model(n_id, x_dict, adjs, edge_type, node_type, local_node_idx, blocks=prebuilt)
    loss = F.nll_loss(out, labels)
    loss.backward()
    allreduce_gradients(list(model.parameters()), world_size)
    optimizer.step()
    return loss.detach(), sum(int(b.src.numel()) for b in blocks)


# ------------------------------------------------------------------------------------------------------------------
# GraphSAINT variant (mag/regnn_saint.py)
class SaintREGCNConv(nn.Module):
    """``REGCNConv`` of mag/regnn_saint.py:195-275: ``aggr='add'`` with the relation weights normalised per destination,
    ``ew = w[etype] / deg[dst]`` (relation-WEIGHTED in-degree, no clamp) or, with ``use_softmax``, mag/utils.py's
    global-max softmax of the relation weights (``+ 1e-16``); ``F.dropout`` on ``ew`` in training; bias after aggregation.

    Both options run on the same fused SpMM: the softmax is a relation table ``exp(w - M)`` (positive, so the kernels'
    LeakyReLU is the identity on it) with the destination-side normaliser ``1 / (sum + 1e-16)``; dropping an edge weight
    is dropping the edge, so the aggregation runs on the kept-edge subgraph (its own CSR) with the survivors scaled by
    ``1 / (1 - p)``, while the normaliser still comes from all edges, as in the reference."""

    def __init__(self, in_channels, out_channels, num_node_types, num_edge_types, scaling_factor=100., gcn=False,
                 dropout=0., use_softmax=False):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.num_node_types, self.num_edge_types = num_node_types, num_edge_types
        self.use_softmax, self.dropout, self.scaling_factor = use_softmax, dropout, scaling_factor
        self.weight = nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.relation_weight = nn.Parameter(torch.empty(num_edge_types), requires_grad=not gcn)
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.xavier_uniform_(self.weight)
        nn.init.zeros_(self.bias)
        nn.init.constant_(self.relation_weight, 1.0 / self.scaling_factor)

    def forward(self, x, edge_index, edge_type, return_weights=False, graph=None, edge_keep=None, block=None):
        """``edge_keep`` (optional bool [E]): the dropout mask to use instead of drawing one (tests).  ``block``: the
        subgraph's ``(Graph, etype1)`` from ``Block.prebuilt`` (``edge_index`` is then not read); its edge-type views are
        already cached for ``etype1``.  ``edge_type`` stays the 0-based type of every edge."""
        x_src, x_target = x if isinstance(x, tuple) else (x, x)
        n_src, n_dst = x_src.shape[0], x_target.shape[0]
        etype1 = None
        if block is not None:
            graph, etype1 = block
        if graph is None:
            graph = Graph(edge_index[0], edge_index[1], n_src)
        r = self.num_edge_types
        etv = graph.etype_views(edge_type + 1 if etype1 is None else etype1, r)
        theta, alpha = self.relation_weight.view(-1, 1), self.scaling_factor
        if self.use_softmax:
            w = F.leaky_relu(theta * alpha)                                   # [R,1]: differentiable, R floats
            present = torch.zeros(r, dtype=torch.bool, device=w.device).index_fill_(0, edge_type, True).view(-1, 1)
            m_glob = torch.where(present, w, torch.full_like(w, float('-inf'))).max()
            theta = torch.where(present, torch.exp(w - m_glob), torch.zeros_like(w))   # table exp(w - M) >= 0
            alpha = 1.0
            deg = RF.weighted_degree_norm(graph, etv, theta, alpha, 1.0, clamp_min=0.0)   # exponent 1: the sum itself
            inv = 1.0 / (deg + 1e-16)
        else:
            inv = RF.weighted_degree_norm(graph, etv, theta, alpha, -1.0, clamp_min=0.0)
        g_agg, etv_agg, scale = graph, etv, 1.0
        if edge_keep is not None or (self.training and self.dropout > 0):
            if edge_keep is None:
                edge_keep = torch.rand(edge_type.numel(), device=edge_type.device) >= self.dropout
            scale = 1.0 / (1.0 - self.dropout)
            src, dst = graph.edges()
            g_agg = Graph(src[edge_keep], dst[edge_keep], n_src)
            etv_agg = g_agg.etype_views((edge_type + 1)[edge_keep], r)
            inv = inv * scale
        if self.in_channels < self.out_channels:
            # aggregation is linear, so A(xW) = (Ax)W: gather the narrower rows (e.g. 128 instead of 349 classes)
            out = RF.propagate(g_agg, etv_agg, x_src, theta, alpha, inv, sides=2)[:n_dst] @ self.weight
        else:
            out = RF.propagate(g_agg, etv_agg, x_src @ self.weight, theta, alpha, inv, sides=2)[:n_dst]
        out = out + self.bias
        if return_weights:
            wr = F.leaky_relu(self.relation_weight * self.scaling_factor)
            ew = _reference_edge_weights(wr[edge_type], graph.edges()[1], n_src, self.use_softmax)
            if edge_keep is not None:
                ew = ew * edge_keep.to(ew.dtype) * scale
            return out, ew
        return out


class SaintREGCN(nn.Module):
    """``REGCN`` of mag/regnn_saint.py:278-361 (full-subgraph forward)."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, scaling_factor, dropout,
                 num_feature_dict, num_edge_types, use_bn, residual, gcn):
        super().__init__()
        self.in_channels, self.hidden_channels, self.out_channels = in_channels, hidden_channels, out_channels
        self.num_layers, self.dropout, self.use_bn, self.residual = num_layers, dropout, use_bn, residual
        self.num_node_types, self.num_edge_types = len(num_feature_dict), num_edge_types
        self.lins = nn.ModuleDict({str(k): nn.Linear(d, hidden_channels) for k, d in num_feature_dict.items()})
        dims = [hidden_channels] * num_layers + [out_channels]
        self.convs = nn.ModuleList([
            SaintREGCNConv(dims[i], dims[i + 1] if i == num_layers - 1 else hidden_channels, self.num_node_types,
                           num_edge_types, scaling_factor, gcn) for i in range(num_layers)])
        self.bns = nn.ModuleList([nn.BatchNorm1d(hidden_channels) for _ in range(num_layers)])

    def group_input(self, x_dict, node_type, local_node_idx, n_id=None):
        if n_id is not None:
            node_type, local_node_idx = node_type[n_id], local_node_idx[n_id]
        return _grouped_input(self.lins, x_dict, node_type, local_node_idx)

    def forward(self, x_dict, edge_index, edge_type, node_type, local_node_idx, block=None):
        """``block``: the subgraph's prebuilt ``(Graph, etype1)`` (``Block.prebuilt``), shared by every layer; without it
        the layers share one ``Graph`` built from ``edge_index``."""
        x = self.group_input(x_dict, node_type, local_node_idx)
        graph = None
        if block is None:
            graph = Graph(edge_index[0], edge_index[1], x.shape[0])     # one CSR for all layers of this subgraph
        for layer, conv in enumerate(self.convs):
            x_pre = x
            x = conv(x, edge_index, edge_type, graph=graph, block=block)
            if layer != self.num_layers - 1:
                if self.residual:
                    x = x + x_pre
                if self.use_bn:
                    x = self.bns[layer](x)
                x = F.dropout(F.relu(x), p=self.dropout, training=self.training)
        return x.log_softmax(dim=-1)


def saint_train_step(model, optimizer, sampler, labels, train_mask, x_dict, edge_type, node_type, local_node_idx,
                     epoch, batch, world_size=1):
    """One GraphSAINT training step (mag/regnn_saint.py:427-443 + gradient all-reduce): loss on the training nodes
    of the sampled subgraph.  On a CUDA device the subgraph reaches the layers with its graph prebuilt from the sample
    (``sample_block`` + ``Block.prebuilt``, no self loops).  Returns (loss, number of subgraph edges)."""
    if sampler.graph.device.type == 'cuda':
        n_id, block = sampler.sample_block(epoch=epoch, batch=batch)
        prebuilt = block.prebuilt(edge_type, node_type, model.num_edge_types, 1, model.num_edge_types)
        edge_index, eid, num_edges = None, block.eid, block.src.numel()
    else:
        n_id, edge_index, eid = sampler.sample(epoch=epoch, batch=batch)
        prebuilt, num_edges = None, edge_index.shape[1]
    optimizer.zero_grad(set_to_none=True)
    out = model(x_dict, edge_index, edge_type[eid], node_type[n_id], local_node_idx[n_id], block=prebuilt)
    mask = train_mask[n_id]
    loss = F.nll_loss(out[mask], labels[n_id][mask])
    loss.backward()
    allreduce_gradients(list(model.parameters()), world_size)
    optimizer.step()
    return loss.detach(), int(num_edges)
