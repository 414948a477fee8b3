"""Multi-GPU execution of the full-batch REGCN aggregation (BASELINE config 4: ogbn-mag-shaped graph over 2/4/8
B200).  The reference has no multi-GPU code (SURVEY.md 2.4); numerics must equal the single-device result (Y and dX
are bit-identical in every scheme below: all kernels add a row's slots in slot order).

Common contract: rank p holds the row block [r_p, r_{p+1}) of X and dL/dY and gets back the same rows of Y and dX;
every rank holds the whole CSR / transposed view (int32 structures, ~0.4 GB at MAG scale) and computes the cheap
relation-degree norm for all rows; the caller sums the R-float relation gradient once (``allreduce_relation_grads``).

1. ``partitioned_propagate`` -- destination-row blocks (owner computes):
   forward:  NCCL all-gather of the owned source rows -> full X; fused SpMM on the owned rows;
   backward: NCCL all-gather of the owned dL/dY rows -> full G; transposed SpMM on the owned SOURCE rows gives the
   owned dX rows (no reduce-scatter, no atomics).  Exchange-bound: (P-1)/P of the [N,F] matrix per rank, twice.
2. ``feature_sliced_propagate`` -- column slabs: every rank propagates ALL rows for F/P columns, so the SpMM and its
   backward need no remote rows; a row<->slab re-partition (N*F/P floats per rank, P times less) sits on each side:
   * ``exchange=None``: ``all_to_all_single`` (NCCL; gloo in the CPU tests) plus pack / unpack copies;
   * ``exchange=SlabExchange(...)``: our own kernels over NVLink peer memory -- ``regnn_rows_to_slabs`` pushes row
     blocks into the peers' slabs, the ``regnn_spmm_*_scatter`` epilogues store finished rows into their owners'
     row blocks; torch symmetric memory supplies the mapped buffers and the device-side barrier.
   The norm gradient's row dots span all columns, but the row owner has complete rows: ``d_norm`` is a local pass.
3. ``halo_propagate`` -- destination-row blocks that exchange only their **halo** (the remote rows their edges
   reference) and hold only local views (``HaloPartition``): every rank gathers E/P edges at the full row width.  The
   degree norm is computed inside from a local relation-count table (halo rows get their owner's bits); the exchange is
   one uneven all-to-all (``exchange=None``) or ``regnn_halo_push`` over peer memory (``exchange=HaloExchange(...)``).
   It pays off on graphs with locality (``synth.hetero_graph_local``, or a real graph after partitioning).
4. ``halo_gat`` -- the REGAT core on the same row blocks (``HaloPartition(..., attention=True)``): the features go
   forward through the in-halo, dL/dY and the softmax statistics backward through the out-halo, and the logit gradient
   of every cut edge goes back to its destination's owner (``regnn_halo_scatter`` or one more uneven all-to-all).
5. ``halo_gatv2`` -- the REGATv2 core on the same row blocks: as ``halo_gat``, plus a per-slot exchange in the forward
   direction -- the logit and sign mask the forward stored in the destination's slot go to the source's owner, whose
   edge pass reads them (``regnn_halo_push_slots`` or one more pair of uneven all-to-alls).
"""
import torch
import torch.distributed as dist

from . import _lib, ops


def row_blocks(indptr, parts, balance='edges'):
    """Row boundaries [r_0=0, ..., r_P=N].  ``balance='edges'``: ~equal in-edge counts per block (prefix sums of
    indptr), uneven row counts.  ``balance='rows'``: ceil(N/P) rows per block -- compute is less balanced, but the
    exchange becomes ONE even ``all_gather_into_tensor`` straight into the row-indexed buffer, which is what
    matters when the step is exchange-bound."""
    n = indptr.numel() - 1
    if balance == 'rows':
        per = (n + parts - 1) // parts
        return [min(n, p * per) for p in range(parts)] + [n]
    e = int(indptr[-1].item())
    targets = torch.arange(1, parts, device=indptr.device, dtype=torch.int64) * e // parts
    cuts = torch.searchsorted(indptr.to(torch.int64), targets)
    bounds = [0] + [int(c) for c in cuts.clamp(max=n).tolist()] + [n]
    for i in range(1, len(bounds)):
        bounds[i] = max(bounds[i], bounds[i - 1])
    return bounds


def _uniform_rows(bounds):
    parts = len(bounds) - 1
    per = bounds[1] - bounds[0]
    return per if per > 0 and all(bounds[p] == min(bounds[-1], p * per) for p in range(parts)) else 0


def _alloc_full(n, f, bounds, like):
    """[N, F] buffer indexed by global row id; over-allocated to P*ceil(N/P) rows for the even all-gather."""
    per = _uniform_rows(bounds)
    rows = max(n, per * (len(bounds) - 1)) if per else n
    return torch.empty((rows, f), dtype=like.dtype, device=like.device)


def _all_gather_rows(full, own, bounds, group):
    """Gathers every rank's row block into ``full`` (global row ids).  Equal-size blocks: one
    ``all_gather_into_tensor``.  Uneven blocks (balanced by edges): ProcessGroupNCCL's grouped broadcasts."""
    per = _uniform_rows(bounds)
    if per and dist.get_backend(group) == 'nccl' and full.shape[0] >= per * (len(bounds) - 1):
        send = own.contiguous()
        if send.shape[0] != per:      # last block: pad to the common size
            send = torch.cat([send, send.new_zeros((per - send.shape[0], send.shape[1]))])
        dist.all_gather_into_tensor(full[:per * (len(bounds) - 1)], send, group=group)
        return full
    views = [full[bounds[p]:bounds[p + 1]] for p in range(len(bounds) - 1)]
    if dist.get_backend(group) == 'nccl':
        dist.all_gather(views, own.contiguous(), group=group)
    else:  # gloo (CPU tests) has no uneven all-gather: one broadcast per owner
        rank = dist.get_rank(group)
        views[rank].copy_(own)
        for p, v in enumerate(views):
            if v.numel():
                dist.broadcast(v, src=dist.get_global_rank(group, p) if group is not None else p, group=group)
    return full


class _PartitionedPropagate(torch.autograd.Function):
    """Rows [rb, re) of  Y = norm (.) A_w (norm (.) X)  with X row-partitioned across ranks."""

    @staticmethod
    def forward(ctx, graph, etv, x_own, theta, alpha, norm, bounds, rank, group):
        csr = graph.csr()
        n = graph.number_of_nodes()
        rb, re = bounds[rank], bounds[rank + 1]
        x_full = _alloc_full(n, x_own.shape[1], bounds, x_own)
        _all_gather_rows(x_full, x_own, bounds, group)
        y_full = torch.empty_like(x_full)
        ops.spmm(csr['indptr'], csr['indices'], etv[0], theta, alpha, norm, norm, x_full, rows=(rb, re), out=y_full,
                 split=csr.get('split'))
        ctx.graph, ctx.etv, ctx.alpha, ctx.bounds, ctx.rank, ctx.group = graph, etv, alpha, bounds, rank, group
        ctx.save_for_backward(x_full, y_full, theta, norm)
        return y_full[rb:re]

    @staticmethod
    def backward(ctx, g_own):
        x_full, y_full, theta, norm = ctx.saved_tensors
        csr = ctx.graph.csr()
        bounds, rank = ctx.bounds, ctx.rank
        rb, re = bounds[rank], bounds[rank + 1]
        g_full = torch.empty_like(x_full)
        _all_gather_rows(g_full, g_own, bounds, ctx.group)
        dx_full = torch.empty_like(x_full)
        # owner computes: the transposed rows [rb, re) are this rank's SOURCE rows; one fused gather pass gives
        # their dX and this rank's share of the relation gradient (each edge belongs to exactly one source row)
        _, d_theta, xdx = ops.spmm_bwd_fused(csr, ctx.etv[1], theta, ctx.alpha, norm, x_full, g_full, rows=(rb, re),
                                             out=dx_full, want_xdx=True)
        d_norm = ops.rowdot_norm_bwd(norm, x_full, y_full, g_full, dx_full, rows=(rb, re), xdx=xdx)
        # d_theta / d_norm hold this rank's rows only; the caller all-reduces the parameter gradient once.
        return None, None, dx_full[rb:re], d_theta.view_as(theta), None, d_norm, None, None, None


def partitioned_propagate(graph, etv, x_own, theta, alpha, norm, bounds, rank, group=None):
    return _PartitionedPropagate.apply(graph, etv, x_own, theta, alpha, norm, bounds, rank, group)


def _rows_to_columns(own, per, parts, group):
    """[rows_own, F] row block (all columns)  ->  [P*per, F/P] column slab (all rows, this rank's columns).
    One all-to-all: block q of the send buffer holds this rank's rows restricted to rank q's columns, and
    lands on rank q at row offset rank*per -- the receive buffer IS the slab, no unpack pass."""
    fc = own.shape[1] // parts
    pad = own if own.shape[0] == per else torch.cat([own, own.new_zeros((per - own.shape[0], own.shape[1]))])
    send = pad.view(per, parts, fc).permute(1, 0, 2).contiguous()
    slab = torch.empty((parts * per, fc), dtype=own.dtype, device=own.device)
    dist.all_to_all_single(slab, send.view(parts * per, fc), group=group)
    return slab


def _columns_to_rows(slab, per, parts, rows_own, group):
    """Inverse of ``_rows_to_columns``: the slab is sent as is (block q = rank q's rows), the received
    [P, per, F/P] pieces are interleaved back into [rows_own, F]."""
    fc = slab.shape[1]
    recv = torch.empty_like(slab)
    dist.all_to_all_single(recv, slab, group=group)
    return recv.view(parts, per, fc).permute(1, 0, 2).reshape(per, parts * fc)[:rows_own]


def _own_rows_norm_grad(norm, x_own, y_own, g_own, dx_own, rb, re):
    """d_norm (length N, zero outside [rb, re)) from the owner's complete rows."""
    d_norm = torch.zeros_like(norm)
    if re > rb:
        d_norm[rb:re] = ops.rowdot_norm_bwd(norm[rb:re].contiguous(), x_own, y_own, g_own, dx_own)
    return d_norm


class _ColumnSlabPropagate(torch.autograd.Function):
    """Same contract as ``_PartitionedPropagate`` (row block in, row block out), but the aggregation itself runs
    feature-sliced: every rank propagates ALL rows for F/P of the columns, so the SpMM and its backward need
    no remote rows at all.  The row<->column re-partition is an all-to-all that moves (P-1)/P of ONE row block
    per rank (N*F/P floats) instead of the all-gather's (P-1) row blocks -- P times less NVLink traffic; the
    norm gradient's row dot products span all columns, but the row owner holds complete rows: a local pass."""

    @staticmethod
    def forward(ctx, graph, etv, x_own, theta, alpha, norm, bounds, rank, group):
        csr = graph.csr()
        parts = len(bounds) - 1
        per = _uniform_rows(bounds)
        if not per or x_own.shape[1] % parts:
            raise ValueError('feature-sliced propagation needs equal row blocks (row_blocks(..., balance="rows")) '
                             'and a feature width divisible by the number of ranks')
        x_cols = _rows_to_columns(x_own, per, parts, group)
        y_cols = torch.empty_like(x_cols)
        weighted = theta is not None
        ops.spmm(csr['indptr'], csr['indices'], etv[0] if weighted else None, theta, alpha, norm, norm, x_cols, out=y_cols,
                 split=csr.get('split'), order=ops.row_order(csr) if x_cols.shape[1] <= ops.NARROW_FEAT else None)
        ctx.graph, ctx.etv, ctx.alpha, ctx.bounds, ctx.rank, ctx.group = graph, etv, alpha, bounds, rank, group
        ctx.weighted = weighted
        y_own = _columns_to_rows(y_cols, per, parts, x_own.shape[0], group)
        ctx.x_own, ctx.y_own = x_own.detach(), y_own
        ctx.save_for_backward(x_cols, theta, norm)
        return y_own

    @staticmethod
    def backward(ctx, g_own):
        x_cols, theta, norm = ctx.saved_tensors
        csr = ctx.graph.csr()
        bounds, rank = ctx.bounds, ctx.rank
        parts, per = len(bounds) - 1, _uniform_rows(bounds)
        rb, re = bounds[rank], bounds[rank + 1]
        g_own = g_own.contiguous()
        g_cols = _rows_to_columns(g_own, per, parts, ctx.group)
        dx_cols = torch.empty_like(x_cols)
        d_theta = None
        if ctx.weighted:
            _, d_theta, _ = ops.spmm_bwd_fused(csr, ctx.etv[1], theta, ctx.alpha, norm, x_cols, g_cols, out=dx_cols)
            d_theta = d_theta.view_as(theta)
        else:   # un-weighted propagation (REMixHop's copy_u): the transposed SpMM alone
            ops.spmm(csr['indptr_t'], csr['indices_t'], None, None, ctx.alpha, norm, norm, g_cols, out=dx_cols,
                     split=csr.get('split_t'), order=ops.row_order(csr, True) if g_cols.shape[1] <= ops.NARROW_FEAT else None)
        dx_own = _columns_to_rows(dx_cols, per, parts, re - rb, ctx.group)
        # the row dot products of d_norm span all columns: the row owner has them all (x, y, dL/dY, dX row blocks),
        # so this is a local pass; the norm's own backward then yields a per-rank share of the relation gradient,
        # like d_theta above (this rank's columns), and the caller all-reduces the parameter gradient once
        d_norm = _own_rows_norm_grad(norm, ctx.x_own, ctx.y_own, g_own, dx_own, rb, re) if norm is not None else None
        return None, None, dx_own, d_theta, None, d_norm, None, None, None


class _PeerBuffers:
    """Peer-mapped buffers (torch symmetric memory over NVLink) of one call site, the device-side barrier across the
    ranks, and a [P, 256]-float table every rank writes its share of the relation gradient into
    (``allreduce_relation_grads``)."""

    GRAD_SLOTS = 256

    def _alloc(self, rows, cols, device, group):
        """-> (local buffer, int64 device tensor [P] of every rank's mapped base address)."""
        import torch.distributed._symmetric_memory as symm
        t = symm.empty((rows, cols), dtype=torch.float32, device=device)
        h = symm.rendezvous(t, group)
        self._handles.append(h)
        return t, torch.tensor([int(p) for p in h.buffer_ptrs], dtype=torch.int64, device=device)

    def barrier(self):
        """Device-side barrier across the ranks on the current stream: everything the ranks wrote into each
        other's buffers before it is visible after it."""
        with _lib.phase('peer_barrier'):
            self._handles[0].barrier()

    def allreduce_small(self, flat):
        """Deterministic sum of a small fp32 vector (<= GRAD_SLOTS) over the ranks: every rank pushes its share into
        row ``rank`` of every peer's table (regnn_rows_to_slabs with a one-row block), a barrier, then each rank
        reduces the P rows with one fixed-shape reduction -- the same order, hence the same bits, on every rank and
        for every topology (no ring / tree of a collective library decides the association)."""
        n = flat.numel()
        if n > self.GRAD_SLOTS:
            raise ValueError('at most %d floats' % self.GRAD_SLOTS)
        if not hasattr(self, '_grad_row'):
            self._grad_row = torch.zeros((1, self.GRAD_SLOTS * self.parts), dtype=torch.float32, device=flat.device)
        self._grad_row.view(self.parts, self.GRAD_SLOTS)[:, :n] = flat.view(1, -1)     # the same share goes to every peer
        ops.rows_to_slabs(self._grad_row, self.parts, self.rank, self.grad_ptrs)
        self.barrier()
        return self.grad_tab[:, :n].sum(dim=0)


class SlabExchange(_PeerBuffers):
    """Peer-mapped buffers of ONE feature-sliced aggregation call site: the
    two column slabs (X and dL/dY, [P*per, F/P]) that peers push their row blocks into, the two row blocks
    (Y and dX, [per, F]) that the SpMM kernels of all ranks store finished rows into, and a [P, 256]-float table
    every rank writes its share of the relation gradient into (``allreduce_relation_grads``).  ``y_cols`` is a plain
    local slab: this rank's columns of Y, kept for the folded norm gradient of the backward kernel.  Create it once
    per layer; a forward must be followed by its backward before the next forward (the buffers are reused)."""

    def __init__(self, feat, bounds, rank, device, group=None):
        group = group if group is not None else dist.group.WORLD
        self.parts, self.per, self.rank, self.feat = len(bounds) - 1, _uniform_rows(bounds), rank, feat
        if not self.per or feat % (4 * self.parts):
            raise ValueError('SlabExchange needs equal row blocks and F divisible by 4 * ranks')
        self.fc = feat // self.parts
        self._handles = []
        self.x_cols, self.x_ptrs = self._alloc(self.parts * self.per, self.fc, device, group)
        self.g_cols, self.g_ptrs = self._alloc(self.parts * self.per, self.fc, device, group)
        self.y_rows, self.y_ptrs = self._alloc(self.per, feat, device, group)
        self.dx_rows, self.dx_ptrs = self._alloc(self.per, feat, device, group)
        self.grad_tab, self.grad_ptrs = self._alloc(self.parts, self.GRAD_SLOTS, device, group)
        self.y_cols = torch.zeros((self.parts * self.per, self.fc), dtype=torch.float32, device=device)
        self.x_cols.zero_()
        self.g_cols.zero_()
        self.grad_tab.zero_()
        self.peer_y = _lib.PeerRows(self.y_ptrs.data_ptr(), self.parts, self.per, feat, rank * self.fc)
        self.peer_dx = _lib.PeerRows(self.dx_ptrs.data_ptr(), self.parts, self.per, feat, rank * self.fc)
        self.barrier()


class _PeerSlabPropagate(torch.autograd.Function):
    """``_ColumnSlabPropagate`` with both re-partitions done by our own kernels over peer memory: row blocks are
    pushed into the peers' column slabs (regnn_rows_to_slabs), and the SpMM kernels store every finished row
    straight into its owner's row block from their epilogue (regnn_spmm_*_scatter) -- no collective library
    call, no pack / unpack pass.  The norm gradient is folded into the backward kernel per column slab (its
    backward is linear, so the shares add up at the R-float level): no row-dot pass and no N-float exchange.
    ``alias=True`` returns views of the exchange buffers (valid until the next step) instead of copies."""

    @staticmethod
    def forward(ctx, graph, etv, x_own, theta, alpha, norm, bounds, rank, xch, alias):
        csr = graph.csr()
        rb, re = bounds[rank], bounds[rank + 1]
        x_own = x_own.contiguous()
        ops.rows_to_slabs(x_own, xch.parts, rank * xch.per, xch.x_ptrs)
        xch.barrier()            # every rank's slice of X has landed in my slab
        weighted = theta is not None
        ops.spmm_scatter(csr, etv[0] if weighted else None, theta, alpha, norm, norm, xch.x_cols, xch.peer_y,
                         y_local=xch.y_cols if (norm is not None and weighted) else None)
        xch.barrier()            # every rank's columns of my rows have landed in my row block
        y_own = xch.y_rows[:re - rb]
        if not alias or not weighted:
            y_own = y_own.clone()
        ctx.graph, ctx.etv, ctx.alpha, ctx.bounds, ctx.rank, ctx.xch, ctx.alias = graph, etv, alpha, bounds, rank, xch, alias
        ctx.weighted = weighted
        if not weighted:   # REMixHop's copy_u propagation: no fused backward to fold the norm gradient into
            ctx.x_own, ctx.y_own = x_own.detach(), y_own
        ctx.save_for_backward(theta, norm)
        return y_own

    @staticmethod
    def backward(ctx, g_own):
        theta, norm = ctx.saved_tensors
        csr, xch, rank = ctx.graph.csr(), ctx.xch, ctx.rank
        rb, re = ctx.bounds[rank], ctx.bounds[rank + 1]
        g_own = g_own.contiguous()
        ops.rows_to_slabs(g_own, xch.parts, rank * xch.per, xch.g_ptrs)
        xch.barrier()
        if not ctx.weighted:   # the transposed SpMM alone, rows scattered to their owners; the owner's row dots are local
            ops.spmm_scatter(csr, None, None, ctx.alpha, norm, norm, xch.g_cols, xch.peer_dx, transposed=True)
            xch.barrier()
            dx_own = xch.dx_rows[:re - rb].clone()
            d_norm = _own_rows_norm_grad(norm, ctx.x_own, ctx.y_own, g_own, dx_own, rb, re) if norm is not None else None
            return None, None, dx_own, None, None, d_norm, None, None, None, None
        # d_norm: every row's norm gradient restricted to this rank's columns (all N rows, a share of the total)
        d_theta, d_norm = ops.spmm_bwd_fused_scatter(csr, ctx.etv[1], theta, ctx.alpha, norm, xch.x_cols, xch.g_cols,
                                                     xch.peer_dx, y_cols=xch.y_cols if norm is not None else None)
        xch.barrier()
        dx_own = xch.dx_rows[:re - rb]
        if not ctx.alias:
            dx_own = dx_own.clone()
        return None, None, dx_own, d_theta.view_as(theta), None, d_norm, None, None, None, None


def feature_sliced_propagate(graph, etv, x_own, theta, alpha, norm, bounds, rank, group=None, exchange=None,
                             alias=False):
    """Row block in, row block out; the aggregation runs on column slabs.  ``exchange`` (a ``SlabExchange``):
    re-partition over peer memory inside our own kernels; None: NCCL / gloo all-to-alls."""
    if exchange is not None:
        return _PeerSlabPropagate.apply(graph, etv, x_own, theta, alpha, norm, bounds, rank, exchange, alias)
    return _ColumnSlabPropagate.apply(graph, etv, x_own, theta, alpha, norm, bounds, rank, group)


def _rows_to_head_slab(own, n, bounds, rank, group, xch, grad=False):
    """Row block [rows_own, H, D] -> this rank's head slab of all N rows [N, H*D/P]: one all-to-all, or (``xch``) pushed
    into every rank's ``x_cols`` (``g_cols`` with ``grad``) over peer memory."""
    own = own.flatten(1).contiguous()      # [0, H*D] for a rank that owns no rows
    if xch is None:
        return _rows_to_columns(own, _uniform_rows(bounds), len(bounds) - 1, group)[:n]
    cols, ptrs = (xch.g_cols, xch.g_ptrs) if grad else (xch.x_cols, xch.x_ptrs)
    ops.rows_to_slabs(own, xch.parts, rank * xch.per, ptrs)
    xch.barrier()            # every rank's rows of my heads have landed in my slab
    return cols[:n]


def _head_slab_to_rows(slab, rows_own, bounds, group, xch, grad=False):
    """Inverse of ``_rows_to_head_slab``: head slab [N, H/P, D] -> this rank's row block [rows_own, H*D], through
    ``xch.y_rows`` (``dx_rows`` with ``grad``) over peer memory."""
    n = slab.shape[0]
    slab = slab.flatten(1)
    if xch is None:
        parts, per = len(bounds) - 1, _uniform_rows(bounds)
        pad = torch.cat([slab, slab.new_zeros((parts * per - n, slab.shape[1]))]) if parts * per > n else slab
        return _columns_to_rows(pad.contiguous(), per, parts, rows_own, group)
    ops.slabs_to_rows(slab, n, xch.peer_dx if grad else xch.peer_y)
    xch.barrier()            # every rank's heads of my rows have landed in my row block
    return (xch.dx_rows if grad else xch.y_rows)[:rows_own].clone()


def _head_slice_grad(param, grad, sl):
    """The gradient of a [*, H, ...] parameter with this rank's head slice ``sl`` filled and zeros elsewhere."""
    if grad is None:
        return None
    full = torch.zeros_like(param)
    full[:, sl] = grad.view(full[:, sl].shape)
    return full


class _HeadSlicedGat(torch.autograd.Function):
    """REGAT core (projection scores + fused logits / edge softmax / aggregation) sharded over the HEADS: attention
    heads are independent (el / er, the softmax statistics and the aggregation never mix heads), so rank q runs all
    rows for heads [q*H/P, (q+1)*H/P) -- the same column-slab scheme as the REGCN aggregation.  The four row <-> slab
    re-partitions (``_rows_to_head_slab``, ``_head_slab_to_rows``) are one all-to-all each (NCCL; gloo in the CPU tests)
    or, with a ``SlabExchange`` ``xch`` of width H*D, our own kernels over peer memory (regnn_rows_to_slabs,
    regnn_slabs_to_rows), where the head slab of the features stays in ``xch.x_cols`` for the backward.  Row block in,
    row block out; parameter gradients (attn_l, attn_r, relation embedding) come back with this rank's head slice filled
    and zeros elsewhere: the caller sums them across ranks (``allreduce_relation_grads``)."""

    @staticmethod
    def forward(ctx, graph, etv, f_own, attn_l, attn_r, theta, alpha, slope, bounds, rank, group, xch, dropout):
        csr = graph.csr()
        n = graph.number_of_nodes()
        rows_own, heads, dim = f_own.shape
        hs = heads // (len(bounds) - 1)
        sl = slice(rank * hs, (rank + 1) * hs)
        # this rank's heads of the full-H mask: the counter hash takes the global head
        dropout = dropout.for_heads(rank * hs, heads) if dropout is not None else None
        f_cols = _rows_to_head_slab(f_own, n, bounds, rank, group, xch).view(n, hs, dim)
        al, ar = attn_l[:, sl].contiguous(), attn_r[:, sl].contiguous()
        th = theta[:, sl].contiguous() if etv is not None else None
        el, er = ops.attn_scores_fwd(f_cols, al, ar)
        out, rowmax, rowsum, _ = ops.gat_fwd(csr, etv[0] if etv is not None else None, th, alpha, f_cols, el, er, slope,
                                             **ops.dropout_kw(dropout))
        ctx.graph, ctx.etv, ctx.alpha, ctx.slope, ctx.bounds, ctx.rank, ctx.group, ctx.xch = \
            graph, etv, alpha, slope, bounds, rank, group, xch
        ctx.dropout = dropout
        ctx.sl = sl
        ctx.save_for_backward(f_cols, el, er, al, ar, th, out, rowmax, rowsum, attn_l, attn_r, theta)
        return _head_slab_to_rows(out, rows_own, bounds, group, xch).view(rows_own, heads, dim)

    @staticmethod
    def backward(ctx, g_own):
        f_cols, el, er, al, ar, th, out, rowmax, rowsum, attn_l, attn_r, theta = ctx.saved_tensors
        n, hs, dim = f_cols.shape
        rows_own, heads, _ = g_own.shape
        g_cols = _rows_to_head_slab(g_own, n, ctx.bounds, ctx.rank, ctx.group, ctx.xch, grad=True).view(n, hs, dim)
        et, et_t = (ctx.etv[0], ctx.etv[1]) if ctx.etv is not None else (None, None)
        d_f, _, _, d_th, d_al, d_ar = ops.gat_bwd(ctx.graph.csr(), et, et_t, th, ctx.alpha, f_cols, el, er, ctx.slope,
                                                   None, out, rowmax, rowsum, g_cols, attn_l=al, attn_r=ar,
                                                   **ops.dropout_kw(ctx.dropout))
        d_f_own = _head_slab_to_rows(d_f, rows_own, ctx.bounds, ctx.group, ctx.xch, grad=True).view(rows_own, heads, dim)
        return (None, None, d_f_own, _head_slice_grad(attn_l, d_al, ctx.sl), _head_slice_grad(attn_r, d_ar, ctx.sl),
                _head_slice_grad(theta, d_th, ctx.sl), None, None, None, None, None, None, None)


def head_sliced_gat(graph, etv, f_own, attn_l, attn_r, theta, alpha, slope, bounds, rank, group=None, exchange=None,
                    dropout=None):
    """f_own [rows_own, H, D] -> out rows [rows_own, H, D]; see ``_HeadSlicedGat``.  ``exchange`` (a ``SlabExchange`` of
    width H*D): the re-partitions run over peer memory inside our own kernels instead of NCCL / gloo all-to-alls.
    ``dropout`` (a ``functional.HashedDropout`` over all H heads): attention dropout; rank q computes the mask of its
    heads from the global head index, so the result is that of ``functional.gat_layer`` with the same ``dropout``."""
    _, heads, dim = f_own.shape
    _check_hashed_dropout(dropout, 'head_sliced_gat')
    if not _uniform_rows(bounds) or heads % (len(bounds) - 1):
        raise ValueError('head-sliced attention needs equal row blocks and num_heads divisible by the number of ranks')
    if exchange is not None and exchange.feat != heads * dim:
        raise ValueError('head-sliced attention over peer memory needs a SlabExchange of width num_heads * head_dim')
    return _HeadSlicedGat.apply(graph, etv, f_own, attn_l, attn_r, theta, alpha, slope, bounds, rank, group, exchange,
                                dropout)


def allreduce_relation_grads(params, group=None, exchange=None):
    """Sums the per-rank relation-embedding gradients (R x H floats each) -- the only cross-rank floating-point
    reduction of the partitioned layer.  ``exchange`` (a ``SlabExchange`` or ``HaloExchange``): all-gather over peer
    memory and a sum in rank order (bit-identical on every rank and topology); otherwise all-gather with the collective
    library (NCCL / gloo) followed by the same fixed-order sum."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    if exchange is not None and flat.numel() <= exchange.GRAD_SLOTS:
        total = exchange.allreduce_small(flat)
    else:
        with _lib.phase('allgather_relation_grads'):
            world = dist.get_world_size(group)
            parts = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(parts, flat, group=group)
        total = parts[0].clone()
        for q in range(1, world):
            total = total + parts[q]
    off = 0
    for g in grads:
        g.copy_(total[off:off + g.numel()].view_as(g))
        off += g.numel()


# ---- destination-row blocks with a halo exchange -------------------------------------------------------------------
def _owner(ids, bounds_t):
    """Rank owning each global row id (empty blocks own nothing)."""
    return torch.bucketize(ids, bounds_t[1:-1], right=True)


def _send_lists(own_local, remote_global, bounds_t, rank, parts, n_own):
    """Unique (peer, own row) pairs of one view, peer-major and row-ascending -> (local row ids int32, counts [P] int64).
    ``own_local``: this rank's row of every entry; ``remote_global``: the other end of the entry."""
    peer = _owner(remote_global, bounds_t)
    keep = peer != rank
    key = torch.unique(peer[keep] * max(n_own, 1) + own_local[keep])
    peer_of = key // max(n_own, 1)
    return (key - peer_of * max(n_own, 1)).to(torch.int32), torch.bincount(peer_of, minlength=parts)


class HaloPartition:
    """Local views of one destination-row block [rb, re) for ``halo_propagate``, built once per
    (graph, e_feat, bounds, rank) from the global ``Graph`` and its ``etype_views``; afterwards only local structures
    are kept.

    * in-view: rows [rb, re) of the destination-sorted CSR (slots ``indptr[rb]:indptr[re]``, global slot order).  An own
      source u is column ``u - rb``; a remote one is ``n_own + k``, k its position in the **in-halo** (remote sources
      sorted by global id, hence grouped by owner).
    * out-view: rows [rb, re) of the transposed view, destinations renumbered the same way into own rows plus an
      **out-halo**.
    * ``csr``: both views in the layout of ``Graph.csr()`` (with their own long-row splits and row orders): row lengths
      are the global ones, so fragments and kernel choice -- and hence every row's bits -- match the single-device run.
    * ``counts``: the [n_own + halo rows, R] relation-count table (own rows, in-halo, then the out-halo unless it is the
      same set): the degree norm of every row this rank touches, computed locally with the owner's bits.
    * send lists: for every peer q, the own rows (local ids) in q's in-halo / out-halo; ``recv_offset_*[q]``: the row of
      q's extended buffer at which this rank's segment lands (one all-gather of the halo counts at setup).

    ``attention=True`` (``halo_gat``) also keeps what the REGAT backward needs to send the logit gradient of an edge back
    to the owner of its destination (the slot belongs to the destination's in-view row):

    * ``eid_in``: global edge ids of the in-view slots (the kernels read them only for attention dropout, so they stay
      out of ``csr``); ``eid_ext``: the same for the extended slots [e_in + tail] that ``csr['slot_t']`` points at --
      ``eid_in``, then the global edge ids of the tail entries in tail order (the backward's dropout factors);
    * ``csr['slot_t']``: for every out-view entry (own source u -> destination v), its position in the **extended dpre
      buffer** [E_in_own + cut_out, H]: v's local in-view slot when v is own, else ``E_in_own + k`` with k its position
      in the **tail** -- grouped by owner, and within an owner by that owner's local slot (global slot order is both);
    * ``tail_ptr`` [P+1] (host, offsets into the tail) and ``tail_dst`` (int32): the owner's local slot of every tail
      entry -- the send side of regnn_halo_scatter;
    * ``dpre_recv`` (int64) and ``dpre_recv_counts`` [P]: per peer, the own in-view slots whose source that peer owns,
      slot-ascending -- the receive side of the all-to-all variant, entry for entry the peer's tail segment;
    * ``max_dpre_rows``: the largest extended dpre buffer over all ranks (the symmetric allocation size), computed from
      the global CSR like the tails, so no collective is needed;
    * ``push_slots`` = (send_slots int32, send_ptr [P+1], recv_offset [P]): the same exchange in the other direction, for
      ``halo_gatv2``, whose edge pass reads the logit and the sign mask that the forward stored in the destination's
      slot: ``send_slots`` is ``dpre_recv`` and lands on peer q from row ``e_in_q + tail_ptr_q[rank]`` of its extended
      buffers, i.e. on q's tail segment of this rank (regnn_halo_push_slots); also from the global CSR.

    Index bookkeeping with device-agnostic torch ops."""

    def __init__(self, graph, etv, bounds, rank, group=None, attention=False):
        self._build(graph, etv, bounds, rank, attention)
        table = self.halo_counts.view(1, -1)
        if self.parts > 1:
            gathered = [torch.empty_like(table) for _ in range(self.parts)]
            dist.all_gather(gathered, table, group=group)
            table = torch.cat(gathered)
        self._set_offsets(table.cpu())

    @classmethod
    def virtual_ranks(cls, graph, etv, bounds, attention=False):
        """All P partitions of ``bounds`` in one process (one device, no process group)."""
        parts = []
        for p in range(len(bounds) - 1):     # the counts exchange is this list: no process group, no collective
            part = cls.__new__(cls)
            part._build(graph, etv, bounds, p, attention)
            parts.append(part)
        table = torch.stack([p.halo_counts for p in parts]).cpu()
        for p in parts:
            p._set_offsets(table)
        return parts

    def _build(self, graph, etv, bounds, rank, attention=False):
        from .graph import SPLIT_THRESHOLD, _row_split
        if etv[2] is None:
            raise ValueError('HaloPartition needs the [N, R] relation-count table of etype_views(), which is not built for '
                             'this graph (N * R * 4 bytes > graph.COUNTS_MAX_BYTES): the halo rows\' norms come from it')
        csr = graph.csr()
        n, parts = graph.number_of_nodes(), len(bounds) - 1
        r = etv[2].numel() // max(n, 1)
        dev = csr['indptr'].device
        rb, re = int(bounds[rank]), int(bounds[rank + 1])
        n_own = re - rb
        self.parts, self.rank, self.bounds, self.n_own, self.num_relations = parts, rank, list(bounds), n_own, r
        bounds_t = torch.tensor(bounds, dtype=torch.int64, device=dev)
        own_rows = torch.arange(n_own, dtype=torch.int64, device=dev)

        def view(indptr, indices, et):
            s0, s1 = int(indptr[rb]), int(indptr[re])
            ip = (indptr[rb:re + 1] - s0).to(torch.int32).contiguous()
            other = indices[s0:s1].to(torch.int64)
            remote = (other < rb) | (other >= re)
            halo = torch.unique(other[remote])
            local = torch.where(remote, n_own + torch.searchsorted(halo, other), other - rb)
            row_of = torch.repeat_interleave(own_rows, (ip[1:] - ip[:-1]).to(torch.int64))
            return ip, local.to(torch.int32).contiguous(), et[s0:s1].clone(), halo, row_of, other

        ip_in, idx_in, self.et_in, self.in_halo, dst_of, src_of = view(csr['indptr'], csr['indices'], etv[0])
        ip_out, idx_out, self.et_out, self.out_halo, src_of_t, dst_of_t = view(csr['indptr_t'], csr['indices_t'], etv[1])
        self.csr = {'indptr': ip_in, 'indices': idx_in, 'indptr_t': ip_out, 'indices_t': idx_out,
                    'split': _row_split(ip_in, SPLIT_THRESHOLD), 'split_t': _row_split(ip_out, SPLIT_THRESHOLD)}
        # q's in-halo from this rank = own sources of an edge into q's block (seen from the out-view), and the other way
        self.send_in, self.send_in_counts = _send_lists(src_of_t, dst_of_t, bounds_t, rank, parts, n_own)
        self.send_out, self.send_out_counts = _send_lists(dst_of, src_of, bounds_t, rank, parts, n_own)
        self.n_in, self.n_out = self.in_halo.numel(), self.out_halo.numel()
        self.same_halo = bool(torch.equal(self.in_halo, self.out_halo))
        own_global = torch.arange(rb, re, dtype=torch.int64, device=dev)
        # global row of every row of the two extended buffers (own rows, then the halo)
        self.rows_in, self.rows_out = torch.cat([own_global, self.in_halo]), torch.cat([own_global, self.out_halo])
        rows = [own_global, self.in_halo]
        if not self.same_halo:
            rows.append(self.out_halo)
        self.counts = etv[2].view(n, r)[torch.cat(rows)].contiguous().view(-1)
        self.n_ext = self.counts.numel() // r
        # [2, P]: rows of my in-halo / out-halo that each rank owns
        self.halo_counts = torch.stack([torch.bincount(_owner(self.in_halo, bounds_t), minlength=parts),
                                        torch.bincount(_owner(self.out_halo, bounds_t), minlength=parts)]).view(-1)
        self.attention = attention
        if attention:
            self._build_attention(csr, bounds_t, src_of, dst_of_t)

    def _build_attention(self, csr, bounds_t, src_of, dst_of_t):
        """The attention views of the class docstring.  ``src_of``: global source of every in-view slot;
        ``dst_of_t``: global destination of every out-view entry."""
        rank, parts, rb, re = self.rank, self.parts, self.bounds[self.rank], self.bounds[self.rank + 1]
        slot_bounds = csr['indptr'].to(torch.int64)[bounds_t]      # global CSR slot range of every row block
        s0, s1 = int(slot_bounds[rank]), int(slot_bounds[rank + 1])
        t0, t1 = int(csr['indptr_t'][rb]), int(csr['indptr_t'][re])
        self.e_in = s1 - s0
        self.eid_in = csr['eid'][s0:s1].clone()
        gslot = csr['slot_t'][t0:t1].to(torch.int64)
        remote = (dst_of_t < rb) | (dst_of_t >= re)
        tail_glob, perm = torch.sort(gslot[remote])                # global slot order = owner-major, owner-slot order
        pos = torch.empty_like(perm)
        pos[perm] = torch.arange(perm.numel(), dtype=torch.int64, device=perm.device)
        slot_t = gslot - s0
        slot_t[remote] = self.e_in + pos
        self.csr['slot_t'] = slot_t.to(torch.int32).contiguous()
        tail_owner = _owner(dst_of_t[remote][perm], bounds_t)
        self.tail_dst = (tail_glob - slot_bounds[tail_owner]).to(torch.int32).contiguous()
        self.eid_ext = torch.cat([self.eid_in, csr['eid'][tail_glob]]).contiguous()
        self.tail_counts = torch.bincount(tail_owner, minlength=parts).tolist()
        self.tail_ptr = [0]
        for c in self.tail_counts:
            self.tail_ptr.append(self.tail_ptr[-1] + c)
        # receive side: own in-view slots by the owner of their source, slot-ascending within an owner
        src_owner = _owner(src_of, bounds_t)
        rem_in = src_owner != rank
        slots = torch.arange(self.e_in, dtype=torch.int64, device=src_of.device)[rem_in]
        key, _ = torch.sort(src_owner[rem_in] * max(self.e_in, 1) + slots)
        self.dpre_recv = key % max(self.e_in, 1)
        self.dpre_recv_counts = torch.bincount(src_owner[rem_in], minlength=parts).tolist()
        # the extended buffer of every rank: its in-view slots plus its cut out-edges (source own, destination not)
        all_src_owner = _owner(csr['indices'].to(torch.int64), bounds_t)
        all_dst_owner = _owner(torch.arange(int(slot_bounds[-1]), dtype=torch.int64, device=src_of.device), slot_bounds)
        cross = all_src_owner != all_dst_owner
        # [P, P] cut edges by (source owner, destination owner): row q is rank q's tail counts
        cut_pairs = torch.bincount(all_src_owner[cross] * parts + all_dst_owner[cross], minlength=parts * parts)
        cut_pairs = cut_pairs.view(parts, parts).cpu()
        e_in_all = (slot_bounds[1:] - slot_bounds[:-1]).cpu()
        self.max_dpre_rows = int((e_in_all + cut_pairs.sum(dim=1)).max())
        # push list of regnn_halo_push_slots (REGATv2): the receive list read the other way -- the stored logit and sign
        # mask of every own in-view slot whose source q owns go to q's tail segment of this rank
        tail_before = torch.cumsum(cut_pairs, dim=1) - cut_pairs      # [q, p]: q's tail entries owned by ranks < p
        self.push_slots = (self.dpre_recv.to(torch.int32).contiguous(),
                           [0] + torch.tensor(self.dpre_recv_counts, dtype=torch.int64).cumsum(0).tolist(),
                           [int(e_in_all[q] + tail_before[q, rank]) for q in range(parts)])

    def _set_offsets(self, table):
        """``table`` [P, 2, P] (host): every rank's ``halo_counts``."""
        table = table.view(self.parts, 2, self.parts).to(torch.int64)
        per = [self.bounds[q + 1] - self.bounds[q] for q in range(self.parts)]
        before = torch.cumsum(table, dim=2) - table           # rows of q's halo owned by ranks < p
        p = self.rank
        self.recv_offset_in = [0 if q == p else per[q] + int(before[q, 0, p]) for q in range(self.parts)]
        self.recv_offset_out = [0 if q == p else per[q] + int(before[q, 1, p]) for q in range(self.parts)]
        self.recv_counts_in = table[p, 0].tolist()
        self.recv_counts_out = table[p, 1].tolist()
        self.max_rows_in = max(per[q] + int(table[q, 0].sum()) for q in range(self.parts))
        self.max_rows_out = max(per[q] + int(table[q, 1].sum()) for q in range(self.parts))
        # push lists of regnn_halo_push: the send lists with this rank's own rows as the self entry (into the head)
        self.push_in = self._push_list(self.send_in, self.send_in_counts, self.recv_offset_in)
        self.push_out = self._push_list(self.send_out, self.send_out_counts, self.recv_offset_out)

    def _push_list(self, rows, counts, offsets):
        counts = counts.tolist()
        counts[self.rank] = self.n_own
        cut = sum(counts[:self.rank])
        own = torch.arange(self.n_own, dtype=torch.int32, device=rows.device)
        ptr = [0]
        for c in counts:
            ptr.append(ptr[-1] + c)
        return torch.cat([rows[:cut], own, rows[cut:]]).contiguous(), ptr, offsets


class HaloExchange(_PeerBuffers):
    """Peer-mapped halo buffers of ONE ``halo_propagate`` call site: X [n_own + in-halo, F] and dL/dY
    [n_own + out-halo, F], own rows in the head, halos in the tail, written by every rank's ``regnn_halo_push``.
    Symmetric allocation needs one size on every rank: the maximum over ranks.  Also carries the [P, 256] table of
    ``allreduce_relation_grads``.  A forward must be followed by its backward before the next forward (the buffers
    are reused).

    ``heads`` (a ``halo_gat`` call site, ``feat`` = heads * head_dim, ``part`` built with ``attention=True``): also the
    softmax statistics of the out-halo [n_own + out-halo, 4 * heads], the extended dpre buffer
    [E_in_own + cut_out, heads] that peers scatter the logit gradients of this rank's in-view slots into, and a gradient
    table wide enough for d_attn_l, d_attn_r and d_theta together (2 * feat + R * heads floats).

    ``gatv2=True`` (a ``halo_gatv2`` call site, with ``heads``): also the extended per-slot buffers of the stored logits
    [E_in_own + cut_out, heads] and sign masks [E_in_own + cut_out, 4 * C] (fp32 storage of int32 [., C, 4] words,
    C = ceil(feat / 128)): the forward writes the head, peers fill the tail with regnn_halo_push_slots.  dl reuses the
    dpre buffer."""

    def __init__(self, part, feat, device, group=None, heads=None, gatv2=False):
        group = group if group is not None else dist.group.WORLD
        self.parts, self.rank, self.feat, self.heads, self.gatv2 = part.parts, part.rank, feat, heads, gatv2
        if gatv2 and heads is None:
            raise ValueError('HaloExchange(gatv2=True) needs heads=H')
        self._handles = []
        self.x_ext, self.x_ptrs = self._alloc(max(part.max_rows_in, 1), feat, device, group)
        self.g_ext, self.g_ptrs = self._alloc(max(part.max_rows_out, 1), feat, device, group)
        if heads is not None:
            if not getattr(part, 'attention', False):
                raise ValueError('HaloExchange(heads=...) needs a HaloPartition built with attention=True')
            self.s_ext, self.s_ptrs = self._alloc(max(part.max_rows_out, 1), 4 * heads, device, group)
            self.dpre, self.dpre_ptrs = self._alloc(max(part.max_dpre_rows, 1), heads, device, group)
            self.GRAD_SLOTS = max(self.GRAD_SLOTS, (2 * feat + part.num_relations * heads + 63) // 64 * 64)
        if gatv2:
            chunks = (feat + 127) // 128
            _check_slot_offsets(part, heads, chunks)
            self.logit_ext, self.logit_ptrs = self._alloc(max(part.max_dpre_rows, 1), heads, device, group)
            mask, self.mask_ptrs = self._alloc(max(part.max_dpre_rows, 1), 4 * chunks, device, group)
            self.mask_ext = mask.view(torch.int32).view(-1, chunks, 4)
        self.grad_tab, self.grad_ptrs = self._alloc(self.parts, self.GRAD_SLOTS, device, group)
        self.grad_tab.zero_()
        self.barrier()


def _fill_halo(part, own, direction, group, xch):
    """[n_own + halo, F] buffer of one direction ('in': X for the forward, 'out': dL/dY for the backward): own rows in
    the head, the halo -- rows pushed by their owners -- in the tail."""
    n_halo = part.n_in if direction == 'in' else part.n_out
    if xch is not None:
        rows, ptr, offsets = part.push_in if direction == 'in' else part.push_out
        buf, ptrs = (xch.x_ext, xch.x_ptrs) if direction == 'in' else (xch.g_ext, xch.g_ptrs)
        if ptr[-1]:              # an empty row block has nothing to send (and no edges)
            ops.halo_push(own, rows, ptr, offsets, ptrs, buf.stride(0), part.rank)
        xch.barrier()            # every owner's rows of my halo have landed
        return buf[:part.n_own + n_halo]
    send = part.send_in if direction == 'in' else part.send_out
    send_counts = part.send_in_counts if direction == 'in' else part.send_out_counts
    recv_counts = part.recv_counts_in if direction == 'in' else part.recv_counts_out
    buf = torch.empty((part.n_own + n_halo, own.shape[1]), dtype=own.dtype, device=own.device)
    buf[:part.n_own] = own
    if part.parts > 1:
        with _lib.phase('halo_all_to_all'):
            dist.all_to_all_single(buf[part.n_own:], own.index_select(0, send.to(torch.int64)),
                                   output_split_sizes=recv_counts, input_split_sizes=send_counts.tolist(), group=group)
    return buf


def _halo_norm(part, theta, alpha):
    """(deg, norm) of every row of the count table: own rows, in-halo, out-halo."""
    if part.n_ext == 0:
        z = theta.new_zeros(0)
        return z, z
    return ops.wdeg_norm_fwd(None, None, theta, alpha, -0.5, counts=part.counts)


def _halo_forward(part, x_ext, theta, alpha, weighted):
    """-> (y_own, deg, norm) from the filled [n_own + in-halo, F] buffer: the degree norm of every count-table row, then
    the SpMM over the in-view."""
    if weighted and not ops.fused_bwd_fits(x_ext.shape[1], theta.numel()):
        raise ValueError('halo_propagate: the weighted backward runs the fused kernel only, which does not cover F=%d '
                         'with %d relations (ops.fused_bwd_fits: F <= 1024 and its shared-memory tile must fit)'
                         % (x_ext.shape[1], theta.numel()))
    deg, norm = _halo_norm(part, theta, alpha)
    if not part.n_own:
        return x_ext.new_zeros((0, x_ext.shape[1])), deg, norm
    csr = part.csr
    norm_in = norm[:part.n_own + part.n_in]
    y_own = ops.spmm(csr['indptr'], csr['indices'], part.et_in if weighted else None, theta if weighted else None,
                     alpha, norm_in, norm_in, x_ext, split=csr['split'],
                     order=ops.row_order(csr) if x_ext.shape[1] <= ops.NARROW_FEAT else None)
    return y_own, deg, norm


def _halo_backward(part, x_own, y_own, g_ext, theta, alpha, weighted, deg, norm):
    """-> (dX own rows, this rank's share of d_theta) from the filled [n_own + out-halo, F] dL/dY buffer."""
    n_own, f = part.n_own, x_own.shape[1]
    if not n_own:
        return x_own.new_zeros(x_own.shape), torch.zeros_like(theta)
    csr = part.csr
    g_own = g_ext[:n_own]
    # norms of the out-view: own rows, then the out-halo (the same rows as the in-halo on a symmetric graph)
    norm_out = norm if part.same_halo else torch.cat([norm[:n_own], norm[n_own + part.n_in:]])
    norm_own = norm[:n_own]
    d_theta = None
    if weighted:
        fold = ops.fused_dnorm_fits(f)
        dx_own, d_theta, extra = ops.spmm_bwd_fused(csr, part.et_out, theta, alpha, norm_out, x_own, g_ext,
                                                    want_xdx=not fold, y=y_own if fold else None, want_dnorm=fold)
        d_norm = extra if fold else ops.rowdot_norm_bwd(norm_own, x_own, y_own, g_own, dx_own, xdx=extra)
    else:   # REMixHop: the transposed SpMM alone, then the owner's row dots
        dx_own = ops.spmm(csr['indptr_t'], csr['indices_t'], None, None, alpha, norm_out, norm_out, g_ext,
                          split=csr['split_t'], order=ops.row_order(csr, True) if f <= ops.NARROW_FEAT else None)
        d_norm = ops.rowdot_norm_bwd(norm_own, x_own, y_own, g_own, dx_own)
    # the norm's share of the relation gradient: own rows only (a halo row's norm gradient is its owner's)
    d_theta_norm = ops.wdeg_norm_bwd(None, None, theta, alpha, -0.5, deg, d_norm, rows=(0, n_own), counts=part.counts)
    return dx_own, (d_theta_norm if d_theta is None else d_theta + d_theta_norm).view_as(theta)


class _HaloPropagate(torch.autograd.Function):
    """Rows [rb, re) of  Y = n (.) A_w (n (.) X)  (``weighted=False``: A instead of A_w, REMixHop) with the degree norm
    n computed inside from the relation weights; X and dL/dY row-partitioned, only halo rows exchanged."""

    @staticmethod
    def forward(ctx, part, x_own, theta, alpha, weighted, group, xch):
        x_own = x_own.contiguous()
        y_own, deg, norm = _halo_forward(part, _fill_halo(part, x_own, 'in', group, xch), theta, alpha, weighted)
        ctx.part, ctx.alpha, ctx.weighted, ctx.group, ctx.xch = part, alpha, weighted, group, xch
        ctx.save_for_backward(x_own, y_own, theta, deg, norm)
        return y_own

    @staticmethod
    def backward(ctx, g_own):
        x_own, y_own, theta, deg, norm = ctx.saved_tensors
        g_ext = _fill_halo(ctx.part, g_own.contiguous(), 'out', ctx.group, ctx.xch)
        dx_own, d_theta = _halo_backward(ctx.part, x_own, y_own, g_ext, theta, ctx.alpha, ctx.weighted, deg, norm)
        return None, dx_own, d_theta, None, None, None, None


def halo_propagate(part, x_own, theta, alpha, weighted=True, group=None, exchange=None):
    """Row block in, row block out (``part``: this rank's ``HaloPartition``): the REGCN aggregation
    Y = n (.) A_w (n (.) X) with n = max(sum_in w, 1)^-1/2 from ``theta`` (``weighted=False``: REMixHop's
    Y = n (.) A (n (.) X)).  Only halo rows are exchanged: ``exchange`` (a ``HaloExchange``) pushes them over peer
    memory with regnn_halo_push; None: one uneven all-to-all (NCCL / gloo).  Y and dX are bit-identical to
    ``functional.propagate``; ``theta.grad`` holds this rank's share (``allreduce_relation_grads``)."""
    return _HaloPropagate.apply(part, x_own, theta, alpha, weighted, group, exchange)


def _check_gat_shape(heads, dim, num_relations, relational, name='halo_gat'):
    """The head widths the fused attention kernels take (check_shape of csrc/gat.cu), refused before any work."""
    if not (1 <= heads <= 32 and 4 <= dim <= 128 and dim & (dim - 1) == 0 and heads * dim <= 1024):
        raise ValueError('%s: the fused attention kernels take 1 <= H <= 32 heads of a power-of-two width D in '
                         '[4, 128] with H * D <= 1024, not H=%d D=%d' % (name, heads, dim))
    if relational and not (1 <= num_relations <= 200 and num_relations * heads <= 4096):
        raise ValueError('%s: the fused attention kernels take 1..200 relations with R * H <= 4096, not R=%d H=%d'
                         % (name, num_relations, heads))


def _check_slot_offsets(part, heads, chunks):
    """The REGATv2 kernels address the per-slot buffers with 32-bit offsets (slot * H, slot * C)."""
    if part.max_dpre_rows * max(heads, chunks) >= 2 ** 32:
        raise ValueError('halo_gatv2: %d extended slots * max(H, ceil(H*D/128)) exceeds the 32-bit slot offsets of the '
                         'REGATv2 kernels' % part.max_dpre_rows)


def _fill_out_halo_gat(part, g_own, stats_own, group, xch, slots=None):
    """dL/dY [n_own + out-halo, H*D] and the softmax statistics [n_own + out-halo, 4H] of the backward: the same rows,
    pushed by their owners (one barrier for both over peer memory, two uneven all-to-alls otherwise).  ``slots``
    (REGATv2: the extended logit and mask buffers): their tails are filled in the same exchange
    (``_push_slot_records``), behind the same barrier."""
    if xch is None:
        g_ext, s_ext = _fill_halo(part, g_own, 'out', group, None), _fill_halo(part, stats_own, 'out', group, None)
        if slots is not None:
            _push_slot_records(part, slots, group, None)
        return g_ext, s_ext
    rows, ptr, offsets = part.push_out
    if ptr[-1]:
        ops.halo_push(g_own, rows, ptr, offsets, xch.g_ptrs, xch.g_ext.stride(0), part.rank)
        ops.halo_push(stats_own, rows, ptr, offsets, xch.s_ptrs, xch.s_ext.stride(0), part.rank)
    if slots is not None:
        _push_slot_records(part, slots, group, xch)
    xch.barrier()
    n = part.n_own + part.n_out
    return xch.g_ext[:n], xch.s_ext[:n]


def _return_dpre(part, dpre, group, xch):
    """Sends the tail of the extended dpre buffer (logit gradients of this rank's out-edges into remote rows) to the
    owners of those rows; afterwards ``dpre[:e_in]`` holds every in-view slot of this rank."""
    e_in = part.e_in
    if xch is not None:
        if part.tail_ptr[-1]:
            ops.halo_scatter(dpre[e_in:], part.tail_ptr, part.tail_dst, xch.dpre_ptrs, xch.dpre.stride(0), part.rank)
        xch.barrier()            # every peer's gradients of my in-view slots have landed
        return
    if part.parts > 1:
        recv = dpre.new_empty((sum(part.dpre_recv_counts), dpre.shape[1]))
        with _lib.phase('halo_all_to_all'):
            dist.all_to_all_single(recv, dpre[e_in:], output_split_sizes=part.dpre_recv_counts,
                                   input_split_sizes=part.tail_counts, group=group)
        dpre.index_copy_(0, part.dpre_recv, recv)


def _dropout_in(part, dropout):
    """Keywords of the forward kernel call over the in-view: the hashed dropout and the global edge ids of its slots."""
    return {} if dropout is None else {'dropout': dropout, 'eid': part.eid_in}


def _dropout_ext(part, dropout):
    """Keywords of the source-major edge pass: the hashed dropout and the global edge ids of the extended slots."""
    return {} if dropout is None else {'dropout': dropout, 'eid': part.eid_ext}


def _gat_forward(part, f_ext, attn_l, attn_r, theta, alpha, slope, dropout=None):
    """-> (out, el, er, rowmax, rowsum) of the own rows from the filled [n_own + in-halo, H, D] feature buffer: el / er
    of own AND halo rows computed here (row-wise, so a halo row carries its owner's bits and el is never exchanged),
    then the fused kernel over the in-view."""
    n_own, heads, dim = part.n_own, f_ext.shape[1], f_ext.shape[2]
    if not n_own:                # an empty row block has no edges and no halo
        z = f_ext.new_zeros((0, heads))
        return f_ext.new_zeros((0, heads, dim)), z, z, z, z
    el, er = ops.attn_scores_fwd(f_ext, attn_l, attn_r)
    out, rowmax, rowsum, _ = ops.gat_fwd(part.csr, part.et_in if theta is not None else None, theta, alpha, f_ext, el,
                                         er, slope, **_dropout_in(part, dropout))
    return out, el[:n_own], er[:n_own], rowmax, rowsum


def _gat_stats(out, g_own, er, rowmax, rowsum):
    """[n_own, 4H] softmax statistics of the own rows (the rows peers' edge passes read through their out-halo)."""
    n_own, heads, _ = out.shape
    if not n_own:
        return out.new_zeros((0, 4 * heads))
    return ops.gat_bwd_stats(out, g_own, er, rowmax, rowsum).view(n_own, 4 * heads)


def _gat_backward_edges(part, f_own, el, attn_l, theta, alpha, slope, g_ext, s_ext, dpre, dropout=None):
    """-> (d_feat without the destination-side score term, d_el) of the own rows; writes the logit gradient of every
    out-view entry into the extended ``dpre`` buffer [e_in + tail, H] through ``csr['slot_t']``."""
    n_own, heads, dim = f_own.shape
    if not n_own:
        return torch.zeros_like(f_own), f_own.new_zeros((0, heads))
    return ops.gat_bwd_edges(part.csr, part.et_out if theta is not None else None, theta, alpha, f_own, el,
                             s_ext.view(-1, heads, 4), slope, g_ext.view(-1, heads, dim), dpre, attn_l=attn_l,
                             **_dropout_ext(part, dropout))


def _gat_backward_reduce(part, f_own, d_feat, d_el, attn_r, theta, alpha, dpre):
    """-> (d_feat, this rank's d_attn_l, d_attn_r [H*D] and d_theta | None) once ``dpre[:e_in]`` holds every in-view
    slot: d_er and the relation bins over the in-view, then the projection-score gradients of the own rows (which add
    d_er * attn_r to d_feat in place)."""
    n_own, heads, dim = f_own.shape
    if not n_own:
        z = f_own.new_zeros(heads * dim)
        return d_feat, z, z.clone(), (f_own.new_zeros(theta.shape) if theta is not None else None)
    d_er, d_theta = ops.gat_bwd_reduce(part.csr, part.et_in if theta is not None else None, theta, alpha,
                                       dpre[:part.e_in])
    d_al, d_ar = ops.attn_scores_bwd(f_own, d_el, d_er, attn_r=attn_r, d_feat=d_feat)
    return d_feat, d_al, d_ar, d_theta


class _HaloGat(torch.autograd.Function):
    """REGAT core (projection scores + fused logits / edge softmax / aggregation) on destination-row blocks with a halo
    exchange.  Forward: the in-halo of the features, then ``_gat_forward``.  Backward: the statistics of own rows; the
    out-halo of dL/dY and of the statistics; the source-major edge pass over the out-view, which writes the logit
    gradient of every out-edge into the extended dpre buffer; the tail of that buffer goes back to the destinations'
    owners (the third exchange); then d_er and the relation bins over the in-view and the projection-score gradients of
    own rows."""

    @staticmethod
    def forward(ctx, part, f_own, attn_l, attn_r, theta, alpha, slope, group, xch, dropout):
        n_own, heads, dim = f_own.shape
        f_own = f_own.contiguous()
        f_ext = _fill_halo(part, f_own.view(n_own, heads * dim), 'in', group, xch).view(-1, heads, dim)
        out, el, er, rowmax, rowsum = _gat_forward(part, f_ext, attn_l, attn_r, theta, alpha, slope, dropout)
        ctx.part, ctx.alpha, ctx.slope, ctx.group, ctx.xch, ctx.dropout = part, alpha, slope, group, xch, dropout
        ctx.save_for_backward(f_own, el, er, attn_l, attn_r, theta, out, rowmax, rowsum)
        return out

    @staticmethod
    def backward(ctx, g_own):
        f_own, el, er, attn_l, attn_r, theta, out, rowmax, rowsum = ctx.saved_tensors
        part, xch = ctx.part, ctx.xch
        n_own, heads, dim = f_own.shape
        g_own = g_own.reshape(n_own, heads, dim).contiguous()
        stats = _gat_stats(out, g_own, er, rowmax, rowsum)
        g_ext, s_ext = _fill_out_halo_gat(part, g_own.view(n_own, heads * dim), stats, ctx.group, xch)
        rows = part.e_in + part.tail_ptr[-1]
        dpre = xch.dpre[:rows] if xch is not None else f_own.new_empty((rows, heads))
        d_feat, d_el = _gat_backward_edges(part, f_own, el, attn_l, theta, ctx.alpha, ctx.slope, g_ext, s_ext, dpre,
                                           ctx.dropout)
        _return_dpre(part, dpre, ctx.group, xch)
        d_feat, d_al, d_ar, d_th = _gat_backward_reduce(part, f_own, d_feat, d_el, attn_r, theta, ctx.alpha, dpre)
        return (None, d_feat, d_al.view_as(attn_l), d_ar.view_as(attn_r),
                d_th.view_as(theta) if d_th is not None else None, None, None, None, None, None)


def _check_hashed_dropout(dropout, name):
    from .dropout import HashedDropout
    if dropout is not None and not isinstance(dropout, HashedDropout):
        raise TypeError('%s: dropout must be a functional.HashedDropout, got %s' % (name, type(dropout).__name__))


def halo_gat(part, f_own, attn_l, attn_r, theta, alpha, slope, group=None, exchange=None, keep=None, dropout=None):
    """f_own [n_own, H, D] -> out [n_own, H, D] (``part``: this rank's ``HaloPartition`` built with ``attention=True``):
    the REGAT core of ``functional.gat_layer`` on destination-row blocks, exchanging only halo rows.  ``exchange`` (a
    ``HaloExchange`` with ``heads=H`` and width H*D): the features, dL/dY and the statistics are pushed over peer memory
    (regnn_halo_push) and the logit gradients of cut edges are scattered to their owners (regnn_halo_scatter); None:
    uneven all-to-alls (NCCL / gloo).  ``theta=None`` drops the relation term.  out and d_feat are bit-identical to
    ``functional.gat_layer``; ``attn_l.grad``, ``attn_r.grad`` and ``theta.grad`` hold this rank's shares
    (``allreduce_relation_grads``).  Attention dropout: ``dropout`` (a ``functional.HashedDropout``), whose mask every
    rank computes from the global edge ids (``part.eid_in`` / ``part.eid_ext``) -- the result is that of
    ``functional.gat_layer`` with the same ``dropout``; an explicit ``keep`` mask is refused."""
    _, heads, dim = f_own.shape
    if keep is not None:
        raise ValueError('halo_gat: an explicit attention dropout mask is not supported (it is in edge-id order over all '
                         'edges); pass dropout=functional.HashedDropout(p, key)')
    _check_hashed_dropout(dropout, 'halo_gat')
    if not getattr(part, 'attention', False):
        raise ValueError('halo_gat needs a HaloPartition built with attention=True')
    _check_gat_shape(heads, dim, part.num_relations, theta is not None)
    if theta is not None and tuple(theta.shape) != (part.num_relations, heads):
        raise ValueError('halo_gat: theta must be [R=%d, H=%d], got %s' % (part.num_relations, heads, tuple(theta.shape)))
    if exchange is not None and (exchange.heads != heads or exchange.feat != heads * dim):
        raise ValueError('halo_gat: the HaloExchange must be built with heads=%d and width %d' % (heads, heads * dim))
    return _HaloGat.apply(part, f_own, attn_l, attn_r, theta, alpha, slope, group, exchange, dropout)


def _virtual_halo_gat(parts, f, gout, attn_l, attn_r, theta, alpha, slope, scatter=False, dropout=None):
    """Every rank of ``HaloPartition.virtual_ranks(..., attention=True)`` one after another in one process (no process
    group), each on its local views: halos filled by indexing the global [N, H, D] arrays, the dpre tails returned with
    ``index_copy_`` at the owners' receive lists or -- ``scatter=True`` -- by regnn_halo_scatter into the P local buffers.
    -> (out, d_feat, d_attn_l, d_attn_r, d_theta | None): rows in global order, parameter gradients summed in rank
    order."""
    n, heads, dim = f.shape
    g2 = gout.reshape(n, heads * dim)
    bounds = parts[0].bounds
    own = [slice(bounds[p], bounds[p + 1]) for p in range(len(parts))]
    fw = [_gat_forward(part, f[part.rows_in], attn_l, attn_r, theta, alpha, slope, dropout) for part in parts]
    stats = torch.cat([_gat_stats(o, gout[s].contiguous(), er, mx, sm) for (o, _, er, mx, sm), s in zip(fw, own)])
    dpres = [f.new_empty((part.e_in + part.tail_ptr[-1], heads)) for part in parts]
    edges = [_gat_backward_edges(part, f[s].contiguous(), fw[p][1], attn_l, theta, alpha, slope, g2[part.rows_out],
                                 stats[part.rows_out], dpres[p], dropout) for p, (part, s) in enumerate(zip(parts, own))]
    if scatter:
        ptrs = torch.tensor([d.data_ptr() for d in dpres], dtype=torch.int64, device=f.device)
        for p, part in enumerate(parts):
            if part.tail_ptr[-1]:
                ops.halo_scatter(dpres[p][part.e_in:], part.tail_ptr, part.tail_dst, ptrs, heads, p)
    else:
        for q, owner in enumerate(parts):
            segs = [dpres[p][part.e_in + part.tail_ptr[q]:part.e_in + part.tail_ptr[q + 1]] for p, part in enumerate(parts)]
            dpres[q].index_copy_(0, owner.dpre_recv, torch.cat(segs))
    outs, d_feats, d_al, d_ar, d_th = [], [], 0, 0, 0
    for p, part in enumerate(parts):
        df, al, ar, th = _gat_backward_reduce(part, f[own[p]].contiguous(), edges[p][0], edges[p][1], attn_r, theta,
                                              alpha, dpres[p])
        outs.append(fw[p][0])
        d_feats.append(df)
        d_al, d_ar = d_al + al, d_ar + ar
        d_th = d_th + th if th is not None else None
    return torch.cat(outs), torch.cat(d_feats), d_al, d_ar, d_th


# ---- REGATv2 on destination-row blocks with a halo exchange --------------------------------------------------------
def _slot_buffers(part, heads, chunks, like, xch):
    """The extended per-slot buffers of the stored logits [e_in + tail, H] and sign masks [e_in + tail, C, 4] (int32):
    the own in-view slots in the head, the cut out-edges of own sources in the tail (``csr['slot_t']`` order).  Views
    of the exchange's symmetric buffers over peer memory, local buffers otherwise."""
    rows = part.e_in + part.tail_ptr[-1]
    if xch is not None:
        return xch.logit_ext[:rows], xch.mask_ext[:rows]
    return (like.new_empty((max(rows, 1), heads))[:rows],        # max(rows, 1): never a NULL pointer
            torch.empty((max(rows, 1), chunks, 4), dtype=torch.int32, device=like.device)[:rows])


def _push_slot_records(part, slots, group, xch):
    """Sends the stored logit and sign mask of every own in-view slot whose source a peer owns to that peer, into its
    tail (the transpose of ``_return_dpre``); afterwards the tails of ``slots`` hold every cut out-edge of this rank's
    sources.  Over peer memory this is the push only: the caller's barrier completes it."""
    logit, mask = slots
    if xch is not None:
        send, ptr, offsets = part.push_slots
        if ptr[-1]:
            ops.halo_push_slots(logit, mask, send, ptr, offsets, xch.logit_ptrs, xch.mask_ptrs, part.rank)
        return
    if part.parts > 1:
        e_in = part.e_in
        with _lib.phase('halo_all_to_all'):
            for buf in (logit, mask.flatten(1)):
                dist.all_to_all_single(buf[e_in:], buf.index_select(0, part.dpre_recv),
                                       output_split_sizes=part.tail_counts, input_split_sizes=part.dpre_recv_counts,
                                       group=group)


def _gatv2_forward(part, fs_ext, fd_own, attn, theta, alpha, slope, slots, dropout=None):
    """-> (out, rowmax, rowsum) of the own rows from the filled [n_own + in-halo, H, D] source features and the own
    rows' destination features; the logit and the sign mask of every in-view slot go to the head of ``slots``."""
    n_own, heads, dim = fd_own.shape
    if not n_own:                # an empty row block has no edges and no halo
        z = fd_own.new_zeros((0, heads))
        return fd_own.new_zeros((0, heads, dim)), z, z
    out, rowmax, rowsum, _, _ = ops.gatv2_fwd(part.csr, part.et_in if theta is not None else None, theta, alpha, fs_ext,
                                              fd_own, attn, slope, saved=slots, **_dropout_in(part, dropout))
    return out, rowmax, rowsum


def _gatv2_backward_edges(part, fs_own, attn, slope, g_ext, s_ext, slots, dl, dropout=None):
    """-> (d_fs, this rank's d_attn_src [H*D]) of the own rows once the tails of ``slots`` are filled; writes the dl of
    every out-view entry into the extended ``dl`` buffer [e_in + tail, H] through ``csr['slot_t']``."""
    n_own, heads, dim = fs_own.shape
    if not n_own:
        return torch.zeros_like(fs_own), fs_own.new_zeros(heads * dim)
    return ops.gatv2_bwd_edges(part.csr, fs_own, s_ext.view(-1, heads, 4), slots[0], slots[1], attn, slope,
                               g_ext.view(-1, heads, dim), dl, **_dropout_ext(part, dropout))


def _gatv2_backward_dst(part, fd_own, attn, theta, alpha, slope, dl, mask):
    """-> (d_fd, this rank's d_attn_dst [H*D], d_theta | None) once ``dl[:e_in]`` holds every in-view slot: the
    streaming destination pass over the in-view."""
    n_own, heads, dim = fd_own.shape
    if not n_own:
        return (torch.zeros_like(fd_own), fd_own.new_zeros(heads * dim),
                fd_own.new_zeros(theta.shape) if theta is not None else None)
    return ops.gatv2_bwd_dst(part.csr, part.et_in if theta is not None else None, theta, alpha, fd_own,
                             dl[:part.e_in], mask[:part.e_in], attn, slope)


class _HaloGatV2(torch.autograd.Function):
    """REGATv2 core (fused logits / edge softmax / aggregation of ``functional.gatv2_aggregate``) on destination-row
    blocks with a halo exchange.  Forward: the in-halo of the source features (the destination features are read for
    own rows only), then the fused kernel over the in-view, which stores the logit and the sign mask of every in-view
    slot in the head of the extended per-slot buffers.  Backward: the statistics of own rows; one exchange of the
    dL/dY and statistics out-halo and of the slot records of cut edges (to the source's owner, into the buffers'
    tails); the source-major edge pass over the out-view, which writes the dl of every out-edge into the extended dl
    buffer; the tail of that buffer goes back to the destinations' owners; then the destination pass over the in-view.

    Over peer memory the exchange's buffers are reused by every call: a forward must be followed by its backward
    before the next forward, as for every ``HaloExchange``."""

    @staticmethod
    def forward(ctx, part, fs_own, fd_own, attn, theta, alpha, slope, group, xch, dropout):
        n_own, heads, dim = fs_own.shape
        fs_own, fd_own = fs_own.contiguous(), fd_own.contiguous()
        fs_ext = _fill_halo(part, fs_own.view(n_own, heads * dim), 'in', group, xch).view(-1, heads, dim)
        slots = _slot_buffers(part, heads, (heads * dim + 127) // 128, fs_own, xch)
        out, rowmax, rowsum = _gatv2_forward(part, fs_ext, fd_own, attn, theta, alpha, slope, slots, dropout)
        ctx.part, ctx.alpha, ctx.slope, ctx.group, ctx.xch, ctx.slots = part, alpha, slope, group, xch, slots
        ctx.dropout = dropout
        ctx.save_for_backward(fs_own, fd_own, attn, theta, out, rowmax, rowsum)
        return out

    @staticmethod
    def backward(ctx, g_own):
        fs_own, fd_own, attn, theta, out, rowmax, rowsum = ctx.saved_tensors
        part, xch, slots = ctx.part, ctx.xch, ctx.slots
        n_own, heads, dim = fs_own.shape
        g_own = g_own.reshape(n_own, heads, dim).contiguous()
        stats = _gat_stats(out, g_own, None, rowmax, rowsum)
        g_ext, s_ext = _fill_out_halo_gat(part, g_own.view(n_own, heads * dim), stats, ctx.group, xch, slots=slots)
        rows = part.e_in + part.tail_ptr[-1]
        dl = xch.dpre[:rows] if xch is not None else fs_own.new_empty((max(rows, 1), heads))[:rows]
        d_fs, d_attn_src = _gatv2_backward_edges(part, fs_own, attn, ctx.slope, g_ext, s_ext, slots, dl, ctx.dropout)
        _return_dpre(part, dl, ctx.group, xch)
        d_fd, d_attn_dst, d_th = _gatv2_backward_dst(part, fd_own, attn, theta, ctx.alpha, ctx.slope, dl, slots[1])
        return (None, d_fs, d_fd, (d_attn_src + d_attn_dst).view_as(attn),
                d_th.view_as(theta) if d_th is not None else None, None, None, None, None, None)


def halo_gatv2(part, fs_own, fd_own, attn, theta, alpha, slope, group=None, exchange=None, keep=None, dropout=None):
    """fs_own, fd_own [n_own, H, D] -> out [n_own, H, D] (``part``: this rank's ``HaloPartition`` built with
    ``attention=True``): the REGATv2 core of ``functional.gatv2_aggregate`` on destination-row blocks, exchanging only
    halo rows and the per-slot records of cut edges.  With shared weights pass the same tensor as ``fs_own`` and
    ``fd_own``.  ``exchange`` (a ``HaloExchange`` with ``heads=H``, width H*D and ``gatv2=True``): the source features,
    dL/dY and the statistics are pushed over peer memory (regnn_halo_push), the stored logits and sign masks of cut
    edges go to the sources' owners (regnn_halo_push_slots) and their dl back to the destinations' owners
    (regnn_halo_scatter); None: uneven all-to-alls (NCCL / gloo).  ``theta=None`` drops the relation term.  out, d_fs
    and d_fd are bit-identical to ``functional.gatv2_aggregate``; ``attn.grad`` and ``theta.grad`` hold this rank's
    shares (``allreduce_relation_grads``).  The MAG stack's ``softmax_eps`` (a global maximum over all logits) is not
    taken.  Attention dropout: ``dropout`` (a ``functional.HashedDropout``), as ``halo_gat``; an explicit ``keep`` mask
    is refused."""
    _, heads, dim = fs_own.shape
    if keep is not None:
        raise ValueError('halo_gatv2: an explicit attention dropout mask is not supported (it is in edge-id order over '
                         'all edges); pass dropout=functional.HashedDropout(p, key)')
    _check_hashed_dropout(dropout, 'halo_gatv2')
    if not getattr(part, 'attention', False):
        raise ValueError('halo_gatv2 needs a HaloPartition built with attention=True')
    _check_gat_shape(heads, dim, part.num_relations, theta is not None, 'halo_gatv2')
    if tuple(fd_own.shape) != tuple(fs_own.shape):
        raise ValueError('halo_gatv2: fs_own and fd_own must both be [n_own, H, D], got %s and %s'
                         % (tuple(fs_own.shape), tuple(fd_own.shape)))
    if theta is not None and tuple(theta.shape) != (part.num_relations, heads):
        raise ValueError('halo_gatv2: theta must be [R=%d, H=%d], got %s' % (part.num_relations, heads, tuple(theta.shape)))
    _check_slot_offsets(part, heads, (heads * dim + 127) // 128)
    if exchange is not None and (exchange.heads != heads or exchange.feat != heads * dim or not exchange.gatv2):
        raise ValueError('halo_gatv2: the HaloExchange must be built with heads=%d, width %d and gatv2=True'
                         % (heads, heads * dim))
    return _HaloGatV2.apply(part, fs_own, fd_own, attn, theta, alpha, slope, group, exchange, dropout)


def _virtual_halo_gatv2(parts, fs, fd, gout, attn, theta, alpha, slope, push=False, dropout=None):
    """Every rank of ``HaloPartition.virtual_ranks(..., attention=True)`` one after another in one process (no process
    group), each on its local views: halos filled by indexing the global [N, H, D] arrays; the slot records of cut
    edges moved to the sources' owners by indexing and the dl tails returned with ``index_copy_`` at the owners'
    receive lists, or -- ``push=True`` -- by regnn_halo_push_slots and regnn_halo_scatter into the P local buffers.
    -> (out, d_fs, d_fd, d_attn, d_theta | None): rows in global order, parameter gradients summed in rank order."""
    n, heads, dim = fs.shape
    g2 = gout.reshape(n, heads * dim)
    bounds = parts[0].bounds
    own = [slice(bounds[p], bounds[p + 1]) for p in range(len(parts))]
    slots = [_slot_buffers(part, heads, (heads * dim + 127) // 128, fs, None) for part in parts]
    fw = [_gatv2_forward(part, fs[part.rows_in], fd[s].contiguous(), attn, theta, alpha, slope, sl, dropout)
          for part, s, sl in zip(parts, own, slots)]
    stats = torch.cat([_gat_stats(o, gout[s].contiguous(), None, mx, sm) for (o, mx, sm), s in zip(fw, own)])
    if push:
        ptrs = [torch.tensor([sl[i].data_ptr() for sl in slots], dtype=torch.int64, device=fs.device) for i in (0, 1)]
        for p, part in enumerate(parts):
            send, ptr, offsets = part.push_slots
            if ptr[-1]:
                ops.halo_push_slots(slots[p][0], slots[p][1], send, ptr, offsets, ptrs[0], ptrs[1], p)
    else:
        for q, owner in enumerate(parts):      # q's tail segment of rank p: p's slots at its receive list from q
            for p, part in enumerate(parts):
                seg = slice(owner.e_in + owner.tail_ptr[p], owner.e_in + owner.tail_ptr[p + 1])
                idx = part.dpre_recv[part.push_slots[1][q]:part.push_slots[1][q + 1]]
                for dst, src in zip(slots[q], slots[p]):
                    dst[seg] = src.index_select(0, idx)
    dls = [fs.new_empty((max(part.e_in + part.tail_ptr[-1], 1), heads))[:part.e_in + part.tail_ptr[-1]] for part in parts]
    edges = [_gatv2_backward_edges(part, fs[s].contiguous(), attn, slope, g2[part.rows_out], stats[part.rows_out],
                                   slots[p], dls[p], dropout) for p, (part, s) in enumerate(zip(parts, own))]
    if push:
        ptrs = torch.tensor([d.data_ptr() for d in dls], dtype=torch.int64, device=fs.device)
        for p, part in enumerate(parts):
            if part.tail_ptr[-1]:
                ops.halo_scatter(dls[p][part.e_in:], part.tail_ptr, part.tail_dst, ptrs, heads, p)
    else:
        for q, owner in enumerate(parts):
            segs = [dls[p][part.e_in + part.tail_ptr[q]:part.e_in + part.tail_ptr[q + 1]] for p, part in enumerate(parts)]
            dls[q].index_copy_(0, owner.dpre_recv, torch.cat(segs))
    outs, d_fss, d_fds, d_attn, d_th = [], [], [], 0, 0
    for p, part in enumerate(parts):
        d_fd, d_at_dst, th = _gatv2_backward_dst(part, fd[own[p]].contiguous(), attn, theta, alpha, slope, dls[p],
                                                 slots[p][1])
        outs.append(fw[p][0])
        d_fss.append(edges[p][0])
        d_fds.append(d_fd)
        d_attn = d_attn + (edges[p][1] + d_at_dst)
        d_th = d_th + th if th is not None else None
    return torch.cat(outs), torch.cat(d_fss), torch.cat(d_fds), d_attn, d_th
