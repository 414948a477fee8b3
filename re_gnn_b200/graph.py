"""``Graph``: the stand-in for the DGLGraph argument of the reference layers.

The reference builds ``g = dgl.DGLGraph(adjM); g = dgl.remove_self_loop(g); g = dgl.add_self_loop(g);
g = g.to(device)`` (run_regnn.py:84-87) and aligns ``e_feat`` to ``g.edges()`` order (:94-99).
This class keeps exactly that contract -- edge k is ``src[k] -> dst[k]``, self loops appended last --
and owns the device-resident structures the CUDA kernels read (built once by ``regnn_csr_build``):

  indptr/indices/eid/row          destination-sorted CSR (slots of a row in edge-id order)
  indptr_t/indices_t/slot_t       source-sorted view for the backward passes
  etype views                     uint8 0-based edge types per CSR slot / per transposed entry,
                                  cached per ``e_feat`` tensor

Methods mirror what layer/*.py and run_regnn.py touch on a DGLGraph: ``local_var``, ``local_scope``,
``num_nodes``/``number_of_nodes``, ``number_of_edges``, ``edges``, ``in_degrees``, ``is_block``, ``to``.
"""
import contextlib
import ctypes

import numpy as np
import torch

from . import _lib


class ZeroInDegreeError(RuntimeError):
    """Raised where the reference raises ``dgl.base.DGLError`` (layer/REGATv2Conv.py:105-115)."""


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


SPLIT_THRESHOLD = 256   # rows with more slots are cut into fragments of this many slots
COUNTS_MAX_BYTES = 4 << 30   # build the [N,R] relation-count table only while it stays below this size


def _row_split(indptr, threshold, sizes=None):
    """Long-row decomposition of one CSR view (``regnn_rowsplit_t``): index bookkeeping with torch ops on the
    device, once per graph.  Returns None when no row exceeds the threshold.  ``sizes``: (long rows, fragments)
    when the caller already knows them, which keeps the host from waiting for the device."""
    deg = (indptr[1:] - indptr[:-1]).to(torch.int64)
    if sizes is not None:
        if sizes[0] == 0:
            return None
        long_rows = torch.nonzero_static(deg > threshold, size=int(sizes[0])).view(-1)
    else:
        long_rows = torch.nonzero(deg > threshold).view(-1)
        if long_rows.numel() == 0:
            return None
    nfr = (deg[long_rows] + threshold - 1) // threshold
    frag_ptr = torch.zeros(long_rows.numel() + 1, dtype=torch.int64, device=indptr.device)
    frag_ptr[1:] = torch.cumsum(nfr, 0)
    total = int(frag_ptr[-1].item()) if sizes is None else int(sizes[1])
    frag_row = torch.repeat_interleave(long_rows, nfr, output_size=total)
    within = torch.arange(total, device=indptr.device) - torch.repeat_interleave(frag_ptr[:-1], nfr, output_size=total)
    frag_begin = indptr.to(torch.int64)[frag_row] + within * threshold
    t = dict(long_rows=long_rows.to(torch.int32), frag_ptr=frag_ptr.to(torch.int32),
             frag_row=frag_row.to(torch.int32), frag_begin=frag_begin.to(torch.int32))
    t['struct'] = _lib.RowSplit(t['long_rows'].data_ptr(), t['frag_ptr'].data_ptr(), t['frag_row'].data_ptr(),
                                t['frag_begin'].data_ptr(), long_rows.numel(), total, threshold)
    return t


class Graph:
    is_block = False

    def __init__(self, src, dst=None, num_nodes=None):
        """``Graph(src, dst, num_nodes)`` from edge arrays, or ``Graph(scipy_sparse)`` where a stored
        entry ``A[i, j]`` is the edge ``i -> j`` in COO order (the ``dgl.DGLGraph(adjM)`` convention)."""
        if dst is None and hasattr(src, 'tocoo'):
            coo = src.tocoo()
            num_nodes = int(coo.shape[0])
            src, dst = coo.row, coo.col
        self._src = torch.as_tensor(np.asarray(src) if not torch.is_tensor(src) else src).to(torch.int64).contiguous()
        self._dst = torch.as_tensor(np.asarray(dst) if not torch.is_tensor(dst) else dst).to(torch.int64).contiguous()
        if self._src.shape != self._dst.shape or self._src.dim() != 1:
            raise ValueError('src and dst must be 1-D arrays of equal length')
        if num_nodes is None:
            num_nodes = int(max(self._src.max().item(), self._dst.max().item())) + 1 if self._src.numel() else 0
        self._n = int(num_nodes)
        self._csr = None
        self._etype_cache = {}
        self._zero_in_degree = None

    @classmethod
    def from_csr(cls, src, dst, num_nodes, csr, etype_views=None, has_zero_in_degree=None):
        """A graph whose device structures are already built (``NeighborSampler`` blocks): ``src`` / ``dst`` in
        edge-id order, ``csr`` the dict ``csr()`` returns (``split`` / ``split_t`` included), ``etype_views`` an
        optional ``(e_feat, num_relations, et_csr, et_t, counts)`` entry of the ``etype_views`` cache and
        ``has_zero_in_degree`` the answer when it is known on the host."""
        g = cls(src, dst, num_nodes)
        g._csr = csr
        g._zero_in_degree = has_zero_in_degree
        if etype_views is not None:
            e_feat, num_relations, et_csr, et_t, counts = etype_views
            g._etype_cache[g._etype_key(e_feat, num_relations)] = (et_csr, et_t, counts, e_feat)
        return g

    # ---- DGLGraph surface ---------------------------------------------------------------------
    @classmethod
    def from_scipy(cls, adj):
        return cls(adj)

    def to(self, device):
        device = torch.device(device)
        if device == self._src.device:
            return self
        g = Graph(self._src.to(device), self._dst.to(device), self._n)
        return g

    @property
    def device(self):
        return self._src.device

    def number_of_nodes(self):
        return self._n

    num_nodes = number_of_nodes
    number_of_dst_nodes = number_of_nodes
    number_of_src_nodes = number_of_nodes

    def number_of_edges(self):
        return int(self._src.numel())

    num_edges = number_of_edges

    def edges(self):
        return self._src, self._dst

    def in_degrees(self):
        if self._src.is_cuda:
            ip = self.csr()['indptr']
            return (ip[1:] - ip[:-1]).to(torch.int64)
        return torch.bincount(self._dst, minlength=self._n)

    def has_zero_in_degree(self):
        if self._zero_in_degree is None:
            self._zero_in_degree = bool((self.in_degrees() == 0).any().item()) if self._n else False
        return self._zero_in_degree

    def local_var(self):
        return self  # frames are never mutated by our layers

    @contextlib.contextmanager
    def local_scope(self):
        yield

    def remove_self_loop(self):
        keep = self._src != self._dst
        return Graph(self._src[keep], self._dst[keep], self._n)

    def add_self_loop(self):
        loop = torch.arange(self._n, dtype=torch.int64, device=self._src.device)
        return Graph(torch.cat([self._src, loop]), torch.cat([self._dst, loop]), self._n)

    # ---- device structures --------------------------------------------------------------------
    def csr(self):
        """Builds (once) and returns the dict of int32 device arrays produced by regnn_csr_build."""
        if self._csr is not None:
            return self._csr
        if not self._src.is_cuda:
            raise RuntimeError('Graph is on %s: move it to a CUDA device with .to(device) before use; '
                               're_gnn_b200 has no CPU path' % self._src.device)
        dev = self._src.device
        n, e = self._n, self.number_of_edges()
        with torch.cuda.device(dev):
            i32 = dict(dtype=torch.int32, device=dev)
            out = {k: torch.empty(n + 1, **i32) for k in ('indptr', 'indptr_t')}
            out.update({k: torch.empty(max(e, 1), **i32)[:e] for k in ('indices', 'eid', 'row', 'indices_t', 'slot_t')})
            lib = _lib.load()
            ws_bytes = lib.regnn_csr_build_workspace_bytes(n, e)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _lib.call('regnn_csr_build', _ptr(self._src), _ptr(self._dst), n, e, _ptr(out['indptr']),
                      _ptr(out['indices']), _ptr(out['eid']), _ptr(out['row']), _ptr(out['indptr_t']),
                      _ptr(out['indices_t']), _ptr(out['slot_t']), _ptr(ws), ws_bytes, _stream())
            out['split'] = _row_split(out['indptr'], SPLIT_THRESHOLD)
            out['split_t'] = _row_split(out['indptr_t'], SPLIT_THRESHOLD)
        self._csr = out
        return out

    @staticmethod
    def _etype_key(e_feat, num_relations):
        return (e_feat.data_ptr(), e_feat._version, int(e_feat.numel()), int(num_relations))

    def etype_views(self, e_feat, num_relations):
        """uint8 0-based edge types in CSR-slot order and transposed-entry order for the reference's
        1-based int64 ``e_feat`` (edge-id order).  Cached per tensor (data_ptr, version); a cached entry holds a
        reference to the tensor, so the key cannot be recycled by the allocator while the entry lives."""
        key = self._etype_key(e_feat, num_relations)
        hit = self._etype_cache.get(key)
        if hit is not None:
            return hit[:3]
        csr = self.csr()
        e = self.number_of_edges()
        if e_feat.numel() != e:
            raise ValueError('e_feat has %d entries but the graph has %d edges' % (e_feat.numel(), e))
        dev = self._src.device
        et = e_feat.to(device=dev, dtype=torch.int64).contiguous().view(-1)
        with torch.cuda.device(dev):
            et_csr = torch.empty(max(e, 1), dtype=torch.uint8, device=dev)[:e]
            et_t = torch.empty(max(e, 1), dtype=torch.uint8, device=dev)[:e]
            scratch = torch.zeros(1, dtype=torch.int32, device=dev)
            _lib.call('regnn_etype_permute', _ptr(et), _ptr(csr['eid']), _ptr(csr['slot_t']), e,
                      int(num_relations), _ptr(et_csr), _ptr(et_t), _ptr(scratch), _stream())
            # per-(row, relation) in-edge counts: turns the degree norm into a dense [N,R] pass (when it fits)
            counts = None
            if self._n * int(num_relations) * 4 <= COUNTS_MAX_BYTES:
                counts = torch.empty(max(self._n * int(num_relations), 1), dtype=torch.int32, device=dev)
                _lib.call('regnn_relation_counts', _ptr(csr['row']), _ptr(et_csr), e, self._n, int(num_relations),
                          _ptr(counts), _stream())
        if len(self._etype_cache) > 8:
            self._etype_cache.clear()
        # the entry keeps ``e_feat`` alive: while it is cached its storage cannot be freed and handed to another
        # tensor with the same address / version (which would be a silent stale hit)
        self._etype_cache[key] = (et_csr, et_t, counts, e_feat)
        return self._etype_cache[key][:3]
