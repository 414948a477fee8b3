"""GPU neighbour sampler for the sampled-minibatch path (BASELINE config 5).

Stands in for ``NeighborSampler(edge_index, node_idx=..., sizes=[25, 20], batch_size=...)`` of
mag/regnn_ns.py:206-214: layer-wise sampling from the seed nodes outwards, up to ``size`` distinct in-edges
per target without replacement, target nodes first in every frontier, blocks returned outermost-first like
PyG's ``adjs``.  The random choice is counter-based (``regnn_sample_neighbors``): a batch is a pure function
of (seed, epoch, rank, batch index), so data-parallel ranks draw independent batches and the CPU oracle
(oracle/sampler_oracle.py) reproduces every sampled edge set bit for bit.

Sampling, relabelling and edge compaction of every layer run on the device (``regnn_sample_layer``) with the
frontier sizes kept there; the host reads them all in ONE small copy per batch.  Each block can then build its
CSR views on the device without another synchronisation (``Block.prebuilt``), so a training step does not
rebuild them from the edge list.  The GraphSAINT sampler hands its induced subgraph over the same way
(``regnn_induced_subgraph_count`` / ``_fill``, one host read per batch).
"""
import ctypes

import torch

from . import _lib
from .graph import COUNTS_MAX_BYTES, SPLIT_THRESHOLD, Graph, _ptr, _row_split, _stream

M32 = 0xFFFFFFFF


def _mix32(z):
    z &= M32
    z ^= z >> 16
    z = (z * 0x7feb352d) & M32
    z ^= z >> 15
    z = (z * 0x846ca68b) & M32
    z ^= z >> 16
    return z


def layer_key(seed, epoch, rank, batch, layer):
    lo = _mix32((seed * 0x9E3779B1 + epoch * 0x85EBCA6B + layer * 0xC2B2AE35) & M32)
    hi = _mix32((rank * 0x27D4EB2F + batch * 0x165667B1 + 0x5bd1e995) & M32)
    return (hi << 32) | lo


class Block:
    """One bipartite message-passing block: edges ``src_local -> dst_local`` between the ``n_src`` nodes of
    the outer frontier and its first ``n_dst`` nodes (the targets); ``eid`` are edge ids of the full graph."""

    def __init__(self, src_local, dst_local, eid, n_src, n_dst):
        self.src, self.dst, self.eid, self.n_src, self.n_dst = src_local, dst_local, eid, int(n_src), int(n_dst)
        self._sample = None     # (targets, row_off, info, status) of blocks sampled on the device

    @property
    def edge_index(self):
        return torch.stack([self.src, self.dst])

    @property
    def size(self):
        return (self.n_src, self.n_dst)

    def prebuilt(self, edge_type, node_type, num_edge_types, self_loop_type, num_relations):
        """``(Graph, etype1)`` of this block as ``mag.REGCNConv.build_block`` returns it -- with the typed self
        loops of ``self_loop_type == 2`` -- built on the device from the sample (``regnn_block_csr_build``) with
        every structure the convolutions read already in place: both CSR views, both row splits and the edge-type
        views for ``num_relations`` relations.  No host synchronisation.  ``edge_type`` / ``node_type``: 0-based
        types of the full graph's edges and nodes.  A type outside [0, num_relations) cannot be reported without a
        synchronisation: the block's edge is typed 0 and the sampler's next batch raises."""
        if self._sample is None:
            raise RuntimeError('Block.prebuilt needs a block sampled on a CUDA device')
        targets, row_off, info, status = self._sample
        dev = self.src.device
        loops = self_loop_type == 2
        n, e = self.n_src, self.src.numel() + (self.n_dst if loops else 0)
        edge_type = edge_type.to(device=dev, dtype=torch.int64).contiguous()
        node_type = node_type.to(device=dev, dtype=torch.int64).contiguous()
        i32, i64 = dict(dtype=torch.int32, device=dev), dict(dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            csr = {k: torch.empty(n + 1, **i32) for k in ('indptr', 'indptr_t')}
            csr.update({k: torch.empty(max(e, 1), **i32)[:e] for k in ('indices', 'eid', 'row', 'indices_t', 'slot_t')})
            src, dst, etype1 = (torch.empty(max(e, 1), **i64)[:e] for _ in range(3))
            et_csr, et_t = (torch.empty(max(e, 1), dtype=torch.uint8, device=dev)[:e] for _ in range(2))
            counts = None
            if n * int(num_relations) * 4 <= COUNTS_MAX_BYTES:
                counts = torch.empty(max(n * int(num_relations), 1), **i32)
            ws_bytes = _lib.load().regnn_csr_build_workspace_bytes(n, e)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _lib.call('regnn_block_csr_build', _ptr(self.src), _ptr(self.dst), _ptr(self.eid), _ptr(row_off),
                      _ptr(targets), n, self.n_dst, self.src.numel(), _ptr(edge_type), _ptr(node_type),
                      int(num_edge_types), int(loops), int(num_relations), _ptr(src), _ptr(dst), _ptr(etype1),
                      _ptr(csr['indptr']), _ptr(csr['indices']), _ptr(csr['eid']), _ptr(csr['row']),
                      _ptr(csr['indptr_t']), _ptr(csr['indices_t']), _ptr(csr['slot_t']), _ptr(et_csr), _ptr(et_t),
                      _ptr(counts), _ptr(status), _ptr(ws), ws_bytes, _stream())
            _lib.count_launches(_block_build_launches(n, e, counts is not None))
            split_in = info[_INFO_IN_SPLIT_LOOPS if loops else _INFO_IN_SPLIT:][:2]
            split_out = info[_INFO_OUT_SPLIT_LOOPS if loops else _INFO_OUT_SPLIT:][:2]
            csr['split'] = _row_split(csr['indptr'], SPLIT_THRESHOLD, split_in)
            csr['split_t'] = _row_split(csr['indptr_t'], SPLIT_THRESHOLD, split_out)
        zero_in = n > self.n_dst or (not loops and info[_INFO_EMPTY_ROWS] > 0)
        g = Graph.from_csr(src, dst, n, csr, (etype1, num_relations, et_csr, et_t, counts), zero_in)
        return g, etype1


# regnn_sample_info words (include/regnn_b200.h)
_INFO_SOURCES, _INFO_EDGES, _INFO_EMPTY_ROWS = 0, 1, 2
_INFO_IN_SPLIT, _INFO_IN_SPLIT_LOOPS, _INFO_OUT_SPLIT, _INFO_OUT_SPLIT_LOOPS = 3, 5, 7, 9
_INFO_WORDS = 16
_SAMPLE_LAYER_LAUNCHES = 12     # 2 memsets, 4 kernels, 2 three-kernel scans
_INDUCED_COUNT_LAUNCHES = 16    # 3 memsets, 4 kernels, 3 three-kernel scans
_INDUCED_FILL_LAUNCHES = 2      # fill, flag reset


def _block_build_launches(n, e, counts):
    """Kernels and memsets of regnn_block_csr_build: fill, the radix sort of the transposed view (5 per 8-bit pass
    of the key bits of regnn_csr_build), its boundaries, the edge-type transpose, the relation counts."""
    passes = (max(1, (n - 1).bit_length()) + 7) // 8 if e else 0
    return 2 + (2 + 5 * passes + 1 if e else 0) + (2 if counts else 0)


class NeighborSampler:
    def __init__(self, graph: Graph, fanouts, seed=0, rank=0):
        self.graph, self.fanouts, self.seed, self.rank = graph, list(fanouts), int(seed), int(rank)
        # (pos_map, flags, status) on the device: the [N] scratch of regnn_sample_layer, which every call leaves as it
        # found it, and the type-check word of regnn_block_csr_build.  Shared by all batches, so one sampler samples on
        # one stream at a time.
        self._maps = None

    def sample_slots(self, targets, fanout, key):
        csr = self.graph.csr()
        t = targets.numel()
        out = torch.empty(max(t * fanout, 1), dtype=torch.int32, device=targets.device)[:t * fanout]
        with torch.cuda.device(targets.device):
            _lib.call('regnn_sample_neighbors', ctypes.c_void_p(csr['indptr'].data_ptr()),
                      ctypes.c_void_p(targets.data_ptr()), t, int(fanout), ctypes.c_uint64(key),
                      ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            _lib.count_launches(1)
        return out.view(t, fanout)

    def sample(self, seeds, epoch=0, batch=0):
        """-> (n_id [int64, global ids of the outermost frontier], [Block, ...] outermost first).
        Seeds are distinct node ids.  On a CUDA device the host waits for the device once, for the frontier sizes.
        Samples on the current stream; a sampler must not be used from two streams at once."""
        n_id = seeds.to(torch.int64).contiguous()
        if not n_id.is_cuda:
            return self.reference_sample(n_id, epoch, batch)
        info, layers = self.sample_on_device(n_id, epoch, batch)
        status = self._maps[2]
        info[-1, :1].copy_(status)
        sizes = info.cpu().tolist()     # the one host synchronisation of the batch
        if sizes.pop()[0]:
            status.zero_()
            raise RuntimeError('Block.prebuilt of an earlier batch of this sampler was given an edge or node type '
                               'outside [0, num_relations): its blocks typed those edges 0')
        blocks, t = [], n_id.numel()
        for (targets, new_n_id, src_local, dst_local, eid, row_off), inf in zip(layers, sizes):
            n_src, e = inf[_INFO_SOURCES], inf[_INFO_EDGES]
            b = Block(src_local[:e], dst_local[:e], eid[:e], n_src, t)
            b._sample = (targets[:t], row_off[:t + 1], inf, status)
            blocks.append(b)
            n_id, t = new_n_id[:n_src], n_src
        return n_id, blocks[::-1]

    def sample_on_device(self, n_id, epoch=0, batch=0):
        """Enqueues every layer of the batch without waiting for the device.  Returns the int32
        [layers + 1, REGNN_SAMPLE_INFO_WORDS] device table of sizes (row ``layer``; the last row is ``sample``'s) and,
        per layer, the capacity-sized device buffers (targets, new_n_id, src_local, dst_local, eid, row_off) of
        ``regnn_sample_layer``.  If a call fails part-way, the scratch maps are dropped and rebuilt by the next call."""
        csr = self.graph.csr()
        dev, n = n_id.device, self.graph.number_of_nodes()
        if self._maps is None:
            self._maps = (torch.full((n,), 0x7fffffff, dtype=torch.int32, device=dev),
                          torch.zeros(n, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev))
        pos_map, flags, _ = self._maps
        lib = _lib.load()
        info = torch.empty((len(self.fanouts) + 1, _INFO_WORDS), dtype=torch.int32, device=dev)
        layers = []
        targets, cap, num_targets = n_id, n_id.numel(), None
        with torch.cuda.device(dev):
            for layer, fanout in enumerate(self.fanouts):
                max_src = cap + min(n, cap * fanout)
                i64 = dict(dtype=torch.int64, device=dev)
                new_n_id = torch.empty(max(max_src, 1), **i64)
                src_local, dst_local, eid = (torch.empty(max(cap * fanout, 1), **i64) for _ in range(3))
                row_off = torch.empty(cap + 1, dtype=torch.int32, device=dev)
                hist = torch.empty(max(max_src, 1), dtype=torch.int32, device=dev)
                ws_bytes = lib.regnn_sample_layer_workspace_bytes(n, cap, int(fanout))
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                try:
                    _lib.call('regnn_sample_layer', _ptr(csr['indptr']), _ptr(csr['indices']), _ptr(csr['eid']), n,
                              _ptr(targets), cap, _ptr(num_targets), int(fanout),
                              ctypes.c_uint64(layer_key(self.seed, epoch, self.rank, batch, layer)), SPLIT_THRESHOLD,
                              _ptr(pos_map), _ptr(flags), _ptr(new_n_id), max_src, _ptr(src_local), _ptr(dst_local),
                              _ptr(eid), _ptr(row_off), _ptr(hist), _ptr(info[layer]), _ptr(ws), ws_bytes, _stream())
                except RuntimeError:
                    self._maps = None       # an earlier layer of this batch may have left them half restored
                    raise
                _lib.count_launches(_SAMPLE_LAYER_LAUNCHES)
                layers.append((targets, new_n_id, src_local, dst_local, eid, row_off))
                targets, cap, num_targets = new_n_id, max_src, info[layer, _INFO_SOURCES:]
        return info, layers

    def reference_sample(self, seeds, epoch=0, batch=0):
        """The same batch relabelled with torch ops (``torch.unique`` over targets and sources, boolean masks that
        wait for the device to learn their sizes): ``sample``'s path for CPU tensors, which only the CPU emulation of
        the operators produces (the library has no CPU path), and the reference the device path is checked and
        timed against (tests/test_device_blocks_gpu.py, scripts/check_ns_step.py)."""
        csr = self.graph.csr()
        n_id = seeds.to(torch.int64).contiguous()
        dev = n_id.device
        blocks = []
        for layer, fanout in enumerate(self.fanouts):
            slots = self.sample_slots(n_id, fanout, layer_key(self.seed, epoch, self.rank, batch, layer))
            valid = slots >= 0
            t = n_id.numel()
            dst_local = torch.arange(t, device=dev).view(-1, 1).expand_as(slots)[valid]
            flat = slots[valid].to(torch.int64)
            src_global = csr['indices'][flat].to(torch.int64)
            uniq, inv = torch.unique(torch.cat([n_id, src_global]), return_inverse=True)
            is_target = torch.zeros(uniq.numel(), dtype=torch.bool, device=dev)
            is_target[inv[:t]] = True
            rest = uniq[~is_target]
            pos = torch.empty(uniq.numel(), dtype=torch.int64, device=dev)
            pos[inv[:t]] = torch.arange(t, device=dev)
            pos[~is_target] = t + torch.arange(rest.numel(), device=dev)
            new_n_id = torch.cat([n_id, rest])
            blocks.append(Block(pos[inv[t:]], dst_local, csr['eid'][flat].to(torch.int64), new_n_id.numel(), t))
            n_id = new_n_id
        return n_id, blocks[::-1]


class SaintRandomWalkSampler:
    """GraphSAINT random-walk sampler (``GraphSAINTRandomWalkSampler(data, batch_size=roots, walk_length=...)``,
    mag/regnn_saint.py:185-190; ``sample_coverage=0`` so no normalisation statistics): ``roots`` random start
    nodes, ``walk_length`` steps along out-edges (``regnn_random_walk``), then the subgraph INDUCED by the visited
    nodes.  On a CUDA device the subgraph is extracted, relabelled and handed over as a ``Block`` whose CSR views
    ``Block.prebuilt`` builds without rebuilding them from the edge list (``regnn_induced_subgraph_count`` / ``_fill``),
    with one host synchronisation per batch."""

    def __init__(self, graph: Graph, roots, walk_length, seed=0, rank=0):
        self.graph, self.roots, self.walk_length = graph, int(roots), int(walk_length)
        self.seed, self.rank = int(seed), int(rank)
        # (flags, status, workspace) on the device: the [N] flag map of regnn_induced_subgraph_count, which the fill
        # leaves as it found it, the type-check word of Block.prebuilt, and the workspace the two calls of a batch share.
        # Shared by all batches, so one sampler samples on one stream at a time.
        self._maps = None

    def walks(self, key):
        csr = self.graph.csr()
        dev = csr['indptr'].device
        out = torch.empty((self.roots, self.walk_length + 1), dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            _lib.call('regnn_random_walk', ctypes.c_void_p(csr['indptr_t'].data_ptr()),
                      ctypes.c_void_p(csr['indices_t'].data_ptr()), self.graph.number_of_nodes(), self.roots,
                      self.walk_length, ctypes.c_uint64(key), ctypes.c_void_p(out.data_ptr()),
                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            _lib.count_launches(1)
        return out

    def _key(self, epoch, batch):
        return layer_key(self.seed, epoch, self.rank, batch, 0x5A1)

    def sample(self, epoch=0, batch=0):
        """-> (n_id sorted ascending, edge_index_local [2, E'], eid): the edges are every in-edge of a subgraph node
        whose source is in the subgraph too, ordered by (destination, CSR slot).  Built from ``sample_block`` on a CUDA
        device."""
        if not self.graph.csr()['indptr'].is_cuda:
            return self.reference_sample(epoch, batch)
        n_id, block = self.sample_block(epoch, batch)
        return n_id, block.edge_index, block.eid

    def sample_block(self, epoch=0, batch=0):
        """-> (n_id, Block) of the batch: ``Block(src_local, dst_local, eid, n_sub, n_sub)`` over the ``sample`` edges.
        The host waits for the device once, for the subgraph's sizes; an out-of-range type given to ``Block.prebuilt``
        of an earlier batch is raised here."""
        return self.induced_block(self.walks(self._key(epoch, batch)).view(-1))

    def induced_block(self, nodes):
        """(n_id, Block) of the subgraph induced by ``nodes`` (int64 CUDA tensor of node ids, repeats allowed).  If a
        call fails part-way, the flag map is dropped and rebuilt by the next call."""
        csr = self.graph.csr()
        n, e = self.graph.number_of_nodes(), self.graph.number_of_edges()
        nodes = nodes.to(torch.int64).contiguous()
        dev, listed = nodes.device, nodes.numel()
        rows = min(n, listed)
        ws_bytes = _lib.load().regnn_induced_subgraph_workspace_bytes(n, e, listed)
        i32, i64 = dict(dtype=torch.int32, device=dev), dict(dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            if self._maps is None:
                self._maps = (torch.zeros(n, **i32), torch.zeros(1, **i32), torch.empty(0, dtype=torch.uint8, device=dev))
            flags, status, ws = self._maps
            if ws.numel() < ws_bytes:
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                self._maps = (flags, status, ws)
            n_id, hist = torch.empty(max(rows, 1), **i64), torch.empty(max(rows, 1), **i32)
            row_off = torch.empty(rows + 1, **i32)
            info = torch.empty((2, _INFO_WORDS), **i32)
            try:
                _lib.call('regnn_induced_subgraph_count', _ptr(csr['indptr']), _ptr(csr['indices']), n, e, _ptr(nodes),
                          listed, SPLIT_THRESHOLD, _ptr(flags), _ptr(n_id), _ptr(row_off), _ptr(hist), _ptr(info[0]),
                          _ptr(ws), ws_bytes, _stream())
                _lib.count_launches(_INDUCED_COUNT_LAUNCHES)
                info[1, :1].copy_(status)
                sizes, checked = info.cpu().tolist()     # the one host synchronisation of the batch
                n_sub, e_sub = sizes[_INFO_SOURCES], sizes[_INFO_EDGES]
                src_local, dst_local, eid = (torch.empty(max(e_sub, 1), **i64)[:e_sub] for _ in range(3))
                _lib.call('regnn_induced_subgraph_fill', _ptr(csr['indptr']), _ptr(csr['indices']), _ptr(csr['eid']), n,
                          e, listed, _ptr(flags), _ptr(n_id), n_sub, e_sub, _ptr(src_local), _ptr(dst_local), _ptr(eid),
                          _ptr(ws), ws_bytes, _stream())
                _lib.count_launches(_INDUCED_FILL_LAUNCHES)
            except BaseException:
                self._maps = None       # the count may have left flags set
                raise
        if checked[0]:
            status.zero_()
            raise RuntimeError('Block.prebuilt of an earlier batch of this sampler was given an edge type outside '
                               '[0, num_relations): its block typed those edges 0')
        b = Block(src_local, dst_local, eid, n_sub, n_sub)
        b._sample = (n_id[:n_sub], row_off[:n_sub + 1], sizes, status)
        return n_id[:n_sub], b

    def reference_sample(self, epoch=0, batch=0):
        """The same batch with torch ops (``torch.unique`` over the walk nodes, a ``.item()`` for the candidate slot
        count and a boolean mask over the candidate edges, each waiting for the device): ``sample``'s path for CPU
        tensors, which only the CPU emulation of the operators produces (the library has no CPU path), and the
        reference the device path is checked and timed against (tests/test_saint_subgraph_gpu.py,
        scripts/check_saint_step.py)."""
        csr = self.graph.csr()
        n = self.graph.number_of_nodes()
        dev = csr['indptr'].device
        n_id = torch.unique(self.walks(self._key(epoch, batch)).view(-1))
        relabel = torch.full((n,), -1, dtype=torch.int64, device=dev)
        relabel[n_id] = torch.arange(n_id.numel(), device=dev)
        indptr = csr['indptr'].to(torch.int64)
        starts, degs = indptr[n_id], indptr[n_id + 1] - indptr[n_id]
        total = int(degs.sum().item())
        first = torch.cumsum(degs, 0) - degs
        slot = torch.repeat_interleave(starts - first, degs) + torch.arange(total, device=dev)
        dst_local = torch.repeat_interleave(torch.arange(n_id.numel(), device=dev), degs)
        src_local = relabel[csr['indices'][slot].to(torch.int64)]
        keep = src_local >= 0
        return n_id, torch.stack([src_local[keep], dst_local[keep]]), csr['eid'][slot[keep]].to(torch.int64)
