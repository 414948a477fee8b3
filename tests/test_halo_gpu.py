"""GPU tests of the halo-exchange row partitioning (``pytest -m gpu``, one B200): the regnn_halo_push kernel against
index_select, P virtual ranks on their local views against the single-device propagation (Y and dX bit for bit), and
``partition.halo_propagate`` in a world-size-1 NCCL group with both exchange variants."""
import ctypes
import os

import numpy as np
import pytest
import torch

from re_gnn_b200 import Graph, _lib, functional as RF, ops, partition, synth

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.mark.parametrize('feat', [4, 64, 128, 1024])
def test_halo_push_matches_index_select(feat):
    """P = 5 local buffers; lists of uneven length, one empty, the self entry among them; rank 2 pushes."""
    gen = torch.Generator(device=DEV).manual_seed(feat)
    x = torch.randn(300, feat, device=DEV, generator=gen)
    counts = [17, 0, 300, 1, 64]
    lists = [torch.randint(0, 300, (c,), device=DEV, generator=gen, dtype=torch.int32) for c in counts]
    lists[2] = torch.arange(300, dtype=torch.int32, device=DEV)
    offsets = [5, 0, 0, 9, 3]
    bufs = [torch.full((o + c + 2, feat), -1.0, device=DEV) for o, c in zip(offsets, counts)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=DEV)
    ptr = [0] + list(np.cumsum(counts))
    ops.halo_push(x, torch.cat(lists), [int(p) for p in ptr], offsets, ptrs, feat, 2)
    torch.cuda.synchronize()
    for b, lst, o, c in zip(bufs, lists, offsets, counts):
        assert torch.equal(b[o:o + c], x.index_select(0, lst.long()))
        assert bool((b[:o] == -1).all()) and bool((b[o + c:] == -1).all())


def test_halo_push_rejects_bad_arguments():
    lib = _lib.load()
    x = torch.zeros(8, 8, device=DEV)
    rows = torch.zeros(4, dtype=torch.int32, device=DEV)
    ptrs = torch.tensor([x.data_ptr(), x.data_ptr()], dtype=torch.int64, device=DEV)

    def call(feat=8, ldx=8, ptr=(0, 2, 4), off=(0, 0), ldb=8, p=2, rank=0, xp=None):
        return lib.regnn_halo_push(ctypes.c_void_p(xp if xp is not None else x.data_ptr()), ldx, feat,
                                   ctypes.c_void_p(rows.data_ptr()), (ctypes.c_int64 * len(ptr))(*ptr),
                                   (ctypes.c_int64 * len(off))(*off), ctypes.c_void_p(ptrs.data_ptr()), ldb, p, rank, None)
    assert call() == 0
    torch.cuda.synchronize()
    assert call(feat=6, ldx=8, ldb=8) == -2                    # not whole 128-bit chunks
    assert call(ldx=6, feat=4) == -2                           # row stride breaks 16-byte alignment
    assert call(xp=x.data_ptr() + 4) == -2                     # misaligned base
    assert call(ptr=(0, 3, 2)) == -1                           # negative count
    assert call(off=(0, -1)) == -1                             # negative receive offset
    assert call(rank=2) == -1
    assert call(ptr=(0,) * 66, off=(0,) * 65, p=65) == -2      # more ranks than the parameter table holds
    assert b'halo_push' in lib.regnn_last_error_string()


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(DEV)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(DEV), d['num_relations'])
    return g, etv


def _single(g, etv, x, gout, theta, weighted):
    xs, th = x.clone().requires_grad_(True), theta.clone().requires_grad_(True)
    out = RF.propagate(g, etv, xs, th if weighted else None, 100.0, RF.weighted_degree_norm(g, etv, th, 100.0, -0.5))
    out.backward(gout)
    return out.detach(), xs.grad, th.grad


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max())


@pytest.mark.parametrize('name,feat,scale', [('mag', 128, 0.04), ('dblp', 48, 1.0), ('dblp', 256, 1.0)])
@pytest.mark.parametrize('parts', [2, 4, 8])
@pytest.mark.parametrize('weighted', [True, False])
def test_virtual_ranks_bit_identical(name, feat, scale, parts, weighted):
    """Every virtual rank on its local views (halos filled with index_select): its rows of Y and dX equal the
    single-device result bit for bit; the relation gradient summed over ranks agrees to 1e-6.  Uneven bounds: the
    generator's communities for the MAG shape, edge-balanced row blocks for DBLP."""
    d = synth.hetero_graph_local(name, parts, 0.9, seed=7, scale=scale)
    g, etv = _setup(d)
    n = d['num_nodes']
    bounds = d['community_bounds'] if name == 'mag' else partition.row_blocks(g.csr()['indptr'], parts)
    part_list = partition.HaloPartition.virtual_ranks(g, etv, bounds)
    if name == 'mag':   # hub rows longer than the split threshold: the fragment path runs on the local views
        assert any(p.csr['split'] is not None for p in part_list) and any(p.csr['split_t'] is not None for p in part_list)
    gen = torch.Generator(device=DEV).manual_seed(parts)
    x = torch.randn(n, feat, device=DEV, generator=gen)
    gout = torch.randn(n, feat, device=DEV, generator=gen)
    theta = (torch.rand(d['num_relations'], 1, device=DEV, generator=gen) + 0.5) / 100
    ry, rdx, rdth = _single(g, etv, x, gout, theta, weighted)
    dth = torch.zeros_like(theta)
    for p, part in enumerate(part_list):
        rb, re = bounds[p], bounds[p + 1]
        y, deg, norm = partition._halo_forward(part, x[part.rows_in], theta, 100.0, weighted)
        dx, dt = partition._halo_backward(part, x[rb:re].contiguous(), y, gout[part.rows_out], theta, 100.0, weighted,
                                          deg, norm)
        assert torch.equal(y, ry[rb:re]), p
        assert torch.equal(dx, rdx[rb:re]), p
        dth += dt
    assert _rel(dth, rdth) < 1e-6


@pytest.mark.parametrize('weighted', [True, False])
def test_halo_propagate_world1_nccl(weighted):
    """Single-rank NCCL group: both exchange variants (uneven all-to-all; regnn_halo_push over a HaloExchange), twice in a
    row so the exchange buffers are reused, against functional.propagate."""
    import torch.distributed as dist
    if not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', str(29000 + os.getpid() % 400))
        dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device(DEV))
    try:
        d = synth.hetero_graph_local('acm', 1, 0.9, seed=4, scale=0.2)
        g, etv = _setup(d)
        n, f = d['num_nodes'], 64
        gen = torch.Generator(device=DEV).manual_seed(8)
        x = torch.randn(n, f, device=DEV, generator=gen)
        gout = torch.randn(n, f, device=DEV, generator=gen)
        theta = (torch.rand(d['num_relations'], 1, device=DEV, generator=gen) + 0.5) / 100
        ry, rdx, rdth = _single(g, etv, x, gout, theta, weighted)
        part = partition.HaloPartition(g, etv, d['community_bounds'], 0)
        xch = partition.HaloExchange(part, f, torch.device(DEV))
        for exchange in (None, None, xch, xch):
            xs, th = x.clone().requires_grad_(True), theta.clone().requires_grad_(True)
            out = partition.halo_propagate(part, xs, th, 100.0, weighted=weighted, exchange=exchange)
            out.backward(gout)
            partition.allreduce_relation_grads([th], exchange=exchange)
            assert torch.equal(out.detach(), ry) and torch.equal(xs.grad, rdx)
            assert _rel(th.grad, rdth) < 1e-6
    finally:
        dist.destroy_process_group()
