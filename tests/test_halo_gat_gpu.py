"""GPU tests of the REGAT halo path (``pytest -m gpu``, one B200): the regnn_halo_scatter kernel against index_put_,
P virtual ranks of ``partition.halo_gat``'s stages on their local views against ``functional.gat_layer`` (out and d_feat
bit for bit), and ``partition.halo_gat`` in a world-size-1 NCCL group with both exchange variants."""
import ctypes
import os

import numpy as np
import pytest
import torch

from re_gnn_b200 import Graph, _lib, functional as RF, ops, partition, synth

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.mark.parametrize('width', [1, 2, 4, 8, 32])
def test_halo_scatter_matches_index_put(width):
    """P = 5 local buffers; segments of uneven length, one empty, the self segment empty; rank 2 scatters."""
    gen = torch.Generator(device=DEV).manual_seed(width)
    counts = [17, 0, 0, 300, 64]
    sizes = [40, 10, 7, 1000, 64]
    x = torch.randn(sum(counts) + 3, width, device=DEV, generator=gen)
    dst = [torch.randperm(s, device=DEV, generator=gen)[:c].to(torch.int32) for s, c in zip(sizes, counts)]
    bufs = [torch.full((s, width), -1.0, device=DEV) for s in sizes]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=DEV)
    ptr = [3] + [3 + int(c) for c in np.cumsum(counts)]          # the rows start at an offset of the source buffer
    rows = torch.cat([torch.zeros(3, dtype=torch.int32, device=DEV)] + dst)
    ops.halo_scatter(x, ptr, rows, ptrs, width, 2)
    torch.cuda.synchronize()
    for q, (b, s) in enumerate(zip(bufs, sizes)):
        want = torch.full((s, width), -1.0, device=DEV)
        want.index_put_((dst[q].long(),), x[ptr[q]:ptr[q + 1]])
        assert torch.equal(b, want), q


def test_halo_scatter_rejects_bad_arguments():
    lib = _lib.load()
    x = torch.zeros(8, 4, device=DEV)
    rows = torch.zeros(4, dtype=torch.int32, device=DEV)
    ptrs = torch.tensor([x.data_ptr(), x.data_ptr()], dtype=torch.int64, device=DEV)

    def call(width=4, ldx=4, ptr=(0, 2, 4), ldb=4, p=2, rank=0, rp=None):
        return lib.regnn_halo_scatter(ctypes.c_void_p(x.data_ptr()), ldx, width, (ctypes.c_int64 * len(ptr))(*ptr),
                                      ctypes.c_void_p(rows.data_ptr() if rp is None else rp), ctypes.c_void_p(ptrs.data_ptr()),
                                      ldb, p, rank, None)
    assert call() == 0
    torch.cuda.synchronize()
    assert call(width=0) == -1
    assert call(ldx=3) == -1                                   # leading dimension below the width
    assert call(ldb=2) == -1
    assert call(ptr=(0, 3, 2)) == -1                           # negative count
    assert call(ptr=(-1, 0, 0)) == -1                          # negative offset
    assert call(rank=2) == -1
    assert call(rp=0) == -1                                    # rows to send but no destination list
    assert call(ptr=(0,) * 66, p=65) == -2                     # more ranks than the parameter table holds
    assert b'halo_scatter' in lib.regnn_last_error_string()
    assert call(ptr=(0, 0, 0), rp=0) == 0                      # nothing to send: no list needed


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(DEV)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(DEV), d['num_relations'])
    return g, etv


def _inputs(d, heads, dim, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    n = d['num_nodes']
    f = torch.randn(n, heads, dim, device=DEV, generator=gen)
    gout = torch.randn(n, heads, dim, device=DEV, generator=gen)
    al = torch.randn(1, heads, dim, device=DEV, generator=gen) * 0.3
    ar = torch.randn(1, heads, dim, device=DEV, generator=gen) * 0.3
    th = (torch.rand(d['num_relations'], heads, device=DEV, generator=gen) + 0.5) / 100
    return f, gout, al, ar, th


def _single(g, etv, f, gout, al, ar, th):
    leaves = [t.clone().requires_grad_(True) for t in (f, al, ar, th)]
    out, _ = RF.gat_layer(g, etv, *leaves, 100.0, 0.2)
    out.backward(gout)
    return (out.detach(),) + tuple(t.grad for t in leaves)


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize('locality', [0.0, 0.9])
@pytest.mark.parametrize('heads,dim', [(8, 16), (2, 64), (4, 8)])
@pytest.mark.parametrize('name,scale', [('mag', 0.04), ('dblp', 1.0), ('acm', 1.0)])
@pytest.mark.parametrize('parts', [2, 4, 8])
def test_virtual_ranks_bit_identical(name, scale, heads, dim, parts, locality):
    """Every virtual rank on its local views (halos filled by indexing, dpre tails returned by regnn_halo_scatter over
    local buffers at locality 0.9, by index_copy_ at the receive lists at 0): out and d_feat equal gat_layer bit for bit;
    the parameter gradients summed over ranks agree norm-wise to 1e-6.  Bounds: the generator's communities for MAG,
    edge-balanced row blocks otherwise."""
    d = synth.hetero_graph_local(name, parts, locality, seed=7, scale=scale)
    g, etv = _setup(d)
    bounds = d['community_bounds'] if name == 'mag' else partition.row_blocks(g.csr()['indptr'], parts)
    plist = partition.HaloPartition.virtual_ranks(g, etv, bounds, attention=True)
    if name == 'mag':   # rows longer than the split threshold: the fragment path runs on both local views
        assert any(p.csr['split'] is not None for p in plist) and any(p.csr['split_t'] is not None for p in plist)
    f, gout, al, ar, th = _inputs(d, heads, dim, parts)
    r_out, r_f, r_al, r_ar, r_th = _single(g, etv, f, gout, al, ar, th)
    out, d_f, d_al, d_ar, d_th = partition._virtual_halo_gat(plist, f, gout, al, ar, th, 100.0, 0.2,
                                                             scatter=locality > 0.5)
    errs = (_rel(d_al, r_al.view(-1)), _rel(d_ar, r_ar.view(-1)), _rel(d_th, r_th))
    print('%s P=%d H=%d D=%d locality=%.1f  d_attn_l %.2e  d_attn_r %.2e  d_theta %.2e' % ((name, parts, heads, dim,
                                                                                         locality) + errs))
    assert torch.equal(out, r_out)
    assert torch.equal(d_f, r_f)
    assert max(errs) < 1e-6


def test_halo_gat_world1_nccl():
    """Single-rank NCCL group: both exchange variants (uneven all-to-alls; regnn_halo_push / regnn_halo_scatter over a
    HaloExchange), each twice in a row so the exchange buffers are reused, against functional.gat_layer."""
    import torch.distributed as dist
    if not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', str(29400 + os.getpid() % 400))
        dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device(DEV))
    try:
        d = synth.hetero_graph_local('acm', 1, 0.9, seed=4, scale=0.2)
        g, etv = _setup(d)
        heads, dim = 8, 16
        f, gout, al, ar, th = _inputs(d, heads, dim, 8)
        r_out, r_f, r_al, r_ar, r_th = _single(g, etv, f, gout, al, ar, th)
        part = partition.HaloPartition(g, etv, d['community_bounds'], 0, attention=True)
        xch = partition.HaloExchange(part, heads * dim, torch.device(DEV), heads=heads)
        assert xch.GRAD_SLOTS >= 2 * heads * dim + d['num_relations'] * heads
        for exchange in (None, None, xch, xch):
            leaves = [t.clone().requires_grad_(True) for t in (f, al, ar, th)]
            out = partition.halo_gat(part, *leaves, 100.0, 0.2, exchange=exchange)
            out.backward(gout)
            partition.allreduce_relation_grads(leaves[1:], exchange=exchange)
            assert torch.equal(out.detach(), r_out) and torch.equal(leaves[0].grad, r_f)
            for a, b in zip(leaves[1:], (r_al, r_ar, r_th)):
                assert _rel(a.grad, b) < 1e-6
    finally:
        dist.destroy_process_group()
