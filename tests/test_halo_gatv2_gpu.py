"""GPU tests of the REGATv2 halo path (``pytest -m gpu``, one B200): the regnn_halo_push_slots kernel against
index_select, P virtual ranks of ``partition.halo_gatv2``'s stages on their local views against
``functional.gatv2_aggregate`` (out, d_fs and d_fd bit for bit), and ``partition.halo_gatv2`` in a world-size-1 NCCL
group with both exchange variants."""
import ctypes
import os

import numpy as np
import pytest
import torch

from re_gnn_b200 import Graph, _lib, functional as RF, ops, partition, synth

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ALPHA, SLOPE = 100.0, 0.2


@pytest.mark.parametrize('heads,feat', [(1, 4), (2, 128), (8, 128), (8, 512), (32, 1024)])
def test_halo_push_slots_matches_index_select(heads, feat):
    """P = 5 local buffer pairs; segments of uneven length, one empty, the self segment empty; rank 2 pushes, from a
    send list that starts at an offset."""
    gen = torch.Generator(device=DEV).manual_seed(heads * 7 + feat)
    chunks = (feat + 127) // 128
    e = 900
    logit = torch.randn(e, heads, device=DEV, generator=gen)
    mask = torch.randint(-2 ** 31, 2 ** 31 - 1, (e, chunks, 4), dtype=torch.int32, device=DEV, generator=gen)
    counts = [17, 0, 0, 300, 64]
    sizes = [40, 10, 7, 1000, 64]
    offsets = [20, 3, 7, 600, 0]                 # rows of each peer's buffers the segment starts at
    send = [torch.randint(0, e, (c,), device=DEV, generator=gen).to(torch.int32) for c in counts]
    lbufs = [torch.full((s, heads), -1.0, device=DEV) for s in sizes]
    mbufs = [torch.full((s, chunks, 4), -1, dtype=torch.int32, device=DEV) for s in sizes]
    lptrs = torch.tensor([b.data_ptr() for b in lbufs], dtype=torch.int64, device=DEV)
    mptrs = torch.tensor([b.data_ptr() for b in mbufs], dtype=torch.int64, device=DEV)
    ptr = [3] + [3 + int(c) for c in np.cumsum(counts)]
    slots = torch.cat([torch.zeros(3, dtype=torch.int32, device=DEV)] + send)
    ops.halo_push_slots(logit, mask, slots, ptr, offsets, lptrs, mptrs, 2)
    torch.cuda.synchronize()
    for q in range(5):
        want_l = torch.full((sizes[q], heads), -1.0, device=DEV)
        want_m = torch.full((sizes[q], chunks, 4), -1, dtype=torch.int32, device=DEV)
        want_l[offsets[q]:offsets[q] + counts[q]] = logit.index_select(0, send[q].long())
        want_m[offsets[q]:offsets[q] + counts[q]] = mask.index_select(0, send[q].long())
        assert torch.equal(lbufs[q], want_l) and torch.equal(mbufs[q], want_m), q


def test_halo_push_slots_rejects_bad_arguments():
    lib = _lib.load()
    logit = torch.zeros(8, 2, device=DEV)
    mask = torch.zeros(8, 1, 4, dtype=torch.int32, device=DEV)
    slots = torch.zeros(4, dtype=torch.int32, device=DEV)
    lptrs = torch.tensor([logit.data_ptr()] * 2, dtype=torch.int64, device=DEV)
    mptrs = torch.tensor([mask.data_ptr()] * 2, dtype=torch.int64, device=DEV)

    def call(heads=2, chunks=1, ptr=(0, 2, 4), off=(4, 4), p=2, rank=0, sp=None, mp=None, lp=None):
        return lib.regnn_halo_push_slots(
            ctypes.c_void_p(logit.data_ptr() if lp is None else lp), heads,
            ctypes.c_void_p(mask.data_ptr() if mp is None else mp), chunks,
            ctypes.c_void_p(slots.data_ptr() if sp is None else sp), (ctypes.c_int64 * len(ptr))(*ptr),
            (ctypes.c_int64 * len(off))(*off), ctypes.c_void_p(lptrs.data_ptr()), ctypes.c_void_p(mptrs.data_ptr()),
            p, rank, None)
    assert call() == 0
    torch.cuda.synchronize()
    assert call(heads=0) == -1
    assert call(chunks=0) == -1
    assert call(ptr=(0, 3, 2)) == -1                           # negative count
    assert call(ptr=(-1, 0, 0)) == -1                          # negative offset
    assert call(off=(0, -1)) == -1                             # negative receive offset
    assert call(rank=2) == -1
    assert call(lp=0) == -1
    assert call(sp=0) == -1                                    # slots to send but no send list
    assert call(mp=mask.data_ptr() + 4) == -2                  # mask rows not 16-byte aligned
    assert call(ptr=(0,) * 66, off=(0,) * 65, p=65) == -2      # more ranks than the parameter table holds
    assert b'halo_push_slots' in lib.regnn_last_error_string()
    assert call(ptr=(0, 0, 0), sp=0) == 0                      # nothing to send: no list needed


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(DEV)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(DEV), d['num_relations'])
    return g, etv


def _inputs(d, heads, dim, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    n = d['num_nodes']
    fs = torch.randn(n, heads, dim, device=DEV, generator=gen)
    fd = torch.randn(n, heads, dim, device=DEV, generator=gen)
    gout = torch.randn(n, heads, dim, device=DEV, generator=gen)
    attn = torch.randn(1, heads, dim, device=DEV, generator=gen) * 0.3
    th = (torch.rand(d['num_relations'], heads, device=DEV, generator=gen) + 0.5) / 100
    return fs, fd, gout, attn, th


def _single(g, etv, fs, fd, gout, attn, th):
    leaves = [t.clone().requires_grad_(True) for t in (fs, fd, attn, th)]
    out, _ = RF.gatv2_aggregate(g, etv, *leaves, ALPHA, SLOPE)
    out.backward(gout)
    return (out.detach(),) + tuple(t.grad for t in leaves)


def _rel(a, b):
    return float((a.reshape(-1) - b.reshape(-1)).norm() / b.norm())


@pytest.mark.parametrize('locality', [0.0, 0.9])
@pytest.mark.parametrize('heads,dim', [(8, 16), (2, 64), (4, 8), (1, 128)])
@pytest.mark.parametrize('name,scale', [('mag', 0.04), ('dblp', 1.0), ('acm', 1.0)])
@pytest.mark.parametrize('parts', [2, 4, 8])
def test_virtual_ranks_bit_identical(name, scale, heads, dim, parts, locality):
    """Every virtual rank on its local views (halos filled by indexing; the slot records and the dl tails moved by
    regnn_halo_push_slots / regnn_halo_scatter over local buffers at locality 0.9, by indexing at 0): out, d_fs and d_fd
    equal gatv2_aggregate bit for bit; d_attn and d_theta summed over ranks agree norm-wise to 1e-6.  Bounds: the
    generator's communities for MAG, edge-balanced row blocks otherwise."""
    d = synth.hetero_graph_local(name, parts, locality, seed=7, scale=scale)
    g, etv = _setup(d)
    bounds = d['community_bounds'] if name == 'mag' else partition.row_blocks(g.csr()['indptr'], parts)
    plist = partition.HaloPartition.virtual_ranks(g, etv, bounds, attention=True)
    if name == 'mag':   # rows longer than the split threshold: the fragment path runs on both local views
        assert any(p.csr['split'] is not None for p in plist) and any(p.csr['split_t'] is not None for p in plist)
    assert sum(p.push_slots[1][-1] for p in plist) > 0
    fs, fd, gout, attn, th = _inputs(d, heads, dim, parts)
    r_out, r_fs, r_fd, r_attn, r_th = _single(g, etv, fs, fd, gout, attn, th)
    out, d_fs, d_fd, d_attn, d_th = partition._virtual_halo_gatv2(plist, fs, fd, gout, attn, th, ALPHA, SLOPE,
                                                                  push=locality > 0.5)
    errs = (_rel(d_attn, r_attn), _rel(d_th, r_th))
    print('%s P=%d H=%d D=%d locality=%.1f  d_attn %.2e  d_theta %.2e' % ((name, parts, heads, dim, locality) + errs))
    assert torch.equal(out, r_out)
    assert torch.equal(d_fs, r_fs)
    assert torch.equal(d_fd, r_fd)
    assert max(errs) < 1e-6


def test_halo_gatv2_world1_nccl():
    """Single-rank NCCL group: both exchange variants (uneven all-to-alls; regnn_halo_push / regnn_halo_push_slots /
    regnn_halo_scatter over a HaloExchange), each twice in a row so the exchange buffers are reused, against
    functional.gatv2_aggregate."""
    import torch.distributed as dist
    if not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', str(28600 + os.getpid() % 400))
        dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device(DEV))
    try:
        d = synth.hetero_graph_local('acm', 1, 0.9, seed=4, scale=0.2)
        g, etv = _setup(d)
        heads, dim = 8, 16
        fs, fd, gout, attn, th = _inputs(d, heads, dim, 8)
        r_out, r_fs, r_fd, r_attn, r_th = _single(g, etv, fs, fd, gout, attn, th)
        part = partition.HaloPartition(g, etv, d['community_bounds'], 0, attention=True)
        xch = partition.HaloExchange(part, heads * dim, torch.device(DEV), heads=heads, gatv2=True)
        assert xch.GRAD_SLOTS >= heads * dim + d['num_relations'] * heads
        assert xch.mask_ext.dtype == torch.int32 and xch.mask_ext.shape[1:] == (1, 4)
        for exchange in (None, None, xch, xch):
            leaves = [t.clone().requires_grad_(True) for t in (fs, fd, attn, th)]
            out = partition.halo_gatv2(part, *leaves, ALPHA, SLOPE, exchange=exchange)
            out.backward(gout)
            partition.allreduce_relation_grads(leaves[2:], exchange=exchange)
            assert torch.equal(out.detach(), r_out) and torch.equal(leaves[0].grad, r_fs)
            assert torch.equal(leaves[1].grad, r_fd)
            for a, b in zip(leaves[2:], (r_attn, r_th)):
                err = _rel(a.grad, b)
                print('exchange=%s  %.2e' % ('peer' if exchange is not None else 'all_to_all', err))
                assert err < 1e-6
    finally:
        dist.destroy_process_group()
