"""GPU tests of ``partition.head_sliced_gatv2`` (``pytest -m gpu``, one B200): the REGATv2 core sharded over its heads.

* World size 1 (an NCCL group of one rank), both exchange variants (all-to-all, peer memory through a
  ``SlabExchange(..., gatv2=True)`` whose only peer is this rank), D in {16, 64, 256}: out, d_fs and d_fd bit-identical
  to ``functional.gatv2_aggregate``, also with shared features and with hashed dropout; parameter gradients norm-wise.
* Virtual head slices: the per-rank slab compute for q = 0..P-1 (P = 2, 4, 8) in one process, stitched along the heads,
  is bit-identical to the full-H call, with and without hashed dropout, on a graph whose hub rows take the long-row
  fragment path in both CSR views.  Every multi-rank run relies on this property.
* The refusals raise before any kernel launch."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist

import helpers
from re_gnn_b200 import Graph, _lib, functional as RF, partition, synth

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
RTOL = 2e-5
ALPHA, SLOPE = 100.0, 0.2
KEY = RF.attn_dropout_key(5, 2, 1)


def _hub_graph(n=2500, e=30000, r=5, seed=0):
    """Random multigraph with hub destinations AND hub sources (rows > 256 slots in the CSR and the transposed view)."""
    d = synth.random_multigraph(n, e, r, seed=seed, hubs=3)
    rng = np.random.RandomState(seed + 1)
    hub = rng.rand(d['src'].size) < 0.15
    d['src'][hub] = n - 1 - rng.randint(0, 3, size=int(hub.sum()))
    return d


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(DEV)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(DEV), d['num_relations'])
    return g, etv


def _inputs(n, r, heads, dim, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    fs = torch.randn(n, heads, dim, device=DEV, generator=gen)
    fd = torch.randn(n, heads, dim, device=DEV, generator=gen) * 0.5
    gout = torch.randn(n, heads, dim, device=DEV, generator=gen)
    attn = torch.randn(1, heads, dim, device=DEV, generator=gen) * (0.3 if dim <= 64 else 0.1)
    th = (torch.rand(r, heads, device=DEV, generator=gen) + 0.5) / 100
    return fs, fd, gout, attn, th


def _single(g, etv, fs, fd, gout, attn, th, shared=False, dropout=None):
    """gatv2_aggregate -> (out, d_fs, d_fd | None, d_attn, d_theta)."""
    leaves = [t.clone().requires_grad_(True) for t in (fs, fd, attn, th)]
    if shared:
        leaves[1] = leaves[0]
    out, _ = RF.gatv2_aggregate(g, etv, *leaves, ALPHA, SLOPE, dropout=dropout)
    out.backward(gout)
    return out.detach(), leaves[0].grad, None if shared else leaves[1].grad, leaves[2].grad, leaves[3].grad


def _check(got, want, what):
    for i, name in ((0, 'out'), (1, 'd_fs'), (2, 'd_fd')):
        if want[i] is not None:
            assert torch.equal(got[i], want[i]), '%s: %s differs (max |diff| %.3g)' % (
                what, name, float((got[i] - want[i]).abs().max()))
    for i, name in ((3, 'd_attn'), (4, 'd_theta')):
        if want[i] is not None:
            helpers.assert_close(got[i].reshape(want[i].shape).cpu(), want[i].cpu(), RTOL, '%s %s' % (what, name))


@pytest.fixture(scope='module')
def world1():
    """An NCCL group of this one rank for the module's tests."""
    if dist.is_initialized():
        yield
        return
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    os.environ.setdefault('MASTER_PORT', str(29700 + os.getpid() % 97))
    dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device(DEV))
    try:
        yield
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('heads,dim', [(8, 16), (2, 64), (2, 256)])
@pytest.mark.parametrize('peer', [False, True])
def test_world1_equals_gatv2_aggregate(world1, peer, heads, dim):
    d = synth.hetero_graph('acm', seed=6, scale=0.2)
    g, etv = _setup(d)
    n, r = d['num_nodes'], d['num_relations']
    fs, fd, gout, attn, th = _inputs(n, r, heads, dim, heads + dim)
    bounds = partition.row_blocks(g.csr()['indptr'], 1, balance='rows')
    xch = partition.SlabExchange(heads * dim, bounds, 0, torch.device(DEV), gatv2=True) if peer else None
    drop = RF.HashedDropout(0.3, KEY)

    def sharded(shared=False, dropout=None):
        leaves = [t.clone().requires_grad_(True) for t in (fs, fd, attn, th)]
        if shared:
            leaves[1] = leaves[0]
        out = partition.head_sliced_gatv2(g, etv, *leaves, ALPHA, SLOPE, bounds, 0, exchange=xch, dropout=dropout)
        out.backward(gout)
        partition.allreduce_relation_grads(leaves[2:], exchange=xch)
        return out.detach(), leaves[0].grad, None if shared else leaves[1].grad, leaves[2].grad, leaves[3].grad
    want = _single(g, etv, fs, fd, gout, attn, th)
    for step in range(2):   # twice: the exchange buffers are reused from step to step
        _check(sharded(), want, 'step %d' % step)
    _check(sharded(shared=True), _single(g, etv, fs, fs, gout, attn, th, shared=True), 'shared')
    _check(sharded(dropout=drop), _single(g, etv, fs, fd, gout, attn, th, dropout=drop), 'dropout')


@pytest.fixture(scope='module')
def hub():
    d = _hub_graph()
    g, etv = _setup(d)
    csr = g.csr()
    assert csr.get('split') is not None and csr.get('split_t') is not None   # the fragment path runs in both views
    return d, g, etv


@pytest.mark.parametrize('dropout', [False, True])
@pytest.mark.parametrize('heads,dim,parts,relational', [(8, 16, 2, True), (8, 16, 4, True), (8, 16, 8, True),
                                                        (8, 16, 8, False), (2, 64, 2, True), (2, 256, 2, True)])
def test_virtual_head_slices_equal_full_heads(hub, heads, dim, parts, relational, dropout):
    d, g, etv = hub
    fs, fd, gout, attn, th = _inputs(d['num_nodes'], d['num_relations'], heads, dim, 7 * parts + dim)
    drop = RF.HashedDropout(0.3, KEY) if dropout else None
    ev = etv if relational else None
    want = _single(g, ev, fs, fd, gout, attn, th, dropout=drop)
    got = partition._virtual_head_sliced_gatv2(g, ev, fs, fd, gout, attn, th if relational else None, ALPHA, SLOPE,
                                               parts, dropout=drop)
    if not relational:
        want = want[:4] + (None,)
        assert got[4] is None
    _check(got, want, 'H=%d D=%d P=%d' % (heads, dim, parts))


def test_refusals_before_any_launch(world1):
    d = synth.hetero_graph('acm', seed=6, scale=0.05)
    g, etv = _setup(d)
    n, r, heads, dim = d['num_nodes'], d['num_relations'], 8, 16
    fs, fd, _, attn, th = _inputs(n, r, heads, dim, 1)
    bounds = partition.row_blocks(g.csr()['indptr'], 1, balance='rows')
    plain = partition.SlabExchange(heads * dim, bounds, 0, torch.device(DEV))
    assert not hasattr(plain, 'fd_cols') and not hasattr(plain, 'dfd_rows')   # allocated only with gatv2=True
    before = _lib.launch_count
    with pytest.raises(ValueError, match='gatv2=True'):
        partition.head_sliced_gatv2(g, etv, fs, fd, attn, th, ALPHA, SLOPE, bounds, 0, exchange=plain)
    with pytest.raises(ValueError, match='divisible'):
        b3 = partition.row_blocks(g.csr()['indptr'], 3, balance='rows')
        partition.head_sliced_gatv2(g, etv, fs[:b3[1]], fd[:b3[1]], attn, th, ALPHA, SLOPE, b3, 0)
    with pytest.raises(ValueError, match='HashedDropout'):
        partition.head_sliced_gatv2(g, etv, fs, fd, attn, th, ALPHA, SLOPE, bounds, 0,
                                    keep=torch.ones(d['src'].size, heads, device=DEV))
    torch.cuda.synchronize()
    assert _lib.launch_count == before
