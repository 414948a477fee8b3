"""Multi-rank path on CPU: world_size-2 ``gloo`` processes run the destination-row-partitioned RE-layer
(re_gnn_b200/partition.py) with the CUDA operators replaced by tests/cpu_shim.py and must reproduce the
single-process result (outputs, feature gradients, relation-embedding gradient)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _single(d, x, gout, theta0):
    from re_gnn_b200 import Graph, functional as RF
    g = Graph(d['src'], d['dst'], d['num_nodes'])
    et = torch.as_tensor(d['etype'])
    etv = g.etype_views(et, d['num_relations'])
    xs = x.clone().requires_grad_(True)
    th = theta0.clone().requires_grad_(True)
    out = RF.propagate(g, etv, xs, th, 100.0, RF.weighted_degree_norm(g, etv, th, 100.0, -0.5))
    out.backward(gout)
    return out.detach(), xs.grad, th.grad


def _worker(rank, world, port, ret, mode='rows'):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import cpu_shim
    from re_gnn_b200 import Graph, functional as RF, graph as G, ops, partition, synth

    class MP:  # minimal monkeypatch stand-in
        @staticmethod
        def setattr(obj, name, val):
            setattr(obj, name, val)
    cpu_shim.install(MP)
    d = synth.hetero_graph('dblp', seed=5, scale=0.03)
    n, r = d['num_nodes'], d['num_relations']
    rng = np.random.RandomState(0)
    x = torch.as_tensor(rng.randn(n, 8))
    gout = torch.as_tensor(rng.randn(n, 8))
    theta0 = torch.as_tensor(rng.uniform(0.5, 1.5, (r, 1)) / 100.0)
    g = Graph(d['src'], d['dst'], n)
    etv = g.etype_views(torch.as_tensor(d['etype']), r)
    bounds = partition.row_blocks(g.csr()['indptr'], world, balance='edges' if mode == 'edges' else 'rows')
    rb, re = bounds[rank], bounds[rank + 1]
    xo = x[rb:re].clone().requires_grad_(True)
    th = theta0.clone().requires_grad_(True)
    nrm = RF.weighted_degree_norm(g, etv, th, 100.0, -0.5)
    fn = partition.feature_sliced_propagate if mode == 'cols' else partition.partitioned_propagate
    out = fn(g, etv, xo, th, 100.0, nrm, bounds, rank)
    out.backward(gout[rb:re])
    partition.allreduce_relation_grads([th])
    ref_out, ref_dx, ref_dth = _single(d, x, gout, theta0)
    ok = (torch.allclose(out.detach(), ref_out[rb:re], rtol=1e-12, atol=1e-12)
          and torch.allclose(xo.grad, ref_dx[rb:re], rtol=1e-12, atol=1e-12)
          and torch.allclose(th.grad, ref_dth, rtol=1e-10, atol=1e-12)
          and re > rb and bounds[-1] == n)
    if not ok:
        print('rank', rank, 'bounds', bounds, 'out', (out.detach() - ref_out[rb:re]).abs().max().item(),
              'dx', (xo.grad - ref_dx[rb:re]).abs().max().item(), 'dth', (th.grad - ref_dth).abs().max().item(),
              file=sys.stderr)
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


def test_row_blocks_balance_edges():
    sys.path.insert(0, ROOT)
    from re_gnn_b200 import partition
    indptr = torch.tensor([0, 10, 10, 11, 30, 31, 40])
    assert partition.row_blocks(indptr, 1) == [0, 6]
    b = partition.row_blocks(indptr, 2)
    assert b[0] == 0 and b[-1] == 6 and all(x <= y for x, y in zip(b, b[1:]))
    b4 = partition.row_blocks(indptr, 4)
    assert len(b4) == 5 and b4[-1] == 6
    assert partition.row_blocks(indptr, 4, balance='rows') == [0, 2, 4, 6, 6]
    assert partition._uniform_rows([0, 2, 4, 6, 6]) == 2 and partition._uniform_rows(b) in (0, b[1])


@pytest.mark.timeout(300)
@pytest.mark.parametrize('mode', ['edges', 'rows', 'cols'])
def test_partitioned_layer_matches_single_process_world2(mode):
    """edges / rows: destination-row blocks + all-gather; cols: feature-sliced aggregation between all-to-alls."""
    world = 2
    port = 29500 + (os.getpid() % 2000) + {'edges': 0, 'rows': 2000, 'cols': 4000}[mode]
    mgr = mp.get_context('spawn').Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, ret, mode), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)


def _attn_worker(rank, world, port, ret, kind):
    """World-size-2 gloo run of the head-sliced REGAT core / the un-weighted (REMixHop) column-slab propagation against
    the single-process result."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import cpu_shim
    from re_gnn_b200 import Graph, functional as RF, partition, synth

    class MP:
        @staticmethod
        def setattr(obj, name, val):
            setattr(obj, name, val)
    cpu_shim.install(MP)
    if kind == 'gat_empty_block':   # 4 rows over 3 ranks: bounds [0, 2, 4, 4], the last rank owns no rows
        d = dict(src=np.array([0, 1, 2, 3, 0, 2]), dst=np.array([1, 2, 3, 0, 0, 1]),
                 etype=np.array([1, 2, 1, 2, 2, 1]), num_nodes=4, num_relations=2)
    else:
        d = synth.hetero_graph('imdb', seed=7, scale=0.02)
    n, r = d['num_nodes'], d['num_relations']
    rng = np.random.RandomState(1)
    g = Graph(d['src'], d['dst'], n)
    etv = g.etype_views(torch.as_tensor(d['etype']), r)
    bounds = partition.row_blocks(g.csr()['indptr'], world, balance='rows')
    rb, re = bounds[rank], bounds[rank + 1]
    if kind != 'mixhop':
        heads, dim = (3, 8) if kind == 'gat_empty_block' else (4, 8)
        f = torch.as_tensor(rng.randn(n, heads, dim) * 0.5)
        gout = torch.as_tensor(rng.randn(n, heads, dim))
        al0, ar0 = torch.as_tensor(rng.randn(1, heads, dim) * 0.3), torch.as_tensor(rng.randn(1, heads, dim) * 0.3)
        th0 = torch.as_tensor(rng.uniform(0.5, 1.5, (r, heads)) / 100.0)
        leaves = [t.clone().requires_grad_(True) for t in (f, al0, ar0, th0)]
        ref, _ = RF.gat_layer(g, etv, *leaves, 100.0, 0.2)
        ref.backward(gout)
        mine = [f[rb:re].clone().requires_grad_(True)] + [t.clone().requires_grad_(True) for t in (al0, ar0, th0)]
        out = partition.head_sliced_gat(g, etv, mine[0], mine[1], mine[2], mine[3], 100.0, 0.2, bounds, rank)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads(mine[1:])
        ok = (torch.allclose(out.detach(), ref.detach()[rb:re], rtol=1e-12, atol=1e-12)
              and torch.allclose(mine[0].grad, leaves[0].grad[rb:re], rtol=1e-11, atol=1e-12)
              and all(torch.allclose(a.grad, b.grad, rtol=1e-10, atol=1e-12) for a, b in zip(mine[1:], leaves[1:])))
    else:   # REMixHop: relation weights enter through the norm only, the propagation itself is un-weighted
        x = torch.as_tensor(rng.randn(n, 8))
        gout = torch.as_tensor(rng.randn(n, 8))
        th0 = torch.as_tensor(rng.uniform(0.5, 1.5, (r, 1)) / 100.0)
        xs, th = x.clone().requires_grad_(True), th0.clone().requires_grad_(True)
        ref = RF.propagate(g, etv, xs, None, 100.0, RF.weighted_degree_norm(g, etv, th, 100.0, -0.5))
        ref.backward(gout)
        xo, th2 = x[rb:re].clone().requires_grad_(True), th0.clone().requires_grad_(True)
        out = partition.feature_sliced_propagate(g, etv, xo, None, 100.0, RF.weighted_degree_norm(g, etv, th2, 100.0, -0.5),
                                                 bounds, rank)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads([th2])
        ok = (torch.allclose(out.detach(), ref.detach()[rb:re], rtol=1e-12, atol=1e-12)
              and torch.allclose(xo.grad, xs.grad[rb:re], rtol=1e-11, atol=1e-12)
              and torch.allclose(th2.grad, th.grad, rtol=1e-10, atol=1e-12))
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize('kind', ['gat', 'mixhop'])
def test_sharded_attention_and_mixhop_match_single_process_world2(kind):
    world = 2
    port = 23500 + (os.getpid() % 2000) + (0 if kind == 'gat' else 2500)
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_attn_worker, args=(world, port, ret, kind), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)


@pytest.mark.timeout(300)
def test_head_sliced_attention_with_an_empty_row_block_world3():
    """A rank whose row block is empty (row_blocks(..., balance='rows') gives [0, 2, 4, 4] for 4 rows over 3 ranks)
    still takes part in every all-to-all of the forward and the backward."""
    world = 3
    port = 19000 + (os.getpid() % 2000)
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_attn_worker, args=(world, port, ret, 'gat_empty_block'), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)
