"""Halo-exchange row partitioning on CPU: world-size-2 ``gloo`` processes run ``partition.halo_propagate`` (uneven
all-to-all of the halo rows) with the CUDA operators replaced by tests/cpu_shim.py and must reproduce the single-process
result (outputs, feature gradients, relation-embedding gradient), at the tolerances of tests/test_partition_gloo.py."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, ret, weighted, layout):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import test_halo_host
    from re_gnn_b200 import Graph, functional as RF, partition, synth

    class MP:  # minimal monkeypatch stand-in
        @staticmethod
        def setattr(obj, name, val):
            setattr(obj, name, val)
    test_halo_host.install_halo_shim(MP)
    d = synth.hetero_graph_local('dblp', world, 0.9, seed=5, scale=0.03)
    n, r = d['num_nodes'], d['num_relations']
    rng = np.random.RandomState(0)
    x = torch.as_tensor(rng.randn(n, 8))
    gout = torch.as_tensor(rng.randn(n, 8))
    theta0 = torch.as_tensor(rng.uniform(0.5, 1.5, (r, 1)) / 100.0)
    g = Graph(d['src'], d['dst'], n)
    etv = g.etype_views(torch.as_tensor(d['etype']), r)
    bounds = d['community_bounds'] if layout == 'community' else partition.row_blocks(g.csr()['indptr'], world)
    rb, re = bounds[rank], bounds[rank + 1]
    part = partition.HaloPartition(g, etv, bounds, rank)
    ok = part.n_in > 0 and part.n_out > 0
    for _ in range(2):      # twice: a partition serves every step
        xo = x[rb:re].clone().requires_grad_(True)
        th = theta0.clone().requires_grad_(True)
        out = partition.halo_propagate(part, xo, th, 100.0, weighted=weighted)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads([th])
        xs, ths = x.clone().requires_grad_(True), theta0.clone().requires_grad_(True)
        ref = RF.propagate(g, etv, xs, ths if weighted else None, 100.0, RF.weighted_degree_norm(g, etv, ths, 100.0, -0.5))
        ref.backward(gout)
        ok = (ok and torch.allclose(out.detach(), ref.detach()[rb:re], rtol=1e-12, atol=1e-12)
              and torch.allclose(xo.grad, xs.grad[rb:re], rtol=1e-11, atol=1e-12)
              and torch.allclose(th.grad, ths.grad, rtol=1e-10, atol=1e-12))
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize('layout', ['community', 'edges'])
@pytest.mark.parametrize('weighted', [True, False])
def test_halo_propagate_matches_single_process_world2(weighted, layout):
    """weighted: REGCN's A_w; un-weighted: REMixHop's A.  community: the generator's bounds; edges: row_blocks."""
    world = 2
    port = 25500 + (os.getpid() % 1500) + (0 if weighted else 1500) + (0 if layout == 'community' else 3000)
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_worker, args=(world, port, ret, weighted, layout), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)
