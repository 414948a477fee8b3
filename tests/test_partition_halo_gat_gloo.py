"""REGAT halo path on CPU: world-size-2 ``gloo`` processes run ``partition.halo_gat`` with the all-to-all exchange
variant (features and dL/dY / statistics halos, then the dpre tails back to the destinations' owners) with the CUDA
operators replaced by the emulations of tests/test_halo_gat_host.py, and must reproduce ``functional.gat_layer``."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, ret, layout):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import test_halo_gat_host
    from re_gnn_b200 import Graph, functional as RF, partition, synth

    class MP:  # minimal monkeypatch stand-in
        @staticmethod
        def setattr(obj, name, val):
            setattr(obj, name, val)
    test_halo_gat_host.install_gat_halo_shim(MP)
    d = synth.hetero_graph_local('dblp', world, 0.9, seed=5, scale=0.03)
    n, r, h, dim = d['num_nodes'], d['num_relations'], 2, 4
    rng = np.random.RandomState(0)
    f = torch.as_tensor(rng.randn(n, h, dim))
    gout = torch.as_tensor(rng.randn(n, h, dim))
    al0, ar0 = (torch.as_tensor(rng.randn(1, h, dim) * 0.3) for _ in range(2))
    th0 = torch.as_tensor(rng.uniform(0.5, 1.5, (r, h)) / 100.0)
    g = Graph(d['src'], d['dst'], n)
    etv = g.etype_views(torch.as_tensor(d['etype']), r)
    bounds = d['community_bounds'] if layout == 'community' else partition.row_blocks(g.csr()['indptr'], world)
    rb, re = bounds[rank], bounds[rank + 1]
    part = partition.HaloPartition(g, etv, bounds, rank, attention=True)
    ok = part.n_in > 0 and part.n_out > 0 and part.tail_ptr[-1] > 0
    leaves = [t.clone().requires_grad_(True) for t in (f, al0, ar0, th0)]
    ref, _ = RF.gat_layer(g, etv, *leaves, 100.0, 0.2)
    ref.backward(gout)
    for _ in range(2):      # twice: a partition serves every step
        fo = f[rb:re].clone().requires_grad_(True)
        al, ar, th = (t.clone().requires_grad_(True) for t in (al0, ar0, th0))
        out = partition.halo_gat(part, fo, al, ar, th, 100.0, 0.2)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads([al, ar, th])
        ok = (ok and torch.allclose(out.detach(), ref.detach()[rb:re], rtol=1e-12, atol=1e-12)
              and torch.allclose(fo.grad, leaves[0].grad[rb:re], rtol=1e-10, atol=1e-12)
              and all(torch.allclose(a.grad, b.grad, rtol=1e-10, atol=1e-12) for a, b in zip((al, ar, th), leaves[1:])))
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize('layout', ['community', 'edges'])
def test_halo_gat_matches_single_process_world2(layout):
    """community: the generator's bounds; edges: row_blocks (uneven row counts)."""
    world = 2
    port = 21500 + (os.getpid() % 1500) + (0 if layout == 'community' else 1700)
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_worker, args=(world, port, ret, layout), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)
