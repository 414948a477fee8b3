"""REGATv2 halo path on CPU: world-size-2 ``gloo`` processes run ``partition.halo_gatv2`` with the all-to-all exchange
variant (source-feature in-halo; dL/dY and statistics out-halo together with the stored logits and sign masks of cut
edges; then the dl tails back to the destinations' owners) with the CUDA operators replaced by the emulations of
tests/test_halo_gatv2_host.py, two steps in a row, and must reproduce ``functional.gatv2_aggregate``."""
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
    import test_halo_gatv2_host as H
    from re_gnn_b200 import Graph, partition, synth

    class MP:  # minimal monkeypatch stand-in
        @staticmethod
        def setattr(obj, name, val):
            setattr(obj, name, val)
    H.install_gatv2_halo_shim(MP)
    d = synth.hetero_graph_local('dblp', world, 0.9, seed=5, scale=0.03)
    n, r, h, dim = d['num_nodes'], d['num_relations'], 2, 4
    rng = np.random.RandomState(0)
    fs, fd, gout = (torch.as_tensor(rng.randn(n, h, dim)) for _ in range(3))
    attn0 = torch.as_tensor(rng.randn(1, h, dim) * 0.3)
    th0 = torch.as_tensor(rng.uniform(0.5, 1.5, (r, h)) / 100.0)
    g = Graph(d['src'], d['dst'], n)
    etv = g.etype_views(torch.as_tensor(d['etype']), r)
    bounds = d['community_bounds'] if layout == 'community' else partition.row_blocks(g.csr()['indptr'], world)
    rb, re = bounds[rank], bounds[rank + 1]
    part = partition.HaloPartition(g, etv, bounds, rank, attention=True)
    ok = part.n_in > 0 and part.push_slots[1][-1] > 0 and part.tail_ptr[-1] > 0
    r_out, r_fs, r_fd, r_attn, r_th = H.single(g, etv, fs, fd, gout, attn0, th0)
    for _ in range(2):      # twice: a partition serves every step
        fso, fdo = fs[rb:re].clone().requires_grad_(True), fd[rb:re].clone().requires_grad_(True)
        attn, th = attn0.clone().requires_grad_(True), th0.clone().requires_grad_(True)
        out = partition.halo_gatv2(part, fso, fdo, attn, th, H.ALPHA, H.SLOPE)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads([attn, th])
        ok = (ok and torch.allclose(out.detach(), r_out[rb:re], rtol=1e-12, atol=1e-12)
              and torch.allclose(fso.grad, r_fs[rb:re], rtol=1e-10, atol=1e-12)
              and torch.allclose(fdo.grad, r_fd[rb:re], rtol=1e-10, atol=1e-12)
              and torch.allclose(attn.grad, r_attn, rtol=1e-10, atol=1e-12)
              and torch.allclose(th.grad, r_th, rtol=1e-10, atol=1e-12))
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize('layout', ['community', 'edges'])
def test_halo_gatv2_matches_single_process_world2(layout):
    """community: the generator's bounds; edges: row_blocks (uneven row counts)."""
    world = 2
    port = 24700 + (os.getpid() % 1500) + (0 if layout == 'community' else 1700)
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_worker, args=(world, port, ret, layout), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)
