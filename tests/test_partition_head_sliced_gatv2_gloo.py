"""REGATv2 sharded over its heads on CPU: ``partition.head_sliced_gatv2`` with the all-to-all exchange variant in
world-size-2 and -3 ``gloo`` processes (the latter with an empty row block), the per-rank slab compute for P virtual
ranks in one process, and the refusals.  The CUDA operators are replaced by the plain-PyTorch stage emulations of
tests/test_attention_dropout_host.py (which apply hashed dropout with the oracle's hash); the reference is
``functional.gatv2_aggregate`` over cpu_shim's whole-graph operators, fed the oracle's explicit mask for dropout."""
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHA, SLOPE = 100.0, 0.2
P_DROP = 0.4


def _graph(kind, synth):
    if kind == 'empty_block':   # 4 rows over 3 ranks: bounds [0, 2, 4, 4], the last rank owns no rows
        return dict(src=np.array([0, 1, 2, 3, 0, 2]), dst=np.array([1, 2, 3, 0, 0, 1]),
                    etype=np.array([1, 2, 1, 2, 2, 1]), num_nodes=4, num_relations=2), 3, 4
    return synth.hetero_graph('imdb', seed=7, scale=0.02), 4, 8


def _inputs(d, heads, dim, seed):
    rng = np.random.RandomState(seed)
    n = d['num_nodes']
    fs, fd, gout = (torch.as_tensor(rng.randn(n, heads, dim)) for _ in range(3))
    attn = torch.as_tensor(rng.randn(1, heads, dim) * 0.3)
    th = torch.as_tensor(rng.uniform(0.5, 1.5, (d['num_relations'], heads)) / 100.0)
    return fs, fd, gout, attn, th


def _reference(g, etv, fs, fd, gout, attn, th, shared=False, keep=None):
    """functional.gatv2_aggregate over cpu_shim's whole-graph operators -> (out, d_fs, d_fd | None, d_attn, d_theta |
    None); ``th=None``: no relation term; ``shared``: one leaf for both sides (its gradient is returned as d_fs)."""
    import test_halo_gatv2_host as V2
    from re_gnn_b200 import functional as RF
    with V2._whole_graph_ops():
        leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (fs, fd, attn, th)]
        if shared:
            leaves[1] = leaves[0]
        out, _ = RF.gatv2_aggregate(g, etv if th is not None else None, *leaves, ALPHA, SLOPE, keep=keep)
        out.backward(gout)
    return (out.detach(), leaves[0].grad, None if shared else leaves[1].grad, leaves[2].grad,
            leaves[3].grad if th is not None else None)


def _close(a, b, rtol=1e-10):
    return torch.allclose(a, b, rtol=rtol, atol=1e-12)


def _oracle_keep(drop, num_edges, heads):
    from oracle import attn_dropout_oracle as AO
    return torch.as_tensor(AO.keep_mask(drop.p, drop.key, num_edges, heads)).double()


class _MP:  # minimal monkeypatch stand-in
    @staticmethod
    def setattr(obj, name, val):
        setattr(obj, name, val)


def _worker(rank, world, port, ret, kind):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import test_attention_dropout_host as T
    from re_gnn_b200 import Graph, functional as RF, partition, synth
    T.install_dropout_shim(_MP)
    d, heads, dim = _graph(kind, synth)
    g = Graph(d['src'], d['dst'], d['num_nodes'])
    etv = g.etype_views(torch.as_tensor(d['etype']), d['num_relations'])
    bounds = partition.row_blocks(g.csr()['indptr'], world, balance='rows')
    rb, re = bounds[rank], bounds[rank + 1]
    fs, fd, gout, attn0, th0 = _inputs(d, heads, dim, 1)
    drop = RF.HashedDropout(P_DROP, RF.attn_dropout_key(4, 1, 0))
    keep = _oracle_keep(drop, d['src'].size, heads)
    ok = True
    # (relation term, one tensor for both sides, hashed dropout)
    for relational, shared, dropout in ((True, False, False), (False, False, False), (True, True, False),
                                        (True, False, True), (False, True, True)):
        th_ref = th0 if relational else None
        want = _reference(g, etv, fs, fd, gout, attn0, th_ref, shared, keep if dropout else None)
        if dropout:   # the mask changed the result
            ok = ok and not _close(want[0], _reference(g, etv, fs, fd, gout, attn0, th_ref, shared)[0])
        fso = fs[rb:re].clone().requires_grad_(True)
        fdo = fso if shared else fd[rb:re].clone().requires_grad_(True)
        attn = attn0.clone().requires_grad_(True)
        th = th0.clone().requires_grad_(True) if relational else None
        out = partition.head_sliced_gatv2(g, etv if relational else None, fso, fdo, attn, th, ALPHA, SLOPE, bounds, rank,
                                          dropout=drop if dropout else None)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads([attn] + ([th] if relational else []))
        good = (_close(out.detach(), want[0][rb:re], 1e-12) and _close(fso.grad, want[1][rb:re])
                and (shared or _close(fdo.grad, want[2][rb:re])) and _close(attn.grad, want[3])
                and (not relational or _close(th.grad, want[4])))
        if not good:
            print('rank', rank, 'case', (relational, shared, dropout), 'out',
                  float((out.detach() - want[0][rb:re]).abs().max()) if re > rb else 0.0, file=sys.stderr)
        ok = ok and good
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize('world,kind', [(2, 'imdb'), (3, 'empty_block')])
def test_head_sliced_gatv2_matches_single_process(world, kind):
    """Every rank's out, d_fs and d_fd rows and the summed d_attn / d_theta equal gatv2_aggregate: with and without the
    relation term, with one tensor for both sides, and with hashed dropout against the oracle's explicit mask.  At world
    size 3 the last rank owns no rows and still takes part in every all-to-all."""
    port = 21500 + (os.getpid() % 1500) + (0 if world == 2 else 1700)
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_worker, args=(world, port, ret, kind), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)


@pytest.fixture
def v2_ops(monkeypatch):
    import test_attention_dropout_host as T
    T.install_dropout_shim(monkeypatch)


@pytest.mark.parametrize('dropout', [False, True])
@pytest.mark.parametrize('parts', [1, 2, 4])
def test_virtual_head_slices(v2_ops, parts, dropout):
    """The per-rank slab compute for q = 0..P-1, stitched along the heads, is the full-H core."""
    from re_gnn_b200 import Graph, functional as RF, partition, synth
    d = synth.hetero_graph('acm', seed=3, scale=0.03)
    g = Graph(d['src'], d['dst'], d['num_nodes'])
    etv = g.etype_views(torch.as_tensor(d['etype']), d['num_relations'])
    fs, fd, gout, attn, th = _inputs(d, 4, 8, 2)
    drop = RF.HashedDropout(P_DROP, 77) if dropout else None
    want = _reference(g, etv, fs, fd, gout, attn, th, keep=_oracle_keep(drop, d['src'].size, 4) if dropout else None)
    got = partition._virtual_head_sliced_gatv2(g, etv, fs, fd, gout, attn, th, ALPHA, SLOPE, parts, dropout=drop)
    for i, (a, b) in enumerate(zip(got, want)):
        assert _close(a, b, 1e-12 if i == 0 else 1e-10), i


def test_head_sliced_gatv2_refusals(monkeypatch):
    """Refused before any exchange or kernel: H not divisible by P, uneven row blocks, mismatched feature shapes, an
    exchange of the wrong width or built without gatv2=True, an explicit keep mask, and a dropout that is not a
    HashedDropout."""
    from re_gnn_b200 import Graph, functional as RF, ops, partition

    def reached(*args, **kwargs):
        raise AssertionError('a refused call reached the exchange or a kernel')
    monkeypatch.setattr(partition, '_rows_to_head_slabs', reached)
    monkeypatch.setattr(ops, 'gatv2_fwd', reached)
    g = Graph(np.array([0, 1, 2, 3]), np.array([1, 2, 3, 0]), 4)

    def call(heads=4, dim=8, bounds=(0, 2, 4), rank=0, fd_rows=None, **kw):
        rows = bounds[rank + 1] - bounds[rank]
        f = torch.zeros(rows, heads, dim)
        fd = torch.zeros(rows if fd_rows is None else fd_rows, heads, dim)
        return partition.head_sliced_gatv2(g, None, f, fd, torch.zeros(1, heads, dim), None, ALPHA, SLOPE,
                                           list(bounds), rank, **kw)
    with pytest.raises(ValueError, match='divisible'):
        call(heads=3)
    with pytest.raises(ValueError, match='equal row blocks'):
        call(heads=6, bounds=(0, 1, 3, 4))
    with pytest.raises(ValueError, match='fd_own'):
        call(fd_rows=3)
    for xch in (types.SimpleNamespace(feat=32, gatv2=False), types.SimpleNamespace(feat=64, gatv2=True)):
        with pytest.raises(ValueError, match='gatv2=True'):
            call(exchange=xch)
    with pytest.raises(ValueError, match='HashedDropout'):
        call(keep=torch.ones(4, 4))
    with pytest.raises(TypeError, match='HashedDropout'):
        call(dropout=0.1)
    with pytest.raises(AssertionError, match='reached'):   # the stand-ins are in place: a valid call gets past the checks
        call(exchange=types.SimpleNamespace(feat=32, gatv2=True), dropout=RF.HashedDropout(0.1, 1))
