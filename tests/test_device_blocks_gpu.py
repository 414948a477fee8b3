"""Device-built minibatch blocks on the B200: ``NeighborSampler.sample`` (regnn_sample_layer) and ``Block.prebuilt``
(regnn_block_csr_build) against the torch relabelling they replace (``NeighborSampler.reference_sample``) and against
``Graph(src, dst, n)`` of the same block, bit for bit; ``mag.train_step`` with prebuilt blocks against the
plain-``adjs`` path; out-of-range types; host synchronisations."""
import copy
import os
import traceback
import warnings

import numpy as np
import pytest
import torch

from oracle import sampler_oracle as S

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def reference_block(block, edge_type, node_type_targets, num_edge_types, self_loop_type, num_relations):
    """What ``mag.REGCNConv.build_block`` + ``Graph.etype_views`` build from the block's edge list."""
    from re_gnn_b200 import mag
    conv = mag.REGCNConv(4, 4, 1, num_edge_types, self_loop_type=self_loop_type)
    g, etype1 = conv.build_block(block.edge_index, edge_type[block.eid], node_type_targets, block.n_src, block.n_dst)
    return g, etype1, g.etype_views(etype1, num_relations)


def assert_same_split(a, b, what):
    assert (a is None) == (b is None), what
    if a is not None:
        for k in ('long_rows', 'frag_ptr', 'frag_row', 'frag_begin'):
            assert torch.equal(a[k], b[k]), '%s %s' % (what, k)
        assert (a['struct'].num_long, a['struct'].num_frags) == (b['struct'].num_long, b['struct'].num_frags), what


def assert_prebuilt_matches(block, n_id, edge_type, node_type, num_edge_types, num_node_types):
    for slt in (1, 2):
        r = num_edge_types + (num_node_types if slt == 2 else 0)
        g, etype1 = block.prebuilt(edge_type, node_type, num_edge_types, slt, r)
        g_ref, etype1_ref, (et_csr, et_t, counts) = reference_block(block, edge_type, node_type[n_id[:block.n_dst]],
                                                                    num_edge_types, slt, r)
        assert torch.equal(etype1, etype1_ref), slt
        assert g.number_of_nodes() == g_ref.number_of_nodes() and g.number_of_edges() == g_ref.number_of_edges()
        for x, y in zip(g.edges(), g_ref.edges()):
            assert torch.equal(x, y), slt
        c, c_ref = g.csr(), g_ref.csr()
        for k in ('indptr', 'indices', 'eid', 'row', 'indptr_t', 'indices_t', 'slot_t'):
            assert torch.equal(c[k], c_ref[k]), (slt, k)
        assert_same_split(c['split'], c_ref['split'], 'split %d' % slt)
        assert_same_split(c['split_t'], c_ref['split_t'], 'split_t %d' % slt)
        v = g.etype_views(etype1, r)      # served from the prefilled cache
        assert torch.equal(v[0], et_csr) and torch.equal(v[1], et_t), slt
        assert (v[2] is None) == (counts is None) and (counts is None or torch.equal(v[2], counts)), slt
        assert torch.equal(g.in_degrees(), g_ref.in_degrees())
        zero = bool((g_ref.in_degrees() == 0).any())
        assert g.has_zero_in_degree() == zero


@pytest.fixture(scope='module')
def mag_graph():
    from re_gnn_b200 import Graph, synth
    d = synth.hetero_graph('mag')
    n = d['num_nodes']
    g = Graph(d['src'][:-n], d['dst'][:-n], n).to(DEV)
    g.csr()
    edge_type = (torch.as_tensor(d['etype'][:-n]) - 1).to(DEV)
    node_type = torch.as_tensor(d['ntype']).to(torch.int64).to(DEV)
    return d, g, edge_type, node_type


def test_mag_batches_bit_identical_to_previous_path(mag_graph):
    from re_gnn_b200.sampling import NeighborSampler
    d, g, edge_type, node_type = mag_graph
    net, nnt = d['num_etype'], len(d['type_sizes'])
    sampler = NeighborSampler(g, [25, 20], seed=123)
    gen = torch.Generator(device=DEV).manual_seed(7)
    hub_splits = 0
    for batch in range(50):
        seeds = torch.randperm(d['type_sizes'][0], device=DEV, generator=gen)[:512]
        n_id, blocks = sampler.sample(seeds, epoch=1, batch=batch)
        n_ref, blocks_ref = sampler.reference_sample(seeds, epoch=1, batch=batch)   # the torch relabelling
        assert torch.equal(n_id, n_ref), batch
        assert len(blocks) == len(blocks_ref)
        for b, r in zip(blocks, blocks_ref):
            assert (b.n_src, b.n_dst) == (r.n_src, r.n_dst), batch
            assert torch.equal(b.src, r.src) and torch.equal(b.dst, r.dst) and torch.equal(b.eid, r.eid), batch
            assert b.edge_index.dtype == torch.int64 and b.size == r.size
            assert_prebuilt_matches(b, n_id, edge_type, node_type, net, nnt)
            hub_splits += b.prebuilt(edge_type, node_type, net, 1, net)[0].csr()['split_t'] is not None
    print('blocks whose transposed view has rows over 256 slots: %d of 100' % hub_splits)


def edge_case_graph():
    """Nodes 0..9: a ring fed only from itself (a batch of them has no new sources).  Node 10: a hub feeding
    20..419 (more than 256 out-edges in one block).  Nodes 20..419 also get 0..2 in-edges from 430..449 (fan-out 3
    above most in-degrees).  Nodes 450..459: no in-edges.  Node 470: 400 in-edges from 0..399 (an in-view row over
    256 slots at fan-out 300, and at fan-out 256 once its self loop is appended)."""
    rng = np.random.RandomState(5)
    src, dst = [], []
    for v in range(10):
        src += [(v + 1) % 10, (v + 3) % 10]
        dst += [v, v]
    for v in range(20, 420):
        src.append(10)
        dst.append(v)
        for _ in range(rng.randint(0, 3)):
            src.append(430 + rng.randint(0, 20))
            dst.append(v)
    src += list(range(20, 40))
    dst += [10] * 20
    src += list(range(400))
    dst += [470] * 400
    return np.array(src), np.array(dst), 480


EDGE_CASES = {'hub_and_empty_targets': (np.concatenate([np.arange(20, 420), np.arange(450, 460)]), [3, 2]),
              'no_new_sources': (np.arange(10), [3, 2]),
              'wide_row_fanout_256': (np.array([470, 5, 30]), [256]),
              'wide_row_fanout_300': (np.array([470, 5, 30]), [300, 2])}


@pytest.mark.parametrize('case', sorted(EDGE_CASES))
def test_edge_cases_against_oracle_and_graph(case):
    from re_gnn_b200 import Graph
    from re_gnn_b200.sampling import NeighborSampler
    src, dst, n = edge_case_graph()
    g = Graph(src, dst, n).to(DEV)
    edge_type = torch.as_tensor(np.arange(len(src)) % 3, device=DEV)
    node_type = torch.as_tensor(np.arange(n) % 2, device=DEV)
    seeds, fanouts = EDGE_CASES[case]
    sampler = NeighborSampler(g, fanouts, seed=9)
    n_id, blocks = sampler.sample(torch.as_tensor(seeds, device=DEV), epoch=0, batch=2)
    c = {k: v.cpu().numpy() for k, v in g.csr().items() if torch.is_tensor(v)}
    n_or, blocks_or = S.sample_blocks(c, seeds, fanouts, seed=9, epoch=0, rank=0, batch=2)
    assert np.array_equal(n_id.cpu().numpy(), n_or)
    for b, (s_l, d_l, e, n_src, n_dst) in zip(blocks, blocks_or):
        assert (b.n_src, b.n_dst) == (n_src, n_dst)
        assert np.array_equal(b.src.cpu().numpy(), s_l) and np.array_equal(b.dst.cpu().numpy(), d_l)
        assert np.array_equal(b.eid.cpu().numpy(), e)
        assert_prebuilt_matches(b, n_id, edge_type, node_type, 3, 2)
    inner = blocks[-1]
    in_split = lambda slt: inner.prebuilt(edge_type, node_type, 3, slt, 5)[0].csr()['split']   # noqa: E731
    if case == 'no_new_sources':
        assert inner.n_src == inner.n_dst == 10
    elif case == 'wide_row_fanout_256':
        assert in_split(1) is None and in_split(2)['struct'].num_frags == 2      # 256 sampled slots + the loop
    elif case == 'wide_row_fanout_300':
        assert in_split(1)['struct'].num_frags == 2 and in_split(2)['struct'].num_frags == 2
    else:
        assert inner.prebuilt(edge_type, node_type, 3, 1, 3)[0].csr()['split_t'] is not None    # the hub's fragments
        assert inner.prebuilt(edge_type, node_type, 3, 1, 3)[0].has_zero_in_degree()            # 450..459


def test_out_of_range_type_is_reported_by_the_next_batch():
    from re_gnn_b200 import Graph
    from re_gnn_b200.sampling import NeighborSampler
    src, dst, n = edge_case_graph()
    g = Graph(src, dst, n).to(DEV)
    edge_type = torch.as_tensor(np.arange(len(src)) % 3, device=DEV)
    node_type = torch.as_tensor(np.arange(n) % 2, device=DEV)
    seeds = torch.arange(20, 60, device=DEV)
    sampler = NeighborSampler(g, [3, 2], seed=9)
    _, blocks = sampler.sample(seeds)
    g_bad, etype1 = blocks[-1].prebuilt(edge_type, node_type, 3, 1, 2)     # edge types go up to 2: outside [0, 2)
    et_csr, et_t, counts = g_bad.etype_views(etype1, 2)
    assert int(et_csr.max()) < 2 and int(et_t.max()) < 2 and int(counts.sum()) == g_bad.number_of_edges()
    with pytest.raises(RuntimeError, match='outside'):
        sampler.sample(seeds, batch=1)
    n_id, blocks = sampler.sample(seeds, batch=1)                            # reported once; the sampler goes on
    assert_prebuilt_matches(blocks[-1], n_id, edge_type, node_type, 3, 2)


def _mag_model_setup(kind, seed=0):
    from re_gnn_b200 import Graph, mag, synth
    from re_gnn_b200.sampling import NeighborSampler
    d = synth.hetero_graph('mag', seed=4, scale=0.02)
    n, net, sizes = d['num_nodes'], d['num_etype'], d['type_sizes']
    nnt = len(sizes)
    g = Graph(d['src'], d['dst'], n).to(DEV)
    edge_type = (torch.as_tensor(d['etype']) - 1).to(DEV)
    node_type = torch.as_tensor(d['ntype']).to(DEV)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    local_idx = torch.as_tensor(np.arange(n) - offs[d['ntype']]).to(DEV)
    torch.manual_seed(seed)
    x_dict = {k: torch.randn(sizes[k], 32, device=DEV) for k in range(nnt)}
    labels = torch.randint(0, 7, (n,), device=DEV)
    heads = 1 if kind == 'regcn' else 2
    model = mag.REGNN(32, 16, 7, heads, 2, 100.0, 0.5, {k: 32 for k in range(nnt)}, net, residual=True, no_re=False,
                      model=kind).to(DEV)
    return NeighborSampler(g, [10, 5], seed=3), model, labels, x_dict, edge_type, node_type, local_idx, sizes[0]


@pytest.mark.parametrize('kind', ['regcn', 'regat', 'regatv2'])
def test_train_step_with_prebuilt_blocks_is_bit_equal(kind):
    import torch.nn.functional as F
    from re_gnn_b200 import mag
    sampler, model, labels, x_dict, edge_type, node_type, local_idx, n_papers = _mag_model_setup(kind)
    plain = copy.deepcopy(model)
    opt_a = torch.optim.Adam(model.parameters(), lr=1e-2)
    opt_b = torch.optim.Adam(plain.parameters(), lr=1e-2)
    seeds = torch.randperm(n_papers, device=DEV)[:128]
    for batch in range(3):
        torch.manual_seed(100 + batch)
        loss_a, ne = mag.train_step(model, opt_a, sampler, seeds, labels[seeds], x_dict, edge_type, node_type, local_idx,
                                    epoch=0, batch=batch)
        torch.manual_seed(100 + batch)
        n_id, blocks = sampler.sample(seeds, epoch=0, batch=batch)
        adjs = [(b.edge_index, b.eid, b.size) for b in blocks]
        opt_b.zero_grad(set_to_none=True)
        loss_b = F.nll_loss(plain(n_id, x_dict, adjs, edge_type, node_type, local_idx), labels[seeds])
        loss_b.backward()
        opt_b.step()
        assert ne == sum(int(b.src.numel()) for b in blocks)
        assert torch.equal(loss_a, loss_b.detach()), (batch, float(loss_a), float(loss_b))
        for (k, p), q in zip(model.named_parameters(), plain.parameters()):
            assert (p.grad is None) == (q.grad is None), k
            assert p.grad is None or torch.equal(p.grad, q.grad), (batch, k)
            assert torch.equal(p, q), (batch, k)


def _count_syncs(fn):
    """Runs fn under torch's sync debug mode -> (result, [package / optimizer line that synchronised, per sync])."""
    where = []

    def record(message, category, filename, lineno, file=None, line=None):
        if 'called a synchronizing CUDA operation' in str(message):
            frames = [f for f in traceback.extract_stack()[:-1] if 're_gnn_b200' in f.filename or 'torch/optim' in f.filename]
            f = frames[-1] if frames else None
            where.append('%s:%d' % (os.path.basename(f.filename), f.lineno) if f else '?')

    with warnings.catch_warnings():
        warnings.simplefilter('always')
        warnings.showwarning = record
        torch.cuda.set_sync_debug_mode('warn')
        try:
            out = fn()
        finally:
            torch.cuda.set_sync_debug_mode(0)
    return out, where


def test_one_host_synchronisation_per_batch(mag_graph):
    from re_gnn_b200.sampling import NeighborSampler
    d, g, edge_type, node_type = mag_graph
    net, nnt = d['num_etype'], len(d['type_sizes'])
    sampler = NeighborSampler(g, [25, 20], seed=1)
    seeds = torch.randperm(d['type_sizes'][0], device=DEV)[:512]
    sampler.sample(seeds)          # first call allocates the sampler's maps

    def assemble():
        n_id, blocks = sampler.sample(seeds, epoch=0, batch=1)
        return [b.prebuilt(edge_type, node_type, net, 2, net + nnt) for b in blocks]

    _, syncs = _count_syncs(assemble)
    assert syncs == ['sampling.py:%d' % _SAMPLE_SYNC_LINE], syncs

    # the entry points themselves never wait: with the stream held busy, they return while it is still running
    torch.cuda.synchronize()
    torch.cuda._sleep(400_000_000)
    sampler.sample_on_device(seeds, epoch=0, batch=2)
    assert not torch.cuda.current_stream().query(), 'regnn_sample_layer waited for the device'
    torch.cuda.synchronize()
    n_id, blocks = sampler.sample(seeds, epoch=0, batch=2)
    torch.cuda.synchronize()
    torch.cuda._sleep(400_000_000)
    for b in blocks:
        b.prebuilt(edge_type, node_type, net, 2, net + nnt)
    assert not torch.cuda.current_stream().query(), 'regnn_block_csr_build waited for the device'
    torch.cuda.synchronize()


def _sample_sync_line():
    import inspect
    from re_gnn_b200.sampling import NeighborSampler
    lines, first = inspect.getsourcelines(NeighborSampler.sample)
    return first + next(i for i, l in enumerate(lines) if 'info.cpu()' in l)


_SAMPLE_SYNC_LINE = _sample_sync_line()


def test_synchronisations_of_a_training_step():
    """Sampling and block assembly make exactly one host synchronisation; the rest of the step is reported."""
    from re_gnn_b200 import mag
    for kind in ('regcn', 'regat'):
        sampler, model, labels, x_dict, edge_type, node_type, local_idx, n_papers = _mag_model_setup(kind)
        opt = torch.optim.Adam(model.parameters(), lr=1e-2)
        seeds = torch.randperm(n_papers, device=DEV)[:128]
        y = labels[seeds]
        for batch in range(2):
            mag.train_step(model, opt, sampler, seeds, y, x_dict, edge_type, node_type, local_idx, 0, batch)
        torch.cuda.synchronize()
        _, syncs = _count_syncs(lambda: mag.train_step(model, opt, sampler, seeds, y, x_dict, edge_type, node_type,
                                                       local_idx, 0, 5))
        print('%s: %d host synchronisations in train_step, at %s' % (kind, len(syncs), syncs))
        assert syncs.count('sampling.py:%d' % _SAMPLE_SYNC_LINE) == 1
