"""GraphSAINT subgraphs built on the B200: ``SaintRandomWalkSampler.sample`` / ``sample_block``
(regnn_induced_subgraph_count / _fill) against the torch path they replace (``reference_sample``) and the sampler
oracle, bit for bit; ``Block.prebuilt`` of the subgraph against ``Graph(src, dst, n)`` + ``etype_views``;
``mag.saint_train_step`` against the same steps on the torch path; out-of-range types; host synchronisations."""
import copy
import ctypes
import os
import traceback
import warnings

import numpy as np
import pytest
import torch

from oracle import sampler_oracle as S

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(autouse=True)
def _restore_global_rng():
    """These tests reseed torch's generators; test modules that run later initialise their layers from them."""
    with torch.random.fork_rng(devices=[0]):
        yield


def assert_same_split(a, b, what):
    assert (a is None) == (b is None), what
    if a is not None:
        for k in ('long_rows', 'frag_ptr', 'frag_row', 'frag_begin'):
            assert torch.equal(a[k], b[k]), '%s %s' % (what, k)
        assert (a['struct'].num_long, a['struct'].num_frags) == (b['struct'].num_long, b['struct'].num_frags), what


def assert_prebuilt_matches(block, edge_type, node_type, num_relations):
    """``Block.prebuilt`` without self loops against ``Graph(src, dst, n_sub)`` + ``etype_views`` of the same edges."""
    from re_gnn_b200 import Graph
    g, etype1 = block.prebuilt(edge_type, node_type, num_relations, 1, num_relations)
    g_ref = Graph(block.src, block.dst, block.n_src)
    etype1_ref = (edge_type[block.eid] + 1).contiguous()
    et_csr, et_t, counts = g_ref.etype_views(etype1_ref, num_relations)
    assert torch.equal(etype1, etype1_ref)
    assert g.number_of_nodes() == g_ref.number_of_nodes() and g.number_of_edges() == g_ref.number_of_edges()
    for x, y in zip(g.edges(), g_ref.edges()):
        assert torch.equal(x, y)
    c, c_ref = g.csr(), g_ref.csr()
    for k in ('indptr', 'indices', 'eid', 'row', 'indptr_t', 'indices_t', 'slot_t'):
        assert torch.equal(c[k], c_ref[k]), k
    assert_same_split(c['split'], c_ref['split'], 'split')
    assert_same_split(c['split_t'], c_ref['split_t'], 'split_t')
    v = g.etype_views(etype1, num_relations)      # served from the prefilled cache
    assert torch.equal(v[0], et_csr) and torch.equal(v[1], et_t)
    assert (v[2] is None) == (counts is None) and (counts is None or torch.equal(v[2], counts))
    assert torch.equal(g.in_degrees(), g_ref.in_degrees())
    assert g.has_zero_in_degree() == bool((g_ref.in_degrees() == 0).any())
    return g


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


def test_mag_batches_bit_identical_to_torch_path(mag_graph):
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    d, g, edge_type, node_type = mag_graph
    net = d['num_etype']
    sampler = SaintRandomWalkSampler(g, roots=20000, walk_length=2, seed=123)
    indptr = g.csr()['indptr'].to(torch.int64)
    fragment_batches = long_row_batches = 0
    for batch in range(24):
        n_ref, ei_ref, eid_ref = sampler.reference_sample(epoch=1, batch=batch)
        n_id, ei, eid = sampler.sample(epoch=1, batch=batch)
        assert torch.equal(n_id, n_ref) and torch.equal(ei, ei_ref) and torch.equal(eid, eid_ref), batch
        n_b, block = sampler.sample_block(epoch=1, batch=batch)
        assert torch.equal(n_b, n_ref) and (block.n_src, block.n_dst) == (n_ref.numel(), n_ref.numel())
        assert torch.equal(block.src, ei_ref[0]) and torch.equal(block.dst, ei_ref[1]) and torch.equal(block.eid, eid_ref)
        g_sub = assert_prebuilt_matches(block, edge_type, node_type, net)
        candidates = int((indptr[n_ref + 1] - indptr[n_ref]).sum())
        longest = int(g_sub.in_degrees().max()) if block.n_src else 0
        fragment_batches += int((indptr[n_ref + 1] - indptr[n_ref]).max()) > 256    # rows cut into 256-slot fragments
        long_row_batches += longest > 256
        print('batch %2d: %d nodes, %d candidate slots, %d induced edges, longest subgraph row %d'
              % (batch, block.n_src, candidates, block.src.numel(), longest))
    assert fragment_batches > 0, 'no batch visited a row of more than 256 in-edges'
    assert long_row_batches > 0, 'no subgraph has a row of more than 256 in-edges'


def edge_case_graph():
    """Nodes 0..9: a ring.  Node 10 feeds 20..419 (a hub source), 420..429 and 450..469 feed them and have no in-edges,
    430..449 and 471..479 have no edges.  Node 470 has 400 in-edges from 0..399 (a row of two fragments) and, like
    400..419, no out-edges: walkers that reach them stay put."""
    rng = np.random.RandomState(5)
    src, dst = [], []
    for v in range(10):
        src += [(v + 1) % 10, (v + 3) % 10]
        dst += [v, v]
    src += [10] * 400
    dst += list(range(20, 420))
    src += list(rng.randint(420, 430, 300))
    dst += list(rng.randint(20, 420, 300))
    src += list(range(20, 40)) + list(range(400))
    dst += [10] * 20 + [470] * 400
    src += list(range(450, 470))
    dst += list(rng.randint(0, 10, 20))
    return np.array(src), np.array(dst), 480


EDGE_CASES = {'walk_length_0': (50, 0), 'one_root': (1, 3), 'roots_over_n': (2000, 2), 'short_walks': (60, 1)}


@pytest.mark.parametrize('case', sorted(EDGE_CASES))
def test_edge_cases_against_oracle(case):
    from re_gnn_b200 import Graph
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    src, dst, n = edge_case_graph()
    g = Graph(src, dst, n).to(DEV)
    edge_type = torch.as_tensor(np.arange(len(src)) % 3, device=DEV)
    node_type = torch.zeros(n, dtype=torch.int64, device=DEV)
    roots, wl = EDGE_CASES[case]
    sampler = SaintRandomWalkSampler(g, roots=roots, walk_length=wl, seed=9)
    c = {k: v.cpu().numpy() for k, v in g.csr().items() if torch.is_tensor(v)}
    for batch in range(3):
        n_id, block = sampler.sample_block(epoch=0, batch=batch)
        w_nid, w_s, w_d, w_e = S.saint_subgraph(c, n, roots, wl, seed=9, epoch=0, rank=0, batch=batch)
        assert np.array_equal(n_id.cpu().numpy(), w_nid), batch
        assert np.array_equal(block.src.cpu().numpy(), w_s) and np.array_equal(block.dst.cpu().numpy(), w_d)
        assert np.array_equal(block.eid.cpu().numpy(), w_e)
        assert_prebuilt_matches(block, edge_type, node_type, 3)
    assert not sampler._maps[0].any()          # the flag map comes back all zero


def test_every_node_listed_gives_the_graph_itself():
    from re_gnn_b200 import Graph
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    src, dst, n = edge_case_graph()
    g = Graph(src, dst, n).to(DEV)
    c = g.csr()
    sampler = SaintRandomWalkSampler(g, roots=1, walk_length=1)
    nodes = torch.cat([torch.arange(n - 1, -1, -1, device=DEV), torch.arange(0, n, 7, device=DEV)])
    n_id, block = sampler.induced_block(nodes)
    assert torch.equal(n_id, torch.arange(n, device=DEV))
    assert torch.equal(block.src, c['indices'].long()) and torch.equal(block.dst, c['row'].long())
    assert torch.equal(block.eid, c['eid'].long())
    edge_type = torch.as_tensor(np.arange(len(src)) % 3, device=DEV)
    g_sub = assert_prebuilt_matches(block, edge_type, torch.zeros(n, dtype=torch.int64, device=DEV), 3)
    assert torch.equal(g_sub.csr()['indptr'], c['indptr']) and g_sub.csr()['split'] is not None   # node 470
    assert g_sub.csr()['split_t'] is not None                                                     # node 10
    assert not sampler._maps[0].any()


def test_graph_without_edges():
    from re_gnn_b200 import Graph
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    g = Graph(np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64), 9).to(DEV)
    sampler = SaintRandomWalkSampler(g, roots=5, walk_length=2, seed=1)
    c = {k: v.cpu().numpy() for k, v in g.csr().items() if torch.is_tensor(v)}
    n_id, block = sampler.sample_block(epoch=0, batch=0)
    w_nid, w_s, _, _ = S.saint_subgraph(c, 9, 5, 2, seed=1, epoch=0, rank=0, batch=0)
    assert np.array_equal(n_id.cpu().numpy(), w_nid) and block.src.numel() == 0 == len(w_s)
    empty = torch.zeros(0, dtype=torch.int64, device=DEV)
    gb = assert_prebuilt_matches(block, empty, torch.zeros(9, dtype=torch.int64, device=DEV), 2)
    assert gb.has_zero_in_degree()


def test_out_of_range_type_is_reported_by_the_next_batch():
    from re_gnn_b200 import Graph
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    src, dst, n = edge_case_graph()
    g = Graph(src, dst, n).to(DEV)
    edge_type = torch.as_tensor(np.arange(len(src)) % 3, device=DEV)
    node_type = torch.zeros(n, dtype=torch.int64, device=DEV)
    sampler = SaintRandomWalkSampler(g, roots=300, walk_length=2, seed=4)
    _, block = sampler.sample_block()
    g_bad, etype1 = block.prebuilt(edge_type, node_type, 2, 1, 2)       # edge types go up to 2: outside [0, 2)
    assert int(etype1.max()) == 3
    et_csr, et_t, counts = g_bad.etype_views(etype1, 2)
    assert int(et_csr.max()) < 2 and int(et_t.max()) < 2 and int(counts.sum()) == g_bad.number_of_edges()
    with pytest.raises(RuntimeError, match='outside'):
        sampler.sample_block(batch=1)
    assert not sampler._maps[0].any()
    n_id, block = sampler.sample_block(batch=1)                          # reported once; the sampler goes on
    assert_prebuilt_matches(block, edge_type, node_type, 3)


def _saint_setup(seed=0):
    from re_gnn_b200 import Graph, mag, synth
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    d = synth.hetero_graph('mag', seed=4, scale=0.02)
    n, net, sizes = d['num_nodes'], d['num_etype'], d['type_sizes']
    nnt = len(sizes)
    g = Graph(d['src'][:-n], d['dst'][:-n], n).to(DEV)
    edge_type = (torch.as_tensor(d['etype'][:-n]) - 1).to(DEV)
    node_type = torch.as_tensor(d['ntype']).to(DEV)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    local_idx = torch.as_tensor(np.arange(n) - offs[d['ntype']]).to(DEV)
    torch.manual_seed(seed)
    x_dict = {k: torch.randn(sizes[k], 32, device=DEV) for k in range(nnt)}
    labels = torch.randint(0, 7, (n,), device=DEV)
    train_mask = (node_type == 0) & (local_idx < int(sizes[0] * 0.8))
    model = mag.SaintREGCN(32, 16, 7, 2, 100.0, 0.5, {k: 32 for k in range(nnt)}, net, use_bn=True, residual=True,
                           gcn=False).to(DEV)
    sampler = SaintRandomWalkSampler(g, roots=600, walk_length=2, seed=3)
    return sampler, model, labels, train_mask, x_dict, edge_type, node_type, local_idx


def test_saint_train_step_is_bit_equal_to_the_torch_path():
    import torch.nn.functional as F
    from re_gnn_b200 import mag
    sampler, model, labels, train_mask, x_dict, edge_type, node_type, local_idx = _saint_setup()
    plain = copy.deepcopy(model)
    opt_a = torch.optim.Adam(model.parameters(), lr=1e-2)
    opt_b = torch.optim.Adam(plain.parameters(), lr=1e-2)
    for batch in range(4):
        torch.manual_seed(100 + batch)          # the model's feature dropout draws from torch's RNG
        loss_a, ne = mag.saint_train_step(model, opt_a, sampler, labels, train_mask, x_dict, edge_type, node_type,
                                          local_idx, epoch=0, batch=batch)
        torch.manual_seed(100 + batch)
        n_id, ei, eid = sampler.reference_sample(epoch=0, batch=batch)
        opt_b.zero_grad(set_to_none=True)
        out = plain(x_dict, ei, edge_type[eid], node_type[n_id], local_idx[n_id])
        mask = train_mask[n_id]
        loss_b = F.nll_loss(out[mask], labels[n_id][mask])
        loss_b.backward()
        opt_b.step()
        assert ne == ei.shape[1]
        assert torch.equal(loss_a, loss_b.detach()), (batch, float(loss_a), float(loss_b))
        for (k, p), q in zip(model.named_parameters(), plain.parameters()):
            assert (p.grad is None) == (q.grad is None), k
            assert p.grad is None or torch.equal(p.grad, q.grad), (batch, k)
            assert torch.equal(p, q), (batch, k)


def test_softmax_layer_on_a_prebuilt_subgraph():
    from re_gnn_b200 import mag
    sampler, _, _, _, _, edge_type, node_type, _ = _saint_setup()
    net = int(edge_type.max()) + 1
    conv = mag.SaintREGCNConv(24, 8, 4, net, 100.0, use_softmax=True).to(DEV)
    with torch.no_grad():
        conv.relation_weight.copy_(torch.linspace(-0.5, 1.5, net) / 100.0)
    n_id, block = sampler.sample_block(epoch=2, batch=1)
    x = torch.randn(block.n_src, 24, device=DEV)
    et = edge_type[block.eid]
    outs, grads = [], []
    for use_block in (True, False):
        conv.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(True)
        if use_block:
            out = conv(xi, None, et, block=block.prebuilt(edge_type, node_type, net, 1, net))
        else:
            out = conv(xi, block.edge_index, et)
        out.backward(torch.ones_like(out))
        outs.append(out.detach())
        grads.append([xi.grad] + [p.grad for p in conv.parameters()])
    assert torch.equal(outs[0], outs[1])
    for a, b in zip(*grads):
        assert torch.equal(a, b)


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


def _sample_sync_line():
    import inspect
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    lines, first = inspect.getsourcelines(SaintRandomWalkSampler.induced_block)
    return 'sampling.py:%d' % (first + next(i for i, l in enumerate(lines) if 'info.cpu()' in l))


def test_one_host_synchronisation_per_batch(mag_graph):
    from re_gnn_b200 import _lib
    from re_gnn_b200.graph import _ptr
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    d, g, edge_type, node_type = mag_graph
    net = d['num_etype']
    sampler = SaintRandomWalkSampler(g, roots=20000, walk_length=2, seed=1)
    sampler.sample_block()          # first call allocates the sampler's maps

    def assemble():
        n_id, block = sampler.sample_block(epoch=0, batch=1)
        return block.prebuilt(edge_type, node_type, net, 1, net)

    _, syncs = _count_syncs(assemble)
    assert syncs == [_sample_sync_line()], syncs

    # the entry points themselves never wait: with the stream held busy, they return while it is still running
    lib, c = _lib.load(), g.csr()
    n, e = g.number_of_nodes(), g.number_of_edges()
    nodes = sampler.walks(sampler._key(0, 2)).view(-1)
    rows = min(n, nodes.numel())
    ws_bytes = lib.regnn_induced_subgraph_workspace_bytes(n, e, nodes.numel())
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    flags = torch.zeros(n, dtype=torch.int32, device=DEV)
    n_id, hist = torch.empty(rows, dtype=torch.int64, device=DEV), torch.empty(rows, dtype=torch.int32, device=DEV)
    row_off, info = torch.empty(rows + 1, dtype=torch.int32, device=DEV), torch.empty(16, dtype=torch.int32, device=DEV)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    torch.cuda._sleep(400_000_000)
    assert lib.regnn_induced_subgraph_count(_ptr(c['indptr']), _ptr(c['indices']), n, e, _ptr(nodes), nodes.numel(), 256,
                                            _ptr(flags), _ptr(n_id), _ptr(row_off), _ptr(hist), _ptr(info), _ptr(ws),
                                            ws_bytes, stream) == 0
    assert not torch.cuda.current_stream().query(), 'regnn_induced_subgraph_count waited for the device'
    torch.cuda.synchronize()
    n_sub, e_sub = int(info[0]), int(info[1])
    out = [torch.empty(max(e_sub, 1), dtype=torch.int64, device=DEV) for _ in range(3)]
    torch.cuda._sleep(400_000_000)
    assert lib.regnn_induced_subgraph_fill(_ptr(c['indptr']), _ptr(c['indices']), _ptr(c['eid']), n, e, nodes.numel(),
                                           _ptr(flags), _ptr(n_id), n_sub, e_sub, *[_ptr(t) for t in out], _ptr(ws),
                                           ws_bytes, stream) == 0
    assert not torch.cuda.current_stream().query(), 'regnn_induced_subgraph_fill waited for the device'
    torch.cuda.synchronize()
    assert not flags.any()
    n_ref, ei_ref, eid_ref = sampler.reference_sample(epoch=0, batch=2)
    assert torch.equal(n_id[:n_sub], n_ref) and torch.equal(out[0][:e_sub], ei_ref[0])
    assert torch.equal(out[1][:e_sub], ei_ref[1]) and torch.equal(out[2][:e_sub], eid_ref)
    _, block = sampler.sample_block(epoch=0, batch=2)
    torch.cuda.synchronize()
    torch.cuda._sleep(400_000_000)
    block.prebuilt(edge_type, node_type, net, 1, net)
    assert not torch.cuda.current_stream().query(), 'Block.prebuilt waited for the device'
    torch.cuda.synchronize()


def test_synchronisations_of_a_saint_training_step():
    """Sampling and block assembly make exactly one host synchronisation; the rest of the step is reported."""
    from re_gnn_b200 import mag
    sampler, model, labels, train_mask, x_dict, edge_type, node_type, local_idx = _saint_setup()
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    for batch in range(2):
        mag.saint_train_step(model, opt, sampler, labels, train_mask, x_dict, edge_type, node_type, local_idx, 0, batch)
    torch.cuda.synchronize()
    _, syncs = _count_syncs(lambda: mag.saint_train_step(model, opt, sampler, labels, train_mask, x_dict, edge_type,
                                                         node_type, local_idx, 0, 5))
    print('%d host synchronisations in saint_train_step, at %s' % (len(syncs), syncs))
    assert syncs.count(_sample_sync_line()) == 1
