"""Device-built minibatch blocks without a GPU: a numpy restatement of regnn_sample_layer's relabelling (position
map + scan of "new source" flags) and of regnn_block_csr_build's arrays, checked against oracle/sampler_oracle.py
and oracle/csr_oracle.py; the host logic of ``Graph.from_csr`` and of the known-size row split."""
import numpy as np
import pytest
import torch

from oracle import csr_oracle, sampler_oracle as S
from re_gnn_b200 import synth

UNMAPPED = 0x7fffffff


def sample_layer_np(c, targets, fanout, key, pos_map, flags):
    """regnn_sample_layer, kernel by kernel."""
    indptr, indices, eid = c['indptr'], c['indices'], c['eid']
    t = len(targets)
    for i, v in enumerate(targets):                                  # frontier_rows_kernel
        pos_map[v] = min(pos_map[v], i)
    k = np.minimum(indptr[targets + 1] - indptr[targets], fanout)
    row_off = np.concatenate([[0], np.cumsum(k)]).astype(np.int64)   # in-place exclusive scan, entry t = E
    slots = S.sample_slots(indptr, targets, fanout, key)             # frontier_slots_kernel
    e_src, dst_local, edge_id = [], [], []
    for i in range(t):
        for j in range(k[i]):
            u = indices[slots[i, j]]
            e_src.append(u)
            dst_local.append(i)
            edge_id.append(eid[slots[i, j]])
            if pos_map[u] == UNMAPPED:
                flags[u] = 1
    excl = np.concatenate([[0], np.cumsum(flags)[:-1]])              # scan over the flags in global-id order
    n_src = t + int(excl[-1] + flags[-1])
    new_n_id = np.empty(n_src, dtype=np.int64)
    new_n_id[:t] = targets
    src_local = np.empty(len(e_src), dtype=np.int64)
    for e, u in enumerate(e_src):                                    # frontier_relabel_kernel
        p = pos_map[u]
        if p == UNMAPPED:
            p = t + excl[u]
            new_n_id[p] = u
        src_local[e] = p
    pos_map[targets] = UNMAPPED                                      # frontier_finish_kernel
    flags[new_n_id[t:]] = 0
    return new_n_id, src_local, np.array(dst_local, dtype=np.int64), np.array(edge_id, dtype=np.int64), row_off


def block_csr_np(src_local, dst_local, row_off, n_src, n_dst, loops):
    """regnn_block_csr_build's in-view: sampled edge x of row v at slot x + v (loops) / x, the loop of v last."""
    e_s = len(src_local)
    total = e_s + (n_dst if loops else 0)
    indices, eid, row = (np.empty(total, dtype=np.int32) for _ in range(3))
    s = np.arange(e_s) + (dst_local if loops else 0)
    indices[s], eid[s], row[s] = src_local, np.arange(e_s), dst_local
    if loops:
        s = row_off[1:] + np.arange(n_dst)
        indices[s], eid[s], row[s] = np.arange(n_dst), e_s + np.arange(n_dst), np.arange(n_dst)
    v = np.arange(n_src + 1)
    indptr = np.where(v <= n_dst, row_off[np.minimum(v, n_dst)] + (v if loops else 0),
                      e_s + (n_dst if loops else 0)).astype(np.int32)
    slot_t = np.argsort(indices, kind='stable').astype(np.int32)     # the stable sort by local source
    indptr_t = np.zeros(n_src + 1, dtype=np.int32)
    np.cumsum(np.bincount(indices, minlength=n_src), out=indptr_t[1:])
    return dict(indptr=indptr, indices=indices, eid=eid, row=row, indptr_t=indptr_t, indices_t=row[slot_t],
                slot_t=slot_t)


@pytest.mark.parametrize('fanouts,seed_range', [([5, 3], (20, 52)), ([30, 2], (0, 90)), ([4], (390, 400))])
def test_relabel_and_block_csr_restatement_match_oracles(fanouts, seed_range):
    d = synth.random_multigraph(400, 9000, 5, seed=2)
    n = 400
    c = csr_oracle.csr_build(d['src'], d['dst'], n)
    seeds = np.arange(*seed_range)
    n_or, blocks_or = S.sample_blocks(c, seeds, fanouts, seed=11, epoch=1, rank=0, batch=4)
    pos_map, flags = np.full(n, UNMAPPED, dtype=np.int64), np.zeros(n, dtype=np.int64)
    targets, layers = seeds.astype(np.int64), []
    for layer, f in enumerate(fanouts):
        out = sample_layer_np(c, targets, f, S.layer_key(11, 1, 0, 4, layer), pos_map, flags)
        layers.append(out + (len(targets),))
        targets = out[0]
        assert np.all(pos_map == UNMAPPED) and not flags.any()          # maps restored for the next layer
    assert np.array_equal(targets, n_or)
    for (new_n_id, src_l, dst_l, edge_id, row_off, t), (s_or, d_or, e_or, n_src, n_dst) in zip(layers[::-1], blocks_or):
        assert (len(new_n_id), t) == (n_src, n_dst)
        assert np.array_equal(src_l, s_or) and np.array_equal(dst_l, d_or) and np.array_equal(edge_id, e_or)
        for loops in (False, True):
            got = block_csr_np(src_l, dst_l, row_off, n_src, n_dst, loops)
            s_all = np.concatenate([src_l, np.arange(n_dst)]) if loops else src_l
            d_all = np.concatenate([dst_l, np.arange(n_dst)]) if loops else dst_l
            want = csr_oracle.csr_build(s_all, d_all, n_src)
            for k in want:
                assert np.array_equal(got[k], want[k]), (loops, k)
            et1 = np.concatenate([d['etype'][edge_id], 7 + np.arange(n_dst) % 2]) if loops else d['etype'][edge_id]
            et_csr, et_t = csr_oracle.etype_permute(et1, got['eid'], got['slot_t'])
            assert np.array_equal(et_t, et_csr[got['slot_t']])


def test_graph_from_csr_host_logic():
    """Graph.from_csr keeps the edge list, serves the prebuilt CSR and etype views without rebuilding them and answers
    has_zero_in_degree from what it was given; the known-size row split equals the one that counts on the device."""
    from re_gnn_b200 import graph as G
    src = torch.tensor([1, 2, 0, 3, 0, 1, 2], dtype=torch.int64)
    dst = torch.tensor([0, 0, 1, 1, 0, 2, 2], dtype=torch.int64)
    c = {k: torch.as_tensor(v) for k, v in csr_oracle.csr_build(src.numpy(), dst.numpy(), 4).items()}
    c['split'] = c['split_t'] = None
    etype1 = torch.tensor([1, 2, 1, 3, 2, 2, 1])
    et_csr, et_t = (torch.as_tensor(a) for a in csr_oracle.etype_permute(etype1.numpy(), c['eid'].numpy(),
                                                                          c['slot_t'].numpy()))
    g = G.Graph.from_csr(src, dst, 4, c, (etype1, 3, et_csr, et_t, None), True)
    assert g.csr() is c and g.number_of_edges() == 7 and g.number_of_nodes() == 4
    s, t = g.edges()
    assert torch.equal(s, src) and torch.equal(t, dst)
    a, b, cnt = g.etype_views(etype1, 3)
    assert a is et_csr and b is et_t and cnt is None
    assert g.has_zero_in_degree() is True
    assert torch.equal(g.in_degrees(), torch.tensor([3, 2, 2, 0]))

    deg = np.array([3, 300, 0, 257, 1000, 256, 513])
    indptr = torch.as_tensor(np.concatenate([[0], np.cumsum(deg)]).astype(np.int32))
    ref = G._row_split(indptr, 256)
    long_ = deg > 256
    known = G._row_split(indptr, 256, (int(long_.sum()), int(((deg[long_] + 255) // 256).sum())))
    for k in ('long_rows', 'frag_ptr', 'frag_row', 'frag_begin'):
        assert torch.equal(ref[k], known[k]), k
    assert (known['struct'].num_long, known['struct'].num_frags) == (ref['struct'].num_long, ref['struct'].num_frags)
    assert G._row_split(indptr[:3], 256, (0, 0)) is None
