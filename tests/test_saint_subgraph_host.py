"""GraphSAINT induced subgraph without a GPU: a numpy restatement of regnn_induced_subgraph_count / _fill, kernel by
kernel (flags, scan, row fragments, ballots, fragment offsets, fill, flag reset), checked against
oracle/sampler_oracle.saint_subgraph, against oracle/csr_oracle.py for the subgraph's CSR, and for the info words the
row splits read."""
import numpy as np
import pytest

from oracle import csr_oracle, sampler_oracle as S
from re_gnn_b200 import synth

FRAG = 256          # kInducedFragSlots
THRESHOLD = 256     # graph.SPLIT_THRESHOLD
INFO = dict(SOURCES=0, EDGES=1, EMPTY_ROWS=2, IN_SPLIT=3, IN_SPLIT_LOOPS=5, OUT_SPLIT=7, OUT_SPLIT_LOOPS=9)


def long_rows(deg):
    deg = np.asarray(deg, dtype=np.int64)
    big = deg > THRESHOLD
    return [int(big.sum()), int(((deg[big] + THRESHOLD - 1) // THRESHOLD).sum())]


def excl_scan(x):
    return np.concatenate([[0], np.cumsum(x)[:-1]]).astype(np.int64) if len(x) else np.zeros(0, dtype=np.int64)


def induced_count_np(c, num_nodes, nodes, flags):
    """regnn_induced_subgraph_count, kernel by kernel.  Returns (n_id, row_off, src_hist, info, workspace)."""
    indptr, indices = c['indptr'].astype(np.int64), c['indices']
    max_rows = min(num_nodes, len(nodes))
    cap = max_rows + (len(indices) + FRAG - 1) // FRAG
    info = np.zeros(16, dtype=np.int64)
    src_hist = np.zeros(max_rows, dtype=np.int64)
    frag_first = np.zeros(max_rows + 1, dtype=np.int64)
    flags[nodes[(nodes >= 0) & (nodes < num_nodes)]] = 1                 # induced_flag_kernel
    excl = excl_scan(flags)                                              # exclusive_scan_u32 over all N
    n_sub = int(excl[-1] + flags[-1])                                    # induced_rows_kernel
    info[INFO['SOURCES']] = n_sub
    n_id = np.empty(max_rows, dtype=np.int64)
    for v in np.nonzero(flags)[0]:
        r = excl[v]
        n_id[r] = v
        deg = indptr[v + 1] - indptr[v]
        frag_first[r] = (deg + FRAG - 1) // FRAG if deg > FRAG else 1
    frag_first = excl_scan(np.append(frag_first, 0))[:max_rows + 1]     # scan over max_rows + 1 entries
    num_frags = int(frag_first[n_sub])
    assert num_frags <= cap
    frag_row = np.zeros(cap, dtype=np.int64)
    frag_cnt = np.zeros(cap + 1, dtype=np.int64)
    for f in range(num_frags):                                           # induced_frag_count_kernel: a warp per fragment
        r = int(np.searchsorted(frag_first[:n_sub + 1], f, side='right') - 1)
        v = n_id[r]
        s0 = indptr[v] + (f - frag_first[r]) * FRAG
        s1 = min(s0 + FRAG, indptr[v + 1])
        kept = 0
        for base in range(s0, s1, 32):
            ballot = [s < s1 and flags[indices[s]] == 1 for s in range(base, base + 32)]
            for s, k in zip(range(base, base + 32), ballot):
                if k:
                    src_hist[excl[indices[s]]] += 1
            kept += sum(ballot)
        frag_row[f], frag_cnt[f] = r, kept
    frag_off = excl_scan(frag_cnt)                                       # scan over frag_cap + 1 entries
    row_off = np.empty(max_rows + 1, dtype=np.int64)                     # induced_rows_finish_kernel
    for r in range(max_rows + 1):
        row_off[r] = frag_off[frag_first[min(r, n_sub)]]
    info[INFO['EDGES']] = row_off[n_sub]
    deg = row_off[1:n_sub + 1] - row_off[:n_sub]
    info[INFO['EMPTY_ROWS']] = int((deg == 0).sum())
    info[INFO['IN_SPLIT']:INFO['IN_SPLIT'] + 2] = long_rows(deg)
    info[INFO['OUT_SPLIT']:INFO['OUT_SPLIT'] + 2] = long_rows(src_hist[:n_sub])
    return n_id, row_off, src_hist, info, (excl, frag_first, frag_row, frag_off)


def induced_fill_np(c, n_id, num_rows, num_sub_edges, flags, workspace):
    """regnn_induced_subgraph_fill: the ballots replayed, each kept slot at its fragment offset plus its rank."""
    indptr, indices, eid = c['indptr'].astype(np.int64), c['indices'], c['eid']
    excl, frag_first, frag_row, frag_off = workspace
    src_local, dst_local, edge_id = (np.full(num_sub_edges, -1, dtype=np.int64) for _ in range(3))
    for f in range(int(frag_first[num_rows])):
        r = frag_row[f]
        v = n_id[r]
        s0 = indptr[v] + (f - frag_first[r]) * FRAG
        s1 = min(s0 + FRAG, indptr[v + 1])
        out = frag_off[f]
        for base in range(s0, s1, 32):
            ballot = [s < s1 and flags[indices[s]] == 1 for s in range(base, base + 32)]
            for lane, k in enumerate(ballot):
                if k:
                    e = out + sum(ballot[:lane])
                    s = base + lane
                    src_local[e], dst_local[e], edge_id[e] = excl[indices[s]], r, eid[s]
            out += sum(ballot)
    flags[n_id[:num_rows]] = 0                                           # induced_clear_flags_kernel
    return src_local, dst_local, edge_id


def hub_graph(seed=3):
    """random_multigraph with hub destinations (about 1 100 in-edges each) plus node 7 feeding 400 nodes (a hub source)."""
    d = synth.random_multigraph(600, 12000, 5, seed=seed, hubs=3, self_loops=False)
    rng = np.random.RandomState(seed)
    src = np.concatenate([d['src'], np.full(400, 7)])
    dst = np.concatenate([d['dst'], rng.choice(600, 400, replace=False)])
    return src, dst, 600


def run_both(c, n, nodes):
    flags = np.zeros(n, dtype=np.int64)
    n_id, row_off, hist, info, ws = induced_count_np(c, n, nodes, flags)
    n_sub, e_sub = int(info[INFO['SOURCES']]), int(info[INFO['EDGES']])
    s_l, d_l, e = induced_fill_np(c, n_id, n_sub, e_sub, flags, ws)
    assert not flags.any()                                               # the map comes back all zero
    return n_id[:n_sub], row_off[:n_sub + 1], hist[:n_sub], info, s_l, d_l, e


@pytest.mark.parametrize('roots,walk_length,batch', [(40, 2, 0), (300, 2, 3), (1500, 1, 1), (7, 0, 2)])
def test_restatement_matches_saint_oracle_and_csr(roots, walk_length, batch):
    src, dst, n = hub_graph()
    c = csr_oracle.csr_build(src, dst, n)
    walks = S.random_walks(c, n, roots, walk_length, S.layer_key(5, 1, 0, batch, 0x5A1))
    n_id, row_off, hist, info, s_l, d_l, e = run_both(c, n, walks.reshape(-1))
    w_nid, w_s, w_d, w_e = S.saint_subgraph(c, n, roots, walk_length, seed=5, epoch=1, rank=0, batch=batch)
    assert np.array_equal(n_id, w_nid)
    assert np.array_equal(s_l, w_s) and np.array_equal(d_l, w_d) and np.array_equal(e, w_e)
    # the edge list is the subgraph's in-CSR already: row_off is its indptr and CSR slot k holds edge k
    n_sub = len(n_id)
    want = csr_oracle.csr_build(s_l, d_l, n_sub)
    assert np.array_equal(row_off, want['indptr'])
    assert np.array_equal(want['eid'], np.arange(len(s_l)))
    assert np.array_equal(hist, np.diff(want['indptr_t']))
    deg = np.diff(want['indptr'])
    assert info[INFO['EMPTY_ROWS']] == (deg == 0).sum()
    assert list(info[INFO['IN_SPLIT']:INFO['IN_SPLIT'] + 2]) == long_rows(deg)
    assert list(info[INFO['OUT_SPLIT']:INFO['OUT_SPLIT'] + 2]) == long_rows(np.diff(want['indptr_t']))
    assert info[INFO['IN_SPLIT_LOOPS']] == info[INFO['OUT_SPLIT_LOOPS']] == 0


def test_hub_rows_and_hub_sources_take_the_fragment_path():
    """Every node listed: the subgraph is the graph itself, hub rows span several 256-slot fragments and node 7's
    out-edges make a long row of the transposed view."""
    src, dst, n = hub_graph()
    c = csr_oracle.csr_build(src, dst, n)
    nodes = np.concatenate([np.arange(n)[::-1], np.arange(0, n, 3)])     # every node, some twice, out of order
    n_id, row_off, hist, info, s_l, d_l, e = run_both(c, n, nodes)
    assert np.array_equal(n_id, np.arange(n)) and np.array_equal(row_off, c['indptr'])
    assert np.array_equal(s_l, c['indices']) and np.array_equal(e, c['eid'])
    assert np.array_equal(d_l, c['row'])
    assert info[INFO['IN_SPLIT']] >= 3 and info[INFO['IN_SPLIT'] + 1] > info[INFO['IN_SPLIT']]
    assert info[INFO['OUT_SPLIT']] >= 1 and hist[7] > THRESHOLD
    assert list(info[INFO['IN_SPLIT']:INFO['IN_SPLIT'] + 2]) == long_rows(np.diff(c['indptr']))
    assert list(info[INFO['OUT_SPLIT']:INFO['OUT_SPLIT'] + 2]) == long_rows(np.diff(c['indptr_t']))


def test_empty_inputs():
    src, dst, n = hub_graph()
    c = csr_oracle.csr_build(src, dst, n)
    n_id, row_off, hist, info, s_l, d_l, e = run_both(c, n, np.zeros(0, dtype=np.int64))
    assert len(n_id) == 0 and list(row_off) == [0] and len(s_l) == 0 and not info.any()
    c0 = csr_oracle.csr_build(np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64), 9)
    n_id, row_off, hist, info, s_l, d_l, e = run_both(c0, 9, np.array([4, 2, 4, 8]))
    assert list(n_id) == [2, 4, 8] and list(row_off) == [0, 0, 0, 0] and len(s_l) == 0
    assert info[INFO['EMPTY_ROWS']] == 3
