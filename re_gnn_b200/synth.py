"""Synthetic heterogeneous graphs of the shapes named in BASELINE.json (SURVEY.md Appendix D).

The reference checkout ships no data (``data/`` is git-ignored), so benchmarks and parity tests run
on seeded synthetic graphs with the public node / edge counts of the named datasets.  Conventions
reproduced from run_regnn.py:84-99: node types occupy contiguous id blocks; every relation is
present in both directions with its own 1-based edge type; duplicates and self loops are removed;
one self loop per node is appended LAST with edge type ``num_etype + 1 + ntype(node)``.

Pure numpy on the host -- this is input generation, not part of the hot path.
"""
import numpy as np

# name -> (node type sizes, relations (src_type, dst_type, n_edges, symmetric_pairs))
SHAPES = {
    # DBLP (HGB): A 4057, P 14328, T 7723, V 20;  A-P 19645, P-T 85810, P-V 14328 (+ reverses)
    'dblp': ([4057, 14328, 7723, 20], [(0, 1, 19645, False), (1, 2, 85810, False), (1, 3, 14328, False)]),
    # ACM (HGB): P 3025, A 5959, S 56, T 1902;  P-P cite/ref 5343, P-A 9949, P-S 3025, P-T 255619
    'acm': ([3025, 5959, 56, 1902], [(0, 0, 5343, False), (0, 1, 9949, False), (0, 2, 3025, False),
                                     (0, 3, 255619, False)]),
    # IMDB (MAGNN): M 4932, D 2393, A 6124, K 7971;  M-D 4932, M-A 14779, M-K 23610
    'imdb': ([4932, 2393, 6124, 7971], [(0, 1, 4932, False), (0, 2, 14779, False), (0, 3, 23610, False)]),
    # ogbn-mag: paper 736389, author 1134649, institution 8740, field 59965.  BASELINE's "21M edges":
    # each bipartite relation's OGB count split between its forward and reverse type, cites symmetrised.
    'mag': ([736389, 1134649, 8740, 59965], [(1, 2, 521999, False), (1, 0, 3572830, False),
                                             (0, 0, 2708135, True), (0, 3, 3752539, False)]),
}


def _draw_relation(rng, n_src, n_dst, n_edges, skew):
    """``n_edges`` distinct (u, v) pairs, u uniform, v with power-law popularity (hub destinations)."""
    got = np.zeros(0, dtype=np.int64)
    perm = rng.permutation(n_dst)
    while got.size < n_edges:
        m = int((n_edges - got.size) * 1.25) + 64
        u = rng.randint(0, n_src, size=m).astype(np.int64)
        v = perm[np.minimum((n_dst * rng.random_sample(m) ** skew).astype(np.int64), n_dst - 1)]
        got = np.unique(np.concatenate([got, u * n_dst + v]))
    if got.size > n_edges:
        got = np.sort(rng.choice(got, size=n_edges, replace=False))
    return got // n_dst, got % n_dst


def hetero_graph(name, seed=123, skew=2.5, scale=1.0):
    """Returns a dict: src, dst (int64, edge-id order), etype (int64, 1-based), num_nodes, ntype (per
    node), type_sizes, num_etype, num_relations (= num_etype + num_ntype, run_regnn.py:91-92,121).
    ``scale`` < 1 shrinks node and edge counts proportionally (parity-test sized copies)."""
    sizes, relations = SHAPES[name]
    sizes = [max(2, int(round(s * scale))) for s in sizes]
    rng = np.random.RandomState(seed)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    srcs, dsts, ets = [], [], []
    et = 0
    for (ts, td, ne, symmetric) in relations:
        ne = max(1, int(round(ne * scale)))
        ne = min(ne, sizes[ts] * sizes[td] // 2)
        u, v = _draw_relation(rng, sizes[ts], sizes[td], ne, skew)
        if ts == td:
            keep = u != v
            u, v = u[keep], v[keep]
        u, v = u + offs[ts], v + offs[td]
        if symmetric:          # one edge type holding both directions (ogbn-mag "cites" symmetrised)
            srcs += [u, v]; dsts += [v, u]; ets += [np.full(2 * u.size, et + 1, dtype=np.int64)]
            et += 1
        else:                  # forward type, then its reverse type
            srcs += [u, v]; dsts += [v, u]
            ets += [np.full(u.size, et + 1, dtype=np.int64), np.full(u.size, et + 2, dtype=np.int64)]
            et += 2
    n = int(offs[-1])
    ntype = np.repeat(np.arange(len(sizes), dtype=np.int64), sizes)
    loop = np.arange(n, dtype=np.int64)
    src = np.concatenate(srcs + [loop])
    dst = np.concatenate(dsts + [loop])
    etype = np.concatenate(ets + [et + 1 + ntype])
    return dict(src=src, dst=dst, etype=etype, num_nodes=n, ntype=ntype, type_sizes=sizes,
                num_etype=et, num_relations=et + len(sizes), name=name)


def _draw_relation_local(rng, n_src, n_dst, n_edges, skew, locality, src_cuts, dst_comm):
    """``_draw_relation`` with locality: with probability ``locality`` the source is drawn uniformly from the
    destination's community (``src_cuts``: community boundaries of the source type's local ids; ``dst_comm``: the
    community of every destination), otherwise from the whole source type."""
    got = np.zeros(0, dtype=np.int64)
    perm = rng.permutation(n_dst)
    while got.size < n_edges:
        m = int((n_edges - got.size) * 1.25) + 64
        v = perm[np.minimum((n_dst * rng.random_sample(m) ** skew).astype(np.int64), n_dst - 1)]
        lo, hi = src_cuts[dst_comm[v]], src_cuts[dst_comm[v] + 1]
        near = (rng.random_sample(m) < locality) & (hi > lo)
        u_near = lo + np.minimum((rng.random_sample(m) * (hi - lo)).astype(np.int64), np.maximum(hi - lo - 1, 0))
        u = np.where(near, u_near, rng.randint(0, n_src, size=m).astype(np.int64))
        got = np.unique(np.concatenate([got, u * n_dst + v]))
    if got.size > n_edges:
        got = np.sort(rng.choice(got, size=n_edges, replace=False))
    return got // n_dst, got % n_dst


def hetero_graph_local(name, parts, locality, seed=123, skew=2.5, scale=1.0):
    """``hetero_graph`` with community structure, for row-block partitioning with halos.  The node-type sizes, relation
    counts, edge-type numbering, de-duplication and the self loops appended last are those of ``hetero_graph``; the
    layout differs: nodes are community-major -- community c holds about 1/``parts`` of every node type in one contiguous
    id range -- so node types are NOT contiguous id blocks any more (``ntype`` is per node, as always).  Destinations
    keep the power-law popularity; with probability ``locality`` a source is drawn from the destination's community
    (same source type), otherwise from all nodes of its type.  Returns ``hetero_graph``'s dict plus
    ``community_bounds`` ([parts + 1] row boundaries, usable as ``bounds`` of ``partition``)."""
    sizes, relations = SHAPES[name]
    sizes = [max(2, int(round(s * scale))) for s in sizes]
    rng = np.random.RandomState(seed)
    # cuts[t][c]: first local id of type t in community c; community c = type blocks in type order
    cuts = [np.array([s * c // parts for c in range(parts + 1)], dtype=np.int64) for s in sizes]
    per_comm = np.array([[cuts[t][c + 1] - cuts[t][c] for t in range(len(sizes))] for c in range(parts)], dtype=np.int64)
    comm_start = np.concatenate([[0], np.cumsum(per_comm.sum(1))]).astype(np.int64)
    gid, comm_of = [], []     # per type: global id / community of every local id
    for t, s in enumerate(sizes):
        c = np.repeat(np.arange(parts, dtype=np.int64), np.diff(cuts[t]))
        within = np.arange(s, dtype=np.int64) - cuts[t][c]
        gid.append(comm_start[c] + per_comm[c, :t].sum(1) + within)
        comm_of.append(c)
    srcs, dsts, ets = [], [], []
    et = 0
    for (ts, td, ne, symmetric) in relations:
        ne = max(1, int(round(ne * scale)))
        ne = min(ne, sizes[ts] * sizes[td] // 2)
        u, v = _draw_relation_local(rng, sizes[ts], sizes[td], ne, skew, locality, cuts[ts], comm_of[td])
        if ts == td:
            keep = u != v
            u, v = u[keep], v[keep]
        u, v = gid[ts][u], gid[td][v]
        if symmetric:
            srcs += [u, v]; dsts += [v, u]; ets += [np.full(2 * u.size, et + 1, dtype=np.int64)]
            et += 1
        else:
            srcs += [u, v]; dsts += [v, u]
            ets += [np.full(u.size, et + 1, dtype=np.int64), np.full(u.size, et + 2, dtype=np.int64)]
            et += 2
    n = int(comm_start[-1])
    ntype = np.empty(n, dtype=np.int64)
    for t in range(len(sizes)):
        ntype[gid[t]] = t
    loop = np.arange(n, dtype=np.int64)
    src = np.concatenate(srcs + [loop])
    dst = np.concatenate(dsts + [loop])
    etype = np.concatenate(ets + [et + 1 + ntype])
    return dict(src=src, dst=dst, etype=etype, num_nodes=n, ntype=ntype, type_sizes=sizes,
                num_etype=et, num_relations=et + len(sizes), name=name,
                community_bounds=[int(b) for b in comm_start])


def random_multigraph(n, e, r, seed=0, hubs=4, self_loops=True):
    """Small adversarial test graph: duplicate edges, a few hub destinations, zero-in-degree nodes
    (when ``self_loops`` is False), 1-based edge types in [1, r]."""
    rng = np.random.RandomState(seed)
    src = rng.randint(0, n, size=e).astype(np.int64)
    dst = rng.randint(0, max(1, n - n // 8), size=e).astype(np.int64)
    if hubs and e:
        hub = rng.rand(e) < 0.3
        dst[hub] = rng.randint(0, min(hubs, n), size=int(hub.sum()))
    etype = rng.randint(1, r + 1, size=e).astype(np.int64)
    if self_loops:
        loop = np.arange(n, dtype=np.int64)
        src, dst = np.concatenate([src, loop]), np.concatenate([dst, loop])
        etype = np.concatenate([etype, rng.randint(1, r + 1, size=n).astype(np.int64)])
    return dict(src=src, dst=dst, etype=etype, num_nodes=n, num_relations=r)
