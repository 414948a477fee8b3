"""Host-side checks of the halo-exchange row partitioning (re_gnn_b200.partition.HaloPartition / halo_propagate) and of
the community-structured generator synth.hetero_graph_local, with the CUDA operators replaced by tests/cpu_shim.py.
``install_halo_shim`` is also used by the two-process gloo test (tests/test_partition_halo_gloo.py)."""
import numpy as np
import pytest
import torch

import cpu_shim
from re_gnn_b200 import Graph, functional as RF, partition, synth


def _etype_views_with_counts(self, e_feat, num_relations):
    a, b, _ = cpu_shim.graph_etype_views(self, e_feat, num_relations)
    cnt = torch.zeros(self._n * num_relations, dtype=torch.int32)
    cnt.index_add_(0, self._dst * num_relations + (e_feat.to(torch.int64) - 1), torch.ones(e_feat.numel(), dtype=torch.int32))
    return a, b, cnt


def _wdeg_fwd(csr, et_csr, theta, alpha, exponent, rows=None, counts=None, clamp_min=1.0):
    if csr is not None:
        return cpu_shim.wdeg_norm_fwd(csr, et_csr, theta, alpha, exponent, rows, counts, clamp_min)
    w = cpu_shim._w(theta.detach().view(-1), alpha)
    deg = counts.view(-1, w.numel()).to(w.dtype) @ w
    return deg, deg.clamp(min=clamp_min) ** exponent


def _wdeg_bwd(csr, et_csr, theta, alpha, exponent, deg, d_norm, rows=None, counts=None, clamp_min=1.0):
    if csr is not None:
        return cpu_shim.wdeg_norm_bwd(csr, et_csr, theta, alpha, exponent, deg, d_norm, rows, counts, clamp_min)
    th = theta.detach().view(-1)
    rb, re = rows
    d = deg[rb:re]
    dd = torch.where(d >= clamp_min, exponent * d.clamp(min=clamp_min) ** (exponent - 1) * d_norm[rb:re], torch.zeros_like(d))
    dw = counts.view(-1, th.numel())[rb:re].to(dd.dtype).t() @ dd
    return dw * alpha * cpu_shim._lgrad(th * alpha, cpu_shim.SLOPE)


_shim_spmm = cpu_shim.spmm


def _spmm(indptr, indices, etype, theta, alpha, norm_src, norm_dst, x, rows=None, out=None, split=None, order=None):
    # the kernels index norm_dst by row: a longer table (own rows first) is fine there, the emulation wants its length
    nd = norm_dst[:indptr.numel() - 1] if norm_dst is not None else None
    return _shim_spmm(indptr, indices, etype, theta, alpha, norm_src, nd, x, rows, out, split, order)


def _spmm_bwd_fused(csr, et_t, theta, alpha, norm, x, g, rows=None, sides=3, out=None, want_xdx=False, y=None,
                    want_dnorm=False):
    dx, dw, xdx = cpu_shim.spmm_bwd_fused(csr, et_t, theta, alpha, norm, x, g, rows, sides, out,
                                          want_xdx=want_xdx or want_dnorm)
    if want_dnorm:   # the folded norm gradient of the rows of this view
        n = csr['indptr_t'].numel() - 1
        xdx = (xdx + (y.detach() * g.detach()[:n]).sum(1)) / norm.detach()[:n]
    return dx, dw, xdx


def install_halo_shim(monkeypatch):
    """cpu_shim plus what the halo path needs: the relation-count table and count-table norms, norm tables longer than
    the row count."""
    from re_gnn_b200 import graph as G, ops
    cpu_shim.install(monkeypatch)
    monkeypatch.setattr(G.Graph, 'etype_views', _etype_views_with_counts)
    monkeypatch.setattr(cpu_shim, 'spmm', _spmm)
    for name, fn in (('wdeg_norm_fwd', _wdeg_fwd), ('wdeg_norm_bwd', _wdeg_bwd), ('spmm', _spmm),
                     ('spmm_bwd_fused', _spmm_bwd_fused)):
        monkeypatch.setattr(ops, name, fn)


@pytest.fixture
def halo_ops(monkeypatch):
    install_halo_shim(monkeypatch)


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes'])
    etv = g.etype_views(torch.as_tensor(d['etype']), d['num_relations'])
    return g, etv


def _check_partitions(g, etv, bounds, parts):
    """Every invariant of the local views against a numpy restatement."""
    csr = {k: v.numpy() for k, v in g.csr().items() if torch.is_tensor(v)}
    n, r = g.number_of_nodes(), etv[2].numel() // g.number_of_nodes()
    counts = etv[2].numpy().reshape(n, r)
    for p, part in enumerate(parts):
        rb, re = bounds[p], bounds[p + 1]
        assert part.n_own == re - rb
        for ip_key, idx_key, et_loc, et_glob, halo in (('indptr', 'indices', part.et_in, etv[0], part.in_halo),
                                                       ('indptr_t', 'indices_t', part.et_out, etv[1], part.out_halo)):
            ip, idx = csr[ip_key], csr[idx_key]
            s0, s1 = ip[rb], ip[re]
            assert np.array_equal(part.csr[ip_key].numpy(), ip[rb:re + 1] - s0)
            glob = idx[s0:s1].astype(np.int64)
            loc = part.csr[idx_key].numpy().astype(np.int64)
            h = halo.numpy()
            back = np.where(loc < part.n_own, loc + rb, h[np.maximum(loc - part.n_own, 0)] if h.size else 0)
            assert np.array_equal(back, glob)                               # every slot maps back to its global id
            assert np.array_equal(et_loc.numpy(), et_glob.numpy()[s0:s1])
            remote = glob[(glob < rb) | (glob >= re)]
            assert np.array_equal(h, np.unique(remote))                     # sorted, unique, hence grouped by owner
            assert not ((h >= rb) & (h < re)).any()
        rows = np.concatenate([np.arange(rb, re), part.in_halo.numpy()] + ([] if part.same_halo else [part.out_halo.numpy()]))
        assert np.array_equal(part.counts.numpy().reshape(-1, r), counts[rows])
        assert part.same_halo == np.array_equal(part.in_halo.numpy(), part.out_halo.numpy())
    # rank p's send list to q is q's halo segment owned by p, landing where q's buffer keeps it
    for p, part in enumerate(parts):
        for direction in ('in', 'out'):
            rows, ptr, offsets = part.push_in if direction == 'in' else part.push_out
            for q, other in enumerate(parts):
                seg = rows[ptr[q]:ptr[q + 1]].numpy().astype(np.int64) + bounds[p]
                ext = (other.rows_in if direction == 'in' else other.rows_out).numpy()
                assert np.array_equal(ext[offsets[q]:offsets[q] + seg.size], seg), (p, q, direction)
                if q != p:
                    halo = (other.in_halo if direction == 'in' else other.out_halo).numpy()
                    assert np.array_equal(seg, halo[(halo >= bounds[p]) & (halo < bounds[p + 1])])


def _virtual_step(g, etv, parts, x, gout, theta, weighted):
    """Every virtual rank on its local views with halos filled by index_select: -> (Y, dX, summed d_theta)."""
    ys, dxs, dth = [], [], torch.zeros_like(theta)
    for part in parts:
        y, deg, norm = partition._halo_forward(part, x[part.rows_in], theta, 100.0, weighted)
        dx, dt = partition._halo_backward(part, x[part.rows_in[:part.n_own]], y, gout[part.rows_out], theta, 100.0,
                                          weighted, deg, norm)
        ys.append(y)
        dxs.append(dx)
        dth = dth + dt
    return torch.cat(ys), torch.cat(dxs), dth


def _single(g, etv, x, gout, theta, weighted):
    xs, th = x.clone().requires_grad_(True), theta.clone().requires_grad_(True)
    out = RF.propagate(g, etv, xs, th if weighted else None, 100.0, RF.weighted_degree_norm(g, etv, th, 100.0, -0.5))
    out.backward(gout)
    return out.detach(), xs.grad, th.grad


@pytest.mark.parametrize('layout', ['community', 'edges', 'empty_block', 'one_part'])
@pytest.mark.parametrize('weighted', [True, False])
def test_halo_partition_invariants_and_virtual_ranks(halo_ops, layout, weighted):
    parts_n = 1 if layout == 'one_part' else 3
    d = synth.hetero_graph_local('dblp', parts_n, 0.8, seed=2, scale=0.04)
    g, etv = _setup(d)
    n = d['num_nodes']
    if layout == 'edges':
        bounds = partition.row_blocks(g.csr()['indptr'], parts_n, balance='edges')
    elif layout == 'empty_block':
        cb = d['community_bounds']
        bounds = [0, cb[1], cb[1], n]
    else:
        bounds = d['community_bounds']
    parts = partition.HaloPartition.virtual_ranks(g, etv, bounds)
    _check_partitions(g, etv, bounds, parts)
    if layout == 'one_part':
        assert parts[0].n_in == parts[0].n_out == 0 and parts[0].send_in.numel() == 0
    if layout == 'empty_block':
        assert parts[1].n_own == 0 and parts[1].n_in == parts[1].n_out == 0
    rng = np.random.RandomState(3)
    x, gout = torch.as_tensor(rng.randn(n, 8)), torch.as_tensor(rng.randn(n, 8))
    theta = torch.as_tensor(rng.uniform(0.5, 1.5, (d['num_relations'], 1)) / 100.0)
    y, dx, dth = _virtual_step(g, etv, parts, x, gout, theta, weighted)
    ry, rdx, rdth = _single(g, etv, x, gout, theta, weighted)
    assert torch.allclose(y, ry, rtol=1e-12, atol=1e-12)
    assert torch.allclose(dx, rdx, rtol=1e-12, atol=1e-12)
    assert torch.allclose(dth, rdth, rtol=1e-10, atol=1e-12)


def test_halo_partition_needs_the_count_table(halo_ops):
    d = synth.hetero_graph_local('dblp', 2, 0.5, seed=1, scale=0.02)
    g, etv = _setup(d)
    with pytest.raises(ValueError, match='relation-count table'):
        partition.HaloPartition.virtual_ranks(g, (etv[0], etv[1], None), d['community_bounds'])


def test_local_generator_properties():
    a = synth.hetero_graph_local('mag', 4, 0.9, seed=5, scale=0.01)
    b = synth.hetero_graph_local('mag', 4, 0.9, seed=5, scale=0.01)
    c = synth.hetero_graph_local('mag', 4, 0.9, seed=6, scale=0.01)
    for k in ('src', 'dst', 'etype', 'ntype'):
        assert np.array_equal(a[k], b[k])
    assert not np.array_equal(a['src'], c['src'])
    ref = synth.hetero_graph('mag', seed=5, scale=0.01)
    n = a['num_nodes']
    assert n == ref['num_nodes'] and a['type_sizes'] == ref['type_sizes']
    assert (a['num_etype'], a['num_relations']) == (ref['num_etype'], ref['num_relations'])
    assert np.array_equal(np.bincount(a['ntype']), np.bincount(ref['ntype']))
    src, dst, et = a['src'], a['dst'], a['etype']
    t = 1
    for (_, _, _, symmetric) in synth.SHAPES['mag'][1]:                     # the pairs drawn per relation are distinct
        m = np.nonzero(et == t)[0]
        m = m[:m.size // 2] if symmetric else m                             # a symmetric type holds both directions
        assert np.unique(src[m] * n + dst[m]).size == m.size
        t += 1 if symmetric else 2
    loops = src[-n:]
    assert np.array_equal(loops, np.arange(n)) and np.array_equal(dst[-n:], np.arange(n))
    assert np.array_equal(et[-n:], a['num_etype'] + 1 + a['ntype'])        # self loops last, typed by node type
    assert not (src[:-n] == dst[:-n]).any() and et[:-n].max() <= a['num_etype']
    # every edge type joins the node types of its relation (forward and reverse)
    for t in range(1, a['num_etype'] + 1):
        m = et == t
        assert np.unique(a['ntype'][src[m]]).size == 1 and np.unique(a['ntype'][dst[m]]).size == 1
    cb = a['community_bounds']
    assert cb[0] == 0 and cb[-1] == n and len(cb) == 5 and all(x < y for x, y in zip(cb, cb[1:]))
    comm = np.searchsorted(np.asarray(cb), np.arange(n), side='right') - 1
    for c in range(4):                                                      # about 1/parts of every node type
        got = np.bincount(a['ntype'][comm == c], minlength=len(a['type_sizes']))
        assert np.all(np.abs(got - np.asarray(a['type_sizes']) / 4) <= 1)
    for loc in (0.0, 0.5, 0.9):
        d = synth.hetero_graph_local('mag', 4, loc, seed=5, scale=0.01)
        s, t = d['src'][:-n], d['dst'][:-n]
        cm = np.searchsorted(np.asarray(d['community_bounds']), np.arange(n), side='right') - 1
        frac = float(np.mean(cm[s] == cm[t]))
        want = loc + (1 - loc) / 4                                          # global draws land inside 1/parts of the time
        assert abs(frac - want) < 0.05, (loc, frac, want)


def test_halo_weighted_rejects_shapes_without_a_fused_backward(halo_ops):
    """The weighted backward runs the fused kernel only: a width it does not cover is refused before any work."""
    d = synth.hetero_graph_local('dblp', 2, 0.5, seed=1, scale=0.02)
    g, etv = _setup(d)
    part = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'])[0]
    theta = torch.full((d['num_relations'], 1), 0.01, dtype=torch.float64)
    with pytest.raises(ValueError, match='fused_bwd_fits'):
        partition._halo_forward(part, torch.zeros(part.n_own + part.n_in, 1028, dtype=torch.float64), theta, 100.0, True)
