"""Host-side checks of the REGAT halo path (``HaloPartition(..., attention=True)``, ``partition.halo_gat``) with the CUDA
operators replaced by plain-PyTorch emulations: the attention views against a numpy restatement, and every virtual rank
against ``functional.gat_layer``.  ``install_gat_halo_shim`` is also used by the two-process gloo test
(tests/test_partition_halo_gat_gloo.py)."""
import numpy as np
import pytest
import torch

import cpu_shim
import test_halo_host
from re_gnn_b200 import Graph, functional as RF, partition, synth


# ---- stage-wise emulations of the attention operators on local views (rows come from indptr, not from feat) ----------
def _rows(indptr):
    return cpu_shim._rows_of(indptr)


def _gat_fwd(csr, et_csr, theta, alpha, feat, el, er, slope, keep=None, want_attn=False, rows=None):
    feat, el, er = feat.detach(), el.detach(), er.detach()
    n = csr['indptr'].numel() - 1
    row, col = _rows(csr['indptr']), csr['indices'].long()
    pre = el[col] + er[row]
    if theta is not None and et_csr is not None:
        pre = pre + cpu_shim._w(theta.detach(), alpha)[et_csr.long()]
    a, mx, sm = cpu_shim._softmax_rows(cpu_shim._leaky(pre, slope), row, n)
    out = torch.zeros((n,) + feat.shape[1:], dtype=feat.dtype).index_add(0, row, a[:, :, None] * feat[col])
    return out, mx, sm, None


def _gat_bwd_stats(out, g, er, rowmax, rowsum):
    inv = torch.where(rowsum > 0, 1.0 / rowsum, torch.zeros_like(rowsum))
    return torch.stack([er.detach(), rowmax, inv, (out.detach() * g.detach()).sum(-1)], dim=-1)


def _gat_bwd_edges(csr, et_t, theta, alpha, feat, el, stats, slope, g, dpre, attn_l=None):
    feat, el, g = feat.detach(), el.detach(), g.detach()
    n = csr['indptr_t'].numel() - 1
    u, v = _rows(csr['indptr_t']), csr['indices_t'].long()
    st = stats[v]
    pre = el[u] + st[..., 0]
    if theta is not None and et_t is not None:
        pre = pre + cpu_shim._w(theta.detach(), alpha)[et_t.long()]
    a = torch.exp(cpu_shim._leaky(pre, slope) - st[..., 1]) * st[..., 2]
    dp = (a * (feat[u] * g[v]).sum(-1) - a * st[..., 3]) * cpu_shim._lgrad(pre, slope)
    dpre[csr['slot_t'].long()] = dp
    d_el = torch.zeros((n, feat.shape[1]), dtype=feat.dtype).index_add(0, u, dp)
    d_feat = torch.zeros((n,) + feat.shape[1:], dtype=feat.dtype).index_add(0, u, a[:, :, None] * g[v])
    if attn_l is not None:
        d_feat = d_feat + d_el[:, :, None] * attn_l.detach().view(1, *feat.shape[1:])
    return d_feat, d_el


def _gat_bwd_reduce(csr, et_csr, theta, alpha, dpre):
    n = csr['indptr'].numel() - 1
    d_er = torch.zeros((n, dpre.shape[1]), dtype=dpre.dtype).index_add(0, _rows(csr['indptr']), dpre)
    if theta is None or et_csr is None:
        return d_er, None
    th = theta.detach()
    dw = torch.zeros_like(th).index_add(0, et_csr.long(), dpre)
    return d_er, dw * alpha * cpu_shim._lgrad(th * alpha, cpu_shim.SLOPE)


def _attn_scores_bwd(feat, d_el, d_er, attn_r=None, d_feat=None):
    feat = feat.detach()
    h, d = feat.shape[1], feat.shape[2]
    if d_feat is not None:
        d_feat += d_er[:, :, None] * attn_r.detach().view(1, h, d)
    return (d_el[:, :, None] * feat).sum(0).reshape(-1), (d_er[:, :, None] * feat).sum(0).reshape(-1)


def install_gat_halo_shim(monkeypatch):
    """The halo shim plus stage-wise attention operators that take local views."""
    from re_gnn_b200 import ops
    test_halo_host.install_halo_shim(monkeypatch)
    for name, fn in (('gat_fwd', _gat_fwd), ('gat_bwd_stats', _gat_bwd_stats), ('gat_bwd_edges', _gat_bwd_edges),
                     ('gat_bwd_reduce', _gat_bwd_reduce), ('attn_scores_bwd', _attn_scores_bwd)):
        monkeypatch.setattr(ops, name, fn)


@pytest.fixture
def gat_ops(monkeypatch):
    install_gat_halo_shim(monkeypatch)


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes'])
    etv = g.etype_views(torch.as_tensor(d['etype']), d['num_relations'])
    return g, etv


def _bounds(g, d, layout, parts):
    n = d['num_nodes']
    if layout == 'edges':        # uneven row counts
        return partition.row_blocks(g.csr()['indptr'], parts, balance='edges')
    if layout == 'empty_block':
        cb = d['community_bounds']
        return [0, cb[1], cb[1]] + list(cb[2:])
    if layout == 'one_part':
        return [0, n]
    return list(d['community_bounds'])


def _check_attention_views(g, bounds, parts):
    csr = {k: v.numpy() for k, v in g.csr().items() if torch.is_tensor(v)}
    ip, ip_t = csr['indptr'].astype(np.int64), csr['indptr_t'].astype(np.int64)
    slot_bounds = ip[np.asarray(bounds)]
    covered = [np.zeros(part.e_in, dtype=np.int64) for part in parts]
    for p, part in enumerate(parts):
        rb, re = bounds[p], bounds[p + 1]
        s0, s1 = ip[rb], ip[re]
        assert part.e_in == s1 - s0
        assert np.array_equal(part.eid_in.numpy(), csr['eid'][s0:s1])
        assert 'eid' not in part.csr
        gslot = csr['slot_t'][ip_t[rb]:ip_t[re]].astype(np.int64)
        st = part.csr['slot_t'].numpy().astype(np.int64)
        own = st < part.e_in
        dst_own = (gslot >= s0) & (gslot < s1)
        assert np.array_equal(own, dst_own)
        assert np.array_equal(st[own] + s0, gslot[own])                 # own destination: its local in-view slot
        np.add.at(covered[p], st[own], 1)
        tail = part.tail_ptr[-1]
        assert np.array_equal(np.sort(st[~own]), part.e_in + np.arange(tail))
        td = part.tail_dst.numpy().astype(np.int64)
        tail_glob = np.empty(tail, dtype=np.int64)
        tail_glob[st[~own] - part.e_in] = gslot[~own]
        assert part.tail_counts[p] == 0 and part.tail_ptr == [0] + list(np.cumsum(part.tail_counts))
        for q in range(len(parts)):
            seg = slice(part.tail_ptr[q], part.tail_ptr[q + 1])
            assert np.all(np.diff(td[seg]) > 0)                           # grouped by owner, slot-ascending
            assert np.array_equal(td[seg] + slot_bounds[q], tail_glob[seg])
            np.add.at(covered[q], td[seg], 1)
    for p, part in enumerate(parts):
        assert np.all(covered[p] == 1), p                                # every in-view slot exactly once
        recv = part.dpre_recv.numpy()
        ptr = np.concatenate([[0], np.cumsum(part.dpre_recv_counts)])
        for q, other in enumerate(parts):                                # the receive list is q's tail segment
            assert np.array_equal(recv[ptr[q]:ptr[q + 1]], other.tail_dst.numpy()[other.tail_ptr[p]:other.tail_ptr[p + 1]])
    assert all(part.max_dpre_rows == max(o.e_in + o.tail_ptr[-1] for o in parts) for part in parts)


def _inputs(d, heads, dim, seed, relational=True):
    rng = np.random.RandomState(seed)
    n = d['num_nodes']
    f = torch.as_tensor(rng.randn(n, heads, dim))
    gout = torch.as_tensor(rng.randn(n, heads, dim))
    al = torch.as_tensor(rng.randn(1, heads, dim) * 0.3)
    ar = torch.as_tensor(rng.randn(1, heads, dim) * 0.3)
    th = torch.as_tensor(rng.uniform(0.5, 1.5, (d['num_relations'], heads)) / 100.0) if relational else None
    return f, gout, al, ar, th


def _single(g, etv, f, gout, al, ar, th):
    leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (f, al, ar, th)]
    out, _ = RF.gat_layer(g, etv, leaves[0], leaves[1], leaves[2], leaves[3], 100.0, 0.2)
    out.backward(gout)
    return (out.detach(),) + tuple(t.grad if t is not None else None for t in leaves)


@pytest.mark.parametrize('layout', ['community', 'edges', 'empty_block', 'one_part'])
@pytest.mark.parametrize('name', ['dblp', 'acm', 'mag'])
def test_attention_views_and_virtual_ranks(gat_ops, name, layout):
    parts_n = 3
    d = synth.hetero_graph_local(name, parts_n, 0.8, seed=2, scale={'dblp': 0.04, 'acm': 0.05, 'mag': 0.002}[name])
    g, etv = _setup(d)
    bounds = _bounds(g, d, layout, parts_n)
    parts = partition.HaloPartition.virtual_ranks(g, etv, bounds, attention=True)
    _check_attention_views(g, bounds, parts)
    if layout == 'empty_block':
        assert parts[1].n_own == 0 and parts[1].e_in == 0 and parts[1].tail_ptr[-1] == 0
    if layout != 'one_part':
        assert sum(p.tail_ptr[-1] for p in parts) > 0
    f, gout, al, ar, th = _inputs(d, 2, 4, 3)
    out, d_f, d_al, d_ar, d_th = partition._virtual_halo_gat(parts, f, gout, al, ar, th, 100.0, 0.2)
    r_out, r_f, r_al, r_ar, r_th = _single(g, etv, f, gout, al, ar, th)
    assert torch.allclose(out, r_out, rtol=1e-12, atol=1e-12)
    assert torch.allclose(d_f, r_f, rtol=1e-10, atol=1e-12)
    assert torch.allclose(d_al, r_al.view(-1), rtol=1e-10, atol=1e-12)
    assert torch.allclose(d_ar, r_ar.view(-1), rtol=1e-10, atol=1e-12)
    assert torch.allclose(d_th, r_th, rtol=1e-10, atol=1e-12)


def test_default_partition_keeps_no_attention_views(gat_ops):
    d = synth.hetero_graph_local('dblp', 2, 0.8, seed=2, scale=0.03)
    g, etv = _setup(d)
    plain = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'])
    att = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'], attention=True)
    for a, b in zip(plain, att):
        assert not a.attention and not hasattr(a, 'tail_dst') and 'slot_t' not in a.csr
        assert set(b.csr) == set(a.csr) | {'slot_t'}
        for k in a.csr:
            if torch.is_tensor(a.csr[k]):
                assert torch.equal(a.csr[k], b.csr[k])
        assert a.push_in[1] == b.push_in[1] and a.push_out[1] == b.push_out[1]


@pytest.mark.parametrize('relational', [True, False])
def test_halo_gat_autograd_one_rank(gat_ops, relational):
    """One row block (no process group needed): halo_gat through autograd equals gat_layer, with and without the
    relation term."""
    d = synth.hetero_graph_local('acm', 1, 0.8, seed=4, scale=0.05)
    g, etv = _setup(d)
    part = partition.HaloPartition.virtual_ranks(g, etv, [0, d['num_nodes']], attention=True)[0]
    f, gout, al, ar, th = _inputs(d, 4, 8, 5, relational)
    leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (f, al, ar, th)]
    out = partition.halo_gat(part, *leaves, 100.0, 0.2)
    out.backward(gout)
    r_out, r_f, r_al, r_ar, r_th = _single(g, etv, f, gout, al, ar, th)
    assert torch.allclose(out.detach(), r_out, rtol=1e-12, atol=1e-12)
    assert torch.allclose(leaves[0].grad, r_f, rtol=1e-10, atol=1e-12)
    assert torch.allclose(leaves[1].grad, r_al, rtol=1e-10, atol=1e-12)
    assert torch.allclose(leaves[2].grad, r_ar, rtol=1e-10, atol=1e-12)
    if relational:
        assert torch.allclose(leaves[3].grad, r_th, rtol=1e-10, atol=1e-12)


def test_halo_gat_refuses_unsupported_inputs(gat_ops):
    d = synth.hetero_graph_local('dblp', 2, 0.8, seed=2, scale=0.03)
    g, etv = _setup(d)
    part = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'], attention=True)[0]
    plain = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'])[0]
    r = d['num_relations']

    def call(p=part, h=2, dim=8, keep=None, th_shape=None):
        f = torch.zeros(p.n_own, h, dim, dtype=torch.float64)
        a = torch.zeros(1, h, dim, dtype=torch.float64)
        th = torch.zeros(th_shape or (r, h), dtype=torch.float64)
        return partition.halo_gat(p, f, a, a, th, 100.0, 0.2, keep=keep)
    with pytest.raises(ValueError, match='dropout'):
        call(keep=torch.ones(3, 2))
    with pytest.raises(ValueError, match='attention=True'):
        call(p=plain)
    for h, dim in ((2, 6), (2, 256), (33, 4), (16, 128)):
        with pytest.raises(ValueError, match='fused attention kernels'):
            call(h=h, dim=dim)
    with pytest.raises(ValueError, match='theta'):
        call(th_shape=(r + 1, 2))
