"""Host-side checks of the REGATv2 halo path (``HaloPartition(..., attention=True).push_slots``, ``partition.halo_gatv2``)
with the CUDA operators replaced by plain-PyTorch emulations of the stage wrappers on local views: the push lists of
the slot records against the receive lists, every virtual rank against ``functional.gatv2_aggregate`` in float64, and
``ops.gatv2_bwd`` rebuilt from its stages.  ``install_gatv2_halo_shim`` is also used by the two-process gloo test
(tests/test_partition_halo_gatv2_gloo.py)."""
import contextlib
import types

import numpy as np
import pytest
import torch

import cpu_shim
import test_halo_gat_host
from re_gnn_b200 import Graph, functional as RF, ops, partition, synth

ALPHA, SLOPE = 100.0, 0.2
_GATV2_BWD = ops.gatv2_bwd       # the real composition, captured before any fixture replaces it


# ---- stage-wise emulations on local views; the sign masks in the kernels' packed layout ------------------------------
def _rows(indptr):
    return cpu_shim._rows_of(indptr)


def _chunks(h, d):
    return (h * d + 127) // 128


def _pack(pos):
    """[E, H, D] bool -> [E, C, 4] int32: bit l of word c is component c of the l-th 128-bit chunk of a 128-float slice
    (qmask of regnn_gatv2_fwd)."""
    e, h, d = pos.shape
    c = _chunks(h, d)
    flat = torch.zeros((e, c * 128), dtype=torch.int64)
    flat[:, :h * d] = pos.reshape(e, h * d).to(torch.int64)
    words = (flat.view(e, c, 32, 4) << torch.arange(32).view(1, 1, 32, 1)).sum(2)
    return torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)


def _unpack(mask, h, d):
    e, c, _ = mask.shape
    words = mask.to(torch.int64) & 0xFFFFFFFF
    bits = (words.unsqueeze(2) >> torch.arange(32).view(1, 1, 32, 1)) & 1
    return bits.reshape(e, c * 128)[:, :h * d].reshape(e, h, d).bool()


def _phi(mask, h, d, slope, dtype):
    return torch.where(_unpack(mask, h, d), torch.ones((), dtype=dtype), torch.full((), slope, dtype=dtype))


def _gatv2_fwd(csr, et_csr, theta, alpha, fs, fd, attn, slope, keep=None, want_attn=False, rows=None, save=False,
               saved=None):
    fs, fd = fs.detach(), fd.detach()
    _, h, d = fs.shape
    n = csr['indptr'].numel() - 1
    row, col = _rows(csr['indptr']), csr['indices'].long()
    q = fs[col] + fd[row]
    lg = (cpu_shim._leaky(q, slope) * attn.detach().view(1, h, d)).sum(-1)
    if theta is not None and et_csr is not None:
        lg = lg + cpu_shim._w(theta.detach(), alpha)[et_csr.long()]
    a, mx, sm = cpu_shim._softmax_rows(lg, row, n)
    out = torch.zeros((n, h, d), dtype=fs.dtype).index_add(0, row, a[:, :, None] * fs[col])
    e = col.numel()
    if saved is None and save:
        saved = (lg.new_empty((e, h)), torch.empty((e, _chunks(h, d), 4), dtype=torch.int32))
    if saved is not None:
        saved[0][:e] = lg
        saved[1][:e] = _pack(q > 0)
    return out, mx, sm, None, saved


def _gat_bwd_stats(out, g, er, rowmax, rowsum):
    inv = torch.where(rowsum > 0, 1.0 / rowsum, torch.zeros_like(rowsum))
    er = er.detach() if er is not None else torch.zeros_like(rowmax)
    return torch.stack([er, rowmax, inv, (out.detach() * g.detach()).sum(-1)], dim=-1)


def _gatv2_bwd_edges(csr, fs, stats, logit_csr, qmask, attn, slope, g, dl, keep=None):
    fs, g = fs.detach(), g.detach()
    _, h, d = fs.shape
    n = csr['indptr_t'].numel() - 1
    u, v, s = _rows(csr['indptr_t']), csr['indices_t'].long(), csr['slot_t'].long()
    st = stats[v]
    a = torch.exp(logit_csr[s] - st[..., 1]) * st[..., 2]
    dls = a * (fs[u] * g[v]).sum(-1) - a * st[..., 3]
    dl[s] = dls
    t_src = torch.zeros((n, h, d), dtype=fs.dtype).index_add(0, u, dls[:, :, None] * _phi(qmask[s], h, d, slope, fs.dtype))
    d_fs = torch.zeros((n, h, d), dtype=fs.dtype).index_add(0, u, a[:, :, None] * g[v]) + attn.detach().view(1, h, d) * t_src
    return d_fs, (fs * t_src).sum(0).reshape(-1)


def _gatv2_bwd_dst(csr, et_csr, theta, alpha, fd, dl, qmask, attn, slope):
    fd = fd.detach()
    n, h, d = fd.shape
    row = _rows(csr['indptr'])
    e = row.numel()
    t_dst = torch.zeros_like(fd).index_add(0, row, dl[:e, :, None] * _phi(qmask[:e], h, d, slope, fd.dtype))
    d_theta = None
    if theta is not None and et_csr is not None:
        th = theta.detach()
        d_theta = torch.zeros_like(th).index_add(0, et_csr.long(), dl[:e]) * alpha * cpu_shim._lgrad(th * alpha, cpu_shim.SLOPE)
    return attn.detach().view(1, h, d) * t_dst, (fd * t_dst).sum(0).reshape(-1), d_theta


def install_gatv2_halo_shim(monkeypatch):
    """The REGAT halo shim plus the REGATv2 stage emulations (packed sign masks, caller-provided slot buffers)."""
    test_halo_gat_host.install_gat_halo_shim(monkeypatch)
    for name, fn in (('gatv2_fwd', _gatv2_fwd), ('gat_bwd_stats', _gat_bwd_stats), ('gatv2_bwd_edges', _gatv2_bwd_edges),
                     ('gatv2_bwd_dst', _gatv2_bwd_dst)):
        monkeypatch.setattr(ops, name, fn)


@pytest.fixture
def v2_ops(monkeypatch):
    install_gatv2_halo_shim(monkeypatch)


@contextlib.contextmanager
def _whole_graph_ops():
    """cpu_shim's whole-graph REGATv2 emulations (boolean masks, their own formulas) for the single-device reference."""
    saved = ops.gatv2_fwd, ops.gatv2_bwd
    ops.gatv2_fwd, ops.gatv2_bwd = cpu_shim.gatv2_fwd, cpu_shim.gatv2_bwd
    try:
        yield
    finally:
        ops.gatv2_fwd, ops.gatv2_bwd = saved


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes'])
    etv = g.etype_views(torch.as_tensor(d['etype']), d['num_relations'])
    return g, etv


def _inputs(d, heads, dim, seed, relational=True):
    rng = np.random.RandomState(seed)
    n = d['num_nodes']
    fs = torch.as_tensor(rng.randn(n, heads, dim))
    fd = torch.as_tensor(rng.randn(n, heads, dim))
    gout = torch.as_tensor(rng.randn(n, heads, dim))
    attn = torch.as_tensor(rng.randn(1, heads, dim) * 0.3)
    th = torch.as_tensor(rng.uniform(0.5, 1.5, (d['num_relations'], heads)) / 100.0) if relational else None
    return fs, fd, gout, attn, th


def single(g, etv, fs, fd, gout, attn, th, shared=False):
    """functional.gatv2_aggregate on the whole graph -> (out, d_fs, d_fd | None, d_attn, d_theta | None); ``shared``:
    fd is fs (one leaf, its gradient returned as d_fs)."""
    with _whole_graph_ops():
        leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (fs, fd, attn, th)]
        if shared:
            leaves[1] = leaves[0]
        out, _ = RF.gatv2_aggregate(g, etv, leaves[0], leaves[1], leaves[2], leaves[3], ALPHA, SLOPE)
        out.backward(gout)
    return (out.detach(), leaves[0].grad, None if shared else leaves[1].grad, leaves[2].grad,
            leaves[3].grad if th is not None else None)


def _check_push_lists(parts):
    """Every tail row of every rank is filled exactly once, by the owner of the edge's destination, with that
    destination's slot; each segment lands at the receiver's tail segment of the sender; the self segment is empty."""
    nparts = len(parts)
    filled = [np.zeros(part.tail_ptr[-1], dtype=np.int64) for part in parts]
    for p, part in enumerate(parts):
        send, ptr, offsets = part.push_slots
        assert send.dtype == torch.int32 and len(ptr) == nparts + 1 and len(offsets) == nparts
        assert ptr[0] == 0 and ptr[-1] == send.numel() and ptr[p] == ptr[p + 1]
        assert np.array_equal(send.numpy(), part.dpre_recv.numpy())
        for q, owner in enumerate(parts):
            cnt = ptr[q + 1] - ptr[q]
            assert cnt == owner.tail_counts[p]
            if q == p:
                continue
            assert offsets[q] == owner.e_in + owner.tail_ptr[p]
            np.add.at(filled[q], offsets[q] - owner.e_in + np.arange(cnt), 1)
            assert np.array_equal(send[ptr[q]:ptr[q + 1]].numpy(),
                                  owner.tail_dst[owner.tail_ptr[p]:owner.tail_ptr[p + 1]].numpy())
    for p, part in enumerate(parts):
        assert np.all(filled[p] == 1), p
        assert part.max_dpre_rows == max(o.e_in + o.tail_ptr[-1] for o in parts)


def _compare(got, want, d_fd=True):
    out, d_fs, d_fd_, d_attn, d_th = got
    r_out, r_fs, r_fd, r_attn, r_th = want
    assert torch.allclose(out, r_out, rtol=1e-12, atol=1e-12)
    assert torch.allclose(d_fs, r_fs, rtol=1e-10, atol=1e-12)
    if d_fd:
        assert torch.allclose(d_fd_, r_fd, rtol=1e-10, atol=1e-12)
    assert torch.allclose(d_attn.reshape(-1), r_attn.reshape(-1), rtol=1e-10, atol=1e-12)
    if r_th is not None:
        assert torch.allclose(d_th, r_th, rtol=1e-10, atol=1e-12)


def test_sign_mask_packing_round_trip():
    rng = np.random.RandomState(0)
    for h, d in ((1, 4), (2, 64), (3, 128), (8, 128)):
        pos = torch.as_tensor(rng.rand(5, h, d) > 0.5)
        packed = _pack(pos)
        assert packed.shape == (5, _chunks(h, d), 4) and packed.dtype == torch.int32
        assert torch.equal(_unpack(packed, h, d), pos)
    one = torch.zeros(1, 1, 128, dtype=torch.bool)
    one[0, 0, 4 * 31 + 2] = True                   # chunk 31, component 2 -> bit 31 of word 2
    assert _pack(one).tolist() == [[[0, 0, -2 ** 31, 0]]]


@pytest.mark.parametrize('layout', ['community', 'edges', 'empty_block', 'one_part'])
@pytest.mark.parametrize('name', ['dblp', 'acm', 'mag'])
def test_push_lists_and_virtual_ranks(v2_ops, name, layout):
    parts_n = 3
    d = synth.hetero_graph_local(name, parts_n, 0.8, seed=2, scale={'dblp': 0.04, 'acm': 0.05, 'mag': 0.002}[name])
    g, etv = _setup(d)
    bounds = test_halo_gat_host._bounds(g, d, layout, parts_n)
    parts = partition.HaloPartition.virtual_ranks(g, etv, bounds, attention=True)
    _check_push_lists(parts)
    if layout != 'one_part':
        assert sum(p.push_slots[1][-1] for p in parts) > 0
    fs, fd, gout, attn, th = _inputs(d, 2, 4, 3)
    got = partition._virtual_halo_gatv2(parts, fs, fd, gout, attn, th, ALPHA, SLOPE)
    _compare(got, single(g, etv, fs, fd, gout, attn, th))


def test_virtual_ranks_two_mask_chunks(v2_ops):
    """H * D = 256: two 128-bit mask words per slot travel with every cut edge."""
    d = synth.hetero_graph_local('acm', 4, 0.5, seed=6, scale=0.03)
    g, etv = _setup(d)
    parts = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'], attention=True)
    fs, fd, gout, attn, th = _inputs(d, 4, 64, 9)
    got = partition._virtual_halo_gatv2(parts, fs, fd, gout, attn, th, ALPHA, SLOPE)
    _compare(got, single(g, etv, fs, fd, gout, attn, th))


def test_gatv2_bwd_is_composed_from_its_stages(v2_ops, monkeypatch):
    """ops.gatv2_bwd = gat_bwd_stats -> gatv2_bwd_edges -> gatv2_bwd_dst, here over the stage emulations on the whole
    graph, against cpu_shim's whole-graph backward."""
    d = synth.hetero_graph_local('dblp', 2, 0.8, seed=4, scale=0.03)
    g, etv = _setup(d)
    fs, fd, gout, attn, th = _inputs(d, 2, 8, 1)
    want = single(g, etv, fs, fd, gout, attn, th)
    monkeypatch.setattr(ops, 'gatv2_bwd', _GATV2_BWD)
    leaves = [t.clone().requires_grad_(True) for t in (fs, fd, attn, th)]
    out, _ = RF.gatv2_aggregate(g, etv, *leaves, ALPHA, SLOPE)
    out.backward(gout)
    _compare((out.detach(),) + tuple(t.grad for t in leaves), want)


@pytest.mark.parametrize('relational', [True, False])
@pytest.mark.parametrize('shared', [False, True])
def test_halo_gatv2_autograd_one_rank(v2_ops, relational, shared):
    """One row block (no process group needed): halo_gatv2 through autograd equals gatv2_aggregate, with and without
    the relation term, and with one tensor for both sides (shared weights)."""
    d = synth.hetero_graph_local('acm', 1, 0.8, seed=4, scale=0.05)
    g, etv = _setup(d)
    part = partition.HaloPartition.virtual_ranks(g, etv, [0, d['num_nodes']], attention=True)[0]
    fs, fd, gout, attn, th = _inputs(d, 4, 8, 5, relational)
    if shared:
        fd = fs
    leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (fs, fd, attn, th)]
    if shared:
        leaves[1] = leaves[0]
    out = partition.halo_gatv2(part, *leaves, ALPHA, SLOPE)
    out.backward(gout)
    got = (out.detach(), leaves[0].grad, None if shared else leaves[1].grad, leaves[2].grad,
           leaves[3].grad if relational else None)
    _compare(got, single(g, etv, fs, fd, gout, attn, th, shared=shared), d_fd=not shared)


def test_halo_gatv2_refuses_unsupported_inputs(v2_ops):
    d = synth.hetero_graph_local('dblp', 2, 0.8, seed=2, scale=0.03)
    g, etv = _setup(d)
    part = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'], attention=True)[0]
    plain = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'])[0]
    r = d['num_relations']

    def call(p=part, h=2, dim=8, keep=None, th_shape=None, fd_rows=None, exchange=None):
        f = torch.zeros(p.n_own, h, dim, dtype=torch.float64)
        fd = torch.zeros(p.n_own if fd_rows is None else fd_rows, h, dim, dtype=torch.float64)
        a = torch.zeros(1, h, dim, dtype=torch.float64)
        th = torch.zeros(th_shape or (r, h), dtype=torch.float64)
        return partition.halo_gatv2(p, f, fd, a, th, ALPHA, SLOPE, keep=keep, exchange=exchange)
    with pytest.raises(ValueError, match='dropout'):
        call(keep=torch.ones(3, 2))
    with pytest.raises(ValueError, match='attention=True'):
        call(p=plain)
    for h, dim in ((2, 6), (2, 256), (33, 4), (16, 128)):
        with pytest.raises(ValueError, match='fused attention kernels'):
            call(h=h, dim=dim)
    with pytest.raises(ValueError, match='theta'):
        call(th_shape=(r + 1, 2))
    with pytest.raises(ValueError, match='fd_own'):
        call(fd_rows=part.n_own + 1)
    for xch in (types.SimpleNamespace(heads=2, feat=16, gatv2=False), types.SimpleNamespace(heads=2, feat=32, gatv2=True),
                types.SimpleNamespace(heads=4, feat=16, gatv2=True)):
        with pytest.raises(ValueError, match='gatv2=True'):
            call(exchange=xch)
    big = types.SimpleNamespace(max_dpre_rows=2 ** 28)
    with pytest.raises(ValueError, match='32-bit'):
        partition._check_slot_offsets(big, 16, 8)
    partition._check_slot_offsets(big, 8, 8)
