"""GPU tests of the counter-based attention dropout of the fused REGAT / REGATv2 kernels (``pytest -m gpu``, one B200).

The hashed mode (``dropout=HashedDropout(p, key)``) must give exactly the bits of the explicit-mask mode fed with the
mask of oracle/attn_dropout_oracle.py -- out, get_attention and every gradient -- on graphs whose hub rows take the
fragment path in both views; p = 0 must be the no-dropout result; a head slice must reproduce its heads of the full
layer; the halo row partitions (virtual ranks) must reproduce the single-device core; and the mask the kernels apply
must look like Bernoulli(1 - p) draws."""
import numpy as np
import pytest
import torch

from oracle import attn_dropout_oracle as AO
from re_gnn_b200 import Graph, functional as RF, partition, synth

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
P_DROP = 0.3
KEY = RF.attn_dropout_key(11, 5, 1)


def _hub_graph(n=2500, e=30000, r=5, seed=0):
    """Random multigraph with hub destinations AND hub sources (rows > 256 slots in the CSR and the transposed view)."""
    d = synth.random_multigraph(n, e, r, seed=seed, hubs=3)
    rng = np.random.RandomState(seed + 1)
    hub = rng.rand(d['src'].size) < 0.15
    d['src'][hub] = n - 1 - rng.randint(0, 3, size=int(hub.sum()))
    return d


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(DEV)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(DEV), d['num_relations'])
    return g, etv


def _mask(num_edges, heads, p=P_DROP, key=KEY, offset=0, total=None):
    return torch.as_tensor(AO.keep_mask(p, key, num_edges, heads, offset, total)).to(DEV)


def _gat_inputs(n, r, heads, dim, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    f = torch.randn(n, heads, dim, device=DEV, generator=gen)
    gout = torch.randn(n, heads, dim, device=DEV, generator=gen)
    al = torch.randn(1, heads, dim, device=DEV, generator=gen) * 0.3
    ar = torch.randn(1, heads, dim, device=DEV, generator=gen) * 0.3
    th = (torch.rand(r, heads, device=DEV, generator=gen) + 0.5) / 100
    return f, gout, al, ar, th


def _run_gat(g, etv, f, gout, al, ar, th, relational=True, **kw):
    leaves = [t.clone().requires_grad_(True) for t in (f, al, ar, th)]
    out, att = RF.gat_layer(g, etv if relational else None, *leaves, 100.0, 0.2, want_attn=True, **kw)
    out.backward(gout)
    return (out.detach(), att) + tuple(t.grad for t in leaves[:3]) + ((leaves[3].grad,) if relational else ())


def _run_gatv2(g, etv, fs, fd, gout, attn, th, relational=True, **kw):
    leaves = [t.clone().requires_grad_(True) for t in (fs, fd, attn, th)]
    out, att = RF.gatv2_aggregate(g, etv if relational else None, *leaves, 100.0, 0.2, want_attn=True, **kw)
    out.backward(gout)
    return (out.detach(), att) + tuple(t.grad for t in leaves[:3]) + ((leaves[3].grad,) if relational else ())


def _assert_equal(got, want, what):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        assert torch.equal(a, b), '%s: result %d differs (max |diff| %.3g)' % (what, i, float((a - b).abs().max()))


@pytest.fixture(scope='module')
def hub():
    d = _hub_graph()
    g, etv = _setup(d)
    csr = g.csr()
    assert csr.get('split') is not None and csr.get('split_t') is not None   # the fragment path runs in both views
    return d, g, etv


@pytest.mark.parametrize('relational', [True, False])
@pytest.mark.parametrize('dim', [4, 16, 64, 128])
@pytest.mark.parametrize('heads', [1, 4, 8])
def test_gat_hashed_equals_explicit_oracle_mask(hub, heads, dim, relational):
    d, g, etv = hub
    e = d['src'].size
    f, gout, al, ar, th = _gat_inputs(d['num_nodes'], d['num_relations'], heads, dim, heads * 131 + dim)
    drop = RF.HashedDropout(P_DROP, KEY)
    got = _run_gat(g, etv, f, gout, al, ar, th, relational, dropout=drop)
    want = _run_gat(g, etv, f, gout, al, ar, th, relational, keep=_mask(e, heads))
    _assert_equal(got, want, 'gat_layer H=%d D=%d' % (heads, dim))
    assert not torch.equal(got[0], _run_gat(g, etv, f, gout, al, ar, th, relational)[0])   # dropout did something
    _assert_equal(_run_gat(g, etv, f, gout, al, ar, th, relational, dropout=drop), got, 'rerun')


@pytest.mark.parametrize('relational', [True, False])
@pytest.mark.parametrize('dim', [4, 16, 64, 128])
@pytest.mark.parametrize('heads', [1, 4, 8])
def test_gatv2_hashed_equals_explicit_oracle_mask(hub, heads, dim, relational):
    d, g, etv = hub
    e, n = d['src'].size, d['num_nodes']
    fs, gout, attn, _, th = _gat_inputs(n, d['num_relations'], heads, dim, heads * 37 + dim)
    fd = fs.roll(1, 0) * 0.5
    drop = RF.HashedDropout(P_DROP, KEY)
    got = _run_gatv2(g, etv, fs, fd, gout, attn, th, relational, dropout=drop)
    want = _run_gatv2(g, etv, fs, fd, gout, attn, th, relational, keep=_mask(e, heads))
    _assert_equal(got, want, 'gatv2_aggregate H=%d D=%d' % (heads, dim))
    _assert_equal(_run_gatv2(g, etv, fs, fd, gout, attn, th, relational, dropout=drop), got, 'rerun')


def test_gat_aggregate_hashed_equals_explicit(hub):
    """The MAG-stack entry (el / er from the caller, with the global-max softmax epsilon)."""
    d, g, etv = hub
    n, e, heads, dim = d['num_nodes'], d['src'].size, 4, 16
    gen = torch.Generator(device=DEV).manual_seed(3)
    feat, gout = (torch.randn(n, heads, dim, device=DEV, generator=gen) for _ in range(2))
    el, er = (torch.randn(n, heads, device=DEV, generator=gen) for _ in range(2))
    th = (torch.rand(d['num_relations'], heads, device=DEV, generator=gen) + 0.5) / 100

    def run(**kw):
        leaves = [t.clone().requires_grad_(True) for t in (feat, el, er, th)]
        out, att = RF.gat_aggregate(g, etv, *leaves, 100.0, 0.2, want_attn=True, softmax_eps=1e-16, **kw)
        out.backward(gout)
        return (out.detach(), att) + tuple(t.grad for t in leaves)
    _assert_equal(run(dropout=RF.HashedDropout(P_DROP, KEY)), run(keep=_mask(e, heads)), 'gat_aggregate')


def test_p_zero_is_no_dropout(hub):
    d, g, etv = hub
    f, gout, al, ar, th = _gat_inputs(d['num_nodes'], d['num_relations'], 4, 16, 5)
    _assert_equal(_run_gat(g, etv, f, gout, al, ar, th, dropout=RF.HashedDropout(0.0, KEY)),
                  _run_gat(g, etv, f, gout, al, ar, th), 'gat_layer p=0')
    _assert_equal(_run_gatv2(g, etv, f, ar.expand_as(f).contiguous(), gout, al, th, dropout=RF.HashedDropout(0.0, KEY)),
                  _run_gatv2(g, etv, f, ar.expand_as(f).contiguous(), gout, al, th), 'gatv2_aggregate p=0')


@pytest.mark.parametrize('offset', [0, 2, 6])
def test_head_slice_reproduces_full_heads(hub, offset):
    """A call over heads [offset, offset + 2) of an 8-head layer (head_offset / num_heads_total) gives that slice of the
    full-H run bit for bit: out, get_attention and the feature gradients (the parameter gradients are reductions over
    another block layout: norm-wise)."""
    d, g, etv = hub
    heads, hs, dim = 8, 2, 16
    sl = slice(offset, offset + hs)
    f, gout, al, ar, th = _gat_inputs(d['num_nodes'], d['num_relations'], heads, dim, 17)
    drop = RF.HashedDropout(P_DROP, KEY)
    full = _run_gat(g, etv, f, gout, al, ar, th, dropout=drop)
    part = _run_gat(g, etv, *(t[:, sl].contiguous() for t in (f, gout, al, ar, th)),
                    dropout=drop.for_heads(offset, heads))
    for i in range(3):
        assert torch.equal(part[i], full[i][:, sl].contiguous()), i
    for i in (3, 4, 5):
        assert float((part[i] - full[i][:, sl]).norm() / full[i][:, sl].norm()) < 1e-6, i
    fv = _run_gatv2(g, etv, f, f.flip(0).contiguous(), gout, al, th, dropout=drop)
    pv = _run_gatv2(g, etv, *(t[:, sl].contiguous() for t in (f, f.flip(0), gout, al, th)),
                    dropout=drop.for_heads(offset, heads))
    for i in range(4):
        assert torch.equal(pv[i], fv[i][:, sl].contiguous()), i


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize('exchange', [False, True])
@pytest.mark.parametrize('parts', [2, 4])
def test_virtual_halo_gat_with_dropout(parts, exchange):
    d = synth.hetero_graph_local('mag', parts, 0.9, seed=7, scale=0.04)
    g, etv = _setup(d)
    plist = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'], attention=True)
    heads, dim = 8, 16
    f, gout, al, ar, th = _gat_inputs(d['num_nodes'], d['num_relations'], heads, dim, parts)
    drop = RF.HashedDropout(P_DROP, KEY)
    r_out, _, r_f, r_al, r_ar, r_th = _run_gat(g, etv, f, gout, al, ar, th, dropout=drop)
    out, d_f, d_al, d_ar, d_th = partition._virtual_halo_gat(plist, f, gout, al, ar, th, 100.0, 0.2, scatter=exchange,
                                                             dropout=drop)
    assert torch.equal(out, r_out)
    assert torch.equal(d_f, r_f)
    assert max(_rel(d_al, r_al.view(-1)), _rel(d_ar, r_ar.view(-1)), _rel(d_th, r_th)) < 1e-6
    assert not torch.equal(out, _run_gat(g, etv, f, gout, al, ar, th)[0])


@pytest.mark.parametrize('exchange', [False, True])
@pytest.mark.parametrize('parts', [2, 4])
def test_virtual_halo_gatv2_with_dropout(parts, exchange):
    d = synth.hetero_graph_local('mag', parts, 0.9, seed=7, scale=0.04)
    g, etv = _setup(d)
    plist = partition.HaloPartition.virtual_ranks(g, etv, d['community_bounds'], attention=True)
    heads, dim = 8, 16
    fs, gout, attn, _, th = _gat_inputs(d['num_nodes'], d['num_relations'], heads, dim, parts + 50)
    fd = fs.roll(1, 0) * 0.5
    drop = RF.HashedDropout(P_DROP, KEY)
    r_out, _, r_fs, r_fd, r_attn, r_th = _run_gatv2(g, etv, fs, fd, gout, attn, th, dropout=drop)
    out, d_fs, d_fd, d_attn, d_th = partition._virtual_halo_gatv2(plist, fs, fd, gout, attn, th, 100.0, 0.2,
                                                                  push=exchange, dropout=drop)
    assert torch.equal(out, r_out)
    assert torch.equal(d_fs, r_fs)
    assert torch.equal(d_fd, r_fd)
    assert max(_rel(d_attn, r_attn.view(-1)), _rel(d_th, r_th)) < 1e-6


def test_kept_fraction_and_independence():
    """The mask the forward kernel applies, read back through get_attention (el = er = 0, no relations: every edge's
    attention is 1/deg > 0 unless dropped): per head the kept fraction is within 5 sigma of 1 - p over E, and the
    indicators of two steps, of two layers and of neighbouring heads are uncorrelated (|r| < 5 / sqrt(E))."""
    n, e, heads, dim, p = 200000, 2000000, 8, 4, 0.25
    d = synth.random_multigraph(n, e, 1, seed=9, hubs=0, self_loops=False)
    g = Graph(d['src'], d['dst'], n).to(DEV)
    feat = torch.zeros(n, heads, dim, device=DEV)
    z = torch.zeros(n, heads, device=DEV)

    def kept(step, layer=0):
        _, att = RF.gat_aggregate(g, None, feat, z, z, None, 1.0, 0.2, want_attn=True,
                                  dropout=RF.HashedDropout(p, RF.attn_dropout_key(3, step, layer)))
        return (att > 0).double()
    k0, k1, k2 = kept(0), kept(1), kept(0, layer=1)
    sigma = (p * (1 - p) / e) ** 0.5
    frac = k0.mean(0)
    assert float((frac - (1 - p)).abs().max()) < 5 * sigma, frac.tolist()

    def corr(a, b):
        a, b = a - a.mean(), b - b.mean()
        return float((a * b).mean() / (a.std() * b.std()))
    bound = 5 / e ** 0.5
    for h in range(heads):
        assert abs(corr(k0[:, h], k1[:, h])) < bound
        assert abs(corr(k0[:, h], k2[:, h])) < bound
    for h in range(heads - 1):
        assert abs(corr(k0[:, h], k0[:, h + 1])) < bound
    # and it is the oracle's mask
    assert torch.equal(k0.float(), (_mask(e, heads, p, RF.attn_dropout_key(3, 0, 0)) > 0).float())
