"""GPU tests of attention heads wider than 128 floats (D = 256 and 512) in the fused REGAT / REGATv2 kernels and layers
(``pytest -m gpu``, one B200).

The functional cores, the DGL-API and MAG-stack modules are held to the float64 oracle on graphs whose hub rows take the
long-row fragment path in both CSR views; get_attention rows sum to one; reruns are bit-identical; hashed attention
dropout gives exactly the bits of the explicit oracle mask; the head-sliced layer at world size 1 equals gat_layer; and
the full MAG-shaped graph is checked once per core at H*D = 512 against a chunked float64 evaluation."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import helpers
import re_gnn_b200
import test_attention_dropout_gpu as AD
from test_gpu_parity import RTOL, _attention_float64_full, _theta, mag_full  # noqa: F401  (mag_full: fixture)
from oracle import regnn_oracle as O
from re_gnn_b200 import functional as RF, mag, ops, partition, synth

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
SHAPES = [(1, 256), (2, 256), (4, 256), (1, 512), (2, 512)]
SLOPE = 0.2


@pytest.fixture(scope='module', autouse=True)
def _strict_fp32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


@pytest.fixture(scope='module')
def hub():
    d = AD._hub_graph()
    g, etv = AD._setup(d)
    csr = g.csr()
    assert csr.get('split') is not None and csr.get('split_t') is not None   # the fragment path runs in both views
    return d, g, etv


def _oracle_attention(logits, dst, n):
    return O.edge_softmax(logits, dst, n)


def _row_sums(att, dst, n):
    return torch.zeros(n, att.shape[1], dtype=att.dtype, device=att.device).index_add_(0, dst, att)


@pytest.mark.parametrize('relational', [True, False])
@pytest.mark.parametrize('core', ['gat_layer', 'gat_aggregate', 'gatv2_aggregate'])
@pytest.mark.parametrize('heads,dim', SHAPES)
def test_cores_vs_oracle(hub, heads, dim, core, relational):
    d, g, etv = hub
    n, r = d['num_nodes'], d['num_relations']
    src, dst, et = torch.as_tensor(d['src']), torch.as_tensor(d['dst']), torch.as_tensor(d['etype'])
    rng = np.random.RandomState(heads * 1000 + dim)
    f64 = helpers.f32_exact(rng.randn(n, heads, dim) * 0.5).requires_grad_(True)
    fd64 = helpers.f32_exact(rng.randn(n, heads, dim) * 0.5).requires_grad_(True)
    a64 = helpers.f32_exact(rng.randn(1, heads, dim) * (0.3 / np.sqrt(dim / 64))).requires_grad_(True)
    b64 = helpers.f32_exact(rng.randn(1, heads, dim) * (0.3 / np.sqrt(dim / 64))).requires_grad_(True)
    th64 = _theta(r, heads, dim).requires_grad_(True)
    rel = O.edge_relation(th64, 100.0, et) if relational else 0.0
    if core == 'gatv2_aggregate':
        logits = (F.leaky_relu(f64[src] + fd64[dst], SLOPE) * a64).sum(-1) + rel
        refs, names = [f64, fd64, a64], ['fs', 'fd', 'attn']
    else:
        logits = F.leaky_relu((f64 * a64).sum(-1)[src] + (f64 * b64).sum(-1)[dst] + rel, SLOPE)
        refs, names = [f64, a64, b64], ['feat', 'attn_l', 'attn_r']
    if relational:
        refs, names = refs + [th64], names + ['theta']
    att64 = _oracle_attention(logits, dst, n)
    ref = O.segment_sum(f64[src] * att64[:, :, None], dst, n)
    gout = torch.as_tensor(rng.randn(n, heads, dim))
    ref.backward(gout)

    leaves = [t.detach().to(DEV, torch.float32).requires_grad_(True) for t in (f64, fd64, a64, b64, th64)]
    f, fd, va, vb, th = leaves
    ev = etv if relational else None

    def run():
        if core == 'gat_layer':
            return RF.gat_layer(g, ev, f, va, vb, th, 100.0, SLOPE, want_attn=True)
        if core == 'gat_aggregate':
            return RF.gat_aggregate(g, ev, f, (f * va).sum(-1), (f * vb).sum(-1), th, 100.0, SLOPE, want_attn=True)
        return RF.gatv2_aggregate(g, ev, f, fd, va, th, 100.0, SLOPE, want_attn=True)
    out, att = run()
    tag = '%s H%d D%d rel=%d ' % (core, heads, dim, relational)
    helpers.assert_close(out.detach().cpu(), ref.detach(), RTOL, tag + 'out')
    helpers.assert_close(att.cpu(), att64.detach(), RTOL, tag + 'attention')
    sums = _row_sums(att.double(), dst.to(DEV), n).cpu()
    has_in = torch.bincount(dst, minlength=n) > 0
    assert torch.allclose(sums[has_in], torch.ones_like(sums[has_in]), atol=1e-5), tag + 'attention rows sum to one'
    out.backward(gout.to(DEV, torch.float32))
    ours = [f, fd, va] if core == 'gatv2_aggregate' else [f, va, vb]
    if relational:
        ours = ours + [th]
    for a, b, name in zip(ours, refs, names):
        helpers.assert_close(a.grad.cpu(), b.grad, 2 * RTOL, tag + 'd_' + name)
    # bit-identical rerun
    grads = [t.grad.clone() for t in ours]
    for t in ours:
        t.grad = None
    out2, att2 = run()
    out2.backward(gout.to(DEV, torch.float32))
    assert torch.equal(out2, out) and torch.equal(att2, att), tag + 'rerun'
    for a, b in zip(ours, grads):
        assert torch.equal(a.grad, b), tag + 'rerun gradients'


@pytest.mark.parametrize('kind,out_feats', [('REGATConv', 200), ('REGATConv', 256), ('REGATConv', 512),
                                            ('REGATv2Conv', 200), ('REGATv2Conv', 256), ('REGATv2Conv', 512)])
def test_dgl_modules_vs_oracle(kind, out_feats):
    """Widths 129 .. 512 at the DGL-API layers: powers of two run as they are, others (200) zero-padded to 256."""
    d = synth.hetero_graph('imdb', seed=out_feats, scale=0.03)
    g, et = re_gnn_b200.Graph(d['src'], d['dst'], d['num_nodes']).to(DEV), torch.as_tensor(d['etype'])
    n, r, heads = d['num_nodes'], d['num_relations'], 2
    rng = np.random.RandomState(out_feats)
    mod = getattr(re_gnn_b200, kind)(r, 100.0, 16, out_feats, heads, negative_slope=SLOPE)
    mod.edge_weight.data.copy_(_theta(r, heads, out_feats))
    p64 = {k: v.detach().double().requires_grad_(True) for k, v in mod.named_parameters()}
    x64 = helpers.f32_exact(rng.randn(n, 16)).requires_grad_(True)
    s64, d64 = torch.as_tensor(d['src']), torch.as_tensor(d['dst'])
    if kind == 'REGATConv':
        ref = O.regat_forward(s64, d64, et, n, x64, p64['attn_l'], p64['attn_r'], p64['edge_weight'], 100.0, SLOPE,
                              p64['fc.weight'])
    else:
        ref = O.regatv2_forward(s64, d64, et, n, x64, p64['attn'], p64['edge_weight'], 100.0, SLOPE,
                                (p64['fc_src.weight'], p64['fc_src.bias']), (p64['fc_dst.weight'], p64['fc_dst.bias']))
    gout = helpers.f32_exact(rng.randn(*ref.shape))
    ref.backward(gout)
    mod = mod.to(DEV)
    x = x64.detach().to(DEV, torch.float32).requires_grad_(True)
    out = mod(g, x, et.to(DEV))
    assert tuple(out.shape) == (n, heads, out_feats)
    out.backward(gout.to(DEV, torch.float32))
    helpers.assert_close(out.detach().cpu(), ref.detach(), RTOL, kind + ' out')
    helpers.assert_close(x.grad.cpu(), x64.grad, 1e-4, kind + ' d_x', 1e-4)
    for k, v in mod.named_parameters():
        helpers.assert_close(v.grad.cpu(), p64[k].grad, 1e-4, kind + ' d_' + k, 1e-4)


@pytest.mark.parametrize('kind', ['REGATConv', 'REGATv2Conv'])
def test_mag_modules_vs_oracle(kind):
    """mag.REGATConv / REGATv2Conv at out_channels = 256 (the global-max softmax with its epsilon) on a sampled-block
    shape with a hub destination of more than 256 in-edges."""
    rng = np.random.RandomState(5)
    n_src, n_dst, e, t, r, heads, c, fin = 700, 300, 6000, 3, 4, 2, 256, 24
    src = rng.randint(0, n_src, size=e)
    dst = rng.randint(0, n_dst, size=e)
    dst[:400] = 7                                          # hub row: fragments in the CSR view
    ei = torch.as_tensor(np.stack([src, dst]))
    ety = torch.as_tensor(rng.randint(0, r, size=e))
    tnt = torch.as_tensor(rng.randint(0, t, size=n_dst))
    conv = getattr(mag, kind)(fin, c, t, r, heads=heads, self_loop_type=2)
    with torch.no_grad():
        conv.relation_weight.copy_(_theta(conv.relation_weight.shape[0], heads, 3))
        conv.bias.copy_(torch.as_tensor(rng.randn(heads * c) * 0.1))
    p64 = {k: v.detach().double().requires_grad_(True) for k, v in conv.named_parameters()}
    x64 = helpers.f32_exact(rng.randn(n_src, fin) * 0.5).requires_grad_(True)
    common = (x64, x64[:n_dst], ei, ety, tnt)
    if kind == 'REGATConv':
        ref = O.mag_regat_forward(*common, p64['lin_src.weight'], p64['att_src'], p64['att_dst'], p64['bias'],
                                  p64['relation_weight'], 100.0, r, heads, c, SLOPE, 2)
    else:
        ref = O.mag_regatv2_forward(*common, p64['lin_src.weight'], p64['att'], p64['bias'], p64['relation_weight'],
                                    100.0, r, heads, c, SLOPE, 2)
    gout = helpers.f32_exact(rng.randn(*ref.shape))
    ref.backward(gout)
    conv = conv.to(DEV)
    x = x64.detach().to(DEV, torch.float32).requires_grad_(True)
    out = conv((x, x[:n_dst]), ei.to(DEV), ety.to(DEV), tnt.to(DEV))
    out.backward(gout.to(DEV, torch.float32))
    helpers.assert_close(out.detach().cpu(), ref.detach(), RTOL, kind + ' out')
    helpers.assert_close(x.grad.cpu(), x64.grad, 1e-4, kind + ' d_x', 1e-4)
    for k, p in conv.named_parameters():
        helpers.assert_close(p.grad.cpu(), p64[k].grad, 1e-4, kind + ' d_' + k, 1e-4)


@pytest.mark.parametrize('heads,dim', [(1, 1024), (4, 512), (3, 512)])
def test_kernels_refuse_unsupported_head_shapes(heads, dim):
    """D = 1024 and H*D > 1024 stay refused by the kernels themselves (``unsupported shape``)."""
    n = 64
    feat = torch.randn(n, heads, dim, device=DEV)
    vec = torch.randn(1, heads, dim, device=DEV)
    with pytest.raises(RuntimeError, match='unsupported shape'):
        ops.attn_scores_fwd(feat, vec, vec)


@pytest.mark.parametrize('relational', [True, False])
@pytest.mark.parametrize('heads,dim', [(1, 256), (4, 256), (1, 512), (2, 512)])
def test_hashed_dropout_equals_explicit_oracle_mask(hub, heads, dim, relational):
    d, g, etv = hub
    e, n = d['src'].size, d['num_nodes']
    drop = RF.HashedDropout(AD.P_DROP, AD.KEY)
    f, gout, al, ar, th = AD._gat_inputs(n, d['num_relations'], heads, dim, heads * 131 + dim)
    got = AD._run_gat(g, etv, f, gout, al, ar, th, relational, dropout=drop)
    want = AD._run_gat(g, etv, f, gout, al, ar, th, relational, keep=AD._mask(e, heads))
    AD._assert_equal(got, want, 'gat_layer H=%d D=%d' % (heads, dim))
    assert not torch.equal(got[0], AD._run_gat(g, etv, f, gout, al, ar, th, relational)[0])   # dropout did something
    fd = f.roll(1, 0) * 0.5
    got = AD._run_gatv2(g, etv, f, fd, gout, al, th, relational, dropout=drop)
    want = AD._run_gatv2(g, etv, f, fd, gout, al, th, relational, keep=AD._mask(e, heads))
    AD._assert_equal(got, want, 'gatv2_aggregate H=%d D=%d' % (heads, dim))
    AD._assert_equal(AD._run_gatv2(g, etv, f, fd, gout, al, th, relational, dropout=drop), got, 'rerun')


def test_head_sliced_gat_world1():
    """partition.head_sliced_gat at world size 1 with D = 256 equals functional.gat_layer bit for bit."""
    import torch.distributed as dist
    if not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', str(29900 + os.getpid() % 97))
        dist.init_process_group('nccl', rank=0, world_size=1, device_id=torch.device(DEV))
    try:
        d = synth.hetero_graph('acm', seed=6, scale=0.2)
        g = re_gnn_b200.Graph(d['src'], d['dst'], d['num_nodes']).to(DEV)
        n, r, heads, dim = d['num_nodes'], d['num_relations'], 2, 256
        etv = g.etype_views(torch.as_tensor(d['etype']).to(DEV), r)
        gen = torch.Generator(device=DEV).manual_seed(9)
        f = torch.randn(n, heads, dim, device=DEV, generator=gen) * 0.5
        gout = torch.randn(n, heads, dim, device=DEV, generator=gen)
        al0 = torch.randn(1, heads, dim, device=DEV, generator=gen) * 0.2
        ar0 = torch.randn(1, heads, dim, device=DEV, generator=gen) * 0.2
        th0 = _theta(r, heads, 6).to(DEV, torch.float32)
        bounds = partition.row_blocks(g.csr()['indptr'], 1, balance='rows')
        res = []
        for sharded in (False, True):
            leaves = [t.clone().requires_grad_(True) for t in (f, al0, ar0, th0)]
            if sharded:
                out = partition.head_sliced_gat(g, etv, *leaves, 100.0, SLOPE, bounds, 0)
            else:
                out, _ = RF.gat_layer(g, etv, *leaves, 100.0, SLOPE)
            out.backward(gout)
            res.append([out.detach().clone()] + [t.grad.clone() for t in leaves])
        assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
        for i, name in ((2, 'd_attn_l'), (3, 'd_attn_r'), (4, 'd_theta')):
            helpers.assert_close(res[1][i].cpu(), res[0][i].cpu(), RTOL, 'head-sliced ' + name)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('kind,heads,dim', [('gat', 2, 256), ('v2', 1, 512)])
def test_mag_full_graph_wide_heads_vs_float64(mag_full, kind, heads, dim):
    """The full MAG-shaped graph (N = 1.94 M, E = 23 M, hub rows through the fragment path of both views) at
    H*D = 512: output and every gradient against the chunked float64 evaluation of the same formulas."""
    d, g, et = mag_full
    n, r = d['num_nodes'], d['num_relations']
    csr = g.csr()
    etv = g.etype_views(et, r)
    gen = torch.Generator(device=DEV).manual_seed(heads * 100 + dim)
    scale = 0.3 / np.sqrt(dim / 64)
    f = (torch.randn(n, heads, dim, device=DEV, generator=gen) * 0.5).requires_grad_(True)
    fd = (torch.randn(n, heads, dim, device=DEV, generator=gen) * 0.5).requires_grad_(True)
    va = (torch.randn(1, heads, dim, device=DEV, generator=gen) * scale).requires_grad_(True)
    vb = (torch.randn(1, heads, dim, device=DEV, generator=gen) * scale).requires_grad_(True)
    th = _theta(r, heads, 5).to(DEV, torch.float32).requires_grad_(True)
    gout = torch.randn(n, heads, dim, device=DEV, generator=gen)
    if kind == 'gat':
        out, _ = RF.gat_layer(g, etv, f, va, vb, th, 100.0, SLOPE)
    else:
        out, _ = RF.gatv2_aggregate(g, etv, f, fd, va, th, 100.0, SLOPE)
    out.backward(gout)
    with torch.no_grad():
        ref = _attention_float64_full(kind, csr, etv[0], f.detach(), fd.detach(), va.detach(), vb.detach(), th.detach(),
                                      gout, SLOPE)
    tag = 'MAG full %s h%dd%d ' % (kind, heads, dim)
    helpers.assert_close(out.detach().cpu(), ref[0].cpu(), 2 * RTOL, tag + 'out')
    helpers.assert_close(f.grad.cpu(), ref[1].cpu(), 2 * RTOL, tag + ('d_feat' if kind == 'gat' else 'd_fs'))
    if kind == 'v2':
        helpers.assert_close(fd.grad.cpu(), ref[2].cpu(), 2 * RTOL, tag + 'd_fd')
    helpers.assert_close(va.grad.view(heads, dim).cpu(), ref[3].cpu(), 5 * RTOL, tag + ('d_attn_l' if kind == 'gat' else 'd_attn'))
    if kind == 'gat':
        helpers.assert_close(vb.grad.view(heads, dim).cpu(), ref[4].cpu(), 5 * RTOL, tag + 'd_attn_r')
    helpers.assert_close(th.grad.cpu(), ref[5].cpu(), 5 * RTOL, tag + 'd_theta')
