"""Every head shape of the fused REGAT / REGATv2 kernels against a float64 reference (``pytest -m gpu``, one B200).

The attention entry points take any H in [1, 32] and any power-of-two D in [4, 512] with H*D <= 1024 (158 shapes), and
dispatch each shape to one of 20 kernel classes (G, LPH, CPL).  Here every shape runs through the three cores --
``gat_layer`` with relations, ``gat_aggregate`` without, ``gatv2_aggregate`` with relations -- on a graph whose rows and
columns have the degrees where the row-group and fragment mappings change (0 .. 9, 31 .. 33, 255 .. 257, 511 .. 513),
with inputs exact in fp32 so that LeakyReLU pre-activations of exactly 0 occur and the reference and the kernels agree
on the side of every kink.  Then: rows whose logits stress the online softmax and the fragment merge (a maximum 45
above the rest in the first or the last fragment, increasing logits, offsets of +-200, all weights but one exactly 0);
the fused d_er + relation-bin reduction of graphs with >= 65,536 rows at every H; relation tables at the ABI limits.

``REGNN_TEST_DEVICE=cpu`` runs the reference and the test logic against tests/cpu_shim.py (no hashed dropout, no
kernel refusals there)."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import helpers
from oracle import attn_dropout_oracle as AO, csr_oracle, regnn_oracle as O
from re_gnn_b200 import Graph, functional as RF, ops

pytestmark = pytest.mark.gpu
DEV = os.environ.get('REGNN_TEST_DEVICE', 'cuda:0')   # 'cpu' + tests/cpu_shim.py = dry run of the test code itself

ALPHA = 4.0          # a power of two: alpha * theta is exact
SLOPE = 0.2
P_DROP = 0.3
KEY = RF.attn_dropout_key(23, 7, 2)
CORES = ('gat_layer', 'gat_aggregate', 'gatv2_aggregate')
# every (H, D) the attention entry points accept
SHAPES = [(h, d) for d in (4 << i for i in range(8)) for h in range(1, 33) if h * d <= 1024]
BOUNDARY_DEGREES = (0, 1, 2, 3, 4, 5, 7, 8, 9, 31, 32, 33, 255, 256, 257, 511, 512, 513)
NODE_GRADS = ('feat', 'el', 'er', 'fs', 'fd')
TOL_OUT, TOL_NODE, TOL_PARAM = 1e-5, 2e-5, 5e-5


def kernel_class(heads, dim):
    """(G, LPH, CPL) of the dispatch in csrc/gat.cu: lanes per row slice rg_lanes(H*D), lanes per head, 128-bit chunks
    per lane."""
    hd = heads * dim
    g = 32 if hd > 64 else 16 if hd > 32 else 8 if hd > 16 else 4
    return g, min(g, dim // 4), dim // 128 if dim > 128 else 1


@pytest.fixture(scope='module', autouse=True)
def _strict_fp32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


@pytest.fixture(scope='module', autouse=True)
def _dry_run_shim():
    """Module scope: the graph fixtures below are module-scoped too."""
    with pytest.MonkeyPatch.context() as mp:
        if DEV == 'cpu':
            import cpu_shim
            cpu_shim.install(mp)
        yield


# ---- graphs --------------------------------------------------------------------------------------------------------
def boundary_graph(num_nodes=3000, bulk_edges=20000, num_relations=5, seed=0):
    """Nodes 0..17 have the in-degrees BOUNDARY_DEGREES, nodes 18..35 those out-degrees; the other nodes carry a random
    multigraph (duplicate edges on purpose), the last 100 of them have no in-edges.  Edge ids are shuffled, so slot
    order is not construction order.  The structure does not depend on ``num_relations``."""
    rng = np.random.RandomState(seed)
    k = len(BOUNDARY_DEGREES)
    fill = np.arange(2 * k, num_nodes)
    fill_dst = np.arange(2 * k, num_nodes - 100)
    src, dst = [], []
    for i, deg in enumerate(BOUNDARY_DEGREES):
        s = rng.choice(fill, size=deg)
        t = rng.choice(fill_dst, size=deg)
        if deg >= 4:              # a duplicate edge in each view
            s[1], t[1] = s[0], t[0]
        src += [s, np.full(deg, k + i)]
        dst += [np.full(deg, i), t]
    src.append(rng.choice(fill, size=bulk_edges))
    dst.append(rng.choice(fill_dst, size=bulk_edges))
    src, dst = np.concatenate(src).astype(np.int64), np.concatenate(dst).astype(np.int64)
    perm = rng.permutation(src.size)
    src, dst = src[perm], dst[perm]
    etype = np.random.RandomState(seed + 1).randint(1, num_relations + 1, size=src.size).astype(np.int64)
    return dict(src=src, dst=dst, etype=etype, num_nodes=num_nodes, num_relations=num_relations,
                dst_nodes=np.arange(k), src_nodes=np.arange(k, 2 * k))


def boundary_degrees(d, csr):
    """(in-degrees of d['dst_nodes'], out-degrees of d['src_nodes']) read from a built CSR (numpy arrays)."""
    ip, ipt = np.asarray(csr['indptr']), np.asarray(csr['indptr_t'])
    return (ip[d['dst_nodes'] + 1] - ip[d['dst_nodes']], ipt[d['src_nodes'] + 1] - ipt[d['src_nodes']])


def large_graph(num_nodes=70000, num_edges=140000, num_relations=7, seed=3):
    """Sparse graph with more than 65,536 rows (the fused d_er + relation-bin pass) and two hub rows (fragments)."""
    rng = np.random.RandomState(seed)
    src = rng.randint(0, num_nodes, size=num_edges).astype(np.int64)
    dst = rng.randint(0, num_nodes, size=num_edges).astype(np.int64)
    dst[rng.permutation(num_edges)[:1000]] = np.repeat([11, 12345], [300, 700])
    etype = rng.randint(1, num_relations + 1, size=num_edges).astype(np.int64)
    return dict(src=src, dst=dst, etype=etype, num_nodes=num_nodes, num_relations=num_relations)


EXTREME_ROWS = (257, 513, 1100, 1, 2, 3, 5, 9, 33)   # rows 0..8: hub rows (fragments) and short rows
CONTROL_ROWS = 64                                     # rows 9..72: 6 in-edges each, ordinary logits


def extreme_graph(seed=5):
    """Rows 0..8 with EXTREME_ROWS in-edges and CONTROL_ROWS rows of 6, every edge from its own source node, edge ids
    shuffled."""
    rng = np.random.RandomState(seed)
    degs = EXTREME_ROWS + (6,) * CONTROL_ROWS
    dst = np.repeat(np.arange(len(degs)), degs)
    src = len(degs) + np.arange(dst.size)
    perm = rng.permutation(dst.size)
    src, dst = src[perm].astype(np.int64), dst[perm].astype(np.int64)
    etype = rng.randint(1, 4, size=dst.size).astype(np.int64)
    return dict(src=src, dst=dst, etype=etype, num_nodes=len(degs) + dst.size, num_relations=3)


def _setup(d):
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(DEV)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(DEV), d['num_relations'])
    idx = {k: torch.as_tensor(d[k]).to(DEV) for k in ('src', 'dst', 'etype')}
    return g, etv, idx


@pytest.fixture(scope='module')
def bgraph():
    d = boundary_graph()
    g, etv, idx = _setup(d)
    csr = g.csr()
    ins, outs = boundary_degrees(d, {k: csr[k].cpu() for k in ('indptr', 'indptr_t')})
    assert ins.tolist() == list(BOUNDARY_DEGREES) and outs.tolist() == list(BOUNDARY_DEGREES)
    if DEV != 'cpu':
        assert csr.get('split') is not None and csr.get('split_t') is not None   # fragments in both views
    return d, g, etv, idx


@pytest.fixture(scope='module')
def lgraph():
    d = large_graph()
    return (d,) + _setup(d)


# ---- inputs exact in fp32 ------------------------------------------------------------------------------------------
def _dyadic(rng, shape, den=8, kmax=8):
    """float64 k / den, |k| <= kmax (den a power of two): exact in fp32, and so are sums of a few thousand of them."""
    return torch.as_tensor(rng.randint(-kmax, kmax + 1, size=shape) / float(den))


def _attn_den(dim):
    """Power-of-two denominator of the attention vectors, growing with sqrt(D): logits stay within a few units."""
    return 2 ** (2 + (int(math.log2(dim)) + 1) // 2)


def _theta(rng, r, heads):
    """k / 64, 0 <= k <= 8, relation 1 all zero: LeakyReLU(alpha * theta) is exact and d_theta meets its kink."""
    t = rng.randint(0, 9, size=(r, heads)) / 64.0
    t[0] = 0.0
    return torch.as_tensor(t)


def make_inputs(core, n, r, heads, dim, seed, relational=True):
    """float64 leaves (CPU) of one core: feat / fs / fd and el / er dyadic k/8; attention vectors dyadic with a
    D-dependent scale; for gat_layer a tenth of the feature rows are 0, so el = er = 0 there and edges between two
    such nodes of relation 1 (theta = 0) have a pre-activation of exactly 0."""
    rng = np.random.RandomState(seed)
    den = _attn_den(dim)
    x = {}
    if core == 'gatv2_aggregate':
        x['fs'] = _dyadic(rng, (n, heads, dim))
        x['fd'] = _dyadic(rng, (n, heads, dim))
        x['attn'] = _dyadic(rng, (1, heads, dim), den)
    else:
        x['feat'] = _dyadic(rng, (n, heads, dim))
        if core == 'gat_layer':
            x['feat'][rng.rand(n) < 0.1] = 0.0
            x['attn_l'] = _dyadic(rng, (1, heads, dim), den)
            x['attn_r'] = _dyadic(rng, (1, heads, dim), den)
        else:
            x['el'] = _dyadic(rng, (n, heads))
            x['er'] = _dyadic(rng, (n, heads))
    if relational:
        x['theta'] = _theta(rng, r, heads)
    gout = helpers.f32_exact(rng.randn(n, heads, dim))
    return x, gout


# ---- float64 reference ---------------------------------------------------------------------------------------------
def reference(core, idx, n, x, gout, alpha=ALPHA, slope=SLOPE, keep=None, device=None):
    """float64 forward and backward of one core by plain autograd on ``device`` (default: the test device), from the
    definitions in oracle/regnn_oracle.py: logits, per-destination softmax with the row maximum subtracted, optional
    [E, H] keep factors applied after the softmax, aggregation.  -> dict(out, attn = a * keep in edge-id order,
    rowmax, rowsum (0 on rows without in-edges, as the kernels), ties = number of exactly-zero LeakyReLU inputs,
    grads = {name: gradient of x[name]})."""
    device = DEV if device is None else device
    src, dst = idx['src'].to(device), idx['dst'].to(device)
    leaves = {k: v.detach().to(device, torch.float64).requires_grad_(True) for k, v in x.items()}
    theta = leaves.get('theta')
    rel = O.edge_relation(theta, alpha, idx['etype'].to(device)) if theta is not None else 0.0
    if core == 'gatv2_aggregate':
        q = leaves['fs'][src] + leaves['fd'][dst]
        ties = int((q == 0).sum())
        logit = (F.leaky_relu(q, slope) * leaves['attn']).sum(-1) + rel
        msg = leaves['fs']
    else:
        if core == 'gat_layer':
            el = (leaves['feat'] * leaves['attn_l']).sum(-1)
            er = (leaves['feat'] * leaves['attn_r']).sum(-1)
        else:
            el, er = leaves['el'], leaves['er']
        pre = el[src] + er[dst] + rel
        ties = int((pre == 0).sum())
        logit = F.leaky_relu(pre, slope)
        msg = leaves['feat']
    h = logit.shape[1]
    rowmax = torch.full((n, h), float('-inf'), dtype=torch.float64, device=device).scatter_reduce(
        0, dst[:, None].expand_as(logit), logit.detach(), 'amax', include_self=True)
    rowmax = torch.where(torch.isinf(rowmax), torch.zeros_like(rowmax), rowmax)
    ex = torch.exp(logit - rowmax[dst])
    rowsum = torch.zeros((n, h), dtype=torch.float64, device=device).index_add(0, dst, ex)
    a = ex / rowsum[dst]
    if keep is not None:
        a = a * keep.to(device, torch.float64)
    out = torch.zeros(msg.shape, dtype=torch.float64, device=device).index_add(0, dst, a[:, :, None] * msg[src])
    out.backward(gout.to(device, torch.float64))
    return dict(out=out.detach(), attn=a.detach(), rowmax=rowmax, rowsum=rowsum.detach(), ties=ties,
                grads={k: v.grad for k, v in leaves.items()})


# ---- kernel runs ---------------------------------------------------------------------------------------------------
def run_core(core, g, etv, x, gout, slope=SLOPE, backward=True, **kw):
    """One call of a functional core on fp32 copies of ``x`` -> (out, attention | None, {name: gradient})."""
    t = {k: v.detach().to(DEV, torch.float32).requires_grad_(True) for k, v in x.items()}
    th = t.get('theta')
    ev = etv if th is not None else None
    if core == 'gat_layer':
        out, att = RF.gat_layer(g, ev, t['feat'], t['attn_l'], t['attn_r'], th, ALPHA, slope, **kw)
    elif core == 'gat_aggregate':
        out, att = RF.gat_aggregate(g, ev, t['feat'], t['el'], t['er'], th, ALPHA, slope, **kw)
    else:
        out, att = RF.gatv2_aggregate(g, ev, t['fs'], t['fd'], t['attn'], th, ALPHA, slope, **kw)
    if not backward:
        return out.detach(), att, {}
    out.backward(gout.to(DEV, torch.float32))
    return out.detach(), att, {k: v.grad for k, v in t.items()}


def check_vs_reference(tag, got, ref, attention=True):
    out, att, grads = got
    helpers.assert_close(out.cpu(), ref['out'].cpu(), TOL_OUT, tag + 'out')
    if attention:
        helpers.assert_close(att.cpu(), ref['attn'].cpu(), TOL_OUT, tag + 'attention')
    assert set(grads) == set(ref['grads'])
    for k, gr in grads.items():
        helpers.assert_close(gr.cpu(), ref['grads'][k].cpu(), TOL_NODE if k in NODE_GRADS else TOL_PARAM, tag + 'd_' + k)


def assert_same_bits(tag, a, b):
    (oa, aa, ga), (ob, ab, gb) = a, b
    assert torch.equal(oa, ob), tag + 'out differs'
    assert torch.equal(aa, ab), tag + 'attention differs'
    for k in ga:
        assert torch.equal(ga[k], gb[k]), tag + 'd_' + k + ' differs'


# ---- the sweep -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('core', CORES)
@pytest.mark.parametrize('heads,dim', SHAPES, ids=['H%dD%d' % s for s in SHAPES])
def test_every_head_shape_vs_float64(bgraph, heads, dim, core):
    d, g, etv, idx = bgraph
    n, e = d['num_nodes'], d['src'].size
    x, gout = make_inputs(core, n, d['num_relations'], heads, dim, seed=heads * 1000 + dim,
                          relational=core != 'gat_aggregate')
    tag = '%s H%d D%d %s ' % (core, heads, dim, kernel_class(heads, dim))
    ref = reference(core, idx, n, x, gout)
    assert ref['ties'] > 0, tag + 'no exactly-zero LeakyReLU input'
    if 'theta' in x:
        assert bool((x['theta'] == 0).any())
    plain = run_core(core, g, etv, x, gout)
    check_vs_reference(tag, plain, ref, attention=False)
    # get_attention without a mask: the same output bits, attention rows of the reference
    out, att, _ = run_core(core, g, etv, x, gout, backward=False, want_attn=True)
    assert torch.equal(out, plain[0]), tag + 'want_attn changed out'
    helpers.assert_close(att.cpu(), ref['attn'].cpu(), TOL_OUT, tag + 'attention')
    # an explicit [E, H] keep mask (the one the hash gives), against the reference with that mask
    keep = torch.as_tensor(AO.keep_mask(P_DROP, KEY, e, heads))
    ref_k = reference(core, idx, n, x, gout, keep=keep)
    masked = run_core(core, g, etv, x, gout, want_attn=True, keep=keep.to(DEV))
    check_vs_reference(tag + 'keep ', masked, ref_k)
    if DEV != 'cpu':
        hashed = run_core(core, g, etv, x, gout, want_attn=True, dropout=RF.HashedDropout(P_DROP, KEY))
        assert_same_bits(tag + 'hashed ', hashed, masked)


# ---- extreme logits and the fragment merge -------------------------------------------------------------------------
PATTERNS = ('late_max', 'early_max', 'increasing', 'offset_plus', 'offset_minus', 'underflow')
X_SLOPE = 0.25   # a power of two: with dyadic inputs every logit below is exact in fp32


def _pattern_logits(pattern, pos, deg, base):
    """Target logit of the slot at position ``pos`` of a row of ``deg`` slots (float64, dyadic); ``base``: ordinary
    logits in [-2, 2]."""
    if pattern == 'late_max':                                          # more than 40 above the rest, last fragment
        return np.where(pos == deg - 1, 45.0, base)
    if pattern == 'early_max':
        return np.where(pos == 0, 45.0, base)
    if pattern == 'increasing':                                        # every batch raises the running maximum
        return -16.0 + pos / 32.0
    if pattern == 'offset_plus':                                       # exp overflows fp32 without the max subtraction
        return base + 200.0
    if pattern == 'offset_minus':                                      # ... and underflows to 0 / 0
        return base - 200.0
    return np.where(pos == deg // 2, 1.0, -1000.0)                     # exp(-1000) is 0 in float64 too


def _inv_leaky(logit, slope):
    return np.where(logit > 0, logit, logit / slope)


def _extreme_inputs(core, d, pattern, heads, dim):
    """Inputs whose logit on each in-edge of rows 0..8 is the pattern's target plus a small exact term (relation
    weight, and for REGATv2 the other components of the attention dot product).  The control rows keep ordinary
    logits: a row dominated by one edge has logit gradients far below the fp32 resolution of the terms they cancel
    from, and the control rows give the norm-wise bound of every gradient an ordinary scale."""
    n, e = d['num_nodes'], d['src'].size
    rng = np.random.RandomState(PATTERNS.index(pattern) * 10 + CORES.index(core))
    c = csr_oracle.csr_build(d['src'], d['dst'], n)
    pos = np.empty(e, dtype=np.int64)                                  # position of every edge in its row's slots
    pos[c['eid']] = np.arange(e) - c['indptr'][c['row']]
    deg = np.diff(c['indptr'])[d['dst']]
    base = rng.randint(-16, 17, size=e) / 8.0
    logit = np.where(d['dst'] < len(EXTREME_ROWS), _pattern_logits(pattern, pos, deg, base), base)
    pre = torch.as_tensor(_inv_leaky(logit, X_SLOPE))
    x, gout = make_inputs(core, n, d['num_relations'], heads, dim, seed=rng.randint(1 << 30))
    src = torch.as_tensor(d['src'])
    if core == 'gat_aggregate':
        x['el'][src] = pre[:, None]
        x['er'][:len(EXTREME_ROWS)] = 0.0
    else:
        # the +-200 offset through fd of the destination, so that the messages fs stay small: the gradient of a constant
        # shift of a row's logits is 0, and its fp32 rounding grows with the messages
        shift = {'offset_plus': 200.0, 'offset_minus': -200.0 / X_SLOPE}.get(pattern, 0.0)
        x['fs'][src, :, 0] = pre[:, None] - torch.as_tensor(np.where(d['dst'] < len(EXTREME_ROWS), shift, 0.0))[:, None]
        x['fd'][:len(EXTREME_ROWS), :, 0] = shift
        x['attn'][..., 0] = 1.0
        x['attn'][..., 1:] = torch.as_tensor(rng.randint(-2, 3, size=(1, heads, dim - 1)) / 1024.0)
    return x, gout


@pytest.mark.parametrize('pattern', PATTERNS)
@pytest.mark.parametrize('core,heads,dim', [('gat_aggregate', 4, 32), ('gatv2_aggregate', 2, 64)])
def test_extreme_logits_and_fragment_merge(core, heads, dim, pattern):
    d = extreme_graph()
    g, etv, idx = _setup(d)
    if DEV != 'cpu':
        assert g.csr().get('split') is not None
    n = d['num_nodes']
    x, gout = _extreme_inputs(core, d, pattern, heads, dim)
    tag = '%s %s ' % (core, pattern)
    ref = reference(core, idx, n, x, gout, slope=X_SLOPE)
    # the row statistics of the forward kernel itself
    t = {k: v.to(DEV, torch.float32) for k, v in x.items()}
    csr = g.csr()
    if core == 'gat_aggregate':
        _, rowmax, rowsum, _ = ops.gat_fwd(csr, etv[0], t['theta'], ALPHA, t['feat'], t['el'], t['er'], X_SLOPE)
        # exact logits: the maximum is one of them
        assert torch.equal(rowmax.double().cpu(), ref['rowmax'].cpu()), tag + 'rowmax'
    else:
        _, rowmax, rowsum, _, _ = ops.gatv2_fwd(csr, etv[0], t['theta'], ALPHA, t['fs'], t['fd'], t['attn'], X_SLOPE)
        # a dot product over D in fp32; the floor of 1 covers logits near 0, whose error is absolute
        err = (rowmax.double().cpu() - ref['rowmax'].cpu()).abs()
        assert bool((err <= 1e-6 * ref['rowmax'].cpu().abs().clamp(min=1.0)).all()), tag + 'rowmax %.3g' % float(err.max())
    helpers.assert_close(rowsum.cpu(), ref['rowsum'].cpu(), TOL_OUT, tag + 'rowsum')
    got = run_core(core, g, etv, x, gout, slope=X_SLOPE, want_attn=True)
    check_vs_reference(tag, got, ref)
    if pattern == 'underflow':   # all weights but one per row are exactly 0
        att = got[1].cpu()
        assert int((att == 0).sum()) == int((ref['attn'].cpu() == 0).sum()) > 0


# ---- the fused d_er + relation-bin reduction (>= 65,536 rows) at every H -------------------------------------------
@pytest.mark.parametrize('heads', range(1, 33))
def test_large_graph_reduction_every_head_count(lgraph, heads):
    d, g, etv, idx = lgraph
    n = d['num_nodes']
    assert n >= 65536
    x, gout = make_inputs('gat_aggregate', n, d['num_relations'], heads, 4, seed=heads)
    ref = reference('gat_aggregate', idx, n, x, gout)
    assert ref['ties'] > 0
    # d_er is the per-row sum of the logit gradients itself, d_theta their relation bins
    check_vs_reference('large N H%d ' % heads, run_core('gat_aggregate', g, etv, x, gout), ref, attention=False)


# ---- relation tables at the ABI limits -----------------------------------------------------------------------------
@pytest.mark.parametrize('which', ['boundary', 'large'])
@pytest.mark.parametrize('core', ['gat_layer', 'gatv2_aggregate'])
@pytest.mark.parametrize('r,heads', [(200, 1), (200, 20), (128, 32)])
def test_relation_table_limits(r, heads, core, which):
    d = boundary_graph(num_relations=r) if which == 'boundary' else large_graph(num_relations=r)
    g, etv, idx = _setup(d)
    n, dim = d['num_nodes'], 8
    assert int(np.unique(d['etype']).size) == r
    x, gout = make_inputs(core, n, r, heads, dim, seed=r + heads)
    ref = reference(core, idx, n, x, gout)
    check_vs_reference('%s %s R%d H%d ' % (which, core, r, heads), run_core(core, g, etv, x, gout), ref,
                       attention=False)


@pytest.mark.parametrize('core', ['gat_layer', 'gatv2_aggregate'])
@pytest.mark.parametrize('r,heads', [(129, 32), (201, 1)])
def test_relation_tables_past_the_limits_are_refused(bgraph, core, r, heads):
    """R * H = 4128 > 4096 and R = 201 > REGNN_MAX_RELATIONS: the kernels refuse (REGNN_ERR_UNSUPPORTED_SHAPE)."""
    if DEV == 'cpu':
        pytest.skip('the refusal is the kernels\'')
    d = boundary_graph(num_relations=min(r, 200))
    g, etv, _ = _setup(d)
    x, gout = make_inputs(core, d['num_nodes'], r, heads, 8, seed=1)
    with pytest.raises(RuntimeError, match='unsupported shape'):
        run_core(core, g, etv, x, gout)
