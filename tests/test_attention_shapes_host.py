"""CPU side of tests/test_attention_shapes_gpu.py: the generated shape list reaches every kernel class the attention
dispatch in csrc/gat.cu instantiates and no other; the float64 reference of that file equals oracle/regnn_oracle.py,
kink ties and keep mask included; the boundary graph has its degrees in both CSR views."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import csr_oracle, regnn_oracle as O
from test_attention_shapes_gpu import (BOUNDARY_DEGREES, SHAPES, boundary_degrees, boundary_graph, kernel_class,
                                       reference)

GAT_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 're_gnn_b200', 'csrc', 'gat.cu')


def _dispatch_cases(macro):
    src = open(GAT_CU).read()
    cases = re.findall(r'\b%s\((\d+), (\d+), (\d+)\)' % macro, src)
    return {tuple(int(v) for v in c) for c in cases if c != ('G_', 'L_', 'C_')}


def test_shape_list_is_every_accepted_shape():
    assert len(SHAPES) == 158 == len(set(SHAPES))
    for h, d in SHAPES:
        assert 1 <= h <= 32 and 4 <= d <= 512 and d & (d - 1) == 0 and h * d <= 1024


@pytest.mark.parametrize('macro', ['REGNN_EDGES_CASE', 'REGNN_V2F_CASE', 'REGNN_V2E_CASE'])
def test_shapes_reach_every_dispatch_case(macro):
    cases = _dispatch_cases(macro)
    assert len(cases) == 20
    assert {kernel_class(h, d) for h, d in SHAPES} == cases


def _tiny_graph():
    """Duplicate edges, a row without in-edges (node 5), a self loop, two relations."""
    src = torch.tensor([0, 1, 1, 2, 3, 4, 4, 0, 2, 3, 6, 6])
    dst = torch.tensor([1, 0, 0, 1, 2, 2, 3, 3, 4, 6, 6, 4])
    et = torch.tensor([1, 2, 2, 1, 1, 2, 1, 2, 2, 1, 1, 2])
    return src, dst, et, 7


def _tie_inputs(core, n, heads, dim, r):
    """Dyadic inputs with exactly-zero LeakyReLU inputs on purpose (relation 1 of head 0 has theta = 0).  REGATv2: fs and
    fd hold the same values (the oracle's layer without fc layers uses the features on both sides)."""
    rng = np.random.RandomState(heads * 10 + dim)
    dy = lambda *s: torch.as_tensor(rng.randint(-4, 5, size=s) / 4.0)   # noqa: E731
    th = torch.as_tensor(rng.randint(0, 5, size=(r, heads)) / 16.0)
    th[0, 0] = 0.0
    if core == 'gatv2_aggregate':
        f = dy(n, heads, dim)
        x = dict(fs=f, fd=f.clone(), attn=dy(1, heads, dim), theta=th)
    else:
        x = dict(feat=dy(n, heads, dim), attn_l=dy(1, heads, dim), attn_r=dy(1, heads, dim), theta=th)
        x['feat'][[0, 1]] = 0.0          # el = er = 0 on nodes 0 and 1: the edges between them have pre = 0 (theta = 0)
    return x, torch.as_tensor(rng.randn(n, heads, dim))


@pytest.mark.parametrize('with_keep', [False, True])
@pytest.mark.parametrize('core', ['gat_layer', 'gatv2_aggregate'])
def test_reference_equals_oracle(core, with_keep):
    src, dst, et, n = _tiny_graph()
    heads, dim, alpha, slope = 2, 4, 4.0, 0.2
    x, gout = _tie_inputs(core, n, heads, dim, 2)
    keep = torch.as_tensor((np.random.RandomState(1).rand(src.numel(), heads) > 0.4) / 0.6) if with_keep else None
    got = reference(core, dict(src=src, dst=dst, etype=et), n, x, gout, alpha, slope, keep=keep, device='cpu')
    assert got['ties'] > 0

    if core == 'gat_layer':
        leaves = {k: v.clone().requires_grad_(True) for k, v in x.items()}
        feat = leaves['feat']
        out, a = O.regat_forward(src, dst, et, n, feat, leaves['attn_l'], leaves['attn_r'], leaves['theta'], alpha, slope,
                                 return_attention=True)
    else:
        leaves = {k: x[k].clone().requires_grad_(True) for k in ('fs', 'attn', 'theta')}
        feat = leaves['fs']
        out, a = O.regatv2_forward(src, dst, et, n, feat, leaves['attn'], leaves['theta'], alpha, slope,
                                   return_attention=True)
    if keep is not None:
        a = a * keep[:, :, None]
        out = O.segment_sum(feat[src] * a, dst, n)
    out.backward(gout)
    assert torch.allclose(got['out'], out.detach(), rtol=1e-12, atol=1e-12)
    assert torch.allclose(got['attn'], a.detach().squeeze(-1), rtol=1e-12, atol=1e-12)
    grads = dict(got['grads'])
    if core == 'gatv2_aggregate':     # fs and fd are the same features in the oracle
        grads['fs'] = grads['fs'] + grads.pop('fd')
    assert set(grads) == set(leaves)
    for k, v in leaves.items():
        assert torch.allclose(grads[k], v.grad, rtol=1e-10, atol=1e-12), k
    has = torch.bincount(dst, minlength=n) > 0
    assert not bool(has.all())
    assert torch.equal(got['rowsum'][~has], torch.zeros_like(got['rowsum'][~has]))
    assert torch.equal(got['rowmax'][~has], torch.zeros_like(got['rowmax'][~has]))


def test_reference_kink_convention():
    """At a pre-activation of exactly 0 the derivative is the negative slope (PyTorch's leaky_relu_backward, and the
    kernels' leaky_grad)."""
    # row 1 has two in-edges: 0 -> 1 with pre = 0 (the tie) and 1 -> 1 with pre = -5; row 0 one edge
    src, dst = torch.tensor([0, 1, 1]), torch.tensor([1, 0, 1])
    x = dict(feat=torch.tensor([[[1.0, 0, 0, 0]], [[0.0, 0, 0, 0]]]), el=torch.tensor([[0.0], [-5.0]]),
             er=torch.zeros(2, 1))
    gout = torch.zeros(2, 1, 4)
    gout[1, 0, 0] = 1.0
    ref = reference('gat_aggregate', dict(src=src, dst=dst, etype=None), 2, x, gout, slope=0.2, device='cpu')
    assert ref['ties'] == 1
    # loss = out[1, 0, 0] = a0 with logits l0 = 0, l1 = -1: dloss/dl0 = a0 (1 - a0), times the slope at the kink
    a0 = 1.0 / (1.0 + np.exp(-1.0))
    assert abs(float(ref['grads']['el'][0, 0]) - 0.2 * a0 * (1 - a0)) < 1e-12


def test_boundary_graph_degrees_cpu():
    d = boundary_graph()
    c = csr_oracle.csr_build(d['src'], d['dst'], d['num_nodes'])
    ins, outs = boundary_degrees(d, c)
    assert ins.tolist() == list(BOUNDARY_DEGREES) and outs.tolist() == list(BOUNDARY_DEGREES)
    assert 20000 <= d['src'].size <= 30000
    deg_in = np.diff(c['indptr'])
    assert (deg_in == 0).sum() >= 100 and deg_in.max() == 513
    assert np.diff(c['indptr_t']).max() == 513
    pairs = d['src'] * d['num_nodes'] + d['dst']
    assert np.unique(pairs).size < pairs.size                       # duplicate edges
    assert np.unique(d['etype']).tolist() == list(range(1, d['num_relations'] + 1))
    # the structure does not depend on the number of relations
    d2 = boundary_graph(num_relations=200)
    assert np.array_equal(d2['src'], d['src']) and np.array_equal(d2['dst'], d['dst'])
