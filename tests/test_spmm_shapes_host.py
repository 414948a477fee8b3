"""CPU side of tests/test_spmm_shapes_gpu.py: its width / alignment lists reach every dispatch case of csrc/spmm.cu
(through a restatement of pick_stream_shape, rowgroup_lanes, pick_shape and ops.fused_bwd_fits); its float64
reference equals oracle/regnn_oracle.py; the boundary graph has its degrees and row positions in both CSR views."""
import numpy as np
import pytest
import torch

from oracle import csr_oracle, regnn_oracle as O
from re_gnn_b200 import ops
import test_spmm_shapes_gpu as S


def test_fwd_widths_reach_every_forward_case():
    want = {k[1] for k in S.instantiated_kernels() if k[0] == 'spmm_stream_kernel' and k[1][2] == 0}
    want_rg = {k[1] for k in S.instantiated_kernels() if k[0] == 'spmm_rowgroup_kernel' and k[1][0] == 0}
    assert len(want) == 15 and len(want_rg) == 4
    seen = set()
    for feat, off in S.FWD_WIDTHS:
        for full, order in ((True, True), (False, True), (True, False)):
            k = S.fwd_kernel(feat, off, feat, full, order)
            assert k is not None, (feat, off)
            seen.add(k)
    assert {k[1:3] + (0,) for k in seen if k[0] == 'stream'} == {(c, vw, 0) for c, vw, _ in want}
    assert {(0, k[2], 0) for k in seen if k[0] == 'rowgroup'} == want_rg


def test_bwd_widths_reach_every_fused_case_with_both_tile_copies():
    inst = S.instantiated_kernels()
    want = {k[1][:2] for k in inst if k[0] == 'spmm_stream_kernel' and k[1][2] == 1}
    rg = {k[1][1] for k in inst if k[0] == 'spmm_rowgroup_kernel' and k[1][0] == 1}
    tma, plain, groups = set(), set(), set()
    for feat, xoff, goff, full in S.BWD_WIDTHS:
        k, t = S.bwd_kernel(feat, xoff, goff, full)
        assert k is not None and ops.fused_bwd_fits(feat, 5), (feat, xoff, goff)
        if k[0] == 'rowgroup':
            groups.add(k[2])
        else:
            (tma if t else plain).add(k[1:3])
    assert groups == rg == {4, 8, 16, 32}
    assert tma == want
    assert plain == {s for s in want if s[1] != 4}      # VW = 4 implies 16-byte aligned X: always TMA


def test_bwd_w_widths_reach_every_class():
    want = {k[1][:3] for k in S.instantiated_kernels() if k[0] == 'spmm_bwd_w_kernel'}
    assert len(want) == 17
    got = {S.pick_shape(feat, off == 0) for feat, off in S.BWDW_WIDTHS}
    assert got == want
    # and no width reaches a class that is not instantiated
    assert {S.pick_shape(f, v) for f in range(1, 1100) for v in (False, True)} - {None} == want


@pytest.mark.parametrize('feat,off', [(257, 0), (1028, 0), (260, 1), (1024, 1), (514, 2), (1024, 2)])
def test_refused_widths_have_no_kernel(feat, off):
    assert S.fwd_kernel(feat, off, feat, True) is None


def test_two_pass_shapes():
    assert not ops.fused_bwd_fits(1000, 5) and not ops.fused_bwd_fits(130, 200)
    assert ops.fused_bwd_fits(128, 200) and ops.fused_bwd_fits(33, 200) and ops.fused_bwd_fits(640, 5)


def test_parse_kernel_names():
    assert S.parse_kernel_name('void regnn::spmm_stream_kernel<4, 2, false>(regnn::StreamArgs)') == \
        ('spmm_stream_kernel', (4, 2, 0))
    assert S.parse_kernel_name('void regnn::spmm_rowgroup_kernel<true, 32, true>(regnn::StreamArgs)') == \
        ('spmm_rowgroup_kernel', (1, 32, 1))
    assert S.parse_kernel_name('regnn::rowdot_norm_kernel(float const*, int)') == ('rowdot_norm_kernel', ())


# ---- the float64 reference against the oracle ------------------------------------------------------------------------
class _Tiny:
    """Duplicate edges, a row without in-edges (node 5), self loops, two relations; the View interface."""

    def __init__(self):
        src = np.array([0, 1, 1, 2, 3, 4, 4, 0, 2, 3, 6, 6, 2])
        dst = np.array([1, 0, 0, 1, 2, 2, 3, 3, 4, 6, 6, 4, 2])
        self.d = dict(src=src, dst=dst, etype=np.array([1, 2, 2, 1, 1, 2, 1, 2, 2, 1, 1, 2, 2]), num_nodes=7)
        c = csr_oracle.csr_build(src, dst, 7)
        self.n, self.r, self.e = 7, 2, src.size
        self.row, self.col = torch.as_tensor(c['row']).long(), torch.as_tensor(c['indices']).long()
        self.et = torch.as_tensor(self.d['etype'][c['eid']] - 1).long()
        self.indeg = torch.as_tensor(np.diff(c['indptr']))
        self.outdeg = torch.as_tensor(np.diff(c['indptr_t']))


@pytest.fixture
def cpu_ref(monkeypatch):
    monkeypatch.setattr(S, 'DEV', 'cpu')


@pytest.mark.parametrize('sides', [0, 1, 2, 3])
def test_reference_equals_oracle(cpu_ref, sides):
    v = _Tiny()
    rng = np.random.RandomState(sides)
    x, g, y = (torch.as_tensor(rng.randn(7, 3)) for _ in range(3))
    theta = torch.tensor([[0.25], [-0.125]], dtype=torch.float64)
    norm = torch.as_tensor(rng.uniform(0.5, 2.0, size=7))
    ns, nd = S.sides_norms(norm, sides)
    src, dst, et = (torch.as_tensor(v.d[k]) for k in ('src', 'dst', 'etype'))
    # oracle: Y = nd . sum w ns X, by autograd for the backward
    xl, tl, nl = x.clone().requires_grad_(True), theta.clone().requires_grad_(True), norm.clone().requires_grad_(True)
    c = O.edge_relation(tl.view(-1), S.ALPHA, et)
    if sides & 1:
        c = c * nl[src]
    yo = O.segment_sum(c[:, None] * xl[src], dst, 7)
    if sides & 2:
        yo = yo * nl[:, None]
    yo.backward(g)
    ref_y = S.ref_spmm(v, x, theta, ns, nd)
    assert torch.allclose(ref_y[0], yo.detach(), rtol=1e-12, atol=1e-12)
    assert ref_y[0][5].abs().sum() == 0 and ref_y[2][5, 0] == 0          # the row without in-edges
    dx, dth, xdx, dn = S.ref_bwd(v, dict(x=x, g=g, y=yo.detach(), theta=theta, norm=norm), sides)
    assert torch.allclose(dx[0], xl.grad, rtol=1e-12, atol=1e-12)
    assert torch.allclose(dth[0], tl.grad.view(-1), rtol=1e-12, atol=1e-12)
    if sides:
        assert torch.allclose(dn[0], nl.grad, rtol=1e-12, atol=1e-12)
    assert torch.allclose(xdx[0], (x * xl.grad).sum(1), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize('clamp_min', [1.0, 0.0])
@pytest.mark.parametrize('exponent', [-0.5, -1.0, -0.25])
def test_degree_norm_reference_equals_oracle(cpu_ref, exponent, clamp_min):
    """The tie deg == clamp_min passes the gradient (torch.clamp's convention); without a clamp a row without in-edges
    has norm 0 and no gradient."""
    v = _Tiny()
    theta = torch.tensor([[0.25], [0.0625]], dtype=torch.float64)   # w = 1, 0.25 at alpha = 4
    d_norm = torch.as_tensor(np.random.RandomState(1).randn(7))
    deg, nm, dth = S.ref_wdeg(v, theta, S.ALPHA, exponent, clamp_min, d_norm)
    assert float(deg[0][0]) == 0.25 * 2 and float(deg[0][1]) == 1.0 + 1.0 and float(deg[0][5]) == 0.0
    tl = theta.clone().requires_grad_(True)
    ew = O.edge_relation(tl.view(-1), S.ALPHA, torch.as_tensor(v.d['etype']))
    dsum = O.segment_sum(ew.reshape(-1, 1), torch.as_tensor(v.d['dst']), 7).squeeze(1)
    if clamp_min > 0:
        no = torch.pow(dsum.clamp(min=clamp_min), exponent)
        if exponent == -0.5 and clamp_min == 1.0:
            assert torch.allclose(no, O.weighted_degree_norm(ew, torch.as_tensor(v.d['dst']), 7, -0.5))
    else:
        no = torch.where(dsum == 0, torch.zeros_like(dsum), torch.where(dsum == 0, torch.ones_like(dsum), dsum) ** exponent)
    no.backward(d_norm)
    assert torch.allclose(nm[0], no.detach(), rtol=1e-12)
    assert torch.allclose(dth[0], tl.grad.view(-1), rtol=1e-12, atol=1e-14)


def test_degree_norm_tie_passes_gradient(cpu_ref):
    """A row of weighted degree exactly clamp_min = 1 contributes q * d_norm to its relation's gradient."""
    v = _Tiny()
    theta = torch.tensor([[0.25], [0.0]], dtype=torch.float64)      # w = 1, 0
    d_norm = torch.zeros(7, dtype=torch.float64)
    d_norm[1] = 1.0                                           # node 1: in-edges 0->1 (rel 1), 2->1 (rel 1): degree 2
    d_norm[3] = 1.0                                           # node 3: 4->3 (rel 1), 0->3 (rel 2): degree exactly 1
    _, _, dth = S.ref_wdeg(v, theta, S.ALPHA, -0.5, 1.0, d_norm)
    # relation 1: node 1 (2 slots) -0.5 * 2^-1.5 each, node 3 (1 slot) -0.5 at the tie; times alpha * 1
    want = S.ALPHA * (2 * -0.5 * 2 ** -1.5 + -0.5)
    assert abs(float(dth[0][0]) - want) < 1e-12


def test_boundary_graph_layout():
    d = S.boundary_graph()
    c = csr_oracle.csr_build(d['src'], d['dst'], d['num_nodes'])
    ins, outs = np.diff(c['indptr']), np.diff(c['indptr_t'])
    assert ins.tolist() == outs.tolist() == S.degree_layout().tolist()
    n = d['num_nodes']
    assert n % 32 and n % 8
    present = set(ins.tolist())
    assert set(S.BOUNDARY_DEGREES) <= present and {768, 769} <= present
    long_ = ins > S.THRESHOLD
    assert long_[32] and long_[63] and long_[64] and long_[65]          # lane 0, lane 31, two adjacent long rows
    assert long_[S.LONG_ITEM[0]:S.LONG_ITEM[1]].all() and S.LONG_ITEM[0] % 32 == 0
    assert (ins[S.EMPTY_ITEM[0]:S.EMPTY_ITEM[1]] == 0).all() and S.EMPTY_ITEM[0] % 32 == 0
    assert (ins[2000:2003] == 0).all() and (ins[-5:] == 0).all()
    pairs = d['src'] * n + d['dst']
    assert np.unique(pairs).size < pairs.size and (d['src'] == d['dst']).any()   # duplicate edges, self loops
    assert not np.array_equal(np.argsort(d['dst'], kind='stable'), np.arange(d['dst'].size))   # shuffled edge ids
    assert ins[S.TIE_ROW] == 1 and d['etype'][d['dst'] == S.TIE_ROW].tolist() == [1]
    d2 = S.boundary_graph(num_relations=200)
    assert np.array_equal(d2['src'], d['src']) and np.array_equal(d2['dst'], d['dst'])
    assert np.unique(d2['etype']).size == 200
