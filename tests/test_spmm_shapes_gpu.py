"""Every dispatch shape of the REGCN / REMixHop SpMM kernels against float64 (``pytest -m gpu``, one B200).

csrc/spmm.cu picks its kernel from the width F, the 16/8/4-byte alignment of every operand, the row order, the row
range, the long-row split, relations or none, the norm sides and whether the fused backward fits in shared memory.
Here every instantiated case of ``regnn_spmm_fwd`` (4 lane-group widths, 15 stream shapes), ``regnn_spmm_bwd_fused``
(lane-group plain / xdx / folded d_norm, stream shapes with TMA staging and with the plain tile copy),
``regnn_spmm_bwd_w`` (17 classes) and the degree-norm kernels runs against a float64 reference on a graph whose rows
sit where the work items of the kernels change (long rows at lane 0 and 31 of an item, adjacent long rows, an item of
long rows only, an item of empty rows, N not a multiple of 32), with degrees in both views at the fragment boundaries.

Tolerance, one rule for every output element: |got - ref| <= (k + 3) * 2^-24 * sum|terms|, k = the number of
roundings on the longest chain of that element's sum (first-order bound of fp32 summation in any order):
  Y, dX           k = the row's slots;                       terms  |nd| * |w_s * ns_s * x_s|
  xdx             k = F + the row's slots;                   terms  sum_f |X_f| * (terms of dX_f)
  d_norm          k = 2F + the row's slots;                  terms  (|Y.G| + |X| . terms of dX) / norm
  d_theta[r]      k = F + slots of relation r + 1;           terms  |alpha w'| * sum_e |ns nd X[src] . G[dst]|
  degree norm     k = slots of the row + 8 (pow / sqrt);     terms  |max(deg, c)^q|  (deg itself is exact)
  its d_theta[r]  k = slots of relation r + 8;               terms  |alpha w'| * sum_e |dd[dst]|
``test_tolerances_reject_one_slot_or_fragment`` shows that each bound rejects one dropped slot or one doubled
fragment.  ``test_every_instantiated_kernel_ran`` reads the launched kernels and their template arguments from
torch.profiler and compares them with the instantiations parsed from csrc/spmm.cu.

``REGNN_TEST_DEVICE=cpu`` runs the reference and the test logic against tests/cpu_shim.py (no refusals, no profiler,
no index-width case there)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import helpers
from oracle import regnn_oracle as O
from re_gnn_b200 import Graph, _lib, functional as RF, ops

pytestmark = pytest.mark.gpu
DEV = os.environ.get('REGNN_TEST_DEVICE', 'cuda:0')
ON_GPU = DEV != 'cpu'
U = 2.0 ** -24
ALPHA = 4.0                     # a power of two: alpha * theta is exact
SPMM_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 're_gnn_b200', 'csrc', 'spmm.cu')

# ---- the dispatch of csrc/spmm.cu, restated (tests/test_spmm_shapes_host.py checks it reaches every case) -----------
THRESHOLD = 256                 # SPLIT_THRESHOLD of graph.py


def common_align(offsets_bytes, lds):
    """common_align of spmm.cu: the largest power of two <= 16 dividing every base offset and leading dimension."""
    al = 16
    for o in offsets_bytes:
        while al > 4 and o % al:
            al >>= 1
    for ld in lds:
        while al > 4 and (ld * 4) % al:
            al >>= 1
    return al


def stream_shape(feat, align):
    """(C, VW) of pick_stream_shape, or None (refused)."""
    vw = 4 if (align >= 16 and feat % 4 == 0 and feat >= 96) else 2 if (align >= 8 and feat % 2 == 0 and feat >= 34) else 1
    c = -(-feat // (32 * vw))
    if c > 8:
        if vw == 1 and align >= 8 and feat % 2 == 0:
            vw, c = 2, -(-feat // 64)
        if c > 8 and align >= 16 and feat % 4 == 0:
            vw, c = 4, -(-feat // 128)
        if c > 8:
            return None
    return (8 if c > 4 else c, vw)


def rowgroup_lanes(feat, has_order, full, align):
    if not has_order or not full or feat > 128 or feat % 4 or align < 16:
        return 0
    return 32 if feat > 64 else 16 if feat > 32 else 8 if feat > 16 else 4


def pick_shape(feat, vec_ok):
    """(G, C, VW) of pick_shape (regnn_spmm_bwd_w), or None."""
    if vec_ok and feat % 4 == 0:
        f4 = feat // 4
        g = 4 if f4 <= 4 else 8 if f4 <= 8 else 16 if f4 <= 16 else \
            16 if (f4 % 32 and f4 % 16 == 0 and f4 // 16 <= 3) else 32
        c, vw = -(-f4 // g), 4
    else:
        g = 4 if feat <= 4 else 8 if feat <= 8 else 16 if feat <= 16 else 32
        c, vw = -(-feat // g), 1
    return None if c > 8 else (g, 8 if c > 4 else c, vw)


def fwd_kernel(feat, off, ld_out, full, order=True):
    """The kernel regnn_spmm_fwd launches for operands at ``off`` floats past 16-byte alignment (X and Y), Y's
    leading dimension ``ld_out``: ('rowgroup', False, G, False) | ('stream', C, VW, False) | None."""
    al = common_align([4 * off, 4 * off], [feat, ld_out, feat])
    g = rowgroup_lanes(feat, order, full, al)
    if g:
        return ('rowgroup', False, g, False)
    s = stream_shape(feat, al)
    return ('stream', s[0], s[1], False) if s else None


def bwd_kernel(feat, xoff, goff, full, dnorm=False):
    """The kernel regnn_spmm_bwd_fused launches (X at ``xoff`` floats, G and dX at ``goff``), and whether the stream
    kernel stages its tile with TMA: (('rowgroup', True, G, dnorm) | ('stream', C, VW, True) | None, tma)."""
    al = common_align([4 * xoff, 4 * goff, 4 * goff], [feat, feat, feat, feat])
    g = rowgroup_lanes(feat, True, full, al)
    if g:
        return ('rowgroup', True, g, dnorm), False
    s = stream_shape(feat, al)
    return (('stream', s[0], s[1], True) if s else None), (feat % 4 == 0 and xoff % 4 == 0)


def fused_bwd_fits(feat, r):
    return ops.fused_bwd_fits(feat, r)


# Forward sweep: (F, offset in floats of X and Y).  Every lane-group width and every stream shape is reached; the
# stream kernel at F <= 128 runs on sub-ranges, without a row order, or at an offset.
FWD_WIDTHS = [(4, 0), (16, 0), (20, 0), (32, 0), (48, 0), (64, 0), (68, 0), (128, 0),
              (1, 0), (7, 0), (33, 0), (65, 0), (95, 0), (127, 0), (255, 0),           # VW 1 (odd widths)
              (64, 1), (96, 1), (128, 1), (256, 1),                                     # VW 1 at a 4-byte offset
              (34, 0), (66, 0), (130, 0), (194, 0), (258, 0),                           # VW 2 (F % 4 == 2)
              (64, 2), (128, 2), (192, 2), (256, 2), (512, 2),                          # VW 2 at an 8-byte offset
              (100, 0), (256, 0), (384, 0), (512, 0), (640, 0), (1024, 0)]              # VW 4
# Fused backward sweep: (F, X offset, G / dX offset, full range).  Stream shapes with VW < 4 run twice: with TMA tile
# staging (X aligned, G at an offset) and with the plain copy (X at an offset or F % 4 != 0).  VW = 4 needs every
# operand 16-byte aligned, so it always stages with TMA.
BWD_WIDTHS = [(8, 0, 0, True), (32, 0, 0, True), (64, 0, 0, True), (128, 0, 0, True),   # lane-group kernels
              (128, 0, 0, False), (256, 0, 0, True), (384, 0, 0, True), (512, 0, 0, True), (640, 0, 0, True),
              (64, 0, 2, True), (64, 2, 2, True), (34, 0, 0, True),
              (128, 0, 2, True), (66, 0, 0, True), (192, 0, 2, True), (130, 0, 0, True),
              (256, 0, 2, True), (194, 0, 0, True), (512, 0, 2, True), (258, 0, 0, True),
              (32, 0, 0, False), (32, 1, 1, True), (7, 0, 0, True), (64, 0, 1, True), (33, 0, 0, True),
              (96, 0, 1, True), (65, 0, 0, True), (128, 0, 1, True), (127, 0, 0, True), (256, 0, 1, True),
              (255, 0, 0, True)]
# regnn_spmm_bwd_w: (F, offset) -- offset 0 gives the 128-bit classes, offset 1 the scalar ones.
BWDW_WIDTHS = [(16, 0), (32, 0), (64, 0), (192, 0), (128, 0), (256, 0), (384, 0), (512, 0), (1000, 0),
               (4, 1), (8, 1), (16, 1), (32, 1), (64, 1), (96, 1), (128, 1), (256, 1)]


# ---- the boundary graph ---------------------------------------------------------------------------------------------
BOUNDARY_DEGREES = tuple(range(10)) + (15, 16, 17, 31, 32, 33, 63, 64, 65, 255, 256, 257, 511, 512, 513, 768, 769)
LONG_DEGREES = (257, 511, 512, 513, 768, 769)
NUM_NODES = 4003               # not a multiple of 32 (nor of 8)
EMPTY_ITEM = (128, 160)        # rows 128..159: an item of the plain kernel (and four of the BINS one) with no slots
LONG_ITEM = (96, 128)          # rows 96..127: an item of long rows only
TIE_ROW = 1                    # one in-edge of relation 1 (w = 1): weighted degree exactly 1


def degree_layout(n=NUM_NODES, seed=0):
    """In-degree (= out-degree) of every row.  Rows 0..29: BOUNDARY_DEGREES; row 32 (lane 0 of the second item) and row
    63 (lane 31) long; rows 64, 65 two adjacent long rows; LONG_ITEM long rows only; EMPTY_ITEM no slots; empty rows
    in the middle (2000..2002) and at the end (the last 5); the rest 0..12 slots, a tenth of them 0."""
    rng = np.random.RandomState(seed)
    deg = rng.randint(0, 13, size=n)
    deg[rng.rand(n) < 0.1] = 0
    deg[:len(BOUNDARY_DEGREES)] = BOUNDARY_DEGREES
    deg[30:32] = (3, 0)
    deg[32], deg[63] = 769, 513
    deg[64:66] = (257, 512)
    deg[LONG_ITEM[0]:LONG_ITEM[1]] = np.resize(LONG_DEGREES, LONG_ITEM[1] - LONG_ITEM[0])
    deg[EMPTY_ITEM[0]:EMPTY_ITEM[1]] = 0
    deg[2000:2003] = 0
    deg[-5:] = 0
    return deg


def boundary_graph(num_relations=5, seed=0):
    """Edges pair the in-slots and the out-slots of degree_layout at random, so every node has the same in- and
    out-degree (both CSR views share the layout); hub-to-hub pairs give duplicate edges and self loops.  Edge ids are
    shuffled.  Edge types (1-based) depend on ``num_relations``, the structure does not; the in-edge of TIE_ROW has
    relation 1."""
    rng = np.random.RandomState(seed)
    deg = degree_layout()
    dst = np.repeat(np.arange(NUM_NODES), deg)
    src = rng.permutation(dst)
    perm = rng.permutation(dst.size)
    src, dst = src[perm].astype(np.int64), dst[perm].astype(np.int64)
    etype = np.random.RandomState(seed + 1 + num_relations).randint(1, num_relations + 1, size=src.size).astype(np.int64)
    etype[dst == TIE_ROW] = 1
    return dict(src=src, dst=dst, etype=etype, num_nodes=NUM_NODES, num_relations=num_relations, deg=deg)


class View:
    """A built graph with its relation views and the float64 reference's edge arrays (in-view slot order)."""

    def __init__(self, d):
        self.d, self.n, self.r = d, d['num_nodes'], d['num_relations']
        self.g = Graph(d['src'], d['dst'], self.n).to(DEV)
        self.etv = self.g.etype_views(torch.as_tensor(d['etype']).to(DEV), self.r)
        self.csr = self.g.csr()
        self.row = self.csr['row'].long()
        self.col = self.csr['indices'].long()
        self.et = self.etv[0].long()
        self.indeg = torch.diff(self.csr['indptr'].long())
        self.outdeg = torch.diff(self.csr['indptr_t'].long())
        self.e = self.row.numel()


_VIEWS = {}


def view(r=5):
    if r not in _VIEWS:
        _VIEWS[r] = View(boundary_graph(r))
    return _VIEWS[r]


@pytest.fixture(scope='module', autouse=True)
def _dry_run_shim():
    with pytest.MonkeyPatch.context() as mp:
        if not ON_GPU:
            import cpu_shim
            cpu_shim.install(mp)
        yield
        _VIEWS.clear()


@pytest.fixture(scope='module')
def bv():
    v = view(5)
    indeg = v.indeg.cpu().numpy()
    assert indeg.tolist() == degree_layout().tolist() and v.outdeg.cpu().numpy().tolist() == indeg.tolist()
    if ON_GPU:
        assert v.csr['split'] is not None and v.csr['split_t'] is not None
    return v


# ---- inputs exact in fp32 -------------------------------------------------------------------------------------------
def dyadic(rng, shape, den=8, kmax=8):
    return torch.as_tensor(rng.randint(-kmax, kmax + 1, size=shape) / float(den))


def theta_of(rng, r):
    """k / 64 with 1 <= |k| <= 16, relation 2 (if any) negative: LeakyReLU(alpha * theta) is exact on the positive
    side; the negative side rounds 0.01 * alpha * theta once."""
    t = rng.randint(1, 17, size=(r, 1)) / 64.0
    if r > 1:
        t[1] = -t[1]
    return torch.as_tensor(t)


def norm_of(rng, n):
    return helpers.f32_exact(rng.uniform(0.25, 2.0, size=n))


def placed(a64, off=0, ld=None, fill=float('nan')):
    """fp32 copy of ``a64`` [n, F] whose first element sits ``off`` floats past a 16-byte boundary and whose rows are
    ``ld`` floats apart; the buffer around it holds ``fill``.  -> (view, whole buffer)."""
    n, f = a64.shape
    ld = f if ld is None else ld
    buf = torch.full((off + max(n * ld, 1) + ld,), fill, dtype=torch.float32, device=DEV)
    t = buf[off:off + n * ld].view(n, ld)[:, :f]
    t.copy_(a64.to(DEV, torch.float32))
    return t, buf


# ---- float64 reference ----------------------------------------------------------------------------------------------
def _seg(idx, n, vals):
    return torch.zeros((n,) + tuple(vals.shape[1:]), dtype=torch.float64, device=vals.device).index_add_(0, idx, vals)


def _d(t):
    return None if t is None else t.detach().to(DEV, torch.float64)


def rel_w(theta, alpha=ALPHA):
    return O.relation_weight(_d(theta).view(-1), alpha)


def rel_w_grad(theta, alpha=ALPHA):
    th = _d(theta).view(-1) * alpha
    return alpha * torch.where(th > 0, torch.ones_like(th), torch.full_like(th, O.RELATION_SLOPE))


def ref_spmm(v, x, theta, ns, nd, transposed=False, es=None):
    """Y[i] = nd[i] * sum_s w_s * ns[j_s] * x[j_s] over the in-slots of i (``transposed``: the out-slots, dX of the
    backward) -> (value, sum of |terms|, k).  ``es``: per-slot factor (the sensitivity checks)."""
    dst, src = (v.col, v.row) if transposed else (v.row, v.col)
    c = rel_w(theta)[v.et] if theta is not None else torch.ones(v.e, dtype=torch.float64, device=DEV)
    if ns is not None:
        c = c * _d(ns)[src]
    if es is not None:
        c = c * es
    m = c[:, None] * _d(x)[src]
    y, a = _seg(dst, v.n, m), _seg(dst, v.n, m.abs())
    if nd is not None:
        y, a = y * _d(nd)[:, None], a * _d(nd).abs()[:, None]
    k = (v.outdeg if transposed else v.indeg).to(torch.float64)[:, None].expand_as(y)
    return y, a, k


def ref_dtheta(v, x, g, theta, ns, nd, es=None, rows=None):
    """d_theta[r] = alpha w'(alpha theta_r) * sum over slots of relation r of ns[src] nd[dst] <X[src], G[dst]>;
    ``rows``: only slots whose source lies in [rows[0], rows[1])."""
    x, g = _d(x), _d(g)
    p = x[v.col] * g[v.row]
    c = torch.ones(v.e, dtype=torch.float64, device=DEV)
    if ns is not None:
        c = c * _d(ns)[v.col]
    if nd is not None:
        c = c * _d(nd)[v.row]
    if es is not None:
        c = c * es
    if rows is not None:
        c = c * ((v.col >= rows[0]) & (v.col < rows[1]))
    r = theta.numel()
    dw = _seg(v.et, r, c * p.sum(1))
    da = _seg(v.et, r, c.abs() * p.abs().sum(1))
    cnt = _seg(v.et, r, (c != 0).to(torch.float64))
    s = rel_w_grad(theta)
    return dw * s, da * s.abs(), cnt + x.shape[1] + 1


def ref_rowdots(v, x, y, g, dx_ref, norm, sides):
    """(xdx, d_norm) of the norm gradient from the reference dX = (value, |terms|, k)."""
    x, y, g = _d(x), _d(y), _d(g)
    dxv, dxa, dxk = dx_ref
    f = x.shape[1]
    xdx = ((x * dxv).sum(1), (x.abs() * dxa).sum(1), dxk[:, 0] + f)
    dn, da = torch.zeros(v.n, dtype=torch.float64, device=DEV), torch.zeros(v.n, dtype=torch.float64, device=DEV)
    if sides & 2:
        dn, da = dn + (y * g).sum(1), da + (y * g).abs().sum(1)
    if sides & 1:
        dn, da = dn + xdx[0], da + xdx[1]
    nm = _d(norm)
    return xdx, (dn / nm, da / nm.abs(), dxk[:, 0] + 2 * f)


def check(tag, got, ref, extra=3.0, rows=None):
    """|got - ref| <= (k + extra) * 2^-24 * sum|terms| elementwise (``rows``: only these rows)."""
    val, a, k = ref
    got = got.detach().to(DEV, torch.float64)
    if rows is not None:
        got, val, a, k = got[rows[0]:rows[1]], val[rows[0]:rows[1]], a[rows[0]:rows[1]], k[rows[0]:rows[1]]
    assert got.shape == val.shape, '%s: shape %s vs %s' % (tag, tuple(got.shape), tuple(val.shape))
    err = (got - val).abs()
    bound = (k + extra) * U * a
    ok = err <= bound
    if not bool(ok.all()):
        i = int(torch.nonzero(~ok.reshape(-1))[0])
        raise AssertionError('%s: %d elements outside the bound; first at flat index %d: got %r ref %r bound %.3g'
                             % (tag, int((~ok).sum()), i, float(got.reshape(-1)[i]), float(val.reshape(-1)[i]),
                                float(bound.reshape(-1)[i])))


# ---- kernel runs ----------------------------------------------------------------------------------------------------
def inputs(v, feat, seed):
    rng = np.random.RandomState(seed)
    return dict(x=dyadic(rng, (v.n, feat)), g=dyadic(rng, (v.n, feat)), y=dyadic(rng, (v.n, feat)),
                theta=theta_of(rng, v.r), norm=norm_of(rng, v.n))


def sides_norms(norm, sides):
    return (norm if sides & 1 else None), (norm if sides & 2 else None)


def run_fwd(v, inp, feat, off, sides, weighted, rows=None, order=True, pad=0, transposed=False):
    """ops.spmm on X and Y at ``off`` floats, Y a column slice of a [n, F + pad] NaN buffer -> (Y view, Y buffer)."""
    sfx = '_t' if transposed else ''
    x, _ = placed(inp['x'], off)
    y, ybuf = placed(torch.full((v.n, feat + pad), float('nan'), dtype=torch.float64), off, fill=float('nan'))
    y = y[:, :feat] if pad else y
    norm = inp['norm'].to(DEV, torch.float32)
    ns, nd = sides_norms(norm, sides)
    th = inp['theta'].to(DEV, torch.float32) if weighted else None
    ops.spmm(v.csr['indptr' + sfx], v.csr['indices' + sfx], v.etv[1 if transposed else 0] if weighted else None, th,
             ALPHA, ns, nd, x, rows=rows, out=y, split=v.csr.get('split' + sfx),
             order=ops.row_order(v.csr, transposed) if order else None)
    return y, ybuf


def run_bwd(v, inp, feat, xoff, goff, sides, rows=None, want_xdx=False, want_dnorm=False):
    x, _ = placed(inp['x'], xoff)
    g, _ = placed(inp['g'], goff)
    dx, _ = placed(torch.full((v.n, feat), float('nan'), dtype=torch.float64), goff)
    if rows is not None:
        dx.zero_()
    y = inp['y'].to(DEV, torch.float32)
    norm = inp['norm'].to(DEV, torch.float32) if sides else None
    dx, d_theta, extra = ops.spmm_bwd_fused(v.csr, v.etv[1], inp['theta'].to(DEV, torch.float32), ALPHA, norm, x, g,
                                            rows=rows, sides=sides, out=dx, want_xdx=want_xdx, y=y,
                                            want_dnorm=want_dnorm)
    return dx, d_theta, extra


def ref_bwd(v, inp, sides, rows=None, es=None):
    ns, nd = sides_norms(inp['norm'], sides)
    dx = ref_spmm(v, inp['g'], inp['theta'], nd, ns, transposed=True, es=es)
    dth = ref_dtheta(v, inp['x'], inp['g'], inp['theta'], ns, nd, es=es, rows=rows)
    xdx, dn = ref_rowdots(v, inp['x'], inp['y'], inp['g'], dx, inp['norm'], sides)
    return dx, dth, xdx, dn


# ---- forward --------------------------------------------------------------------------------------------------------
SUB_RANGES = [(31, 33), (32, 64), (33, 66), (64, 65), (97, 3001), (100, 2999), (0, NUM_NODES - 1)]


@pytest.mark.parametrize('feat,off', FWD_WIDTHS, ids=['F%d_off%d' % w for w in FWD_WIDTHS])
def test_forward_every_shape_vs_float64(bv, feat, off):
    v = bv
    inp = inputs(v, feat, seed=feat * 10 + off)
    kern = fwd_kernel(feat, off, feat, True)
    assert kern is not None
    for weighted in (True, False):
        for sides in (0, 1, 2, 3):
            ns, nd = sides_norms(inp['norm'], sides)
            ref = ref_spmm(v, inp['x'], inp['theta'] if weighted else None, ns, nd)
            tag = 'fwd F%d off%d %s w%d s%d ' % (feat, off, kern, weighted, sides)
            full, _ = run_fwd(v, inp, feat, off, sides, weighted)
            check(tag + 'full', full, ref)
            # every variant gives the same bits: without row order, aligned, Y with ldy > F, sub-ranges
            variants = [run_fwd(v, inp, feat, off, sides, weighted, order=False)[0]]
            if off:
                variants.append(run_fwd(v, inp, feat, 0, sides, weighted)[0])
            padded, pbuf = run_fwd(v, inp, feat, off, sides, weighted, pad=4)
            assert bool(torch.isnan(pbuf.view(-1)[off:off + v.n * (feat + 4)].view(v.n, feat + 4)[:, feat:]).all()), \
                tag + 'padding columns written'
            variants.append(padded)
            for i, y in enumerate(variants):
                assert torch.equal(y, full), tag + 'variant %d differs' % i
            for rb, re_ in (SUB_RANGES if sides == 3 else SUB_RANGES[:3]):
                part, _ = run_fwd(v, inp, feat, off, sides, weighted, rows=(rb, re_))
                assert torch.equal(part[rb:re_], full[rb:re_]), tag + 'rows %d..%d differ' % (rb, re_)
                outside = torch.cat([part[:rb], part[re_:]])
                assert bool(torch.isnan(outside).all()), tag + 'rows outside %d..%d written' % (rb, re_)
        # the un-weighted backward of REMixHop: the same kernels over the transposed view
        ns, nd = sides_norms(inp['norm'], 3)
        got, _ = run_fwd(v, inp, feat, off, 3, False, transposed=True)
        check('fwd F%d transposed ' % feat, got, ref_spmm(v, inp['x'], None, ns, nd, transposed=True))


def test_forward_leading_dimension_past_feat(bv):
    """The ABI with ldx > F and ldy > F (X and Y column slices of wider matrices)."""
    if not ON_GPU:
        pytest.skip('the C ABI itself')
    v = bv
    for feat in (64, 96, 256):
        inp = inputs(v, feat, seed=feat)
        xw, _ = placed(torch.cat([inp['x'], torch.ones(v.n, 8, dtype=torch.float64)], 1))
        yw, _ = placed(torch.full((v.n, feat + 8), float('nan'), dtype=torch.float64))
        norm, th = inp['norm'].to(DEV, torch.float32), inp['theta'].to(DEV, torch.float32).view(-1)
        split = v.csr['split']
        ws = torch.empty(split['struct'].num_frags * feat, dtype=torch.float32, device=DEV)
        p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
        _lib.call('regnn_spmm_fwd', p(v.csr['indptr']), p(v.csr['indices']), p(v.etv[0]), p(th), ALPHA, v.r, p(norm),
                  p(norm), p(xw), feat + 8, p(yw), feat + 8, 0, v.n, feat, ctypes.byref(split['struct']), p(ws),
                  p(ops.row_order(v.csr)), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        ns, nd = sides_norms(inp['norm'], 3)
        check('ld F%d ' % feat, yw[:, :feat], ref_spmm(v, inp['x'], inp['theta'], ns, nd))
        assert bool(torch.isnan(yw[:, feat:]).all())
        assert torch.equal(yw[:, :feat], run_fwd(v, inp, feat, 0, 3, True)[0])


# ---- fused backward -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('feat,xoff,goff,full', BWD_WIDTHS, ids=['F%d_x%d_g%d_%s' % (w[0], w[1], w[2], 'full' if w[3]
                                                                                          else 'sub') for w in BWD_WIDTHS])
def test_fused_backward_every_shape_vs_float64(bv, feat, xoff, goff, full):
    v = bv
    inp = inputs(v, feat, seed=feat * 100 + xoff * 10 + goff)
    rows = None if full else (0, v.n - 1)
    kern, tma = bwd_kernel(feat, xoff, goff, full)
    assert kern is not None and fused_bwd_fits(feat, v.r)
    tag = 'bwd F%d x%d g%d %s tma%d ' % (feat, xoff, goff, kern, tma)
    for sides in (3, 1, 2, 0):
        dx_r, dth_r, xdx_r, dn_r = ref_bwd(v, inp, sides, rows=rows)
        dx, dth, xdx = run_bwd(v, inp, feat, xoff, goff, sides, rows=rows, want_xdx=bool(sides))
        t = tag + 's%d ' % sides
        check(t + 'dX', dx, dx_r, rows=rows or (0, v.n))
        check(t + 'd_theta', dth, dth_r)
        if sides:
            check(t + 'xdx', xdx, xdx_r, rows=rows or (0, v.n))
        if rows is not None:
            assert bool((dx[rows[1]:] == 0).all()), t + 'rows outside written'
            assert xdx is None or bool((xdx[rows[1]:] == 0).all()), t + 'xdx outside written'
        if kern[0] == 'rowgroup' and sides:
            dx2, dth2, dn = run_bwd(v, inp, feat, xoff, goff, sides, want_dnorm=True)
            check(t + 'folded d_norm', dn, dn_r)
            assert torch.equal(dx2, dx), t + 'dX differs with the folded norm gradient'
            check(t + 'd_theta (folded)', dth2, dth_r)
    # d_theta of row sub-ranges adds up to the full result; each share against the reference of its source rows
    if full and kern[0] == 'stream':
        total = torch.zeros(v.r, dtype=torch.float64, device=DEV)
        for rb, re_ in ((0, 33), (33, 65), (65, 128), (128, v.n)):
            _, share, _ = run_bwd(v, inp, feat, xoff, goff, 3, rows=(rb, re_))
            check(tag + 'd_theta rows %d..%d' % (rb, re_), share, ref_bwd(v, inp, 3, rows=(rb, re_))[1])
            total += share.double()
        check(tag + 'd_theta summed over sub-ranges', total, ref_bwd(v, inp, 3)[1], extra=7.0)


@pytest.mark.parametrize('r', [1, 46, 200])
def test_fused_backward_relation_counts(r):
    """R = 46 is the first relation count whose bins need the shared-memory opt-in; R = 200 the ABI's maximum."""
    v = view(r)
    assert int(v.et.max()) + 1 == r
    widths = [(64, 0, 0, True), (8, 0, 0, True), (7, 0, 0, True), (33, 0, 0, True)]
    if r < 200:
        widths += [(256, 0, 0, True), (128, 0, 2, True)]
    for feat, xoff, goff, full in widths:
        assert fused_bwd_fits(feat, r)
        inp = inputs(v, feat, seed=r + feat)
        kern, _ = bwd_kernel(feat, xoff, goff, full)
        dx_r, dth_r, xdx_r, dn_r = ref_bwd(v, inp, 3)
        tag = 'R%d F%d %s ' % (r, feat, kern)
        dx, dth, xdx = run_bwd(v, inp, feat, xoff, goff, 3, want_xdx=True)
        check(tag + 'dX', dx, dx_r)
        check(tag + 'd_theta', dth, dth_r)
        check(tag + 'xdx', xdx, xdx_r)
        if kern[0] == 'rowgroup':
            check(tag + 'folded d_norm', run_bwd(v, inp, feat, xoff, goff, 3, want_dnorm=True)[2], dn_r)


# ---- two-pass fallback: regnn_spmm_bwd_w and regnn_rowdot_norm_bwd --------------------------------------------------
@pytest.mark.parametrize('feat,off', BWDW_WIDTHS, ids=['F%d_off%d' % w for w in BWDW_WIDTHS])
def test_bwd_w_every_class_vs_float64(bv, feat, off):
    v = bv
    inp = inputs(v, feat, seed=feat * 7 + off)
    cls = pick_shape(feat, off == 0)
    x, _ = placed(inp['x'], off)
    y, _ = placed(inp['y'], off)
    g, _ = placed(inp['g'], off)
    dx_in, _ = placed(inp['y'].flip(0), off)     # any dX: d_norm takes it as given
    norm = inp['norm'].to(DEV, torch.float32)
    th = inp['theta'].to(DEV, torch.float32)
    for sides in (3, 1, 2):
        ns, nd = sides_norms(inp['norm'], sides)
        _, dn_r = ref_rowdots(v, inp['x'], inp['y'], inp['g'], (_d(dx_in), _d(dx_in).abs(), torch.zeros_like(_d(x))),
                              inp['norm'], sides)
        dth_r = ref_dtheta(v, inp['x'], inp['g'], inp['theta'], ns, nd)
        tag = 'bwd_w F%d %s s%d ' % (feat, cls, sides)
        for weighted in (True, False):
            dth, dn = ops.spmm_bwd_w(v.csr, v.etv[0], th if weighted else None, ALPHA, norm, x, y, g, dx_in,
                                     sides=sides, split=v.csr.get('split'))
            check(tag + 'w%d d_norm' % weighted, dn, dn_r)
            if weighted:
                check(tag + 'd_theta', dth, dth_r)
            else:
                assert dth is None


@pytest.mark.parametrize('feat,off', [(64, 0), (64, 1), (33, 0), (256, 0), (256, 2)])
def test_rowdot_norm_vector_and_scalar_paths(bv, feat, off):
    v = bv
    inp = inputs(v, feat, seed=feat + off)
    ref_dx = ref_spmm(v, inp['g'], inp['theta'], inp['norm'], inp['norm'], transposed=True)
    x, _ = placed(inp['x'], off)
    y, _ = placed(inp['y'], off)
    g, _ = placed(inp['g'], off)
    dx, _ = placed(ref_dx[0], off)
    norm = inp['norm'].to(DEV, torch.float32)
    for sides in (3, 1, 2):
        # dX enters as given (fp32 of the reference): its own error is not part of this kernel's
        _, dn_r = ref_rowdots(v, inp['x'], inp['y'], inp['g'], (_d(dx), _d(dx).abs(), torch.zeros_like(_d(x))),
                              inp['norm'], sides)
        check('rowdot F%d off%d s%d' % (feat, off, sides), ops.rowdot_norm_bwd(norm, x, y, g, dx, sides=sides), dn_r)
        xdx = (x.double() * dx.double()).sum(1).float()
        _, dn_x = ref_rowdots(v, inp['x'], inp['y'], inp['g'], (_d(dx), _d(dx).abs(), torch.zeros_like(_d(x))),
                              inp['norm'], sides)
        check('rowdot xdx F%d off%d s%d' % (feat, off, sides),
              ops.rowdot_norm_bwd(norm, x, y, g, dx, sides=sides, xdx=xdx), dn_x)
        part = ops.rowdot_norm_bwd(norm, x, y, g, dx, sides=sides, rows=(33, 2999))
        check('rowdot rows F%d s%d' % (feat, sides), part, dn_r, rows=(33, 2999))
        assert bool((part[:33] == 0).all()) and bool((part[2999:] == 0).all())


# ---- degree norm ----------------------------------------------------------------------------------------------------
def ref_wdeg(v, theta, alpha, exponent, clamp_min, d_norm, es=None):
    """(deg, norm, d_theta) references: deg exact; norm = max(deg, c)^q (c <= 0: deg^q, 0 without in-edges);
    d_theta through dd = [deg >= c] q max(deg, c)^(q-1) d_norm (the tie passes, PyTorch's convention)."""
    w = rel_w(theta, alpha)[v.et]
    if es is not None:
        w = w * es
    deg = _seg(v.row, v.n, w)
    deg_ref = (deg, _seg(v.row, v.n, w.abs()), v.indeg.to(torch.float64))
    k = v.indeg.to(torch.float64) + 8
    if clamp_min > 0:
        c = deg.clamp(min=clamp_min)
        nm = c ** exponent
        dd = torch.where(deg >= clamp_min, exponent * c ** (exponent - 1), torch.zeros_like(deg))
    else:
        safe = torch.where(deg == 0, torch.ones_like(deg), deg)
        nm = torch.where(deg == 0, torch.zeros_like(deg), safe ** exponent)
        dd = torch.where(deg == 0, torch.zeros_like(deg), exponent * safe ** (exponent - 1))
    dd = dd * _d(d_norm)
    r = theta.numel()
    s = rel_w_grad(theta, alpha)
    dth = (_seg(v.et, r, dd[v.row]) * s, _seg(v.et, r, dd[v.row].abs()) * s.abs(),
           _seg(v.et, r, torch.ones(v.e, dtype=torch.float64, device=DEV)) + 8)
    return deg_ref, (nm, nm.abs(), k), dth


WDEG_CASES = [(r, kind, q, c) for r, kind in ((5, 'counts'), (5, 'slots'), (46, 'generic'))
              for q in (-0.5, -1.0, -0.25) for c in (1.0, 0.0)]


@pytest.mark.parametrize('r,kind,exponent,clamp_min', WDEG_CASES,
                         ids=['R%d_%s_q%g_c%g' % w for w in WDEG_CASES])
def test_degree_norm_vs_float64(r, kind, exponent, clamp_min):
    """The count kernel (etype_views' table), the slot walk (R <= 32) and the generic kernel (R > 32), forward and
    backward; relation 2 negative (LeakyReLU branch); rows of weighted degree exactly clamp_min = 1 (the tie)."""
    v = view(r)
    rng = np.random.RandomState(r + int(-4 * exponent) + int(clamp_min))
    theta = theta_of(rng, r)
    theta[0] = 1.0 / ALPHA                       # w = 1 for relation 1: TIE_ROW has weighted degree exactly 1
    if clamp_min == 0.0:
        theta = theta.abs()                      # without the clamp a negative degree has no real power
    d_norm = dyadic(rng, v.n)
    counts = v.etv[2] if kind == 'counts' else None
    if kind == 'counts' and ON_GPU:
        assert counts is not None
    th = theta.to(DEV, torch.float32)
    deg, norm = ops.wdeg_norm_fwd(v.csr, v.etv[0], th, ALPHA, exponent, counts=counts, clamp_min=clamp_min)
    d_theta = ops.wdeg_norm_bwd(v.csr, v.etv[0], th, ALPHA, exponent, deg, d_norm.to(DEV, torch.float32),
                                counts=counts, clamp_min=clamp_min)
    deg_r, norm_r, dth_r = ref_wdeg(v, theta, ALPHA, exponent, clamp_min, d_norm)
    tag = 'wdeg R%d %s q%g c%g ' % (r, kind, exponent, clamp_min)
    assert float(deg_r[0][TIE_ROW]) == 1.0
    if clamp_min == 0.0:
        assert bool((deg_r[0] == 0).any())       # rows without in-edges: norm 0, no gradient
    check(tag + 'deg', deg, deg_r)
    check(tag + 'norm', norm, norm_r)
    check(tag + 'd_theta', d_theta, dth_r)


# ---- end to end through functional.propagate ------------------------------------------------------------------------
def e2e_reference(v, x, theta, alpha, gout, weighted):
    """float64 autograd of Y = n (.) A_w (n (.) X), n = max(deg, 1)^-1/2 from the oracle's definitions (on the CPU, where
    the oracle allocates) -> (Y, sum of |terms| of Y, dX, d_theta) on the test device."""
    src, dst, et = torch.as_tensor(v.d['src']), torch.as_tensor(v.d['dst']), torch.as_tensor(v.d['etype'])
    x, theta, gout = (t.detach().cpu().double() for t in (x, theta, gout))
    xl = x.clone().requires_grad_(True)
    tl = theta.clone().requires_grad_(True)
    ew = O.edge_relation(tl.view(-1), alpha, et)
    nm = O.weighted_degree_norm(ew, dst, v.n, -0.5)
    coef = (ew if weighted else torch.ones_like(ew)) * nm[src]
    y = O.segment_sum(coef[:, None] * xl[src], dst, v.n) * nm[:, None]
    y.backward(gout)
    ya = O.segment_sum((coef.abs()[:, None] * xl[src].abs()).detach(), dst, v.n) * nm[:, None].detach()
    return tuple(t.to(DEV) for t in (y.detach(), ya, xl.grad, tl.grad))


E2E_CASES = [('fused_fold', 64, 5), ('fused_xdx', 256, 5), ('two_pass', 1000, 5), ('two_pass', 130, 200),
             ('unweighted', 64, 5), ('unweighted', 256, 5)]


def _e2e(v, case, feat, gmode='plain', seed=0):
    rng = np.random.RandomState(seed + feat)
    x = dyadic(rng, (v.n, feat))
    theta = helpers.f32_exact(rng.uniform(0.5, 1.5, size=(v.r, 1)) / 100.0)
    theta[min(1, v.r - 1)] = -theta[min(1, v.r - 1)]
    gout = dyadic(rng, (v.n, feat))
    weighted = case != 'unweighted'
    xs = x.to(DEV, torch.float32).requires_grad_(True)
    th = theta.to(DEV, torch.float32).requires_grad_(True)
    nm = RF.weighted_degree_norm(v.g, v.etv, th, 100.0, -0.5)
    y = RF.propagate(v.g, v.etv, xs, th if weighted else None, 100.0, nm)
    if gmode == 'misaligned':
        # d loss / d y reaches backward as a narrow view of the cat gradient: 4 bytes past the buffer's start
        t = torch.zeros(1, device=DEV, requires_grad=True)
        wts = torch.cat([torch.zeros(1, dtype=torch.float64), gout.reshape(-1)]).to(DEV, torch.float32)
        (torch.cat([t, y.view(-1)]) * wts).sum().backward()
    else:
        y.backward(gout.to(DEV, torch.float32))
    return x, theta, gout, weighted, y.detach(), xs.grad, th.grad


@pytest.mark.parametrize('case,feat,r', E2E_CASES, ids=['%s_F%d_R%d' % c for c in E2E_CASES])
def test_propagate_end_to_end_vs_oracle(case, feat, r):
    """functional.propagate at each branch of its backward, alpha = 100 (the reference default), against float64
    autograd of the oracle.  Y elementwise, with the rounding of the two norm factors added to k; the gradients, which
run through the degree norm's own backward, norm-wise."""
    v = view(r)
    if case != 'unweighted':
        assert (case == 'two_pass') == (not ops.fused_bwd_fits(feat, r))
        assert (case == 'fused_fold') == (ops.fused_bwd_fits(feat, r) and ops.fused_dnorm_fits(feat))
    x, theta, gout, weighted, y, dx, dth = _e2e(v, case, feat)
    ry, ya, rdx, rdth = e2e_reference(v, x.to(DEV, torch.float64), theta.to(DEV, torch.float64), 100.0,
                                      gout.to(DEV, torch.float64), weighted)
    tag = 'e2e %s F%d R%d ' % (case, feat, r)
    # the norms come from fp32 degree sums of non-dyadic weights: |q| = 1/2 of a row's slots per norm factor
    k = 1.5 * v.indeg.double() + 0.5 * float(v.indeg.max())
    check(tag + 'Y', y, (ry, ya, k[:, None].expand_as(ry)), extra=9.0)
    _assert_rel(tag + 'dX', dx, rdx, 1e-5)
    _assert_rel(tag + 'd_theta', dth, rdth, 1e-4)


def _assert_rel(tag, got, ref, rtol):
    helpers.assert_close(got.detach().cpu(), ref.detach().cpu(), rtol, tag)


def test_propagate_misaligned_gradient():
    """F = 64 with d loss / d y 4 bytes past 16-byte alignment: the folded norm gradient cannot run (the lane-group
    kernel needs every operand 16-byte aligned), and backward takes the xdx + row-dot path instead of failing.  The
    gradients equal the aligned run's: dX bit for bit, d_theta to fp32 rounding (its bins sum in another order)."""
    v = view(5)
    x, theta, gout, _, y, dx, dth = _e2e(v, 'fused_fold', 64, gmode='misaligned')
    _, _, _, _, y0, dx0, dth0 = _e2e(v, 'fused_fold', 64)
    assert torch.equal(y, y0) and torch.equal(dx, dx0)
    _assert_rel('misaligned d_theta', dth, dth0, 1e-5)
    _, _, rdx, rdth = e2e_reference(v, x.to(DEV, torch.float64), theta.to(DEV, torch.float64), 100.0,
                                    gout.to(DEV, torch.float64), True)
    _assert_rel('misaligned d_theta vs oracle', dth, rdth, 1e-4)


def test_fused_dnorm_fits_checks_every_operand():
    a = torch.zeros(16 * 64 + 4, device=DEV)
    ok, off = a[:16 * 64].view(16, 64), a[1:1 + 16 * 64].view(16, 64)
    assert ops.fused_dnorm_fits(64, ok, ok, ok, None)
    assert not ops.fused_dnorm_fits(64, ok, off, ok)
    assert not ops.fused_dnorm_fits(64, ok, ok, off)
    assert not ops.fused_dnorm_fits(64, off, ok, ok)
    assert not ops.fused_dnorm_fits(64, ok, torch.zeros(16 * 66, device=DEV).view(16, 66)[:, :64], ok)
    assert not ops.fused_dnorm_fits(62, ok) and not ops.fused_dnorm_fits(132, ok)
    assert not ops.fused_dnorm_fits(64, ok, rows_full=False)


# ---- refusals -------------------------------------------------------------------------------------------------------
REFUSALS = [('fwd', 257, 0), ('fwd', 1028, 0), ('fwd', 260, 1), ('fwd', 1024, 1), ('fwd', 514, 2), ('fwd', 1024, 2),
            ('bwd', 257, 0), ('bwd', 1028, 0), ('bwd', 300, 1), ('bwd', 600, 2)]


@pytest.mark.parametrize('which,feat,off', REFUSALS, ids=['%s_F%d_off%d' % c for c in REFUSALS])
def test_unsupported_widths_are_refused(bv, which, feat, off):
    if not ON_GPU:
        pytest.skip('the refusal is the kernels\'')
    v = bv
    inp = inputs(v, feat, seed=1)
    if which == 'fwd':
        assert fwd_kernel(feat, off, feat, True) is None
        with pytest.raises(RuntimeError, match='too wide'):
            run_fwd(v, inp, feat, off, 3, True)
        y, ybuf = placed(torch.zeros(v.n, feat, dtype=torch.float64), off, fill=7.0)
        y.fill_(-3.0)
        with pytest.raises(RuntimeError, match='too wide'):
            ops.spmm(v.csr['indptr'], v.csr['indices'], v.etv[0], inp['theta'].to(DEV, torch.float32), ALPHA, None, None,
                     placed(inp['x'], off)[0], out=y, split=v.csr['split'], order=ops.row_order(v.csr))
        torch.cuda.synchronize()
        assert bool((y == -3.0).all()) and bool((ybuf[:off] == 7.0).all())
    else:
        assert bwd_kernel(feat, off, off, True)[0] is None
        dx, dbuf = placed(torch.full((v.n, feat), -3.0, dtype=torch.float64), off, fill=7.0)
        with pytest.raises(RuntimeError, match='too wide'):
            ops.spmm_bwd_fused(v.csr, v.etv[1], inp['theta'].to(DEV, torch.float32), ALPHA, None,
                               placed(inp['x'], off)[0], placed(inp['g'], off)[0], out=dx)
        torch.cuda.synchronize()
        assert bool((dx == -3.0).all()) and bool((dbuf[:off] == 7.0).all())


def test_relation_count_past_the_limit_is_refused(bv):
    if not ON_GPU:
        pytest.skip('the refusal is the kernels\'')
    v = bv
    inp = inputs(v, 64, seed=2)
    th = torch.full((201,), 0.25, device=DEV)
    y = torch.full((v.n, 64), -3.0, device=DEV)
    x = inp['x'].to(DEV, torch.float32)
    with pytest.raises(RuntimeError, match='num_relations=201'):
        ops.spmm(v.csr['indptr'], v.csr['indices'], v.etv[0], th, ALPHA, None, None, x, out=y)
    with pytest.raises(RuntimeError, match='num_relations=201'):
        ops.spmm_bwd_fused(v.csr, v.etv[1], th, ALPHA, None, x, x, out=y)
    with pytest.raises(RuntimeError, match='num_relations=201'):
        ops.spmm_bwd_w(v.csr, v.etv[0], th, ALPHA, None, x, x, x, x, sides=0)
    with pytest.raises(RuntimeError, match='num_relations=201'):
        ops.wdeg_norm_fwd(v.csr, v.etv[0], th, ALPHA, -0.5)
    torch.cuda.synchronize()
    assert bool((y == -3.0).all())


# ---- index width ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('feat', [128, 256])
def test_index_width_past_2_31_elements(feat):
    """N * F > 2^31 with hub rows at the top of the row range gathering rows at the top of the index range:
    rowgroup at F = 128, stream at F = 256.  Sampled rows against float64."""
    if not ON_GPU:
        pytest.skip('needs the device')
    n = (1 << 31) // feat + 4099
    need = 2 * n * feat * 4 + (4 << 30)
    if torch.cuda.mem_get_info()[0] < max(need, 40 << 30):
        pytest.skip('needs about 40 GB of free device memory')
    rng = np.random.RandomState(feat)
    top = np.arange(n - 3000, n)
    hubs = np.array([n - 1, n - 2, n - 40])
    dst = np.concatenate([np.repeat(hubs, [769, 513, 257]), rng.randint(0, n, size=5000)])
    src = np.concatenate([rng.choice(top, size=769 + 513 + 257), rng.randint(0, n, size=5000)])
    src[:100] = n - 1
    etype = rng.randint(1, 4, size=src.size)
    g = Graph(src.astype(np.int64), dst.astype(np.int64), n).to(DEV)
    etv = g.etype_views(torch.as_tensor(etype).to(DEV), 3)
    csr = g.csr()
    theta = torch.tensor([[0.25], [0.5], [0.125]], device=DEV)
    x = torch.empty((n, feat), device=DEV).random_(-8, 9).mul_(0.125)
    y = ops.spmm(csr['indptr'], csr['indices'], etv[0], theta, ALPHA, None, None, x, split=csr['split'],
                 order=ops.row_order(csr) if feat <= 128 else None)
    sample = torch.as_tensor(np.unique(np.concatenate([hubs, dst[-50:], [0, n // 2, n - 3]])), device=DEV)
    w = rel_w(theta)
    rows, cols, et = csr['row'].long(), csr['indices'].long(), etv[0].long()
    for v_ in sample.tolist():
        b, e = int(csr['indptr'][v_]), int(csr['indptr'][v_ + 1])
        terms = w[et[b:e]][:, None] * x[cols[b:e]].double()
        ref = (terms.sum(0), terms.abs().sum(0), torch.full((feat,), float(e - b), dtype=torch.float64, device=DEV))
        check('index width F%d row %d' % (feat, v_), y[v_:v_ + 1], tuple(t[None] for t in ref))
    del x, y


# ---- sensitivity of every tolerance ---------------------------------------------------------------------------------
def test_tolerances_reject_one_slot_or_fragment(bv):
    """Each bound above rejects a reference that drops one slot of the heaviest row or counts one fragment of it twice
    -- the kernels' results would fail the check by the same margin if they made that mistake."""
    v = bv
    feat = 64
    inp = inputs(v, feat, seed=99)
    indptr, indptr_t = v.csr['indptr'].long(), v.csr['indptr_t'].long()
    heavy, heavy_t = int(torch.argmax(v.indeg)), int(torch.argmax(v.outdeg))
    slot_t = v.csr['slot_t'].long()

    def es_of(slots, factor):
        es = torch.ones(v.e, dtype=torch.float64, device=DEV)
        es[slots] = factor
        return es

    # a slot of relation 1 (a positive weight) of the heaviest row of each view; the second fragment of that row
    hs = torch.arange(int(indptr[heavy]), int(indptr[heavy + 1]), device=DEV)
    hs_t = slot_t[int(indptr_t[heavy_t]):int(indptr_t[heavy_t + 1])]
    drop, drop_t = int(hs[v.et[hs] == 0][0]), int(hs_t[v.et[hs_t] == 0][0])
    frag, frag_t = hs[THRESHOLD:2 * THRESHOLD], hs_t[THRESHOLD:2 * THRESHOLD]
    ns, nd = sides_norms(inp['norm'], 3)
    y, _ = run_fwd(v, inp, feat, 0, 3, True)
    dx, dth, xdx = run_bwd(v, inp, feat, 0, 0, 3, want_xdx=True)
    dn = run_bwd(v, inp, feat, 0, 0, 3, want_dnorm=True)[2]
    th = inp['theta'].to(DEV, torch.float32)
    d_norm = dyadic(np.random.RandomState(3), v.n)
    d_norm[heavy] = 2.0 ** 16                    # the heaviest row dominates the relation sums of the norm gradient
    deg, nrm = ops.wdeg_norm_fwd(v.csr, v.etv[0], th, ALPHA, -0.5, counts=v.etv[2])
    dthn = ops.wdeg_norm_bwd(v.csr, v.etv[0], th, ALPHA, -0.5, deg, d_norm.to(DEV, torch.float32), counts=v.etv[2])
    # the unperturbed references pass
    check('Y', y, ref_spmm(v, inp['x'], inp['theta'], ns, nd))
    dx_r, dth_r, xdx_r, dn_r = ref_bwd(v, inp, 3)
    check('dX', dx, dx_r)
    check('d_theta', dth, dth_r)
    check('xdx', xdx, xdx_r)
    check('d_norm', dn, dn_r)
    wd = ref_wdeg(v, inp['theta'], ALPHA, -0.5, 1.0, d_norm)
    check('deg', deg, wd[0])
    check('norm', nrm, wd[1])
    check('wdeg d_theta', dthn, wd[2])
    # ... and every perturbed one fails
    for name, es_y, es_t in (('dropped slot', es_of([drop], 0.0), es_of([drop_t], 0.0)),
                             ('doubled fragment', es_of(frag, 2.0), es_of(frag_t, 2.0))):
        with pytest.raises(AssertionError):
            check('Y ' + name, y, ref_spmm(v, inp['x'], inp['theta'], ns, nd, es=es_y))
        b = ref_bwd(v, inp, 3, es=es_t)
        for label, got, ref in (('dX', dx, b[0]), ('xdx', xdx, b[2]), ('d_norm', dn, b[3])):
            with pytest.raises(AssertionError):
                check(label + ' ' + name, got, ref)
        wd = ref_wdeg(v, inp['theta'], ALPHA, -0.5, 1.0, d_norm, es=es_y)
        for label, got, ref in (('deg', deg, wd[0]), ('norm', nrm, wd[1])):
            with pytest.raises(AssertionError):
                check(label + ' ' + name, got, ref)
    # d_theta sums every slot of a relation: one slot is below its resolution, one fragment is not -- with terms of
    # one sign (random signs would cancel the fragment's share down to the rounding of the whole sum)
    pos = dict(inp, x=inp['x'].abs(), g=inp['g'].abs())
    dth_pos = run_bwd(v, pos, feat, 0, 0, 3)[1]
    check('d_theta', dth_pos, ref_bwd(v, pos, 3)[1])
    with pytest.raises(AssertionError):
        check('d_theta doubled fragment', dth_pos, ref_bwd(v, pos, 3, es=es_of(frag_t, 2.0))[1])
    with pytest.raises(AssertionError):
        check('wdeg d_theta doubled fragment', dthn,
              ref_wdeg(v, inp['theta'], ALPHA, -0.5, 1.0, d_norm, es=es_of(frag, 2.0))[2])


# ---- the kernels that actually ran ----------------------------------------------------------------------------------
TEMPLATED = ('spmm_stream_kernel', 'spmm_rowgroup_kernel', 'spmm_bwd_w_kernel')
PLAIN_KERNELS = ('spmm_frag_finalize_kernel', 'long_row_dnorm_kernel', 'rowdot_norm_kernel', 'relation_count_kernel',
                 'wdeg_norm_fwd_kernel', 'wdeg_norm_bwd_kernel', 'wdeg_norm_fwd_slot_kernel',
                 'wdeg_norm_bwd_slot_kernel', 'wdeg_norm_fwd_cnt_kernel', 'wdeg_norm_bwd_cnt_kernel')


def instantiated_kernels(src=None):
    """{(kernel, template arguments)} that the dispatch macros of spmm.cu instantiate (bools as 0 / 1)."""
    src = open(SPMM_CU).read() if src is None else src
    stream = re.findall(r'REGNN_STREAM_CASE\((\d+), (\d+), BINS_, CALL\)', src)
    rowgroup = re.findall(r'REGNN_ROWGROUP_CASE\((\d+), BINS_, CALL\)', src)
    gc = re.findall(r'REGNN_DISPATCH_GC\((\d+), (\d+), (\d+), CALL\)', src)
    out = set()
    for c, vw in stream:
        out |= {('spmm_stream_kernel', (int(c), int(vw), b)) for b in (0, 1)}
    for g in rowgroup:
        out |= {('spmm_rowgroup_kernel', t) for t in ((0, int(g), 0), (1, int(g), 0), (1, int(g), 1))}
    for g, c, vw in gc:
        out |= {('spmm_bwd_w_kernel', (int(g), int(c), int(vw), b)) for b in (0, 1)}
    return out


def parse_kernel_name(name):
    """'void regnn::spmm_stream_kernel<4, 4, false>(regnn::StreamArgs)' -> ('spmm_stream_kernel', (4, 4, 0))."""
    m = re.search(r'(\w+)<([^<>]*)>\(', name)
    if m is None:
        m2 = re.search(r'(\w+)\(', name)
        return (m2.group(1), ()) if m2 else (name, ())
    args = []
    for a in m.group(2).split(','):
        a = a.strip()
        a = {'true': '1', 'false': '0', '(bool)1': '1', '(bool)0': '0'}.get(a, a)
        args.append(int(a.rstrip('uU')))
    return m.group(1), tuple(args)


def test_every_instantiated_kernel_ran():
    """Runs one call of every case of the sweeps above under torch.profiler and compares the launched SpMM kernels,
    with their template arguments, with the instantiations of spmm.cu."""
    if not ON_GPU:
        pytest.skip('torch.profiler on the device')
    from torch.profiler import ProfilerActivity, profile
    v = view(5)
    v46 = view(46)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for feat, off in FWD_WIDTHS:
            inp = inputs(v, feat, seed=feat)
            run_fwd(v, inp, feat, off, 3, True)
            run_fwd(v, inp, feat, off, 3, True, rows=(33, 3001))
        for feat, xoff, goff, full in BWD_WIDTHS:
            inp = inputs(v, feat, seed=feat)
            run_bwd(v, inp, feat, xoff, goff, 3, rows=None if full else (0, v.n - 1), want_xdx=True)
            if bwd_kernel(feat, xoff, goff, full)[0][0] == 'rowgroup':
                run_bwd(v, inp, feat, xoff, goff, 3, want_dnorm=True)
        for feat, off in BWDW_WIDTHS:
            inp = inputs(v, feat, seed=feat)
            x = placed(inp['x'], off)[0]
            for th in (inp['theta'].to(DEV, torch.float32), None):
                ops.spmm_bwd_w(v.csr, v.etv[0], th, ALPHA, inp['norm'].to(DEV, torch.float32), x, x, x, x,
                               split=v.csr['split'])
        for w in (v, v46):
            th = theta_of(np.random.RandomState(0), w.r).to(DEV, torch.float32)
            fresh = w.g.etype_views(torch.as_tensor(w.d['etype']).to(DEV).clone(), w.r)   # relation_count_kernel
            for counts in (fresh[2], None):
                deg, _ = ops.wdeg_norm_fwd(w.csr, w.etv[0], th, ALPHA, -0.5, counts=counts)
                ops.wdeg_norm_bwd(w.csr, w.etv[0], th, ALPHA, -0.5, deg, torch.ones_like(deg), counts=counts)
        x = torch.ones(v.n, 64, device=DEV)
        ops.rowdot_norm_bwd(torch.ones(v.n, device=DEV), x, x, x, x)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    seen = {parse_kernel_name(nm) for nm in names}
    seen_templated = {k for k in seen if k[0] in TEMPLATED}
    want = instantiated_kernels()
    assert len(want) == 30 + 12 + 34
    assert seen_templated == want, 'missing %s, unexpected %s' % (sorted(want - seen_templated),
                                                                 sorted(seen_templated - want))
    missing = set(PLAIN_KERNELS) - {k[0] for k in seen}
    assert not missing, 'not launched: %s' % sorted(missing)
