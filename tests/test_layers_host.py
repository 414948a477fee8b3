"""Host-logic tests (no GPU): the package's modules + autograd stitching, with the CUDA operators
replaced by tests/cpu_shim.py, must reproduce the golden vectors recorded from the reference's own
layer / model code (tests/golden/make_golden.py) in float64."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

import helpers
import re_gnn_b200
from re_gnn_b200 import Graph

LAYER_CASES = [c for c in helpers.golden_cases() if not c.startswith('model_')]
MODEL_CASES = helpers.golden_cases('model_')
REF = os.environ.get('REGNN_REFERENCE', '')   # a checkout of the reference RE-GNN repository, if one is at hand


def run_layer_case(case, device='cpu', dtype=torch.float64):
    meta = case['meta']
    mod = helpers.load_params(helpers.build_layer(re_gnn_b200, meta), case, dtype, device)
    g = Graph(case['src'], case['dst'], int(case['num_nodes'])).to(device)
    et = torch.as_tensor(case['etype']).to(device)
    x = torch.as_tensor(case['in::x']).to(device=device, dtype=dtype).requires_grad_(True)
    if meta.get('no_etype'):
        out = mod(g, x, None)
    elif meta.get('get_attention'):
        out = mod(g, x, et, get_attention=True)
    else:
        out = mod(g, x, et)
    outs = out if isinstance(out, tuple) else (out,)
    outs[0].backward(torch.as_tensor(case['gout']).to(device=device, dtype=dtype))
    return mod, x, outs


def check_layer_case(case, mod, x, outs, rtol):
    for i, o in enumerate(outs):
        helpers.assert_close(o.detach().cpu(), case['out%d' % i], rtol, 'out%d' % i)
    helpers.assert_close(x.grad.cpu(), case['gin::x'], rtol, 'd_x')
    for k, p in mod.named_parameters():
        got = p.grad if p.grad is not None else torch.zeros_like(p)
        helpers.assert_close(got.cpu(), case['grad::' + k], rtol, 'd_' + k)


@pytest.mark.parametrize('name', LAYER_CASES)
def test_layer_matches_reference_golden(name, cpu_ops):
    case = helpers.load_case(name)
    mod, x, outs = run_layer_case(case)
    check_layer_case(case, mod, x, outs, 1e-9)


def test_parameter_names_match_reference_checkpoints():
    """State-dict keys/shapes must equal the reference's (checkpoint compatibility, SURVEY.md sec. 5)."""
    for name in LAYER_CASES:
        case = helpers.load_case(name)
        mod = helpers.build_layer(re_gnn_b200, case['meta'])
        ours = {k: tuple(v.shape) for k, v in mod.state_dict().items()}
        ref = {k.split('::', 1)[1]: tuple(v.shape) for k, v in case.items() if k.startswith('param::')}
        assert ours == ref, name


def test_gatv2_zero_in_degree_raises(cpu_ops):
    g = Graph([0, 1], [1, 2], 3)
    conv = re_gnn_b200.REGATv2Conv(2, 100.0, 4, 4, 1)
    with pytest.raises(re_gnn_b200.ZeroInDegreeError):
        conv(g, torch.randn(3, 4), torch.tensor([1, 2]))
    conv.set_allow_zero_in_degree(True)
    assert conv(g, torch.randn(3, 4), torch.tensor([1, 2])).shape == (3, 1, 4)


def test_bad_edge_type_raises(cpu_ops):
    g = Graph([0, 1], [1, 0], 2)
    conv = re_gnn_b200.REGraphConv(2, 100.0, 4, 4)
    with pytest.raises(RuntimeError):
        conv(g, torch.randn(2, 4), torch.tensor([1, 3]))


def test_graph_self_loop_conventions():
    """remove_self_loop keeps order; add_self_loop appends (i,i) for i=0..N-1 last (run_regnn.py:84-99)."""
    g = Graph([0, 1, 1, 2], [1, 1, 2, 0], 3).remove_self_loop().add_self_loop()
    s, d = g.edges()
    assert s.tolist() == [0, 1, 2, 0, 1, 2] and d.tolist() == [1, 2, 0, 0, 1, 2]
    assert g.in_degrees().tolist() == [2, 2, 2] and g.number_of_nodes() == 3 and not g.is_block
    import scipy.sparse as sp
    a = sp.coo_matrix((np.ones(3), ([0, 2, 1], [1, 0, 2])), shape=(3, 3))
    s, d = Graph(a).edges()
    assert s.tolist() == [0, 2, 1] and d.tolist() == [1, 0, 2]


def test_product_path_has_no_cpu_fallback():
    """Without the shim a CPU graph must fail loudly, not fall back."""
    g = Graph([0, 1], [1, 0], 2)
    conv = re_gnn_b200.REGraphConv(2, 100.0, 4, 4)
    with pytest.raises(RuntimeError):
        conv(g, torch.randn(2, 4), torch.tensor([1, 2]))


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, 'model')),
                    reason='needs REGNN_REFERENCE set to a checkout of the reference RE-GNN repository')
@pytest.mark.parametrize('name', MODEL_CASES)
def test_reference_models_run_unmodified_on_our_layers(name, cpu_ops, monkeypatch):
    """model/REGCN.py, REGAT.py, REMixHop.py, REGIN.py imported from the reference, with OUR package registered
    as ``layer`` (and a name-only ``dgl`` for REMixHop.py's unused imports), must reproduce the
    reference-over-DGL-stub goldens."""
    import torch.nn.functional as F
    from re_gnn_b200 import layer as our_layer
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for m in [k for k in sys.modules if k == 'model' or k.startswith('model.') or k == 'layer' or k.startswith('layer.')
              or k == 'dgl' or k.startswith('dgl.')]:
        monkeypatch.delitem(sys.modules, m)
    monkeypatch.setitem(sys.modules, 'layer', our_layer)
    monkeypatch.syspath_prepend(os.path.join(root, 'oracle', 'dgl_stub'))  # only for `import dgl` in REMixHop.py
    monkeypatch.syspath_prepend(REF)
    case = helpers.load_case(name)
    meta = case['meta']
    g = Graph(case['src'], case['dst'], int(case['num_nodes']))
    args = [helpers.ACT.get(a, a) if isinstance(a, str) else a for a in meta['args']]
    if meta['kind'] == 'REGCN':
        net = importlib.import_module('model.REGCN').REGCN(g, *args)
    elif meta['kind'] == 'REGAT':
        net = importlib.import_module('model.REGAT').REGAT(g, *args, use_gatv2=meta.get('use_gatv2', False))
    elif meta['kind'] == 'REGIN':
        net = importlib.import_module('model.REGIN').REGIN(g, *args)
    else:
        net = importlib.import_module('model.REMixHop').REMixHop(g, *args, activation=F.elu)
    net = helpers.load_params(net, case)
    feats = [torch.as_tensor(case['in::f%d' % i]).requires_grad_(True) for i in range(3)]
    out, _ = net(feats, torch.as_tensor(case['etype']))
    helpers.assert_close(out.detach(), case['out0'], 1e-9, 'logits')
    out.backward(torch.as_tensor(case['gout']))
    for i, f in enumerate(feats):
        helpers.assert_close(f.grad, case['gin::f%d' % i], 1e-9, 'd_f%d' % i)
    for k, p in net.named_parameters():
        got = p.grad if p.grad is not None else torch.zeros_like(p)
        helpers.assert_close(got, case['grad::' + k], 1e-8, 'd_' + k)


@pytest.mark.parametrize('name', MODEL_CASES)
def test_mirrored_models_match_reference_golden(name, cpu_ops):
    """re_gnn_b200.model.{REGCN,REGAT,REMixHop} (used where the reference checkout is absent) against
    the goldens recorded from the reference's own model files."""
    from re_gnn_b200 import model as our_model
    case = helpers.load_case(name)
    net, feats, out = helpers.run_model_case(our_model, Graph, case)
    helpers.check_model_case(case, net, feats, out, 1e-9, 1e-8)


def test_row_order_lists_short_rows_by_descending_slot_count():
    """ops.row_order: the work list of the narrow-row kernels (host-side index bookkeeping, device-independent)."""
    import ctypes
    from re_gnn_b200 import _lib, ops
    indptr = torch.tensor([0, 3, 3, 10, 11, 11, 16, 19], dtype=torch.int32)     # slot counts 3 0 7 1 0 5 3
    csr = {'indptr': indptr, 'indptr_t': indptr, 'split': None, 'split_t': None}
    assert ops.row_order(csr).tolist() == [2, 5, 0, 6, 3, 1, 4]                 # stable: ties by ascending row id
    assert ops.row_order(csr) is csr['order'] and ops.row_order(csr).dtype == torch.int32
    # rows cut into fragments (more slots than the threshold) are not in the list
    split = {'struct': _lib.RowSplit(None, None, None, None, 2, 4, 4)}          # two long rows at threshold 4
    csr_t = {'indptr': indptr, 'indptr_t': indptr, 'split': None, 'split_t': split}
    assert ops.row_order(csr_t, True).tolist() == [0, 6, 3, 1, 4]
