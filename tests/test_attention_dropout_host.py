"""Host-side checks of the counter-based attention dropout (``functional.HashedDropout``, ``regnn_attn_dropout_t``): the
oracle hash against a hand-computed table, the C struct's layout against its ctypes mirror, the Python surface, and --
in world-size-2 gloo processes with the CUDA operators replaced by the plain-PyTorch emulations defined here --
``partition.halo_gat`` / ``halo_gatv2`` / ``head_sliced_gat`` with dropout against the single-process layers fed the
oracle's explicit mask."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import attn_dropout_oracle as AO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = 0xFFFFFFFF


def _mix32_int(z):
    z &= M32
    z ^= z >> 16
    z = (z * 0x7feb352d) & M32
    z ^= z >> 15
    z = (z * 0x846ca68b) & M32
    z ^= z >> 16
    return z


def _hash_int(key, c):
    """The header's formula on Python ints."""
    x = _mix32_int((c & M32) ^ (key & M32))
    return _mix32_int(x + ((c >> 32) * 0x9E3779B1) + (key >> 32))


# (key, counter) -> hash, worked out with _hash_int once and kept as literals: the statement of the hash may not drift
TABLE = [
    (0x0000000000000000, 0, 0x00000000),
    (0x0000000000000000, 1, 0x58f54975),
    (0x0123456789ABCDEF, 0, 0xe47fa7e2),
    (0x0123456789ABCDEF, 7, 0xc4fbe3e2),
    (0xFFFFFFFFFFFFFFFF, 123456789, 0x96adc98a),
    (0x0123456789ABCDEF, (5 << 32) + 3, 0x022629f7),
]


def test_hash_table_is_the_header_formula():
    for key, c, want in TABLE:
        assert _hash_int(key, c) == want, (hex(key), c, hex(_hash_int(key, c)))


def test_oracle_hash_is_bit_exact_with_the_table():
    keys = {k for k, _, _ in TABLE}
    for key in keys:
        rows = [(c, h) for k, c, h in TABLE if k == key]
        got = AO.attn_dropout_hash(key, np.array([c for c, _ in rows], dtype=np.uint64))
        assert [int(x) for x in got] == [h for _, h in rows]
    rng = np.random.RandomState(0)
    for key in (0x9E3779B97F4A7C15, 3):
        c = rng.randint(0, 2 ** 62, size=200, dtype=np.int64).astype(np.uint64)
        got = AO.attn_dropout_hash(key, c)
        assert [int(x) for x in got] == [_hash_int(key, int(v)) for v in c]


def test_oracle_mask_threshold_scale_and_head_slices():
    p, key = 0.3, 0xABCDEF0123456789
    t, scale = AO.threshold_scale(p)
    assert t == int(np.floor(0.3 * 2 ** 32)) and scale == np.float32(1 / 0.7)
    m = AO.keep_mask(p, key, 50, 8)
    assert m.dtype == np.float32 and set(np.unique(m).tolist()) <= {0.0, float(scale)}
    for e, h in ((0, 0), (17, 5), (49, 7)):
        assert (m[e, h] != 0) == (_hash_int(key, e * 8 + h) >= t)
    assert np.array_equal(AO.keep_mask(p, key, 50, 3, head_offset=4, num_heads_total=8), m[:, 4:7])
    assert np.all(AO.keep_mask(0.0, key, 50, 8) == 1.0)


def test_hashed_dropout_surface():
    from re_gnn_b200 import functional as RF
    d = RF.HashedDropout(0.3, RF.attn_dropout_key(1, 2, 3))
    t, scale = AO.threshold_scale(0.3)
    s = d.struct(8)
    assert (s.threshold, s.head_offset, s.num_heads_total) == (t, 0, 8) and np.float32(s.scale) == scale
    s = d.for_heads(2, 8).struct(2)
    assert (s.head_offset, s.num_heads_total, s.key) == (2, 8, d.key)
    with pytest.raises(ValueError):
        d.for_heads(7, 8).struct(2)
    for p in (-0.1, 1.0, 1.5):
        with pytest.raises(ValueError):
            RF.HashedDropout(p, 0)
    s0 = RF.HashedDropout(0.0, 5).struct(1)
    assert s0.threshold == 0 and s0.scale == 1.0
    keys = {RF.attn_dropout_key(seed, step, layer) for seed in range(3) for step in range(50) for layer in range(3)}
    assert len(keys) == 450 and all(0 <= k < 2 ** 64 for k in keys)
    assert RF.attn_dropout_key(7, 9, 1) == RF.attn_dropout_key(7, 9, 1)
    # both halves change with the step (a change of one half only would make the masks permuted copies)
    a, b = RF.attn_dropout_key(7, 9, 1), RF.attn_dropout_key(7, 10, 1)
    assert (a & M32) != (b & M32) and (a >> 32) != (b >> 32)


def test_keep_and_dropout_are_exclusive():
    from re_gnn_b200 import Graph, functional as RF
    g = Graph(np.array([0, 1]), np.array([1, 0]), 2)
    f = torch.zeros(2, 1, 4)
    with pytest.raises(ValueError, match='not both'):
        RF.gat_layer(g, None, f, f[:1], f[:1], None, 1.0, 0.2, keep=torch.ones(2, 1), dropout=RF.HashedDropout(0.1, 1))
    with pytest.raises(TypeError, match='HashedDropout'):
        RF.gatv2_aggregate(g, None, f, f, f[:1], None, 1.0, 0.2, dropout=0.1)


def test_struct_layout_matches_the_c_compiler(tmp_path):
    """The header compiles as plain C and ``_lib.AttnDropout`` has the C compiler's size and field offsets."""
    import ctypes
    from re_gnn_b200 import _lib
    src = tmp_path / 'layout.c'
    src.write_text('''#include <stdio.h>
#include <stddef.h>
#include "regnn_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(regnn_attn_dropout_t), offsetof(regnn_attn_dropout_t, key),
         offsetof(regnn_attn_dropout_t, threshold), offsetof(regnn_attn_dropout_t, scale),
         offsetof(regnn_attn_dropout_t, head_offset), offsetof(regnn_attn_dropout_t, num_heads_total));
  return 0;
}
''')
    exe = tmp_path / 'layout'
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)],
                   check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = _lib.AttnDropout
    assert got == [ctypes.sizeof(S)] + [getattr(S, f).offset for f in
                                        ('key', 'threshold', 'scale', 'head_offset', 'num_heads_total')]


# ---- dropout-aware emulations of the attention operators (whole graph and local views) ----------------------------
def _slot_keep(dropout, eid, heads, dtype):
    """[slots, heads] keep factors of the slots whose global edge ids are ``eid`` (the oracle's hash)."""
    total = dropout.num_heads_total if dropout.num_heads_total is not None else dropout.head_offset + heads
    c = (eid.numpy().astype(np.uint64)[:, None] * np.uint64(total) + np.uint64(dropout.head_offset)
         + np.arange(heads, dtype=np.uint64)[None, :])
    t, scale = AO.threshold_scale(dropout.p)
    return torch.as_tensor(np.where(AO.attn_dropout_hash(dropout.key, c) >= np.uint32(t), scale, 0.0)).to(dtype)


def _keep_slots(csr, keep, dropout, eid, heads, dtype):
    if dropout is not None:
        return _slot_keep(dropout, csr['eid'] if eid is None else eid, heads, dtype)
    return None if keep is None else keep.detach()[csr['eid'].long()]


def _gat_fwd(csr, et_csr, theta, alpha, feat, el, er, slope, keep=None, want_attn=False, rows=None, dropout=None,
             eid=None):
    import cpu_shim
    feat, el, er = feat.detach(), el.detach(), er.detach()
    n = csr['indptr'].numel() - 1
    row, col = cpu_shim._rows_of(csr['indptr']), csr['indices'].long()
    pre = el[col] + er[row]
    if theta is not None and et_csr is not None:
        pre = pre + cpu_shim._w(theta.detach(), alpha)[et_csr.long()]
    a, mx, sm = cpu_shim._softmax_rows(cpu_shim._leaky(pre, slope), row, n)
    kc = _keep_slots(csr, keep, dropout, eid, feat.shape[1], feat.dtype)
    at = a if kc is None else a * kc
    out = torch.zeros((n,) + feat.shape[1:], dtype=feat.dtype).index_add(0, row, at[:, :, None] * feat[col])
    return out, mx, sm, None


def _gat_bwd_edges(csr, et_t, theta, alpha, feat, el, stats, slope, g, dpre, attn_l=None, keep=None, dropout=None,
                   eid=None):
    import cpu_shim
    feat, el, g = feat.detach(), el.detach(), g.detach()
    n = csr['indptr_t'].numel() - 1
    u, v, s = cpu_shim._rows_of(csr['indptr_t']), csr['indices_t'].long(), csr['slot_t'].long()
    st = stats[v]
    pre = el[u] + st[..., 0]
    if theta is not None and et_t is not None:
        pre = pre + cpu_shim._w(theta.detach(), alpha)[et_t.long()]
    a = torch.exp(cpu_shim._leaky(pre, slope) - st[..., 1]) * st[..., 2]
    at = a
    if dropout is not None:
        at = a * _slot_keep(dropout, (csr['eid'] if eid is None else eid)[s], feat.shape[1], feat.dtype)
    dp = (at * (feat[u] * g[v]).sum(-1) - a * st[..., 3]) * cpu_shim._lgrad(pre, slope)
    dpre[s] = dp
    d_el = torch.zeros((n, feat.shape[1]), dtype=feat.dtype).index_add(0, u, dp)
    d_feat = torch.zeros((n,) + feat.shape[1:], dtype=feat.dtype).index_add(0, u, at[:, :, None] * g[v])
    if attn_l is not None:
        d_feat = d_feat + d_el[:, :, None] * attn_l.detach().view(1, *feat.shape[1:])
    return d_feat, d_el


def _edge_order_keep(csr, dropout, heads, dtype):
    eid = csr['eid'].long()
    keep = torch.zeros((eid.numel(), heads), dtype=dtype)
    keep[eid] = _slot_keep(dropout, csr['eid'], heads, dtype)
    return keep


def _gat_bwd(csr, et_csr, et_t, theta, alpha, feat, el, er, slope, keep, out, rowmax, rowsum, g, attn_l=None,
             attn_r=None, dropout=None):
    import cpu_shim
    if dropout is not None:
        keep = _edge_order_keep(csr, dropout, feat.shape[1], feat.dtype)
    return cpu_shim.gat_bwd(csr, et_csr, et_t, theta, alpha, feat, el, er, slope, keep, out, rowmax, rowsum, g,
                            attn_l=attn_l, attn_r=attn_r)


def _gatv2_fwd(csr, et_csr, theta, alpha, fs, fd, attn, slope, keep=None, want_attn=False, rows=None, save=False,
               saved=None, dropout=None, eid=None):
    import cpu_shim
    import test_halo_gatv2_host as V2
    fs, fd = fs.detach(), fd.detach()
    _, h, d = fs.shape
    n = csr['indptr'].numel() - 1
    row, col = cpu_shim._rows_of(csr['indptr']), csr['indices'].long()
    q = fs[col] + fd[row]
    lg = (cpu_shim._leaky(q, slope) * attn.detach().view(1, h, d)).sum(-1)
    if theta is not None and et_csr is not None:
        lg = lg + cpu_shim._w(theta.detach(), alpha)[et_csr.long()]
    a, mx, sm = cpu_shim._softmax_rows(lg, row, n)
    kc = _keep_slots(csr, keep, dropout, eid, h, fs.dtype)
    at = a if kc is None else a * kc
    out = torch.zeros((n, h, d), dtype=fs.dtype).index_add(0, row, at[:, :, None] * fs[col])
    e = col.numel()
    if saved is None and save:
        saved = (lg.new_empty((e, h)), torch.empty((e, V2._chunks(h, d), 4), dtype=torch.int32))
    if saved is not None:
        saved[0][:e] = lg
        saved[1][:e] = V2._pack(q > 0)
    return out, mx, sm, None, saved


def _gatv2_bwd_edges(csr, fs, stats, logit_csr, qmask, attn, slope, g, dl, keep=None, dropout=None, eid=None):
    import test_halo_gatv2_host as V2
    fs, g = fs.detach(), g.detach()
    _, h, d = fs.shape
    n = csr['indptr_t'].numel() - 1
    u, v, s = V2._rows(csr['indptr_t']), csr['indices_t'].long(), csr['slot_t'].long()
    st = stats[v]
    a = torch.exp(logit_csr[s] - st[..., 1]) * st[..., 2]
    at = a
    if dropout is not None:
        at = a * _slot_keep(dropout, (csr['eid'] if eid is None else eid)[s], h, fs.dtype)
    elif keep is not None:
        at = a * keep.detach()[csr['eid'].long()[s]]
    dls = at * (fs[u] * g[v]).sum(-1) - a * st[..., 3]
    dl[s] = dls
    t_src = torch.zeros((n, h, d), dtype=fs.dtype).index_add(0, u, dls[:, :, None] * V2._phi(qmask[s], h, d, slope, fs.dtype))
    d_fs = torch.zeros((n, h, d), dtype=fs.dtype).index_add(0, u, at[:, :, None] * g[v]) + attn.detach().view(1, h, d) * t_src
    return d_fs, (fs * t_src).sum(0).reshape(-1)


def install_dropout_shim(monkeypatch):
    """The REGATv2 halo shim (which includes the REGAT and REGCN halo shims) with the attention stages replaced by the
    dropout-aware emulations above; ops.gat_bwd / ops.gatv2_bwd: cpu_shim's whole-graph backward with the mask, and the
    real composition of the stages for REGATv2."""
    import test_halo_gatv2_host as V2
    from re_gnn_b200 import ops
    gatv2_bwd = ops.gatv2_bwd          # the library's composition of the stages (no device work of its own)
    V2.install_gatv2_halo_shim(monkeypatch)
    for name, fn in (('gat_fwd', _gat_fwd), ('gat_bwd_edges', _gat_bwd_edges), ('gat_bwd', _gat_bwd),
                     ('gatv2_fwd', _gatv2_fwd), ('gatv2_bwd_edges', _gatv2_bwd_edges), ('gatv2_bwd', gatv2_bwd)):
        monkeypatch.setattr(ops, name, fn)


def _close(a, b, rtol=1e-10):
    return torch.allclose(a, b, rtol=rtol, atol=1e-12)


def _worker(rank, world, port, ret, layout):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import test_attention_dropout_host as T
    from oracle import attn_dropout_oracle as O
    from re_gnn_b200 import Graph, functional as RF, partition, synth

    class MP:  # minimal monkeypatch stand-in
        @staticmethod
        def setattr(obj, name, val):
            setattr(obj, name, val)
    T.install_dropout_shim(MP)
    d = synth.hetero_graph_local('dblp', world, 0.9, seed=5, scale=0.03)
    n, r, h, dim = d['num_nodes'], d['num_relations'], 2, 4
    e = d['src'].size
    rng = np.random.RandomState(0)
    f, fd, gout = (torch.as_tensor(rng.randn(n, h, dim)) for _ in range(3))
    al0, ar0 = (torch.as_tensor(rng.randn(1, h, dim) * 0.3) for _ in range(2))
    th0 = torch.as_tensor(rng.uniform(0.5, 1.5, (r, h)) / 100.0)
    g = Graph(d['src'], d['dst'], n)
    etv = g.etype_views(torch.as_tensor(d['etype']), r)
    bounds = d['community_bounds'] if layout == 'community' else partition.row_blocks(g.csr()['indptr'], world)
    rb, re = bounds[rank], bounds[rank + 1]
    part = partition.HaloPartition(g, etv, bounds, rank, attention=True)
    ok = part.tail_ptr[-1] > 0 and part.push_slots[1][-1] > 0
    drop = RF.HashedDropout(0.4, RF.attn_dropout_key(2, 3, 0))
    keep = torch.as_tensor(O.keep_mask(drop.p, drop.key, e, h)).double()
    # REGAT on row blocks
    leaves = [t.clone().requires_grad_(True) for t in (f, al0, ar0, th0)]
    ref, _ = RF.gat_layer(g, etv, *leaves, 100.0, 0.2, keep=keep)
    ref.backward(gout)
    plain, _ = RF.gat_layer(g, etv, f, al0, ar0, th0, 100.0, 0.2)
    ok = ok and not torch.allclose(plain, ref)
    for _ in range(2):
        fo = f[rb:re].clone().requires_grad_(True)
        al, ar, th = (t.clone().requires_grad_(True) for t in (al0, ar0, th0))
        out = partition.halo_gat(part, fo, al, ar, th, 100.0, 0.2, dropout=drop)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads([al, ar, th])
        ok = (ok and _close(out.detach(), ref.detach()[rb:re], 1e-12) and _close(fo.grad, leaves[0].grad[rb:re])
              and all(_close(a.grad, b.grad) for a, b in zip((al, ar, th), leaves[1:])))
    # REGATv2 on row blocks
    leaves = [t.clone().requires_grad_(True) for t in (f, fd, al0, th0)]
    ref, _ = RF.gatv2_aggregate(g, etv, *leaves, 100.0, 0.2, keep=keep)
    ref.backward(gout)
    for _ in range(2):
        fso, fdo = f[rb:re].clone().requires_grad_(True), fd[rb:re].clone().requires_grad_(True)
        attn, th = al0.clone().requires_grad_(True), th0.clone().requires_grad_(True)
        out = partition.halo_gatv2(part, fso, fdo, attn, th, 100.0, 0.2, dropout=drop)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads([attn, th])
        ok = (ok and _close(out.detach(), ref.detach()[rb:re], 1e-12) and _close(fso.grad, leaves[0].grad[rb:re])
              and _close(fdo.grad, leaves[1].grad[rb:re]) and _close(attn.grad, leaves[2].grad)
              and _close(th.grad, leaves[3].grad))
    # REGAT sharded over the heads (equal row blocks): rank q draws heads [q*H/P, (q+1)*H/P) of the full-H mask
    hb = partition.row_blocks(g.csr()['indptr'], world, balance='rows')
    leaves = [t.clone().requires_grad_(True) for t in (f, al0, ar0, th0)]
    ref, _ = RF.gat_layer(g, etv, *leaves, 100.0, 0.2, keep=keep)
    ref.backward(gout)
    mine = [f[hb[rank]:hb[rank + 1]].clone().requires_grad_(True)] + [t.clone().requires_grad_(True)
                                                                      for t in (al0, ar0, th0)]
    out = partition.head_sliced_gat(g, etv, *mine, 100.0, 0.2, hb, rank, dropout=drop)
    out.backward(gout[hb[rank]:hb[rank + 1]])
    partition.allreduce_relation_grads(mine[1:])
    ok = (ok and _close(out.detach(), ref.detach()[hb[rank]:hb[rank + 1]], 1e-12)
          and _close(mine[0].grad, leaves[0].grad[hb[rank]:hb[rank + 1]])
          and all(_close(a.grad, b.grad) for a, b in zip(mine[1:], leaves[1:])))
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize('layout', ['community', 'edges'])
def test_partitioned_attention_with_dropout_matches_single_process_world2(layout):
    """halo_gat, halo_gatv2 (all-to-all exchange variant, two steps on one partition) and head_sliced_gat with a
    HashedDropout reproduce gat_layer / gatv2_aggregate fed the oracle's explicit mask."""
    world = 2
    port = 25500 + (os.getpid() % 1500) + (0 if layout == 'community' else 1700)
    ret = mp.get_context('spawn').Manager().dict()
    mp.spawn(_worker, args=(world, port, ret, layout), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world)), dict(ret)
