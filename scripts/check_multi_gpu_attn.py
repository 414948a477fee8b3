"""Multi-rank GPU check + timing of the sharded attention / REMixHop paths (run under torchrun, one rank per GPU):
``partition.head_sliced_gat`` (REGAT core, heads = column slabs), ``partition.head_sliced_gatv2`` (REGATv2 core, the
same over fs and fd) and ``partition.feature_sliced_propagate(theta=None)`` (REMixHop's un-weighted propagation over
column slabs), each with the NCCL all-to-all and the peer-memory exchange, against the single-device
``functional.gat_layer`` / ``functional.gatv2_aggregate`` / ``functional.propagate`` on every rank: outputs and feature
gradients on the rank's row block, parameter gradients after ``allreduce_relation_grads``.  Then the step is timed (CUDA
events, max over ranks) next to the single-device step on the same graph; at world size 1 the difference is the cost of
the exchange path itself.

    torchrun ... scripts/check_multi_gpu_attn.py [graph_scale=1.0] [heads=8] [dim=16] [iters=10]"""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from re_gnn_b200 import Graph, functional as RF, partition, synth  # noqa: E402


def timed(fn, iters, dev):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b) / iters], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def main():
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
    heads = int(sys.argv[2]) if len(sys.argv) > 2 else 8
    dim = int(sys.argv[3]) if len(sys.argv) > 3 else 16
    iters = int(sys.argv[4]) if len(sys.argv) > 4 else 10
    d = synth.hetero_graph('mag', seed=3, scale=scale)
    n, r, e = d['num_nodes'], d['num_relations'], d['src'].size
    g = Graph(d['src'], d['dst'], n).to(dev)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(dev), r)
    gen = torch.Generator(device=dev).manual_seed(11)
    f = torch.randn(n, heads, dim, device=dev, generator=gen) * 0.5
    gout = torch.randn(n, heads, dim, device=dev, generator=gen)
    al0 = torch.randn(1, heads, dim, device=dev, generator=gen) * 0.3
    ar0 = torch.randn(1, heads, dim, device=dev, generator=gen) * 0.3
    th0 = (torch.rand(r, heads, device=dev, generator=gen) + 0.5) / 100
    thn0 = (torch.rand(r, 1, device=dev, generator=gen) + 0.5) / 100
    fd0 = torch.randn(n, heads, dim, device=dev, generator=gen) * 0.5
    bounds = partition.row_blocks(g.csr()['indptr'], world, balance='rows')
    rb, re = bounds[rank], bounds[rank + 1]
    res = {'n_gpus': world, 'num_nodes': int(n), 'num_edges': int(e), 'heads': heads, 'head_dim': dim}
    ok_all = True

    # ---- REGAT core, heads sharded
    def gat_single():
        leaves = [t.clone().requires_grad_(True) for t in (f, al0, ar0, th0)]
        out, _ = RF.gat_layer(g, etv, *leaves, 100.0, 0.2)
        out.backward(gout)
        return out.detach(), [t.grad for t in leaves]

    xch = partition.SlabExchange(heads * dim, bounds, rank, dev)

    def gat_sharded(exchange=None):
        mine = [f[rb:re].clone().requires_grad_(True)] + [t.clone().requires_grad_(True) for t in (al0, ar0, th0)]
        out = partition.head_sliced_gat(g, etv, mine[0], mine[1], mine[2], mine[3], 100.0, 0.2, bounds, rank,
                                        exchange=exchange)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads(mine[1:])
        return out.detach(), [t.grad for t in mine]
    ref_out, ref_g = gat_single()
    t1 = timed(lambda: gat_single(), iters, dev)
    res['regat'] = {'single_gpu_ms': t1}
    for name, ex in (('nccl_all_to_all', None), ('peer_memory', xch)):
        for rep in range(2):   # twice: the exchange buffers are reused
            out, grads = gat_sharded(ex)
        chk = {'out_equal': bool(torch.equal(out, ref_out[rb:re])), 'd_feat_equal': bool(torch.equal(grads[0], ref_g[0][rb:re])),
               'out_rel': rel(out, ref_out[rb:re]), 'd_feat_rel': rel(grads[0], ref_g[0][rb:re]),
               'd_attn_l_rel': rel(grads[1], ref_g[1]), 'd_attn_r_rel': rel(grads[2], ref_g[2]),
               'd_theta_rel': rel(grads[3], ref_g[3])}
        ok = (max(chk['out_rel'], chk['d_feat_rel']) < 1e-5 and
              max(chk['d_attn_l_rel'], chk['d_attn_r_rel'], chk['d_theta_rel']) < 5e-5)
        flag = torch.tensor([int(ok)], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_all = ok_all and bool(flag.item())
        chk['all_ranks_ok'] = bool(flag.item())
        del out, grads
        tp = timed(lambda: gat_sharded(ex), iters, dev)
        res['regat'][name] = {'check': chk, 'sharded_ms': tp, 'speedup': t1 / tp, 'gteps_sharded': e / tp / 1e6}
    del ref_out, ref_g

    # ---- REGATv2 core, heads sharded
    def gatv2_single():
        leaves = [t.clone().requires_grad_(True) for t in (f, fd0, al0, th0)]
        out, _ = RF.gatv2_aggregate(g, etv, *leaves, 100.0, 0.2)
        out.backward(gout)
        return out.detach(), [t.grad for t in leaves]

    xch2 = partition.SlabExchange(heads * dim, bounds, rank, dev, gatv2=True)

    def gatv2_sharded(exchange=None):
        mine = [t[rb:re].clone().requires_grad_(True) for t in (f, fd0)] + [t.clone().requires_grad_(True)
                                                                            for t in (al0, th0)]
        out = partition.head_sliced_gatv2(g, etv, *mine, 100.0, 0.2, bounds, rank, exchange=exchange)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads(mine[2:])
        return out.detach(), [t.grad for t in mine]
    ref_out, ref_g = gatv2_single()
    t1 = timed(lambda: gatv2_single(), iters, dev)
    res['regatv2'] = {'single_gpu_ms': t1}
    for name, ex in (('nccl_all_to_all', None), ('peer_memory', xch2)):
        for rep in range(2):   # twice: the exchange buffers are reused
            out, grads = gatv2_sharded(ex)
        chk = {'out_equal': bool(torch.equal(out, ref_out[rb:re])),
               'd_fs_equal': bool(torch.equal(grads[0], ref_g[0][rb:re])),
               'd_fd_equal': bool(torch.equal(grads[1], ref_g[1][rb:re])),
               'out_rel': rel(out, ref_out[rb:re]), 'd_fs_rel': rel(grads[0], ref_g[0][rb:re]),
               'd_fd_rel': rel(grads[1], ref_g[1][rb:re]), 'd_attn_rel': rel(grads[2], ref_g[2]),
               'd_theta_rel': rel(grads[3], ref_g[3])}
        ok = (max(chk['out_rel'], chk['d_fs_rel'], chk['d_fd_rel']) < 1e-5 and
              max(chk['d_attn_rel'], chk['d_theta_rel']) < 5e-5)
        flag = torch.tensor([int(ok)], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_all = ok_all and bool(flag.item())
        chk['all_ranks_ok'] = bool(flag.item())
        del out, grads
        tp = timed(lambda: gatv2_sharded(ex), iters, dev)
        res['regatv2'][name] = {'check': chk, 'sharded_ms': tp, 'speedup': t1 / tp, 'gteps_sharded': e / tp / 1e6}
    del ref_out, ref_g

    # ---- REMixHop propagation: relation weights enter through the norm only, un-weighted column slabs
    x = f.view(n, heads * dim)
    gx = gout.view(n, heads * dim)

    def mix_single():
        xs, th = x.clone().requires_grad_(True), thn0.clone().requires_grad_(True)
        out = RF.propagate(g, etv, xs, None, 100.0, RF.weighted_degree_norm(g, etv, th, 100.0, -0.5))
        out.backward(gx)
        return out.detach(), xs.grad, th.grad

    def mix_sharded(exchange=None):
        xo, th = x[rb:re].clone().requires_grad_(True), thn0.clone().requires_grad_(True)
        out = partition.feature_sliced_propagate(g, etv, xo, None, 100.0, RF.weighted_degree_norm(g, etv, th, 100.0, -0.5),
                                                 bounds, rank, exchange=exchange)
        out.backward(gx[rb:re])
        partition.allreduce_relation_grads([th])
        return out.detach(), xo.grad, th.grad
    ref = mix_single()
    t1 = timed(lambda: mix_single(), iters, dev)
    res['remixhop_propagate'] = {'single_gpu_ms': t1}
    for name, ex in (('nccl_all_to_all', None), ('peer_memory', xch)):
        for rep in range(2):
            got = mix_sharded(ex)
        chk = {'out_equal': bool(torch.equal(got[0], ref[0][rb:re])), 'dx_equal': bool(torch.equal(got[1], ref[1][rb:re])),
               'out_rel': rel(got[0], ref[0][rb:re]), 'dx_rel': rel(got[1], ref[1][rb:re]), 'd_theta_rel': rel(got[2], ref[2])}
        ok = max(chk['out_rel'], chk['dx_rel']) < 1e-5 and chk['d_theta_rel'] < 5e-5
        flag = torch.tensor([int(ok)], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_all = ok_all and bool(flag.item())
        chk['all_ranks_ok'] = bool(flag.item())
        del got
        tp = timed(lambda: mix_sharded(ex), iters, dev)
        res['remixhop_propagate'][name] = {'check': chk, 'sharded_ms': tp, 'speedup': t1 / tp, 'gteps_sharded': e / tp / 1e6}
    del ref
    if rank == 0:
        print(json.dumps(res), flush=True)
        print('MULTI_GPU_ATTN_CHECK', 'OK' if ok_all else 'FAIL', flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok_all else 1)


if __name__ == '__main__':
    main()
