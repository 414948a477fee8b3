"""Cost of attention dropout in the fused REGAT / REGATv2 cores on the MAG-shaped graph (synth.hetero_graph('mag')).

For each core (functional.gat_layer, functional.gatv2_aggregate) at H x D = 8 x 16 and 2 x 64, forward + backward is
timed three ways, alternated step by step inside one window per way after a warm-up:
  none      no attention dropout;
  explicit  a mask drawn with torch every step, keep = (rand(E, H) >= p) / (1 - p) (the draw is part of the step),
            passed as ``keep`` (the kernels read it in edge-id order, forward and backward);
  hashed    ``dropout=HashedDropout(p, key)`` with a new key every step: the kernels compute the factor from the edge id.
Then, on the community-structured MAG-shaped graph (synth.hetero_graph_local, P virtual ranks on one GPU), the per-rank
compute of partition.halo_gat / halo_gatv2 (halos pre-filled; forward, statistics, edge pass, reduction) with and
without hashed dropout.  One JSON line per measurement; the GPU name and power limit are read in the same run.

Options: --steps K (timed steps per way, default 20), --p P (drop probability, default 0.2), --scale S (graph size)."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from check_halo import gpu_info  # noqa: E402
from re_gnn_b200 import Graph, functional as RF, partition, synth  # noqa: E402

ALPHA, SLOPE = 100.0, 0.2


def inputs(n, r, heads, dim, dev, seed=11):
    gen = torch.Generator(device=dev).manual_seed(seed)
    f = torch.randn(n, heads, dim, device=dev, generator=gen)
    f2 = torch.randn(n, heads, dim, device=dev, generator=gen)
    gout = torch.randn(n, heads, dim, device=dev, generator=gen)
    al = torch.randn(1, heads, dim, device=dev, generator=gen) * 0.3
    ar = torch.randn(1, heads, dim, device=dev, generator=gen) * 0.3
    th = (torch.rand(r, heads, device=dev, generator=gen) + 0.5) / 100
    return f, f2, gout, al, ar, th


def core_step(kind, g, etv, x, e, p, mode, step):
    f, f2, gout, al, ar, th = x
    heads = f.shape[1]
    kw = {}
    if mode == 'explicit':
        kw['keep'] = (torch.rand(e, heads, device=f.device) >= p).float().mul_(1.0 / (1.0 - p))
    elif mode == 'hashed':
        kw['dropout'] = RF.HashedDropout(p, RF.attn_dropout_key(0, step, 0))
    if kind == 'regat':
        leaves = [t.requires_grad_(True) for t in (f, al, ar, th)]
        out, _ = RF.gat_layer(g, etv, *leaves, ALPHA, SLOPE, **kw)
    else:
        leaves = [t.requires_grad_(True) for t in (f, f2, al, th)]
        out, _ = RF.gatv2_aggregate(g, etv, *leaves, ALPHA, SLOPE, **kw)
    out.backward(gout)
    for t in leaves:
        t.grad = None


def time_modes(fns, steps, warmup=3):
    """{name: ms per step}: every function warmed up, then the ways alternated step by step, each with its own pair of
    events around its step (the steps of one way are summed)."""
    for fn in fns.values():
        for i in range(warmup):
            fn(i)
    total = {k: 0.0 for k in fns}
    for i in range(steps):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(warmup + i)
            b.record()
            torch.cuda.synchronize()
            total[k] += a.elapsed_time(b)
    return {k: v / steps for k, v in total.items()}


def cores(args, dev, info):
    d = synth.hetero_graph('mag', scale=args.scale)
    n, r, e = d['num_nodes'], d['num_relations'], int(d['src'].size)
    g = Graph(d['src'], d['dst'], n).to(dev)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(dev), r)
    for heads, dim in ((8, 16), (2, 64)):
        x = inputs(n, r, heads, dim, dev)
        for kind in ('regat', 'regatv2'):
            fns = {m: (lambda i, m=m: core_step(kind, g, etv, x, e, args.p, m, i)) for m in ('none', 'explicit', 'hashed')}
            ms = time_modes(fns, args.steps)
            print(json.dumps({'mode': 'single_device_core', 'core': kind, 'graph': 'mag', 'num_nodes': n, 'num_edges': e,
                              'heads': heads, 'head_dim': dim, 'p': args.p, 'steps': args.steps,
                              'fwd_bwd_ms_none': ms['none'], 'fwd_bwd_ms_explicit_mask': ms['explicit'],
                              'fwd_bwd_ms_hashed': ms['hashed'], 'explicit_mask_bytes': e * heads * 4, **info}),
                  flush=True)
        del x
        torch.cuda.empty_cache()
    del g, etv
    torch.cuda.empty_cache()


def halo(args, dev, info, parts=4, heads=8, dim=16):
    d = synth.hetero_graph_local('mag', parts, 0.9, seed=3, scale=args.scale)
    n, r = d['num_nodes'], d['num_relations']
    g = Graph(d['src'], d['dst'], n).to(dev)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(dev), r)
    bounds = d['community_bounds']
    plist = partition.HaloPartition.virtual_ranks(g, etv, bounds, attention=True)
    f, f2, gout, al, ar, th = inputs(n, r, heads, dim, dev)
    g2 = gout.view(n, heads * dim)
    chunks = (heads * dim + 127) // 128
    for kind in ('regat', 'regatv2'):
        # statistics of every own row once (what the exchange would bring), then each rank's compute timed alone
        stats = []
        for i, p in enumerate(plist):
            own = slice(bounds[i], bounds[i + 1])
            if kind == 'regat':
                o, _, er, mx, sm = partition._gat_forward(p, f[p.rows_in], al, ar, th, ALPHA, SLOPE)
            else:
                sl = partition._slot_buffers(p, heads, chunks, f, None)
                (o, mx, sm), er = partition._gatv2_forward(p, f[p.rows_in], f2[own].contiguous(), al, th, ALPHA, SLOPE,
                                                           sl), None
            stats.append(partition._gat_stats(o, gout[own].contiguous(), er, mx, sm))
        stats = torch.cat(stats)
        res = {'none': [], 'hashed': []}
        for i, p in enumerate(plist):
            own = slice(bounds[i], bounds[i + 1])
            f_ext, f_own, fd_own = f[p.rows_in], f[own].contiguous(), f2[own].contiguous()
            g_own, g_ext, s_ext = gout[own].contiguous(), g2[p.rows_out], stats[p.rows_out]
            buf = torch.zeros((p.e_in + p.tail_ptr[-1], heads), device=dev)
            slots = partition._slot_buffers(p, heads, chunks, f, None)

            def step(step_i, drop):
                dr = RF.HashedDropout(args.p, RF.attn_dropout_key(0, step_i, 0)) if drop else None
                if kind == 'regat':
                    o, el, er, mx, sm = partition._gat_forward(p, f_ext, al, ar, th, ALPHA, SLOPE, dr)
                    partition._gat_stats(o, g_own, er, mx, sm)
                    df, de = partition._gat_backward_edges(p, f_own, el, al, th, ALPHA, SLOPE, g_ext, s_ext, buf, dr)
                    partition._gat_backward_reduce(p, f_own, df, de, ar, th, ALPHA, buf)
                else:
                    o, mx, sm = partition._gatv2_forward(p, f_ext, fd_own, al, th, ALPHA, SLOPE, slots, dr)
                    partition._gat_stats(o, g_own, None, mx, sm)
                    partition._gatv2_backward_edges(p, f_own, al, SLOPE, g_ext, s_ext, slots, buf, dr)
                    partition._gatv2_backward_dst(p, fd_own, al, th, ALPHA, SLOPE, buf, slots[1])
            ms = time_modes({'none': lambda s: step(s, False), 'hashed': lambda s: step(s, True)}, args.steps)
            for k in res:
                res[k].append(ms[k])
        print(json.dumps({'mode': 'halo_virtual_ranks', 'core': kind, 'graph': 'mag_local', 'locality': 0.9,
                          'parts': parts, 'num_nodes': n, 'num_edges': int(d['src'].size), 'heads': heads,
                          'head_dim': dim, 'p': args.p, 'steps': args.steps,
                          'rank_compute_ms_max_none': max(res['none']), 'rank_compute_ms_max_hashed': max(res['hashed']),
                          'rank_compute_ms_mean_none': sum(res['none']) / parts,
                          'rank_compute_ms_mean_hashed': sum(res['hashed']) / parts, **info}), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--p', type=float, default=0.2)
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--skip-halo', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('check_attn_dropout.py measures on the GPU; no CUDA device found')
    dev = torch.device('cuda:0')
    info = gpu_info(dev)
    cores(args, dev, info)
    if not args.skip_halo:
        halo(args, dev, info)


if __name__ == '__main__':
    main()
