"""REGATv2 on destination-row blocks with a halo exchange (partition.HaloPartition(..., attention=True) / halo_gatv2) on
the community-structured MAG-shaped graph (synth.hetero_graph_local, H x D = 8 x 16 by default, locality 0, 0.9, 0.99):
halo sizes, cut edges, exchanged bytes, parity and time.  One JSON line per configuration.

  python scripts/check_halo_gatv2.py                      one GPU: P = 2, 4, 8 virtual ranks one after another, halos
                                                          filled by indexing, the slot records and dl tails moved by
                                                          regnn_halo_push_slots / regnn_halo_scatter over local
                                                          buffers; out / d_fs / d_fd are checked bit for bit against
                                                          functional.gatv2_aggregate, and each rank's kernel time on its
                                                          local views with the halos pre-filled (its compute share of a
                                                          step) is timed.  Exchange time cannot be measured on one GPU.
  torchrun --nproc_per_node N scripts/check_halo_gatv2.py N ranks: parity of halo_gatv2 with both exchange variants on
                                                          every rank against a single-device run on its own GPU, then
                                                          the two variants timed, alternated.

Options: --heads H, --head-dim D, --scale S (graph size, default 1.0), --steps K (timed steps, default 20),
--localities 0,0.9,0.99."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))
from check_halo import gpu_info, timed  # noqa: E402
from check_halo_gat import rel  # noqa: E402
from re_gnn_b200 import Graph, functional as RF, partition, synth  # noqa: E402

ALPHA = 100.0
SLOPE = 0.2


def build(locality, parts, args, dev):
    d = synth.hetero_graph_local('mag', parts, locality, seed=3, scale=args.scale)
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(dev)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(dev), d['num_relations'])
    gen = torch.Generator(device=dev).manual_seed(11)
    n, h, dim = d['num_nodes'], args.heads, args.head_dim
    fs = torch.randn(n, h, dim, device=dev, generator=gen)
    fd = torch.randn(n, h, dim, device=dev, generator=gen)
    gout = torch.randn(n, h, dim, device=dev, generator=gen)
    attn = torch.randn(1, h, dim, device=dev, generator=gen) * 0.3
    th = (torch.rand(d['num_relations'], h, device=dev, generator=gen) + 0.5) / 100
    return d, g, etv, (fs, fd, gout, attn, th)


def single_device(g, etv, fs, fd, gout, attn, th):
    leaves = [t.clone().requires_grad_(True) for t in (fs, fd, attn, th)]
    out, _ = RF.gatv2_aggregate(g, etv, *leaves, ALPHA, SLOPE)
    out.backward(gout)
    return (out.detach(),) + tuple(t.grad for t in leaves)


def byte_stats(parts, hd, heads):
    """Bytes a rank receives per step: the source-feature in-halo, the dL/dY and statistics out-halo, the stored logits
    and sign masks of its cut out-edges (slot records, H floats + ceil(H*D/128) 16-byte words each) and the dl of its
    in-view slots whose source is remote."""
    record = heads * 4 + (hd + 127) // 128 * 16
    rows = {'features': [p.n_in * hd * 4 for p in parts], 'grad_out': [p.n_out * hd * 4 for p in parts],
            'stats': [p.n_out * 4 * heads * 4 for p in parts], 'slot_records': [p.tail_ptr[-1] * record for p in parts],
            'dl': [sum(p.dpre_recv_counts) * heads * 4 for p in parts]}
    total = [sum(v) for v in zip(*rows.values())]
    line = {'bytes_%s_max' % k: max(v) for k, v in rows.items()}
    line.update({'bytes_%s_mean' % k: sum(v) / len(v) for k, v in rows.items()})
    line.update({'halo_bytes_per_rank_max': max(total), 'halo_bytes_per_rank_mean': sum(total) / len(total)})
    return line


def virtual(args, dev):
    info = gpu_info(dev)
    hd = args.heads * args.head_dim
    chunks = (hd + 127) // 128
    for loc in args.localities:
        for parts in (2, 4, 8):
            d, g, etv, (fs, fd, gout, attn, th) = build(loc, parts, args, dev)
            n = d['num_nodes']
            bounds = d['community_bounds']
            ref = single_device(g, etv, fs, fd, gout, attn, th)
            plist = partition.HaloPartition.virtual_ranks(g, etv, bounds, attention=True)
            out, d_fs, d_fd, d_attn, d_th = partition._virtual_halo_gatv2(plist, fs, fd, gout, attn, th, ALPHA, SLOPE,
                                                                          push=True)
            exact = [all(bool(torch.equal(a[bounds[p]:bounds[p + 1]], b[bounds[p]:bounds[p + 1]]))
                         for a, b in ((out, ref[0]), (d_fs, ref[1]), (d_fd, ref[2]))) for p in range(parts)]
            # per-rank compute with the halos and the slot tails pre-filled: forward, statistics, edge pass, dst pass
            stats, slots = [], []
            for i, p in enumerate(plist):
                sl = partition._slot_buffers(p, args.heads, chunks, fs, None)
                o, mx, sm = partition._gatv2_forward(p, fs[p.rows_in], fd[bounds[i]:bounds[i + 1]].contiguous(), attn,
                                                     th, ALPHA, SLOPE, sl)
                stats.append(partition._gat_stats(o, gout[bounds[i]:bounds[i + 1]].contiguous(), None, mx, sm))
                slots.append(sl)
            stats = torch.cat(stats)
            g2 = gout.view(n, hd)
            ms = []
            for i, p in enumerate(plist):
                fs_ext, fs_own = fs[p.rows_in], fs[bounds[i]:bounds[i + 1]].contiguous()
                fd_own = fd[bounds[i]:bounds[i + 1]].contiguous()
                g_own = gout[bounds[i]:bounds[i + 1]].contiguous()
                g_ext, s_ext = g2[p.rows_out], stats[p.rows_out]
                sl = slots[i]
                dl = torch.zeros((p.e_in + p.tail_ptr[-1], args.heads), device=dev)

                def step():
                    # the forward rewrites only the head of the slot buffers: the tails stay as filled above
                    o, mx, sm = partition._gatv2_forward(p, fs_ext, fd_own, attn, th, ALPHA, SLOPE, sl)
                    partition._gat_stats(o, g_own, None, mx, sm)
                    partition._gatv2_backward_edges(p, fs_own, attn, SLOPE, g_ext, s_ext, sl, dl)
                    partition._gatv2_backward_dst(p, fd_own, attn, th, ALPHA, SLOPE, dl, sl[1])
                ms.append(timed(step, args.steps))

            def one_gpu():
                single_device(g, etv, fs, fd, gout, attn, th)
            ms_full = timed(one_gpu, args.steps)
            cut = [p.tail_ptr[-1] for p in plist]
            line = {'mode': 'virtual_ranks', 'graph': 'mag_local', 'num_nodes': n, 'num_edges': int(d['src'].size),
                    'heads': args.heads, 'head_dim': args.head_dim, 'parts': parts, 'locality': loc,
                    'in_halo_rows_max': max(p.n_in for p in plist), 'in_halo_rows_mean': sum(p.n_in for p in plist) / parts,
                    'out_halo_rows_max': max(p.n_out for p in plist),
                    'out_halo_rows_mean': sum(p.n_out for p in plist) / parts,
                    'cut_edges_total': sum(cut), 'cut_out_edges_per_rank_max': max(cut),
                    **byte_stats(plist, hd, args.heads),
                    'parity_bit_exact_every_rank': all(exact),
                    'd_attn_rel': rel(d_attn, ref[3].view(-1)), 'd_theta_rel': rel(d_th, ref[4]),
                    'rank_compute_ms_max': max(ms), 'rank_compute_ms_mean': sum(ms) / len(ms),
                    'one_gpu_gatv2_aggregate_step_ms': ms_full, 'halo_step_ms': 'not measured (one GPU)', **info}
            print(json.dumps(line), flush=True)
            del g, etv, fs, fd, gout, plist, stats, slots
            torch.cuda.empty_cache()


def distributed(args):
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    info = gpu_info(dev)
    hd = args.heads * args.head_dim
    ok_all = True
    for loc in args.localities:
        d, g, etv, (fs, fd, gout, attn, th) = build(loc, world, args, dev)
        n = d['num_nodes']
        ref = single_device(g, etv, fs, fd, gout, attn, th)
        bounds = d['community_bounds']
        rb, re = bounds[rank], bounds[rank + 1]
        part = partition.HaloPartition(g, etv, bounds, rank, attention=True)
        hx = partition.HaloExchange(part, hd, dev, heads=args.heads, gatv2=True)

        def halo_step(exchange):
            leaves = [t.clone().requires_grad_(True) for t in (fs[rb:re], fd[rb:re], attn, th)]
            out = partition.halo_gatv2(part, *leaves, ALPHA, SLOPE, exchange=exchange)
            out.backward(gout[rb:re])
            partition.allreduce_relation_grads(leaves[2:], exchange=exchange)
            return (out,) + tuple(t.grad for t in leaves)
        ok = True
        for exchange in (None, hx, None, hx):     # each variant twice: the exchange buffers are reused
            out, dfs, dfd, dat, dth = halo_step(exchange)
            ok = ok and torch.equal(out.detach(), ref[0][rb:re]) and torch.equal(dfs, ref[1][rb:re]) and \
                torch.equal(dfd, ref[2][rb:re]) and max(rel(dat, ref[3]), rel(dth, ref[4])) < 1e-6
        flag = torch.tensor([int(ok)], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_all = ok_all and bool(flag.item())
        t_a2a, t_peer = [], []
        for _ in range(3):      # alternate the variants
            dist.barrier()
            t_a2a.append(timed(lambda: halo_step(None), args.steps))
            dist.barrier()
            t_peer.append(timed(lambda: halo_step(hx), args.steps))
        times = torch.tensor([min(t_a2a), min(t_peer)], dtype=torch.float64, device=dev)
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        if rank == 0:
            line = {'mode': 'torchrun', 'graph': 'mag_local', 'num_nodes': n, 'num_edges': int(d['src'].size),
                    'heads': args.heads, 'head_dim': args.head_dim, 'parts': world, 'locality': loc,
                    'parity_bit_exact_all_ranks_both_variants': bool(flag.item()),
                    'halo_a2a_step_ms': float(times[0]), 'halo_peer_step_ms': float(times[1]), **info}
            print(json.dumps(line), flush=True)
        del hx, part, g, etv, fs, fd, gout
        torch.cuda.empty_cache()
    dist.barrier()
    dist.destroy_process_group()
    return ok_all


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--heads', type=int, default=8)
    ap.add_argument('--head-dim', type=int, default=16)
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--localities', default='0,0.9,0.99')
    args = ap.parse_args()
    args.localities = [float(v) for v in args.localities.split(',')]
    if not torch.cuda.is_available():
        sys.exit('check_halo_gatv2.py measures on a CUDA device; none is visible')
    if 'RANK' in os.environ:
        sys.exit(0 if distributed(args) else 1)
    virtual(args, torch.device('cuda', 0))


if __name__ == '__main__':
    main()
