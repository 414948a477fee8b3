"""Halo-exchange row partitioning (partition.HaloPartition / halo_propagate) on the community-structured MAG-shaped graph
(synth.hetero_graph_local, F = 128, locality 0, 0.9, 0.99): halo sizes, exchanged bytes, parity and time.  One JSON line
per configuration.

  python scripts/check_halo.py                      one GPU: P = 2, 4, 8 virtual ranks one after another, halos filled
                                                    with index_select; every rank's Y / dX rows are checked bit for bit
                                                    against the single-device run, and each rank's kernel time on its
                                                    local views (forward + backward: its compute share of a step) is
                                                    timed.  Exchange time cannot be measured on one GPU.
  torchrun --nproc_per_node N scripts/check_halo.py N ranks: parity of halo_propagate (peer-memory variant) on every rank
                                                    against a single-device run on its own GPU, then the halo step and
                                                    feature_sliced_propagate with a SlabExchange, alternated.

Options: --scale S (graph size, default 1.0), --steps K (timed steps, default 20), --localities 0,0.9,0.99."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from re_gnn_b200 import Graph, functional as RF, partition, synth  # noqa: E402

FEAT = 128
ALPHA = 100.0


def gpu_info(dev):
    """Card name and power limit, read in the same run (NVML, else a read-only nvidia-smi query)."""
    info = {'gpu': torch.cuda.get_device_name(dev), 'power_limit_w': None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev.index or 0)
        info['power_limit_w'] = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
        return info
    except Exception as e:
        why = 'NVML: %s' % e
    try:
        import subprocess
        r = subprocess.run(['nvidia-smi', '-i', str(dev.index or 0), '--query-gpu=power.limit',
                            '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=30)
        info['power_limit_w'] = float(r.stdout.strip().splitlines()[0])
    except Exception as e:
        info['power_limit_missing'] = '%s; nvidia-smi: %s' % (why, e)
    return info


def halo_stats(parts, feat):
    n_in = [p.n_in for p in parts]
    n_out = [p.n_out for p in parts]
    halo_bytes = [(a + b) * feat * 4 for a, b in zip(n_in, n_out)]     # received per step: X halo + dL/dY halo
    return {'in_halo_rows_max': max(n_in), 'in_halo_rows_mean': sum(n_in) / len(n_in),
            'out_halo_rows_max': max(n_out), 'out_halo_rows_mean': sum(n_out) / len(n_out),
            'halo_bytes_per_rank_max': max(halo_bytes), 'halo_bytes_per_rank_mean': sum(halo_bytes) / len(halo_bytes)}


def exchange_bytes_other_schemes(n, parts, feat):
    """Bytes a rank receives per step in the column-slab scheme (four row <-> slab re-partitions, each (P-1)/P of a
    row block) and in the row-block scheme with all-gathers (two, each the N - N/P remote rows)."""
    per = (n + parts - 1) // parts
    return {'slab_bytes_per_rank': 4 * per * feat * 4 * (parts - 1) // parts,
            'allgather_bytes_per_rank': 2 * (n - per) * feat * 4}


def timed(fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def single_device(g, etv, x, gout, theta):
    xs, th = x.clone().requires_grad_(True), theta.clone().requires_grad_(True)
    out = RF.propagate(g, etv, xs, th, ALPHA, RF.weighted_degree_norm(g, etv, th, ALPHA, -0.5))
    out.backward(gout)
    return out.detach(), xs.grad, th.grad


def build(locality, parts, scale, dev):
    d = synth.hetero_graph_local('mag', parts, locality, seed=3, scale=scale)
    g = Graph(d['src'], d['dst'], d['num_nodes']).to(dev)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(dev), d['num_relations'])
    gen = torch.Generator(device=dev).manual_seed(11)
    x = torch.randn(d['num_nodes'], FEAT, device=dev, generator=gen)
    gout = torch.randn(d['num_nodes'], FEAT, device=dev, generator=gen)
    theta = (torch.rand(d['num_relations'], 1, device=dev, generator=gen) + 0.5) / 100
    return d, g, etv, x, gout, theta


def virtual(args, dev):
    info = gpu_info(dev)
    for loc in args.localities:
        for parts in (2, 4, 8):
            d, g, etv, x, gout, theta = build(loc, parts, args.scale, dev)
            n = d['num_nodes']
            bounds = d['community_bounds']
            ref = single_device(g, etv, x, gout, theta)
            full = partition.HaloPartition.virtual_ranks(g, etv, [0, n])[0]
            plist = partition.HaloPartition.virtual_ranks(g, etv, bounds)
            exact, ms, dth = True, [], torch.zeros_like(theta)

            def step(part, x_ext, x_own, g_ext):
                y, deg, norm = partition._halo_forward(part, x_ext, theta, ALPHA, True)
                return y, partition._halo_backward(part, x_own, y, g_ext, theta, ALPHA, True, deg, norm)
            for p, part in enumerate(plist):
                rb, re = bounds[p], bounds[p + 1]
                x_ext, x_own, g_ext = x[part.rows_in], x[rb:re].contiguous(), gout[part.rows_out]
                y, (dx, dt) = step(part, x_ext, x_own, g_ext)
                exact = exact and torch.equal(y, ref[0][rb:re]) and torch.equal(dx, ref[1][rb:re])
                dth += dt
                ms.append(timed(lambda: step(part, x_ext, x_own, g_ext), args.steps))
            ms_full = timed(lambda: step(full, x, x, gout), args.steps)
            line = {'mode': 'virtual_ranks', 'graph': 'mag_local', 'num_nodes': n, 'num_edges': int(d['src'].size),
                    'feat': FEAT, 'parts': parts, 'locality': loc, **halo_stats(plist, FEAT),
                    **exchange_bytes_other_schemes(n, parts, FEAT),
                    'parity_bit_exact': bool(exact), 'd_theta_rel': float((dth - ref[2]).abs().max() / ref[2].abs().max()),
                    'rank_compute_ms_max': max(ms), 'rank_compute_ms_mean': sum(ms) / len(ms),
                    'one_gpu_step_ms': ms_full, 'halo_step_ms': 'not measured (one GPU)',
                    'slab_step_ms': 'not measured (one GPU)', **info}
            print(json.dumps(line), flush=True)
            del g, etv, x, gout, plist, full
            torch.cuda.empty_cache()


def distributed(args):
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    info = gpu_info(dev)
    ok_all = True
    for loc in args.localities:
        d, g, etv, x, gout, theta = build(loc, world, args.scale, dev)
        n = d['num_nodes']
        ref = single_device(g, etv, x, gout, theta)
        bounds = d['community_bounds']
        rb, re = bounds[rank], bounds[rank + 1]
        part = partition.HaloPartition(g, etv, bounds, rank)
        hx = partition.HaloExchange(part, FEAT, dev)
        sb = partition.row_blocks(g.csr()['indptr'], world, balance='rows')
        sx = partition.SlabExchange(FEAT, sb, rank, dev)

        def halo_step():
            xo, th = x[rb:re].clone().requires_grad_(True), theta.clone().requires_grad_(True)
            out = partition.halo_propagate(part, xo, th, ALPHA, exchange=hx)
            out.backward(gout[rb:re])
            partition.allreduce_relation_grads([th], exchange=hx)
            return out, xo.grad, th.grad

        def slab_step():
            xo, th = x[sb[rank]:sb[rank + 1]].clone().requires_grad_(True), theta.clone().requires_grad_(True)
            out = partition.feature_sliced_propagate(g, etv, xo, th, ALPHA, RF.weighted_degree_norm(g, etv, th, ALPHA, -0.5),
                                                     sb, rank, exchange=sx)
            out.backward(gout[sb[rank]:sb[rank + 1]])
            partition.allreduce_relation_grads([th], exchange=sx)
        out, dx, dth = halo_step()
        ok = torch.equal(out.detach(), ref[0][rb:re]) and torch.equal(dx, ref[1][rb:re]) and \
            float((dth - ref[2]).abs().max() / ref[2].abs().max()) < 1e-6
        flag = torch.tensor([int(ok)], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_all = ok_all and bool(flag.item())
        t_halo, t_slab = [], []
        for _ in range(3):      # alternate the two schemes
            dist.barrier()
            t_halo.append(timed(halo_step, args.steps))
            dist.barrier()
            t_slab.append(timed(slab_step, args.steps))
        stats = torch.tensor([part.n_in, part.n_out], dtype=torch.float64, device=dev)
        gathered = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(gathered, stats)
        times = torch.tensor([min(t_halo), min(t_slab)], dtype=torch.float64, device=dev)
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        if rank == 0:
            n_in = [int(s[0]) for s in gathered]
            n_out = [int(s[1]) for s in gathered]
            hb = [(a + b) * FEAT * 4 for a, b in zip(n_in, n_out)]
            line = {'mode': 'torchrun', 'graph': 'mag_local', 'num_nodes': n, 'num_edges': int(d['src'].size),
                    'feat': FEAT, 'parts': world, 'locality': loc,
                    'in_halo_rows_max': max(n_in), 'in_halo_rows_mean': sum(n_in) / world,
                    'out_halo_rows_max': max(n_out), 'out_halo_rows_mean': sum(n_out) / world,
                    'halo_bytes_per_rank_max': max(hb), 'halo_bytes_per_rank_mean': sum(hb) / world,
                    **exchange_bytes_other_schemes(n, world, FEAT), 'parity_bit_exact_all_ranks': bool(flag.item()),
                    'halo_step_ms': float(times[0]), 'slab_step_ms': float(times[1]), **info}
            print(json.dumps(line), flush=True)
        del hx, sx, part, g, etv, x, gout
        torch.cuda.empty_cache()
    dist.barrier()
    dist.destroy_process_group()
    return ok_all


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--localities', default='0,0.9,0.99')
    args = ap.parse_args()
    args.localities = [float(v) for v in args.localities.split(',')]
    if not torch.cuda.is_available():
        sys.exit('check_halo.py measures on a CUDA device; none is visible')
    if 'RANK' in os.environ:
        sys.exit(0 if distributed(args) else 1)
    virtual(args, torch.device('cuda', 0))


if __name__ == '__main__':
    main()
