"""Neighbour-sampled training step on the MAG-shaped graph (BASELINE config 5: 512 seeds, fan-out [25, 20], hidden 512)
with device-built blocks against the previous assembly (torch relabelling of the sample, every conv building its
block's CSR from the edge list), alternated in one process, for model='regcn' and 'regat'.

Prints one JSON line per model: ms per step (median over rounds of 20 steps, host clock around a device
synchronise), library launches per step (``_lib.count_launches``: the entry points that report their launches),
every CUDA kernel, memset and copy per step (torch.profiler), host synchronisations per step and the lines that make
them (``torch.cuda.set_sync_debug_mode``) -- both counted on separate, untimed steps -- whether the two paths give
bit-equal losses, and the card name and power limit read in the same run.

    python scripts/check_ns_step.py [--rounds 5] [--steps 20] [--warmup 10]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import traceback
import warnings

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from re_gnn_b200 import Graph, _lib, mag, synth  # noqa: E402
from re_gnn_b200.sampling import NeighborSampler  # noqa: E402


def previous_step(model, opt, sampler, seeds, labels, x_dict, edge_type, node_type, local_idx, batch):
    n_id, blocks = sampler.reference_sample(seeds, 0, batch)    # torch relabelling; each boolean mask syncs
    adjs = [(b.edge_index, b.eid, b.size) for b in blocks]
    opt.zero_grad(set_to_none=True)
    loss = F.nll_loss(model(n_id, x_dict, adjs, edge_type, node_type, local_idx), labels)
    loss.backward()
    opt.step()
    return loss.detach()


def new_step(model, opt, sampler, seeds, labels, x_dict, edge_type, node_type, local_idx, batch):
    return mag.train_step(model, opt, sampler, seeds, labels, x_dict, edge_type, node_type, local_idx, 0, batch)[0]


def count_syncs(fn):
    """-> {package / optimizer line: host synchronisations} of fn, from torch's sync debug mode."""
    where = {}

    def record(message, category, filename, lineno, file=None, line=None):
        if 'called a synchronizing CUDA operation' in str(message):
            frames = [f for f in traceback.extract_stack()[:-1] if 're_gnn_b200' in f.filename
                      or 'torch/optim' in f.filename or 'check_ns_step' in f.filename]
            f = frames[-1] if frames else None
            key = '%s:%d' % (os.path.basename(f.filename), f.lineno) if f else '?'
            where[key] = where.get(key, 0) + 1

    with warnings.catch_warnings():
        warnings.simplefilter('always')
        warnings.showwarning = record
        torch.cuda.set_sync_debug_mode('warn')
        try:
            fn()
        finally:
            torch.cuda.set_sync_debug_mode(0)
    return where


def count_kernels(fn, steps):
    """CUDA kernels, memsets and copies per step, from torch.profiler (every launch, torch's and the library's)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.device_type == torch.autograd.DeviceType.CUDA for e in prof.events()) / steps


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--models', default='regcn,regat')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('check_ns_step.py measures on a CUDA device; none is available')
    dev = 'cuda:0'
    torch.backends.cuda.matmul.allow_tf32 = False
    d = synth.hetero_graph('mag')
    n, net, sizes = d['num_nodes'], d['num_etype'], d['type_sizes']
    nnt = len(sizes)
    g = Graph(d['src'][:-n], d['dst'][:-n], n).to(dev)
    g.csr()
    edge_type = (torch.as_tensor(d['etype'][:-n]) - 1).to(dev)
    node_type = torch.as_tensor(d['ntype']).to(dev)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    local_idx = torch.as_tensor(np.arange(n) - offs[d['ntype']]).to(dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    x_dict = {k: torch.randn(sizes[k], 128, device=dev, generator=gen) for k in range(nnt)}
    labels = torch.randint(0, 349, (n,), device=dev, generator=gen)
    perm = torch.randperm(int(sizes[0] * 0.855), generator=torch.Generator().manual_seed(1000))
    batches = [perm[i * 512:(i + 1) * 512].to(dev) for i in range(64)]
    who = card()
    for kind in args.models.split(','):
        torch.manual_seed(123)
        model = mag.REGNN(128, 512, 349, 1, 2, 100.0, 0.5, {k: 128 for k in range(nnt)}, net, residual=True,
                          no_re=False, self_loop_type=2, model=kind).to(dev)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        sampler = NeighborSampler(g, [25, 20], seed=123)
        paths = {'device_blocks': new_step, 'previous_assembly': previous_step}

        def run(fn, i):
            s = batches[i % 64]
            return fn(model, opt, sampler, s, labels[s], x_dict, edge_type, node_type, local_idx, i)

        # the two paths on the same model state, batch and RNG state must give the same loss, bit for bit
        state = ({k: v.clone() for k, v in model.state_dict().items()}, opt.state_dict())
        losses = {}
        for name, fn in paths.items():
            model.load_state_dict(state[0])
            opt.load_state_dict(state[1])
            torch.manual_seed(5)
            losses[name] = run(fn, 0)
        bit_equal = bool(torch.equal(losses['device_blocks'], losses['previous_assembly']))
        for name, fn in paths.items():
            for i in range(args.warmup):
                run(fn, i)
        torch.cuda.synchronize()
        res = {name: dict(ms=[], launches=0) for name in paths}
        for r in range(args.rounds):
            for name, fn in paths.items():
                l0 = _lib.launch_count
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for i in range(args.steps):
                    run(fn, r * args.steps + i)
                torch.cuda.synchronize()
                res[name]['ms'].append((time.perf_counter() - t0) * 1e3 / args.steps)
                res[name]['launches'] = (_lib.launch_count - l0) / args.steps
        for name, fn in paths.items():
            where = count_syncs(lambda: [run(fn, 900 + i) for i in range(5)])
            res[name]['syncs_per_step'] = sum(where.values()) / 5
            res[name]['syncs_per_step_at'] = {k: v / 5 for k, v in sorted(where.items())}
            res[name]['device_ops_per_step'] = count_kernels(lambda: [run(fn, 950 + i) for i in range(5)], 5)
            ms = res[name].pop('ms')
            res[name].update(ms_per_step=statistics.median(ms), ms_rounds=[round(x, 3) for x in ms])
        line = dict(model=kind, seeds=512, fanouts=[25, 20], hidden=512, steps_per_round=args.steps,
                    rounds=args.rounds, card=who, losses_bit_equal=bit_equal, **res)
        print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
