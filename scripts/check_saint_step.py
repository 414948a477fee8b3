"""GraphSAINT training step on the MAG-shaped graph (BASELINE config 5: 20 000 random-walk roots x walk length 2, hidden
128, 2 layers, batch norm + residual, Adam -- the bench's configuration) with the subgraph extracted on the device and
its CSR views prebuilt from it, against the previous step (torch relabelling in ``reference_sample``, the model
building the subgraph's ``Graph`` from the edge list), alternated in one process.

Prints one JSON line: ms per step (median over rounds of 20 steps, host clock around a device synchronise), library
launches per step (``_lib.count_launches``: the entry points that report their launches), every CUDA kernel, memset
and copy per step (torch.profiler), host synchronisations per step and the lines that make them
(``torch.cuda.set_sync_debug_mode``) -- both counted on separate, untimed steps -- the candidate slots (in-edges of the
subgraph's rows) and induced edges of the batches, whether the two paths give bit-equal first losses, and the card
name and power limit read in the same run.

    python scripts/check_saint_step.py [--rounds 5] [--steps 20] [--warmup 10]
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
from re_gnn_b200.sampling import SaintRandomWalkSampler  # noqa: E402


def previous_step(model, opt, sampler, labels, train_mask, x_dict, edge_type, node_type, local_idx, batch):
    n_id, edge_index, eid = sampler.reference_sample(0, batch)
    opt.zero_grad(set_to_none=True)
    out = model(x_dict, edge_index, edge_type[eid], node_type[n_id], local_idx[n_id])
    mask = train_mask[n_id]
    loss = F.nll_loss(out[mask], labels[n_id][mask])
    loss.backward()
    opt.step()
    return loss.detach()


def new_step(model, opt, sampler, labels, train_mask, x_dict, edge_type, node_type, local_idx, batch):
    return mag.saint_train_step(model, opt, sampler, labels, train_mask, x_dict, edge_type, node_type, local_idx, 0,
                                batch)[0]


def count_syncs(fn):
    """-> {package / optimizer line: host synchronisations} of fn, from torch's sync debug mode."""
    where = {}

    def record(message, category, filename, lineno, file=None, line=None):
        if 'called a synchronizing CUDA operation' in str(message):
            frames = [f for f in traceback.extract_stack()[:-1] if 're_gnn_b200' in f.filename
                      or 'torch/optim' in f.filename or 'check_saint_step' in f.filename]
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
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('check_saint_step.py measures on a CUDA device; none is available')
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
    train_mask = (node_type == 0) & (local_idx < int(sizes[0] * 0.855))
    who = card()
    torch.manual_seed(123)
    model = mag.SaintREGCN(128, 128, 349, 2, 100.0, 0.5, {k: 128 for k in range(nnt)}, net, use_bn=True, residual=True,
                           gcn=False).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=5e-3)
    sampler = SaintRandomWalkSampler(g, roots=20000, walk_length=2, seed=123)
    paths = {'device_subgraph': new_step, 'previous_step': previous_step}

    def run(fn, i):
        return fn(model, opt, sampler, labels, train_mask, x_dict, edge_type, node_type, local_idx, i)

    # the two paths on the same model state, batch and RNG state must give the same loss, bit for bit
    state = ({k: v.clone() for k, v in model.state_dict().items()}, opt.state_dict())
    losses = {}
    for name, fn in paths.items():
        model.load_state_dict(state[0])
        opt.load_state_dict(state[1])
        torch.manual_seed(5)
        losses[name] = run(fn, 0)
    bit_equal = bool(torch.equal(losses['device_subgraph'], losses['previous_step']))
    # subgraph sizes of the batches the timed rounds use
    indptr = g.csr()['indptr'].to(torch.int64)
    cand, induced, nodes = [], [], []
    for i in range(args.rounds * args.steps):
        n_id, block = sampler.sample_block(0, i)
        cand.append(int((indptr[n_id + 1] - indptr[n_id]).sum()))
        induced.append(block.src.numel())
        nodes.append(block.n_src)
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
    stats = lambda xs: dict(min=min(xs), median=statistics.median(xs), max=max(xs))   # noqa: E731
    line = dict(workload='mag_saint', roots=20000, walk_length=2, hidden=128, layers=2, steps_per_round=args.steps,
                rounds=args.rounds, card=who, losses_bit_equal=bit_equal, subgraph_nodes=stats(nodes),
                candidate_slots=stats(cand), induced_edges=stats(induced), **res)
    print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
