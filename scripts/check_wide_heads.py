"""Cost of wide attention heads (D = 256, 512) against narrow twins of equal H*D on the MAG-shaped graph
(synth.hetero_graph('mag'), 1.94 M nodes, 23 M edges).

For each core (functional.gat_layer, functional.gatv2_aggregate) and each group of twins
  H*D = 512:  (4, 128)  (2, 256)  (1, 512)
  H*D = 1024: (8, 128)  (4, 256)  (2, 512)
forward + backward is timed with CUDA events after a warm-up, the configurations of a group alternated step by step.
A second pass over a few steps under ``_lib.Trace`` gives the time of every ABI call per step.  One JSON line per
(core, H, D); the GPU name and power limit are read in the same run.

Options: --steps K (timed steps per configuration, default 20), --scale S (graph size), --out PATH (JSONL, also
printed)."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from check_attn_dropout import core_step, inputs, time_modes  # noqa: E402
from check_halo import gpu_info  # noqa: E402
from re_gnn_b200 import Graph, _lib, synth  # noqa: E402

TWINS = (((4, 128), (2, 256), (1, 512)), ((8, 128), (4, 256), (2, 512)))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--trace-steps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('check_wide_heads.py measures on the GPU; no CUDA device found')
    dev = torch.device('cuda:0')
    info = gpu_info(dev)
    d = synth.hetero_graph('mag', scale=args.scale)
    n, r, e = d['num_nodes'], d['num_relations'], int(d['src'].size)
    g = Graph(d['src'], d['dst'], n).to(dev)
    etv = g.etype_views(torch.as_tensor(d['etype']).to(dev), r)
    out = open(args.out, 'w') if args.out else None
    for kind in ('regat', 'regatv2'):
        for group in TWINS:
            xs = {hd: inputs(n, r, hd[0], hd[1], dev) for hd in group}
            fns = {hd: (lambda i, x=xs[hd]: core_step(kind, g, etv, x, e, 0.0, 'none', i)) for hd in group}
            ms = time_modes(fns, args.steps)
            for hd in group:
                with _lib.Trace() as tr:
                    for i in range(args.trace_steps):
                        fns[hd](i)
                per_call = {k: round(v, 4) for k, v in tr.summary(args.trace_steps).items()}
                rec = {'core': kind, 'graph': 'mag', 'num_nodes': n, 'num_edges': e, 'heads': hd[0], 'head_dim': hd[1],
                       'hd': hd[0] * hd[1], 'steps': args.steps, 'fwd_bwd_ms': round(ms[hd], 4),
                       'trace_ms_per_step': per_call, **info}
                line = json.dumps(rec)
                print(line, flush=True)
                if out:
                    out.write(line + '\n')
                    out.flush()
            del xs, fns
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == '__main__':
    main()
