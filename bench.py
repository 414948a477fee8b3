#!/usr/bin/env python
"""bench.py -- headline benchmark of the RE-GNN hot path on B200.

Metric (BASELINE.json): GTEPS forward+backward per RE-layer (+ % of the HBM roofline).  A "step" is
one forward + backward of one RE-layer (REGraphConv aggregation core: relation-weighted degree norm
+ fused norm*SpMM*norm, gradients w.r.t. the features and the relation embedding) over the whole
synthetic ogbn-mag-shaped graph (BASELINE config 4; 1.94 M nodes, 23.05 M edges incl. self loops,
F = 128 fp32).  With --gpus N the same step is sharded over N ranks (strong scaling): feature-sliced aggregation with
the row<->slab exchange inside our kernels over NVLink peer memory by default (--partition, DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload mag_regcn]
                    [--dump-outputs DIR]

One JSON line on stdout from rank 0.  `--impl reference` times the CPU restatement of the reference
(oracle/regnn_oracle.py; DGL itself cannot be installed) on the box's host cores.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALPHA = 100.0
FEAT = 128


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='mag_regcn', choices=['mag_regcn', 'mag_ns', 'mag_saint'])
    ap.add_argument('--feat', type=int, default=FEAT)
    ap.add_argument('--scale', type=float, default=1.0, help='shrink the graph (debug only; reported in config)')
    ap.add_argument('--partition', default='auto', choices=['auto', 'peer', 'cols', 'rows', 'edges'],
                    help='multi-GPU scheme: peer = feature-sliced aggregation, re-partition over peer memory inside our '
                         'kernels; cols = the same between NCCL all-to-alls; rows / edges = destination-row blocks '
                         '(equal rows / equal in-edge counts) fed by all-gathers; auto = peer, else cols (>= 4 ranks) / rows')
    ap.add_argument('--no-others', action='store_true', help='skip the secondary HGB-shaped workloads')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='multi-GPU: run the step eagerly instead of replaying a CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed to DIR/<name>.npy (float32): y and d_x '
                         '(the output and the feature gradient, on a fixed seeded sample of rows) and d_theta (the '
                         'relation-embedding gradient, whole); single GPU, --workload mag_regcn, --impl ours')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and (args.impl != 'ours' or args.workload != 'mag_regcn'):
        ap.error('--dump-outputs covers the default workload only (--workload mag_regcn --impl ours)')
    return args


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # NVML missing: report nulls rather than fail the bench
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
            getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap',
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def dump_outputs(path, y, dx, d_theta):
    """Writes one step's results for output-for-output comparison of two builds: ``y`` and ``d_x`` on the same seeded
    sample of rows (at most 16 MB each), ``d_theta`` whole, all float32."""
    n, f = y.shape
    rows = np.sort(np.random.RandomState(0).choice(n, min(n, (16 << 20) // (4 * f)), replace=False))
    idx = torch.as_tensor(rows, device=y.device)
    os.makedirs(path, exist_ok=True)
    for name, t in (('y', y[idx]), ('d_x', dx[idx]), ('d_theta', d_theta)):
        np.save(os.path.join(path, name + '.npy'), t.detach().float().cpu().numpy())


def theta_init(r, w, seed=0):
    rng = np.random.RandomState(seed)
    return torch.as_tensor(rng.uniform(0.5, 1.5, size=(r, w)) / ALPHA, dtype=torch.float32)


def algorithmic_bytes_spmm(n, e, f):
    """SURVEY.md 8(d) gather model, forward SpMM: per edge source row + col idx + etype + norm[src];
    per row output row + indptr + norm[dst]."""
    return e * (4 * f + 4 + 1 + 4) + n * (4 * f + 4 + 4)


def compulsory_bytes_spmm(n, e, f):
    """SURVEY.md 8(d) companion figure: every source row read once, every output row written once, the edge
    structure streamed once -- a lower bound on DRAM traffic that no kernel can beat (fraction <= 1 always)."""
    return 2 * 4 * n * f + 5 * e + 12 * n


# ------------------------------------------------------------------------------------------------------
def cpu_reference_sample(d, feat, steps, warmup, max_edges=1_500_000):
    """Times the CPU restatement of the reference layer (oracle) forward+backward on a bounded sample:
    the destination-row block [0, k) of the same graph holding ~max_edges in-edges."""
    from oracle import regnn_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dst = d['dst']
    order = np.argsort(dst, kind='stable')
    k_edges = min(max_edges, dst.size)
    sel = np.sort(order[:k_edges])
    src, dsts, et = (torch.as_tensor(d[k][sel]) for k in ('src', 'dst', 'etype'))
    n = d['num_nodes']
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n, feat, generator=g).requires_grad_(True)
    th = theta_init(d['num_relations'], 1).requires_grad_(True)
    gout = torch.randn(n, feat, generator=g)
    times = []
    for i in range(warmup + steps):
        x.grad = th.grad = None
        t0 = time.perf_counter()
        out = O.regraphconv_forward(src, dsts, et, n, x, th, ALPHA)
        out.backward(gout)
        times.append(time.perf_counter() - t0)
    t = float(np.median(times[warmup:]))
    return {'value': k_edges / t / 1e9, 'unit': 'GTEPS', 'cores': cores, 'kind': 'port',
            'sample': 'oracle/regnn_oracle.py REGraphConv fwd+bwd (PyTorch CPU, fp32) on the destination-row block '
                      'holding the first %d in-edges (%.1f %% of the edges) of the same graph, median of %d runs after %d '
                      'warm-ups, %.3f s per run; GTEPS = sample edges / sample time, i.e. the whole graph is assumed to '
                      'run at the sample\'s per-edge rate (the oracle\'s cost is linear in E: index_select + index_add_)'
                      % (k_edges, 100.0 * k_edges / dst.size, steps, warmup, t)}, t


def run_reference(args, d):
    steps, warmup = max(1, args.steps), max(0, args.warmup)   # the driver's --steps / --warmup, as given
    cb, t = cpu_reference_sample(d, args.feat, steps, warmup)
    line = {
        'impl': 'reference', 'metric': 'GTEPS fwd+bwd per RE-layer', 'value': cb['value'], 'unit': 'GTEPS',
        'n_gpus': args.gpus, 'steps': steps, 'warmup': warmup, 'ms_per_step': t * 1e3, 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, d), 'cpu_baseline': cb,
        'e2e': {'value': cb['value'], 'unit': 'GTEPS', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


PARTITION_HOW = {
    'none': 'single GPU',
    'peer': 'feature-sliced over --gpus (column slabs; rows<->slabs re-partition over NVLink peer memory inside the kernels, '
            'outputs alias the exchange buffers)',
    'cols': 'feature-sliced over --gpus (column slabs between NCCL all-to-alls)',
    'rows': 'dst-row blocks (equal rows) over --gpus, NCCL all-gather of source rows',
    'edges': 'dst-row blocks (equal in-edges) over --gpus, NCCL all-gather of source rows'}


def workload_config(args, d):
    """The workload both arms measure (identical for ``--impl ours`` and ``--impl reference`` at every N: how the repo
    arm shards the step over the GPUs is reported beside it, in the line's ``partition`` key)."""
    return {'workload': 'REGraphConv RE-layer fwd+bwd, full-batch, synthetic ogbn-mag-shaped graph (BASELINE config 4)',
            'num_nodes': int(d['num_nodes']), 'num_edges': int(d['src'].size), 'num_relations': int(d['num_relations']),
            'feat': args.feat, 'graph_scale': args.scale,
            'l2': 'inputs larger than L2 (source matrix %.0f MB vs 126 MB L2); no flush needed'
                  % (d['num_nodes'] * args.feat * 4 / 1e6)}


# ------------------------------------------------------------------------------------------------------
def timed(fn, steps, warmup, sync, barrier=None):
    """W untimed warm-ups, then exactly K steps between CUDA events on the current stream."""
    for _ in range(warmup):
        fn()
    sync()
    if barrier:
        barrier()
    sync()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    sync()
    if barrier:
        barrier()
    return t0.elapsed_time(t1) / 1e3  # seconds for K steps


def others(dev, steps, warmup):
    """Secondary workloads (BASELINE configs 1-3; L2-resident, so each timed iteration is preceded by an
    L2 flush and timed on its own): GTEPS fwd+bwd of one layer call."""
    import torch.nn.functional as F
    import re_gnn_b200
    from re_gnn_b200 import Graph, synth
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    res = {}
    cases = [
        ('dblp_regcn_f64', 'dblp', lambda r: re_gnn_b200.REGraphConv(r, ALPHA, 64, 64, bias=False, weight=False), 64),
        ('acm_regat_h8d64', 'acm', lambda r: re_gnn_b200.REGATConv(r, ALPHA, 512, 64, 8, negative_slope=0.01,
                                                                   use_weight=False), 512),
        ('imdb_remixhop_p012_f64', 'imdb', lambda r: re_gnn_b200.REMixHopConv(r, ALPHA, 64, 64, p=[0, 1, 2]), 64),
        ('imdb_regatv2_h8d64', 'imdb', lambda r: re_gnn_b200.REGATv2Conv(r, ALPHA, 512, 64, 8, negative_slope=0.01,
                                                                         use_weight=False), 512),
    ]
    for name, shape, ctor, fin in cases:
        d = synth.hetero_graph(shape)
        g = Graph(d['src'], d['dst'], d['num_nodes']).to(dev)
        et = torch.as_tensor(d['etype']).to(dev)
        mod = ctor(d['num_relations']).to(dev)
        mod.edge_weight.data.copy_(theta_init(d['num_relations'], mod.edge_weight.shape[1]))
        x = torch.randn(d['num_nodes'], fin, device=dev, requires_grad=True)
        with torch.no_grad():
            gout = torch.randn_like(mod(g, x, et))   # no autograd graph kept alive (its AccumulateGrad node would pin x's
        ts = []                                      # gradient accumulation to this stream and break the capture below)
        for i in range(warmup + steps):
            x.grad = None
            mod.zero_grad(set_to_none=True)
            flush.zero_()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            mod(g, x, et).backward(gout)
            t1.record()
            torch.cuda.synchronize()
            ts.append(t0.elapsed_time(t1) / 1e3)
        t = float(np.median(ts[warmup:]))
        res[name] = {'gteps_fwd_bwd': d['src'].size / t / 1e9, 'ms': t * 1e3, 'num_edges': int(d['src'].size),
                     'l2': 'flushed between iterations', 'l2_resident': True}   # whole working set < 126 MB L2: not an HBM statement
        # the same forward + backward replayed as ONE CUDA graph: these layers are a dozen launches of a few microseconds
        # each, so the eager number above is host time (Python, autograd, allocator), this one is device time
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    x.grad = None
                    mod.zero_grad(set_to_none=True)
                    mod(g, x, et).backward(gout)
            torch.cuda.current_stream().wait_stream(side)
            cg = torch.cuda.CUDAGraph()
            x.grad = None
            mod.zero_grad(set_to_none=True)
            with torch.cuda.graph(cg):
                mod(g, x, et).backward(gout)
            tg = []
            for i in range(warmup + steps):
                flush.zero_()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                cg.replay()
                t1.record()
                torch.cuda.synchronize()
                tg.append(t0.elapsed_time(t1) / 1e3)
            tgm = float(np.median(tg[warmup:]))
            res[name]['ms_cuda_graph'] = tgm * 1e3
            res[name]['gteps_fwd_bwd_cuda_graph'] = d['src'].size / tgm / 1e9
            del cg
        except Exception as exc:   # report, do not hide
            res[name]['ms_cuda_graph'] = None
            res[name]['cuda_graph_error'] = str(exc)[:200]
            torch.cuda.synchronize()
    return res


def attention_at_hbm_scale(dev, d, g, et, steps, warmup):
    """Fused REGAT / REGATv2 on the ogbn-mag-shaped graph, H*D = 128 (gathered matrix 993 MB >> L2): the HBM-bound case
    the north-star's '>= 70 % of HBM roofline for fused REGAT edge-softmax+aggregate' is about.  Per shape: GTEPS of
    the layer's forward+backward through the module API (use_weight=False: no dense projection in front), and a
    ``roofline`` object for the forward kernel launch timed alone, on SURVEY 8(d)'s gather-model bytes."""
    import re_gnn_b200
    from re_gnn_b200 import ops
    hbm, how = peaks()
    n, e, r = d['num_nodes'], d['src'].size, d['num_relations']
    csr = g.csr()
    etv = g.etype_views(et, r)
    res = {}
    traffic = {}
    tp = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tp):
        with open(tp) as fh:
            traffic = json.load(fh)
    gen = torch.Generator(device=dev).manual_seed(99)
    for kind, heads, dim in (('regat', 8, 16), ('regat', 2, 64), ('regatv2', 8, 16), ('regatv2', 2, 64)):
        hd = heads * dim
        cls = re_gnn_b200.REGATConv if kind == 'regat' else re_gnn_b200.REGATv2Conv
        kw = dict(negative_slope=0.01, use_weight=False)
        mod = cls(r, ALPHA, hd, dim, heads, **kw).to(dev)
        mod.edge_weight.data.copy_(theta_init(r, heads))
        x = (torch.randn(n, hd, device=dev, generator=gen) * 0.5).requires_grad_(True)
        gout = torch.randn(n, heads, dim, device=dev, generator=gen)

        def layer():
            x.grad = None
            mod.zero_grad(set_to_none=True)
            mod(g, x, et).backward(gout)
        t = timed(layer, steps, warmup, torch.cuda.synchronize) / steps
        with torch.no_grad():
            f3 = x.detach().view(n, heads, dim)
            th = mod.edge_weight.detach()
            if kind == 'regat':
                el, er = (f3 * mod.attn_l).sum(-1), (f3 * mod.attn_r).sum(-1)
                fwd = lambda: ops.gat_fwd(csr, etv[0], th, ALPHA, f3, el, er, 0.01)
                alg = e * (4 * hd + 4 * heads + 4 + 1) + n * (4 * hd + 4 * heads + 4 + 8 * heads)
                kname = 'regnn::gat_fwd (fused logits + LeakyReLU + online edge-softmax + aggregation)'
            else:
                at = mod.attn.detach().reshape(-1)
                # the training forward: also stores the logits and LeakyReLU' sign masks the backward reads
                fwd = lambda: ops.gatv2_fwd(csr, etv[0], th, ALPHA, f3, f3, at, 0.01, save=True)
                alg = (e * (4 * hd + 4 + 1 + 4 * heads + 16 * ((hd + 127) // 128)) + n * (2 * 4 * hd + 8 * heads + 4)
                       + 4 * hd)
                kname = ('regnn::gatv2_fwd (fused logits + online edge-softmax + aggregation; training variant that '
                         'stores per-slot logits and sign masks)')
            tk = timed(fwd, steps, warmup, torch.cuda.synchronize) / steps
        res['mag_%s_h%dd%d' % (kind, heads, dim)] = {
            'gteps_fwd_bwd': e / t / 1e9, 'ms': t * 1e3, 'fwd_kernel_ms': tk * 1e3, 'gteps_fwd': e / tk / 1e9,
            'num_edges': int(e), 'l2': 'gathered matrix %.0f MB vs 126 MB L2; no flush needed' % (n * hd * 4 / 1e6),
            'roofline': {'bound': 'hbm', 'kernel': kname, 'achieved': alg / tk / 1e9, 'peak': hbm, 'peak_source': how,
                         'unit': 'GB/s', 'frac': alg / tk / 1e9 / hbm,
                         'traffic': traffic.get({'regat': 'gat_fwd_mag_h8d16_bytes', 'regatv2': 'gatv2_fwd_mag_h8d16_bytes'}[kind])
                         if (heads, dim) == (8, 16) else None,
                         'algorithmic_bytes_per_launch': int(alg), 'launch_ms': tk * 1e3, 'l2_resident': False}}
        del mod, x, gout
        torch.cuda.empty_cache()
    return res


def epoch_times(dev, steps, warmup):
    """Epoch time in the reference's own definition (run_regnn.py:144-159): one training step (forward, cross-entropy
    on the training nodes, backward, Adam) plus one no-grad evaluation forward, full batch, for the three callers
    of the hot path on their HGB-shaped graphs with the reference's default hyper-parameters
    (hidden 64, 4 heads x 4 layers for REGAT, 2 layers for REGCN / REMixHop, dropout as in scripts/*.sh)."""
    import torch.nn.functional as F
    from re_gnn_b200 import Graph, model as M, synth
    in_dims = {'dblp': [334, 4231, 50, 20], 'acm': [1902, 1902, 1902, 1902], 'imdb': [3066, 3066, 3066, 3066]}
    classes = {'dblp': 4, 'acm': 3, 'imdb': 5}
    res = {}
    for name, shape, build in [
        ('dblp_regcn_2layer', 'dblp', lambda g, r, dims, c: M.REGCN(g, r, ALPHA, 64, 64, c, 2, F.elu, 0.5, dims)),
        ('acm_regat_4layer_8head', 'acm', lambda g, r, dims, c: M.REGAT(g, r, ALPHA, 4, 64, 64, c, [8] * 4 + [1], F.elu,
                                                                       0.6, 0.6, 0.01, False, dims)),
        ('imdb_remixhop_2layer', 'imdb', lambda g, r, dims, c: M.REMixHop(g, r, ALPHA, 64, 64, c, 2, dims,
                                                                           input_dropout=0.6, activation=F.elu)),
    ]:
        d = synth.hetero_graph(shape)
        g = Graph(d['src'], d['dst'], d['num_nodes']).to(dev)
        et = torch.as_tensor(d['etype']).to(dev)
        net = build(g, d['num_relations'], in_dims[shape], classes[shape]).to(dev)
        feats = [torch.randn(sz, dim, device=dev) for sz, dim in zip(d['type_sizes'], in_dims[shape])]
        labels = torch.randint(0, classes[shape], (d['type_sizes'][0],), device=dev)
        train_idx = torch.arange(0, d['type_sizes'][0], 2, device=dev)
        opt = torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-3, capturable=True)

        def epoch():
            net.train()
            logits, _ = net(feats, et)
            loss = F.cross_entropy(logits[train_idx], labels[train_idx])
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            net.eval()
            with torch.no_grad():
                net(feats, et)

        t = timed(epoch, steps, warmup, torch.cuda.synchronize) / steps
        res[name] = {'epoch_ms': t * 1e3, 'num_edges': int(d['src'].size), 'num_nodes': int(d['num_nodes']),
                     'definition': 'train step + no-grad eval forward (run_regnn.py:144-159); dense projections in true '
                                   'fp32 (TF32 off), as the parity runs'}
        # the same epoch with PyTorch's TF32 tensor-core GEMMs for the dense projections (what a user who does not need
        # 1e-5 parity would run; our kernels are unaffected: they have no GEMM)
        torch.backends.cuda.matmul.allow_tf32 = True
        res[name]['epoch_ms_tf32_projections'] = timed(epoch, steps, warmup, torch.cuda.synchronize) / steps * 1e3
        torch.backends.cuda.matmul.allow_tf32 = False
        # the same epoch captured once into a CUDA graph and replayed: these graphs are launch-bound
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    epoch()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                epoch()
            tg = timed(graph.replay, steps, warmup, torch.cuda.synchronize) / steps
            res[name]['epoch_ms_cuda_graph'] = tg * 1e3
        except Exception as exc:  # report, do not hide
            res[name]['epoch_ms_cuda_graph'] = None
            res[name]['cuda_graph_error'] = str(exc)[:200]
            torch.cuda.synchronize()
    return res


def bind_to_gpu_numa_node(index):
    """Pins this process to the CPUs of the NUMA node its GPU hangs off, BEFORE the pinned host buffers are allocated
    (first touch places them): with N ranks on one host the H2D streams of the e2e arm otherwise cross the socket
    interconnect and contend.  Best effort: returns the node id or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = '/sys/bus/pci/devices/%s/numa_node' % bus.lower()[-12:]
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open('/sys/devices/system/node/node%d/cpulist' % node).read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus += list(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def run_ours(args, d):
    import torch.distributed as dist
    import re_gnn_b200  # noqa: F401  (fails loudly if the CUDA library is missing)
    from re_gnn_b200 import Graph, _lib, functional as RF, ops, partition

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.dump_outputs and world > 1:
        raise SystemExit('bench.py: --dump-outputs runs on one GPU')
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    sync = torch.cuda.synchronize
    barrier = (lambda: dist.barrier()) if world > 1 else None

    n, e, r, f = d['num_nodes'], d['src'].size, d['num_relations'], args.feat
    g = Graph(d['src'], d['dst'], n).to(dev)
    et = torch.as_tensor(d['etype']).to(dev)
    t_build0 = time.perf_counter()
    csr = g.csr()
    etv = g.etype_views(et, r)
    sync()
    build_s = time.perf_counter() - t_build0
    theta = theta_init(r, 1).to(dev).requires_grad_(True)
    gen = torch.Generator(device=dev).manual_seed(1234)
    x_full = torch.randn(n, f, device=dev, generator=gen)
    g_full = torch.randn(n, f, device=dev, generator=gen)

    xch = None
    if world == 1:
        args.partition = 'none'
        x = x_full.clone().requires_grad_(True)
        gout = g_full
        last = {}     # --dump-outputs: the output of the latest step; x.grad and theta.grad hold its gradients

        def step():
            x.grad = theta.grad = None
            nrm = RF.weighted_degree_norm(g, etv, theta, ALPHA, -0.5)
            y = RF.propagate(g, etv, x, theta, ALPHA, nrm)
            y.backward(gout)
            if args.dump_outputs:   # kept only then: otherwise Y is freed before the next step, as a caller would
                last['y'] = y
    else:
        bounds = partition.row_blocks(csr['indptr'], world, balance='edges' if args.partition == 'edges' else 'rows')
        rb, re = bounds[rank], bounds[rank + 1]
        mode = args.partition
        if mode in ('auto', 'peer'):
            xch, why = None, ''
            try:
                if f % (4 * world) or f // world > ops.NARROW_FEAT:
                    raise ValueError('F=%d does not split into 128-bit slabs of <= %d columns over %d ranks'
                                     % (f, ops.NARROW_FEAT, world))
                xch = partition.SlabExchange(f, bounds, rank, dev)
            except Exception as ex:   # no peer mapping on this box / shape: every rank falls back together
                why = '%s: %s' % (type(ex).__name__, ex)
            flag = torch.tensor([int(xch is not None)], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()):
                mode = 'peer'
            else:
                if rank == 0:
                    print('[bench] peer-memory exchange unavailable (%s); using collectives' % why, file=sys.stderr)
                xch, mode = None, ('cols' if world >= 4 and f % world == 0 else 'rows')
        args.partition = mode
        if mode == 'peer':
            def dist_propagate(g_, etv_, x_, th_, al_, nrm_, b_, r_):
                return partition.feature_sliced_propagate(g_, etv_, x_, th_, al_, nrm_, b_, r_, exchange=xch, alias=True)
        elif mode == 'cols':
            dist_propagate = partition.feature_sliced_propagate
        else:
            dist_propagate = partition.partitioned_propagate
        x = x_full[rb:re].clone().requires_grad_(True)
        gout = g_full[rb:re].clone()

        def step():
            x.grad = theta.grad = None
            nrm = RF.weighted_degree_norm(g, etv, theta, ALPHA, -0.5)
            out = dist_propagate(g, etv, x, theta, ALPHA, nrm, bounds, rank)
            out.backward(gout)
            partition.allreduce_relation_grads([theta], exchange=xch if mode == 'peer' else None)
            return out

        # ---- self-check before any timing: this rank's rows of Y and dX against a single-device run of the same step
        # on this GPU (bit-equal: every kernel adds a row's slots in slot order), the relation gradient within 1e-6
        xs = x_full.clone().requires_grad_(True)
        th1 = theta.detach().clone().requires_grad_(True)
        y1 = RF.propagate(g, etv, xs, th1, ALPHA, RF.weighted_degree_norm(g, etv, th1, ALPHA, -0.5))
        y1.backward(g_full)
        y_d = step().detach()
        rel = float(((theta.grad - th1.grad).abs().max() / th1.grad.abs().max()).item())
        flags = torch.tensor([int(torch.equal(y_d, y1.detach()[rb:re])), int(torch.equal(x.grad, xs.grad[rb:re])),
                              int(rel <= 1e-6)], device=dev)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        relt = torch.tensor([rel], device=dev, dtype=torch.float64)
        dist.all_reduce(relt, op=dist.ReduceOp.MAX)
        parity_check = {'y_equal': bool(flags[0].item()), 'dx_equal': bool(flags[1].item()),
                        'd_theta_max_rel_err': float(relt.item()), 'd_theta_ok': bool(flags[2].item()),
                        'against': 'single-device run of the same step on every rank, rows [r_p, r_p+1) of Y and dX '
                                   'compared bit for bit, relation gradient to 1e-6 (all ranks must agree: MIN / MAX)'}
        del x_full, g_full, xs, y1, y_d

    # launches per step, counted on one eager step (a replayed CUDA graph issues the same kernels without going
    # through the Python wrappers that count them)
    l0 = _lib.launch_count
    step()
    launches_per_step = _lib.launch_count - l0
    # ---- multi-GPU: the whole step (4 device-side barriers, ~14 launches of 0.02-0.5 ms) replayed as ONE CUDA graph, so
    # that host launch latency and Python overhead sit outside the measurement's critical path
    timed_step, graphed = step, False
    if world > 1 and args.partition == 'peer' and not args.no_graph:
        ok = 1
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    step()
            torch.cuda.current_stream().wait_stream(side)
            sync()
            cg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(cg):
                step()
            sync()
        except Exception as ex:   # report, do not hide: every rank must take the same path
            ok = 0
            if rank == 0:
                print('[bench] CUDA-graph capture of the multi-GPU step failed (%s: %s); running it eagerly'
                      % (type(ex).__name__, str(ex)[:200]), file=sys.stderr)
        flag = torch.tensor([ok], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()):
            timed_step, graphed = cg.replay, True
    sampler = ClockSampler(local)
    sampler.start()
    total = timed(timed_step, args.steps, args.warmup, sync, barrier)
    launches = launches_per_step * args.steps
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last['y'], x.grad, theta.grad)
    # ---- per-phase device timeline of a few extra (eager) steps: CUDA events around every ABI call, barrier and
    # collective (re_gnn_b200._lib.Trace); max over ranks per phase
    with _lib.Trace() as tr:
        for _ in range(3):
            step()
    phases = tr.summary(3)
    if world > 1:
        keys = sorted(phases)
        pv = torch.tensor([phases[k] for k in keys], device=dev, dtype=torch.float64)
        dist.all_reduce(pv, op=dist.ReduceOp.MAX)
        phases = {k: float(v) for k, v in zip(keys, pv.tolist())}
    phases = {k: round(v, 4) for k, v in phases.items()}
    if world > 1:
        t = torch.tensor([total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())
    ms = total / args.steps * 1e3
    value = e / (total / args.steps) / 1e9

    # ---- end-to-end arm: host buffers, H2D of the step's inputs and D2H of its result inside the timed region
    x_h = torch.randn(x.shape, dtype=torch.float32).pin_memory()
    g_h = torch.randn(gout.shape, dtype=torch.float32).pin_memory()
    res_h = torch.empty(r + 1, dtype=torch.float32).pin_memory()
    # double-buffered on a copy stream: the inputs of step i+1 stream in over PCIe behind the kernels of step i
    copy_stream = torch.cuda.Stream(device=dev)
    x_bufs = [torch.empty_like(x, requires_grad=True) for _ in range(2)]
    g_bufs = [torch.empty_like(gout) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]    # the slot's copies have landed
    freed = [torch.cuda.Event() for _ in range(2)]    # the step that used the slot has finished with it
    state = {'i': 0}

    def prefetch(slot):
        copy_stream.wait_event(freed[slot])           # no-op until the slot has been used once
        with torch.cuda.stream(copy_stream), torch.no_grad():
            x_bufs[slot].copy_(x_h, non_blocking=True)
            g_bufs[slot].copy_(g_h, non_blocking=True)
            ready[slot].record(copy_stream)

    def step_e2e():
        i = state['i']
        slot = i % 2
        if i == 0:
            prefetch(slot)
        prefetch(1 - slot)
        cur = torch.cuda.current_stream()
        cur.wait_event(ready[slot])
        x_e, g_e = x_bufs[slot], g_bufs[slot]
        x_e.grad = theta.grad = None
        nrm = RF.weighted_degree_norm(g, etv, theta, ALPHA, -0.5)
        if world == 1:
            out = RF.propagate(g, etv, x_e, theta, ALPHA, nrm)
        else:
            out = dist_propagate(g, etv, x_e, theta, ALPHA, nrm, bounds, rank)
        out.backward(g_e)
        if world > 1:
            partition.allreduce_relation_grads([theta], exchange=xch if args.partition == 'peer' else None)
        res_h.copy_(torch.cat([theta.grad.view(-1), out.detach().sum().view(1)]), non_blocking=True)
        freed[slot].record(cur)
        state['i'] = i + 1

    e2e_total = timed(step_e2e, max(3, args.steps // 2), 3, sync, barrier)
    if world > 1:
        t = torch.tensor([e2e_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_total = float(t.item())
    e2e_steps = max(3, args.steps // 2)
    e2e = {'value': e / (e2e_total / e2e_steps) / 1e9, 'unit': 'GTEPS',
           'h2d_bytes_per_step': int(x_h.numel() * 4 + g_h.numel() * 4), 'd2h_bytes_per_step': int(res_h.numel() * 4),
           'ms_per_step': e2e_total / e2e_steps * 1e3, 'numa_node_rank0': numa_node,
           'note': 'per rank, every step: pinned-host X and dL/dY rows copied in (double-buffered on a copy stream, so '
                   'step i+1 streams in behind the kernels of step i; K+1 input copies for K timed steps), relation '
                   'gradient + output checksum copied out'}

    # ---- BASELINE config 5 beside the headline, at the same N: neighbour-sampled minibatch training, data-parallel (weak
    # scaling).  Every rank takes part; the numbers ride in the line's `others` so the driver's per-N runs record them.
    ns = None
    if not args.no_others:
        try:
            ns = ns_measure(d, dev, world, rank, 10, 3, sync, barrier)
        except Exception as ex:   # report, do not hide (all ranks fail or succeed together: same code, same shapes)
            ns = {'error': '%s: %s' % (type(ex).__name__, str(ex)[:200])}

    # ---- the fused REGAT core on the same graph, sharded over the heads (N > 1, peer exchange, F = H*D = 128)
    regat_sharded = None
    if world > 1 and not args.no_others and args.partition == 'peer' and xch is not None and f == 128 and 8 % world == 0:
        try:
            regat_sharded = regat_sharded_measure(g, etv, dev, world, rank, bounds, xch, n, r, e, sync, barrier)
        except Exception as ex:
            regat_sharded = {'error': '%s: %s' % (type(ex).__name__, str(ex)[:200])}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (forward SpMM launch, timed alone on the launching stream)
    hbm, how = peaks()
    with torch.no_grad():
        nrm = RF.weighted_degree_norm(g, etv, theta, ALPHA, -0.5).detach()
        sliced = world > 1 and args.partition in ('cols', 'peer')
        fk = f // world if sliced else f      # feature-sliced: this rank's launch covers all rows x F/P columns
        xs = x_bufs[0].detach() if world == 1 else torch.randn(n, fk, device=dev)
        y = torch.empty(n, fk, device=dev)
        rows = None if world == 1 or sliced else (bounds[rank], bounds[rank + 1])

        def k():
            ops.spmm(csr['indptr'], csr['indices'], etv[0], theta.detach(), ALPHA, nrm, nrm, xs, rows=rows, out=y,
                     split=csr.get('split'), order=ops.row_order(csr) if fk <= ops.NARROW_FEAT else None)
        tk = timed(k, 20, 5, sync) / 20
        rows_n = n if rows is None else rows[1] - rows[0]
        edges_n = e if rows is None else int(csr['indptr'][rows[1]].item() - csr['indptr'][rows[0]].item())
    alg = algorithmic_bytes_spmm(rows_n, edges_n, fk)
    traffic = None
    tp = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tp) and world == 1 and args.scale == 1.0 and f == FEAT:
        with open(tp) as fh:
            traffic = json.load(fh).get('spmm_kernel_fwd_mag_f128_bytes')
    vw = 4 if fk >= 96 and fk % 4 == 0 else 2 if fk >= 34 and fk % 2 == 0 else 1
    kname = 'regnn::spmm_stream_kernel<%d,%d,false> (forward launch)' % (max(1, -(-fk // (32 * vw))), vw)
    if fk <= ops.NARROW_FEAT and fk % 4 == 0 and rows is None:
        kname = 'regnn::spmm_rowgroup_kernel<false,%d> (forward launch)' % (32 if fk > 64 else 16 if fk > 32 else 8 if fk > 16 else 4)
    roofline = {'bound': 'hbm', 'kernel': kname, 'achieved': alg / tk / 1e9,
                'peak': hbm, 'peak_source': how, 'unit': 'GB/s', 'frac': alg / tk / 1e9 / hbm, 'traffic': traffic,
                'algorithmic_bytes_per_launch': int(alg), 'launch_ms': tk * 1e3,
                # SURVEY 8(d) companions: the compulsory-traffic bound and whether the gathered matrix fits in L2
                'compulsory_bytes_per_launch': int(compulsory_bytes_spmm(rows_n, edges_n, fk)),
                'frac_compulsory': compulsory_bytes_spmm(rows_n, edges_n, fk) / tk / 1e9 / hbm,
                'l2_resident': bool(n * fk * 4 <= 126 * 2 ** 20)}

    # ---- the same for the kernel that is dominant BY TIME: the fused backward pass (gather + relation bins + folded
    # norm gradient), timed alone; algorithmic bytes per DESIGN.md section 4: E*(4F+13) + N*(3*4F+8)
    roofline_bwd = None
    if world == 1:
        try:
            with torch.no_grad():
                k()                                                       # y = the forward result of xs
                gk = torch.randn(n, f, device=dev)
                dxk = torch.empty(n, f, device=dev)

                def kb():
                    ops.spmm_bwd_fused(csr, etv[1], theta.detach(), ALPHA, nrm, xs, gk, out=dxk, y=y, want_dnorm=True)
                tb = timed(kb, 20, 5, sync) / 20
                del gk, dxk
            alg_b = e * (4 * f + 13) + n * (3 * 4 * f + 8)
            roofline_bwd = {'bound': 'hbm', 'kernel': 'regnn::spmm_rowgroup_kernel<true,32,true> (fused backward launch: dX, '
                                                      'relation bins, folded norm gradient; + its finalize kernels)',
                            'achieved': alg_b / tb / 1e9, 'peak': hbm, 'peak_source': how, 'unit': 'GB/s',
                            'frac': alg_b / tb / 1e9 / hbm, 'traffic': None, 'algorithmic_bytes_per_launch': int(alg_b),
                            'launch_ms': tb * 1e3}
        except Exception as ex:   # never lose the line over the companion measurement
            roofline_bwd = {'error': '%s: %s' % (type(ex).__name__, str(ex)[:200])}

    line = {
        'metric': 'GTEPS fwd+bwd per RE-layer', 'value': value, 'unit': 'GTEPS', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, d), 'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches),
        'roofline': roofline, 'graph_build_s': build_s,
        'partition': {'mode': args.partition, 'how': PARTITION_HOW.get(args.partition, args.partition),
                      'cuda_graph_replay': graphed},
        'phases_ms': dict(phases, note='eager steps with CUDA events around every C-ABI call / barrier / collective, '
                                       'max over ranks per phase; (gaps) = step time outside them (launch gaps, autograd, '
                                       'torch glue); the timed region itself runs without these events'),
    }
    if roofline_bwd is not None:
        line['roofline_backward'] = roofline_bwd
    if world > 1:
        line['parity_check'] = parity_check
    if ns is not None:
        line.setdefault('others', {})['mag_ns_data_parallel'] = dict(
            ns, n_gpus=world, scaling='weak',
            workload='BASELINE config 5: RE-GCN (MAG stack) neighbour-sampled minibatch training, 512 seeds per rank, '
                     'fan-out [25, 20], hidden 512, gradient all-reduce per step')
    if regat_sharded is not None:
        line.setdefault('others', {})['mag_regat_h8d16_head_sliced'] = regat_sharded
    if world == 1 and not args.no_cpu_baseline:
        line['cpu_baseline'], _ = cpu_reference_sample(d, f, 3, 1)
    if world == 1 and not args.no_others:
        del x_bufs, g_bufs, xs, y
        torch.cuda.empty_cache()
        line.setdefault('others', {}).update(others(dev, 10, 3))
        line['others'].update(attention_at_hbm_scale(dev, d, g, et, 5, 3))
        line['epoch_time'] = epoch_times(dev, 10, 3)
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def regat_sharded_measure(g, etv, dev, world, rank, bounds, xch, n, r, e, sync, barrier, heads=8, dim=16, steps=10):
    """The fused REGAT core (projection scores + logits + edge softmax + aggregation, forward + backward) on the same graph,
    sharded over the attention heads across the ranks (partition.head_sliced_gat over peer memory: heads are independent
    column slabs) next to the single-device layer on this rank: bit-equality of the rank's rows of the output and of the
    feature gradient, parameter gradients to 5e-5, then both timed.  Collective: every rank calls it."""
    import torch.distributed as dist
    from re_gnn_b200 import functional as RF, partition
    gen = torch.Generator(device=dev).manual_seed(4242)
    f = torch.randn(n, heads, dim, device=dev, generator=gen) * 0.5
    gout = torch.randn(n, heads, dim, device=dev, generator=gen)
    al0 = torch.randn(1, heads, dim, device=dev, generator=gen) * 0.3
    ar0 = torch.randn(1, heads, dim, device=dev, generator=gen) * 0.3
    th0 = theta_init(r, heads).to(dev)
    rb, re = bounds[rank], bounds[rank + 1]

    def single():
        leaves = [t.clone().requires_grad_(True) for t in (f, al0, ar0, th0)]
        out, _ = RF.gat_layer(g, etv, *leaves, ALPHA, 0.2)
        out.backward(gout)
        return out.detach(), [t.grad for t in leaves]

    def sharded():
        mine = [f[rb:re].clone().requires_grad_(True)] + [t.clone().requires_grad_(True) for t in (al0, ar0, th0)]
        out = partition.head_sliced_gat(g, etv, mine[0], mine[1], mine[2], mine[3], ALPHA, 0.2, bounds, rank, exchange=xch)
        out.backward(gout[rb:re])
        partition.allreduce_relation_grads(mine[1:])
        return out.detach(), [t.grad for t in mine]

    ref_out, ref_g = single()
    out, grads = sharded()
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))  # noqa: E731
    prel = max(rel(grads[i], ref_g[i]) for i in (1, 2, 3))
    chk = torch.tensor([int(torch.equal(out, ref_out[rb:re])), int(torch.equal(grads[0], ref_g[0][rb:re])), int(prel < 5e-5)],
                       device=dev)
    dist.all_reduce(chk, op=dist.ReduceOp.MIN)
    pmax = torch.tensor([prel], device=dev, dtype=torch.float64)
    dist.all_reduce(pmax, op=dist.ReduceOp.MAX)
    del ref_out, ref_g, out, grads
    t = torch.tensor([timed(single, steps, 3, sync, barrier), timed(sharded, steps, 3, sync, barrier)], device=dev,
                     dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t1, tp = float(t[0].item()) / steps, float(t[1].item()) / steps
    return {'gteps_fwd_bwd': e / tp / 1e9, 'ms': tp * 1e3, 'single_gpu_ms_same_boxes': t1 * 1e3, 'speedup_vs_one_gpu': t1 / tp,
            'n_gpus': world, 'heads': heads, 'head_dim': dim, 'scaling': 'strong',
            'how': 'heads sharded over the ranks (H/P heads x all rows per rank), row<->head-slab re-partition by '
                   'regnn_rows_to_slabs / regnn_slabs_to_rows over NVLink peer memory, gradient all-gather of the '
                   'attention vectors and the relation embedding included',
            'parity_check': {'y_equal': bool(chk[0].item()), 'd_feat_equal': bool(chk[1].item()),
                             'param_grad_max_rel_err': float(pmax.item()), 'param_grads_ok': bool(chk[2].item()),
                             'against': 'the single-device RF.gat_layer on every rank, its rows compared bit for bit'}}


def ns_measure(d, dev, world, rank, steps, warmup, sync, barrier):
    """Neighbour-sampled minibatch training of the MAG-stack RE-GCN, data-parallel (BASELINE config 5): batch 512 seeds per
    rank, fan-out [25, 20], 2 layers, hidden 512, 349 classes (mag/regnn_ns.py:41-51,200-208), one gradient all-reduce
    per step; weak scaling (every rank draws its own batches).  Collective: every rank must call it.  Returns the
    timing dict (identical on all ranks)."""
    import torch.distributed as dist
    from re_gnn_b200 import Graph, _lib, mag
    from re_gnn_b200.sampling import NeighborSampler
    n, net, sizes = d['num_nodes'], d['num_etype'], d['type_sizes']
    nnt = len(sizes)
    g = Graph(d['src'][:-n], d['dst'][:-n], n).to(dev)        # MAG stack: no stored self loops (self_loop_type 2 adds them)
    g.csr()
    edge_type0 = (torch.as_tensor(d['etype'][:-n]) - 1).to(dev)
    node_type = torch.as_tensor(d['ntype']).to(dev)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    local_idx = torch.as_tensor(np.arange(n) - offs[d['ntype']]).to(dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    x_dict = {k: torch.randn(sizes[k], 128, device=dev, generator=gen) for k in range(nnt)}
    labels = torch.randint(0, 349, (n,), device=dev, generator=gen)
    torch.manual_seed(123)
    model = mag.REGNN(128, 512, 349, 1, 2, ALPHA, 0.5, {k: 128 for k in range(nnt)}, net, residual=True, no_re=False,
                      self_loop_type=2).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    sampler = NeighborSampler(g, [25, 20], seed=123, rank=rank)
    batch_size, n_train = 512, int(sizes[0] * 0.855)          # 629,571 of 736,389 papers are training nodes in ogbn-mag
    perm = torch.randperm(n_train, generator=torch.Generator().manual_seed(1000 + rank))
    seeds_h = perm[:batch_size * 64].view(64, batch_size).pin_memory()
    loss_h = torch.empty(1).pin_memory()
    state = {'i': 0, 'edges': 0}

    def step():
        i = state['i']
        seeds = seeds_h[i % 64].to(dev, non_blocking=True)     # the step's input comes from pinned host memory
        loss, ne = mag.train_step(model, opt, sampler, seeds, labels[seeds], x_dict, edge_type0, node_type, local_idx,
                                  epoch=0, batch=i, world_size=world)
        loss_h.copy_(loss.view(1), non_blocking=True)          # the step's result goes back to the host
        state['i'] += 1
        state['edges'] += ne

    l0 = _lib.launch_count
    for _ in range(warmup):
        step()
    state['edges'] = 0
    total = timed(step, steps, 0, sync, barrier)
    launches = (_lib.launch_count - l0) * steps // (steps + warmup)
    edges = torch.tensor([float(state['edges']), total], device=dev, dtype=torch.float64)
    if world > 1:
        tmax = edges[1:].clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        esum = edges[:1].clone()
        dist.all_reduce(esum, op=dist.ReduceOp.SUM)
        total, all_edges = float(tmax.item()), float(esum.item())
    else:
        all_edges = float(state['edges'])
    return {'gteps_sampled': all_edges / total / 1e9, 'ms_per_step': total / steps * 1e3,
            'steps_per_s_all_ranks': steps / total * world, 'sampled_edges_per_step': all_edges / steps,
            'params': sum(p.numel() for p in model.parameters()), 'launches': int(launches), 'batch_size_per_rank': batch_size}


def run_ns(args, d):
    """``--workload mag_ns``: the line of BASELINE config 5 on its own (see ``ns_measure``).  value = sampled edges / s."""
    import torch.distributed as dist
    world, rank, local = (int(os.environ.get(k, '0' if k != 'WORLD_SIZE' else '1')) for k in ('WORLD_SIZE', 'RANK', 'LOCAL_RANK'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    sync = torch.cuda.synchronize
    barrier = (lambda: dist.barrier()) if world > 1 else None
    sampler_clk = ClockSampler(local)
    sampler_clk.start()
    m = ns_measure(d, dev, world, rank, args.steps, args.warmup, sync, barrier)
    clocks = sampler_clk.stop()
    if rank == 0:
        line = {'metric': 'GTEPS (sampled edges) per neighbour-sampled train step, data-parallel', 'value': m['gteps_sampled'],
                'unit': 'GTEPS', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': m['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': 'RE-GCN (MAG stack) neighbour-sampled minibatch training, BASELINE config 5',
                           'batch_size_per_rank': m['batch_size_per_rank'], 'fanout': [25, 20], 'hidden': 512, 'classes': 349,
                           'params': m['params'], 'sampled_edges_per_step': m['sampled_edges_per_step'],
                           'l2': 'every step touches a new random batch; feature tables (993 MB) exceed L2'},
                'clocks': clocks,
                'e2e': {'value': m['gteps_sampled'], 'unit': 'GTEPS', 'h2d_bytes_per_step': m['batch_size_per_rank'] * 8,
                        'd2h_bytes_per_step': 4,
                        'note': 'the timed step already starts from pinned-host seed ids and ends with the loss on the host'},
                'gpu_launches': m['launches'], 'steps_per_s': m['steps_per_s_all_ranks']}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_saint(args, d):
    """BASELINE config 5, GraphSAINT variant: 20 000 random-walk roots x walk length 2 per step, RE-GCN (SAINT flavour)
    with hidden 128, 2 layers, batch norm + residual (mag/regnn_saint.py:37-46,185-190), data-parallel, one gradient
    all-reduce per step.  Weak scaling.  value = subgraph edges processed / s."""
    import torch.distributed as dist
    from re_gnn_b200 import Graph, _lib, mag
    from re_gnn_b200.sampling import SaintRandomWalkSampler
    world, rank, local = (int(os.environ.get(k, '0' if k != 'WORLD_SIZE' else '1')) for k in ('WORLD_SIZE', 'RANK', 'LOCAL_RANK'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    sync = torch.cuda.synchronize
    barrier = (lambda: dist.barrier()) if world > 1 else None
    n, net, sizes = d['num_nodes'], d['num_etype'], d['type_sizes']
    nnt = len(sizes)
    g = Graph(d['src'][:-n], d['dst'][:-n], n).to(dev)
    g.csr()
    edge_type0 = (torch.as_tensor(d['etype'][:-n]) - 1).to(dev)
    node_type = torch.as_tensor(d['ntype']).to(dev)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    local_idx = torch.as_tensor(np.arange(n) - offs[d['ntype']]).to(dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    x_dict = {k: torch.randn(sizes[k], 128, device=dev, generator=gen) for k in range(nnt)}
    labels = torch.randint(0, 349, (n,), device=dev, generator=gen)
    train_mask = (node_type == 0) & (local_idx < int(sizes[0] * 0.855))
    torch.manual_seed(123)
    model = mag.SaintREGCN(128, 128, 349, 2, ALPHA, 0.5, {k: 128 for k in range(nnt)}, net, use_bn=True, residual=True,
                           gcn=False).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=5e-3)
    sampler = SaintRandomWalkSampler(g, roots=20000, walk_length=2, seed=123, rank=rank)
    loss_h = torch.empty(1).pin_memory()
    state = {'i': 0, 'edges': 0}

    def step():
        loss, ne = mag.saint_train_step(model, opt, sampler, labels, train_mask, x_dict, edge_type0, node_type, local_idx,
                                        epoch=0, batch=state['i'], world_size=world)
        loss_h.copy_(loss.view(1), non_blocking=True)
        state['i'] += 1
        state['edges'] += ne

    clk = ClockSampler(local)
    clk.start()
    l0 = _lib.launch_count
    for _ in range(args.warmup):
        step()
    state['edges'] = 0
    total = timed(step, args.steps, 0, sync, barrier)
    clocks = clk.stop()
    launches = (_lib.launch_count - l0) * args.steps // (args.steps + args.warmup)
    all_edges = float(state['edges'])
    if world > 1:
        t = torch.tensor([total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        es = torch.tensor([all_edges], device=dev, dtype=torch.float64)
        dist.all_reduce(es, op=dist.ReduceOp.SUM)
        total, all_edges = float(t.item()), float(es.item())
    if rank == 0:
        val = all_edges / total / 1e9
        print(json.dumps({
            'metric': 'GTEPS (subgraph edges) per GraphSAINT train step, data-parallel', 'value': val, 'unit': 'GTEPS',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total / args.steps * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'RE-GCN GraphSAINT random-walk minibatch training, BASELINE config 5',
                       'roots_per_rank': 20000, 'walk_length': 2, 'hidden': 128, 'classes': 349,
                       'subgraph_edges_per_step': all_edges / args.steps,
                       'l2': 'every step touches a new random subgraph; feature tables (993 MB) exceed L2'},
            'clocks': clocks,
            'e2e': {'value': val, 'unit': 'GTEPS', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 4,
                    'note': 'sampling starts from counter-based keys on the device; the loss is copied to the host every step'},
            'gpu_launches': int(launches), 'steps_per_s': args.steps / total * world}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get('RANK', '0'))
    if args.impl == 'reference' and rank != 0:
        return
    from re_gnn_b200 import synth
    d = synth.hetero_graph('mag', scale=args.scale)
    if args.impl == 'reference':
        run_reference(args, d)
    elif args.workload == 'mag_ns':
        run_ns(args, d)
    elif args.workload == 'mag_saint':
        run_saint(args, d)
    else:
        run_ours(args, d)


if __name__ == '__main__':
    main()
