"""ctypes binding of ``libregnn_b200.so`` (C ABI declared in ``include/regnn_b200.h``).

There is deliberately no fallback: if the shared library is missing or a call fails, a
``RuntimeError`` is raised.  Nothing here touches ``oracle/``.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# REGNN_B200_LIB: development knob, points the binding at an A/B build of the same C ABI (scripts/build_variants.sh)
LIB_PATH = os.environ.get('REGNN_B200_LIB') or os.path.join(_HERE, 'lib', 'libregnn_b200.so')

_p = ctypes.c_void_p
_i64 = ctypes.c_int64
_i32 = ctypes.c_int
_f32 = ctypes.c_float
_sz = ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/regnn_b200.h one to one
SIGNATURES = {
    'regnn_version': (_i32, []),
    'regnn_status_string': (ctypes.c_char_p, [_i32]),
    'regnn_last_error_string': (ctypes.c_char_p, []),
    'regnn_max_partial_blocks': (_i32, []),
    'regnn_csr_build_workspace_bytes': (_sz, [_i64, _i64]),
    'regnn_csr_build': (_i32, [_p, _p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    'regnn_etype_permute': (_i32, [_p, _p, _p, _i64, _i32, _p, _p, _p, _p]),
    'regnn_relation_counts': (_i32, [_p, _p, _i64, _i64, _i32, _p, _p]),
    'regnn_wdeg_norm_fwd': (_i32, [_p, _p, _p, _p, _f32, _i32, _f32, _f32, _i64, _i64, _p, _p, _p]),
    'regnn_wdeg_norm_bwd': (_i32, [_p, _p, _p, _p, _f32, _i32, _f32, _f32, _i64, _i64, _p, _p, _p, _p, _p]),
    'regnn_spmm_fwd': (_i32, [_p, _p, _p, _p, _f32, _i32, _p, _p, _p, _i64, _p, _i64, _i64, _i64, _i32, _p, _p, _p, _p]),
    'regnn_spmm_bwd_w': (_i32, [_p, _p, _p, _p, _f32, _i32, _p, _i32, _p, _i64, _p, _i64, _p, _i64, _p, _i64,
                                _i64, _i64, _i32, _p, _p, _p, _p, _p]),
    'regnn_spmm_bwd_fused': (_i32, [_p, _p, _p, _p, _f32, _i32, _p, _i32, _p, _i64, _p, _i64, _p, _i64, _i64, _i64,
                                    _i32, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p]),
    'regnn_rows_to_slabs': (_i32, [_p, _i64, _i64, _i32, _i32, _i64, _p, _p]),
    'regnn_slabs_to_rows': (_i32, [_p, _i64, _i64, _i32, _p, _p]),
    'regnn_halo_push': (_i32, [_p, _i64, _i32, _p, _p, _p, _p, _i64, _i32, _i32, _p]),
    'regnn_halo_scatter': (_i32, [_p, _i64, _i32, _p, _p, _p, _i64, _i32, _i32, _p]),
    'regnn_halo_push_slots': (_i32, [_p, _i32, _p, _i32, _p, _p, _p, _p, _p, _i32, _i32, _p]),
    'regnn_spmm_fwd_scatter': (_i32, [_p, _p, _p, _p, _f32, _i32, _p, _p, _p, _i64, _i64, _i32, _p, _p, _p, _p, _p, _i64,
                                      _p]),
    'regnn_spmm_bwd_fused_scatter': (_i32, [_p, _p, _p, _p, _f32, _i32, _p, _i32, _p, _i64, _p, _i64, _i64, _i32,
                                            _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _p]),
    'regnn_rowdot_norm_bwd': (_i32, [_p, _i32, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _i64, _i32, _p, _p]),
    'regnn_random_walk': (_i32, [_p, _p, _i64, _i64, _i32, ctypes.c_uint64, _p, _p]),
    'regnn_sample_neighbors': (_i32, [_p, _p, _i64, _i32, ctypes.c_uint64, _p, _p]),
    'regnn_gat_fwd': (_i32, [_p, _p, _p, _p, _p, _f32, _i32, _p, _p, _p, _f32, _p, _p, _i32, _i32, _i64, _i64,
                             _p, _p, _p, _p, _p, _p, _p, _p]),
    'regnn_gat_bwd_stats': (_i32, [_p, _p, _p, _p, _p, _i64, _i32, _i32, _p, _p]),
    'regnn_gat_bwd_edges': (_i32, [_p, _p, _p, _p, _p, _p, _f32, _i32, _p, _p, _p, _f32, _p, _p, _p, _i32, _i32, _i64,
                                   _i64, _p, _p, _p, _p, _p, _p, _p, _p]),
    'regnn_gat_bwd_reduce': (_i32, [_p, _p, _p, _f32, _i32, _p, _i32, _i64, _i64, _p, _p, _p, _p, _p, _p]),
    'regnn_attn_scores_fwd': (_i32, [_p, _p, _p, _i64, _i32, _i32, _p, _p, _p]),
    'regnn_attn_scores_bwd': (_i32, [_p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _p, _p]),
    'regnn_grouped_linear_fwd': (_i32, [_i32, _p, _p, _p, _p, _p, _i32, _i64, _p, _p, _p, _p, _i64, _p]),
    'regnn_grouped_linear_bwd': (_i32, [_i32, _p, _p, _p, _i32, _i64, _p, _p, _p, _p, _i64, _i32, _p, _p, _p]),
    'regnn_gatv2_fwd': (_i32, [_p, _p, _p, _p, _p, _f32, _i32, _p, _p, _p, _f32, _p, _p, _i32, _i32, _i64, _i64,
                               _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    'regnn_gatv2_bwd_edges_blocks': (_i64, [_i64, _i32, _i32, _i32, _i32, _i32]),
    'regnn_gatv2_bwd_edges': (_i32, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _f32, _p, _p, _p, _i32, _i32, _i64, _i64,
                                     _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    'regnn_gatv2_bwd_dst': (_i32, [_p, _p, _p, _f32, _i32, _p, _p, _p, _p, _f32, _i32, _i32, _i64, _i64,
                                   _p, _p, _p, _p, _p, _p, _p]),
}



class RowSplit(ctypes.Structure):
    """Mirror of ``regnn_rowsplit_t`` (include/regnn_b200.h)."""
    _fields_ = [('long_rows', _p), ('frag_ptr', _p), ('frag_row', _p), ('frag_begin', _p),
                ('num_long', ctypes.c_int32), ('num_frags', ctypes.c_int32), ('threshold', ctypes.c_int32)]


class AttnDropout(ctypes.Structure):
    """Mirror of ``regnn_attn_dropout_t`` (include/regnn_b200.h)."""
    _fields_ = [('key', ctypes.c_uint64), ('threshold', ctypes.c_uint32), ('scale', ctypes.c_float),
                ('head_offset', ctypes.c_int32), ('num_heads_total', ctypes.c_int32)]


class PeerRows(ctypes.Structure):
    """Mirror of ``regnn_peer_rows_t`` (include/regnn_b200.h)."""
    _fields_ = [('base', _p), ('num_ranks', ctypes.c_int32), ('rows_per_rank', ctypes.c_int64),
                ('ld', ctypes.c_int64), ('col_offset', ctypes.c_int64)]


_lib = None


def load():
    """Loads the shared library (once) and returns the ctypes handle; raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'libregnn_b200.so is missing (%s). Build it with `python -m re_gnn_b200.build` or '
            '`__graft_entry__.build()`; re_gnn_b200 has no CPU or eager fallback.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


# Kernel launches issued through the C ABI since import (bench.py reports the count of a timed region).
# Each wrapper in ops.py adds the number of kernels its entry point launches.
launch_count = 0


def count_launches(n):
    global launch_count
    launch_count += n


# ---- tracing: NVTX ranges around every ABI call, and an optional CUDA-event timeline -----------------------------
# NVTX costs well under a microsecond per call when no profiler is attached; REGNN_NVTX=0 turns it off.
_NVTX = os.environ.get('REGNN_NVTX', '1') != '0'
_trace = None   # active Trace or None


class Trace:
    """Per-phase device timeline of a region: while active, every ABI call (and every ``phase(name)`` block, used by
    partition.py around barriers / collectives) is bracketed by CUDA events on the current stream.
    ``summary(steps)`` -> {name: milliseconds per step}, plus ``'(gaps)'`` = region time not covered by any phase
    (launch gaps, allocator and autograd overhead, torch glue kernels).  Costs two event records per call: use it
    on a few extra steps, never inside a timed region."""

    def __init__(self):
        self.events = []      # (name, start, end)
        self.t0 = self.t1 = None

    def __enter__(self):
        global _trace
        import torch
        self.t0 = torch.cuda.Event(enable_timing=True)
        self.t0.record()
        _trace = self
        return self

    def __exit__(self, *exc):
        global _trace
        import torch
        _trace = None
        self.t1 = torch.cuda.Event(enable_timing=True)
        self.t1.record()

    def summary(self, steps=1):
        import torch
        torch.cuda.synchronize()
        out, covered = {}, 0.0
        for name, a, b in self.events:
            ms = a.elapsed_time(b)
            out[name] = out.get(name, 0.0) + ms / steps
            covered += ms
        total = self.t0.elapsed_time(self.t1)
        out['(gaps)'] = max(0.0, total - covered) / steps
        out['(total)'] = total / steps
        return out


class phase:
    """``with _lib.phase('barrier'): ...`` -- NVTX range + (when a Trace is active) a timeline entry."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        global _NVTX
        import torch
        if _NVTX:
            try:
                torch.cuda.nvtx.range_push(self.name)
                self.pushed = True
            except Exception:   # no NVTX in this build / no CUDA runtime: switch the ranges off, keep going
                _NVTX = False
        if _trace is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        import torch
        if _trace is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _trace.events.append((self.name, self.a, b))
        if getattr(self, 'pushed', False):
            torch.cuda.nvtx.range_pop()


def call(name, *args):
    """Calls a status-returning entry point; raises RuntimeError with the library's message on failure."""
    lib = load()
    if _NVTX or _trace is not None:
        with phase(name):
            rc = getattr(lib, name)(*args)
    else:
        rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.regnn_last_error_string().decode() or lib.regnn_status_string(rc).decode()
        raise RuntimeError('%s failed (%d: %s): %s' % (name, rc, lib.regnn_status_string(rc).decode(), msg))


def partial_blocks(rows=None):
    """Number of per-block partial slots to allocate for any reduction entry point (an upper bound)."""
    return load().regnn_max_partial_blocks()
