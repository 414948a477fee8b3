"""Numpy restatement of the counter-based attention dropout of the fused REGAT / REGATv2 kernels
(``regnn_attn_dropout_t`` in include/regnn_b200.h, ``hashed_keep`` in re_gnn_b200/csrc/gat.cu).  No torch, no
package imports: the GPU tests hold the kernels' hashed mode bit-exact against the explicit mask built here.

  c    = e * num_heads_total + head_offset + h          (64-bit counter; e the global edge id, h the call's head)
  x    = mix32(lo32(c) ^ lo32(key))
  x    = mix32(x + hi32(c) * 0x9E3779B1 + hi32(key))    (uint32, wrapping)
  keep = x >= threshold ? scale : 0,   threshold = floor(p * 2^32),  scale = fp32(1 / (1 - p))
"""
import math

import numpy as np

M32 = 0xFFFFFFFF


def mix32(z):
    """The 32-bit finaliser of the samplers (vectorised over uint32 arrays, or a Python int)."""
    if isinstance(z, int):
        z &= M32
        z ^= z >> 16
        z = (z * 0x7feb352d) & M32
        z ^= z >> 15
        z = (z * 0x846ca68b) & M32
        z ^= z >> 16
        return z
    z = np.asarray(z, dtype=np.uint32)
    with np.errstate(over='ignore'):
        z = z ^ (z >> np.uint32(16))
        z = z * np.uint32(0x7feb352d)
        z = z ^ (z >> np.uint32(15))
        z = z * np.uint32(0x846ca68b)
        z = z ^ (z >> np.uint32(16))
    return z


def attn_dropout_hash(key, counter):
    """uint32 hash of uint64 counters under a 64-bit key."""
    c = np.asarray(counter, dtype=np.uint64)
    lo = (c & np.uint64(M32)).astype(np.uint32)
    hi = (c >> np.uint64(32)).astype(np.uint32)
    with np.errstate(over='ignore'):
        x = mix32(lo ^ np.uint32(key & M32))
        x = mix32(x + hi * np.uint32(0x9E3779B1) + np.uint32((key >> 32) & M32))
    return x


def threshold_scale(p):
    return min(int(math.floor(p * 4294967296.0)), M32), np.float32(1.0 / (1.0 - p))


def keep_mask(p, key, num_edges, heads, head_offset=0, num_heads_total=None):
    """[num_edges, heads] float32 keep factors in edge-id order (0 or scale)."""
    total = head_offset + heads if num_heads_total is None else num_heads_total
    t, scale = threshold_scale(p)
    e = np.arange(num_edges, dtype=np.uint64)[:, None]
    h = np.arange(heads, dtype=np.uint64)[None, :]
    x = attn_dropout_hash(key, e * np.uint64(total) + np.uint64(head_offset) + h)
    return np.where(x >= np.uint32(t), scale, np.float32(0)).astype(np.float32)
