"""Counter-based attention dropout of the fused REGAT / REGATv2 kernels (``regnn_attn_dropout_t``).

The keep factor of edge id e and head h is a pure function of (key, e, global head): the kernels compute it in
registers from the edge id they already load, so no [E, H] mask is drawn, stored or read, and every rank and every
partition of the graph (head slices, halo row blocks) sees the same bits without exchanging anything.  The hash is
stated in include/regnn_b200.h and restated in oracle/attn_dropout_oracle.py.  A key is derived from
(seed, step, layer) with the mixing function of the samplers (``sampling._mix32``).
"""
import math

from . import _lib
from .sampling import M32, _mix32


def attn_dropout_key(seed, step, layer=0):
    """64-bit key of one layer's attention-dropout mask at one training step.  Both halves depend on all three
    inputs, so masks of different steps or layers are unrelated (not shifted or permuted copies of each other)."""
    seed = (int(seed) ^ (int(seed) >> 32)) & M32
    step, layer = int(step) & M32, int(layer) & M32
    lo = _mix32((seed * 0x9E3779B1 + step * 0x85EBCA6B + layer * 0xC2B2AE35 + 0x2545F491) & M32)
    hi = _mix32(((lo ^ (seed * 0x27D4EB2F + step * 0x165667B1 + layer * 0x5BD1E995)) + 0x68E31DA4) & M32)
    return (hi << 32) | lo


class HashedDropout:
    """Attention dropout with drop probability ``p`` (0 <= p < 1) drawn by the counter hash under ``key``: a kept
    edge's attention is scaled by 1 / (1 - p), a dropped one is 0 -- what ``nn.Dropout`` does to the attention
    weights, with the mask a function of (key, edge id, head).  ``head_offset`` / ``num_heads_total``: the call covers
    heads [head_offset, head_offset + H) of a layer with ``num_heads_total`` heads (None: the call's H), so a head
    slice reproduces that slice of the full-H mask."""

    __slots__ = ('p', 'key', 'head_offset', 'num_heads_total')

    def __init__(self, p, key, head_offset=0, num_heads_total=None):
        p = float(p)
        if not 0.0 <= p < 1.0:
            raise ValueError('HashedDropout: p must be in [0, 1), got %r' % p)
        self.p, self.key = p, int(key) & 0xFFFFFFFFFFFFFFFF
        self.head_offset, self.num_heads_total = int(head_offset), num_heads_total

    def __repr__(self):
        return 'HashedDropout(p=%r, key=%#x, head_offset=%d, num_heads_total=%r)' % (
            self.p, self.key, self.head_offset, self.num_heads_total)

    @property
    def threshold(self):
        """floor(p * 2^32): a hash value below it drops the edge."""
        return min(int(math.floor(self.p * 4294967296.0)), M32)

    @property
    def scale(self):
        """The keep factor 1 / (1 - p), rounded to fp32 by the struct."""
        return 1.0 / (1.0 - self.p)

    def for_heads(self, head_offset, num_heads_total):
        """The same mask seen by a call over heads [head_offset, ...) of a ``num_heads_total``-head layer."""
        return HashedDropout(self.p, self.key, head_offset, num_heads_total)

    def struct(self, heads):
        """-> ``_lib.AttnDropout`` for a call over ``heads`` heads."""
        total = self.num_heads_total if self.num_heads_total is not None else self.head_offset + heads
        if self.head_offset < 0 or total < self.head_offset + heads:
            raise ValueError('HashedDropout: heads [%d, %d) outside a %d-head layer'
                             % (self.head_offset, self.head_offset + heads, total))
        return _lib.AttnDropout(self.key, self.threshold, self.scale, self.head_offset, total)
