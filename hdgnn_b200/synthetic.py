"""Synthetic commits in the compact wire format of the hot path.

The shipped dataset blob (Adjset/glide.zip) is absent from the reference mount, so every
benchmark and parity case uses commits generated here (BASELINE.md section 3, SURVEY 8(d)):
directed Bernoulli entity adjacency, small-integer node attribute on the diagonal
(utils2.py:35 reads x_i = A_ii), an entity->hunk map with 'null' entries and ids beyond the
Nc cut (utils2.py:129-136), some commits with fewer index lines than Ne (utils2.py:121-124)
and a planted, learnable hunk adjacency.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np


@dataclass
class CommitBatch:
    """Compact form of the nine dense feeds of model_2.py:54-82.

    adj  (B,Ne,Ne) uint8  off-diagonal entity adjacency, diagonal 0      (utils2.py:46)
    x    (B,Ne)    float32 node attribute = raw diagonal                 (utils2.py:35)
    hmap (B,Ne)    int32  hunk id of entity line i; -1 = 'null' or id >= Nc (utils2.py:129-136)
    L    (B,)      int32  number of index lines read, <= Ne              (utils2.py:121)
    Y    (B,Nc,Nc) uint8  off-diagonal hunk adjacency = label            (utils2.py:47)
    nh   (B,)      int32  number of real hunks, rows 0 .. nh-1 of Y; None = not known (every Nc hunk counts)
    """
    adj: np.ndarray
    x: np.ndarray
    hmap: np.ndarray
    L: np.ndarray
    Y: np.ndarray
    nh: Optional[np.ndarray] = None

    @property
    def B(self):
        return self.adj.shape[0]

    @property
    def Ne(self):
        return self.adj.shape[1]

    @property
    def Nc(self):
        return self.Y.shape[1]

    def slice(self, lo, hi):
        return CommitBatch(self.adj[lo:hi], self.x[lo:hi], self.hmap[lo:hi], self.L[lo:hi], self.Y[lo:hi],
                           None if self.nh is None else self.nh[lo:hi])


def make_commits(B, Ne, Nc, seed=20260, p_edge=0.05, p_null=0.15, p_short=0.2, p_noise=0.02,
                 x_max=9) -> CommitBatch:
    rng = np.random.default_rng(seed)
    adj = (rng.random((B, Ne, Ne)) < p_edge).astype(np.uint8)
    idx = np.arange(Ne)
    adj[:, idx, idx] = 0
    x = rng.integers(0, x_max + 1, size=(B, Ne)).astype(np.float32)
    raw = rng.integers(0, Nc + 4, size=(B, Ne)).astype(np.int32)       # ids >= Nc exercise the cut rule
    hmap = np.where(rng.random((B, Ne)) < p_null, -1, raw).astype(np.int32)
    hmap[hmap >= Nc] = -1
    L = np.full(B, Ne, dtype=np.int32)
    short = rng.random(B) < p_short
    lo = max(2, Ne // 2)
    L[short] = rng.integers(lo, max(lo + 1, Ne), size=int(short.sum())).astype(np.int32)
    Y = (rng.random((B, Nc, Nc)) < p_noise).astype(np.uint8)
    for b in range(B):                                                   # planted: edge between hunks
        ii, jj = np.nonzero(adj[b])
        hs, ht = hmap[b, ii], hmap[b, jj]
        ok = (hs >= 0) & (ht >= 0) & (hs != ht)
        Y[b, hs[ok], ht[ok]] = 1
    cidx = np.arange(Nc)
    Y[:, cidx, cidx] = 0
    return CommitBatch(adj, x, hmap, L, Y)
