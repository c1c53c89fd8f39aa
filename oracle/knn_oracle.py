"""CPU oracle for the kNN graph build.  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED: the reference contains no kNN at all (edges are built offline from
Geant4 ancestry, /root/reference/utils/data.py:847-929, and only offset-concatenated at
batch time, :1228-1261).  kNN is the new capability BASELINE.json's north_star names;
this numpy restatement *defines* its semantics and the CUDA kernel must reproduce it
bit-exactly:

  * per cloud (contiguous rows offsets[b]:offsets[b+1]), for every centre i the k
    nearest other points j != i by squared L2 distance over the position columns;
  * distance arithmetic is float32, evaluated as ((dx*dx + dy*dy) + dz*dz) with each
    product and sum rounded to float32 (no fused multiply-add), so that every platform
    gets the same bits;
  * ordering: ascending distance, ties broken by the lower point index (stable sort);
  * clouds with fewer than k+1 points pad the missing slots with -1;
  * edge list convention is GraphConv's (graph_net.py:73 via _graph_collate,
    data.py:1228-1261): row 0 = neighbour j (source), row 1 = centre i (target),
    centre-major order, global (batch-offset) node ids.

The Gaussian edge weight follows /root/reference/utils/data.py:835-845:
  w = exp(-d^2 / (2 sigma^2)), sigma = median(d) + 1e-6 over the edges of one graph,
  d = Euclidean length of the edge.
"""
from __future__ import annotations

import numpy as np


def _sq_dist(q: np.ndarray, p: np.ndarray) -> np.ndarray:
    """d2[i, j] = ((dx*dx + dy*dy) + dz*dz) between rows q[i] and p[j], every product and sum rounded to float32"""
    dx = q[:, None, 0] - p[None, :, 0]
    dy = q[:, None, 1] - p[None, :, 1]
    dz = q[:, None, 2] - p[None, :, 2]
    d2 = (dx * dx + dy * dy).astype(np.float32) + (dz * dz).astype(np.float32)
    return d2.astype(np.float32)


def knn_neighbours(pos: np.ndarray, offsets: np.ndarray, k: int, rows_per_chunk: int = None):
    """pos[n,3] float32, offsets[B+1] int64 -> (nbr[n,k] int64 (-1 pad), d2[n,k] float32 (inf pad)).

    rows_per_chunk: evaluate the centres of a cloud that many at a time, so memory stays at rows_per_chunk x cloud
    size instead of cloud size squared (clouds of 16384 points).  Same float32 distances and the same selection,
    so the result is identical: the k-th smallest distance of a row is found with a partition, every candidate at or
    below it is kept in ascending id order (all ties at the boundary included) and a stable sort by distance of those
    candidates keeps the first k."""
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    n = pos.shape[0]
    nbr = np.full((n, k), -1, dtype=np.int64)
    d2o = np.full((n, k), np.inf, dtype=np.float32)
    for b in range(len(offsets) - 1):
        s, e = int(offsets[b]), int(offsets[b + 1])
        p = pos[s:e]
        m = e - s
        kk = min(k, m - 1)
        if m == 0:
            continue
        if rows_per_chunk is None:
            d2 = _sq_dist(p, p)
            np.fill_diagonal(d2, np.inf)
            order = np.argsort(d2, axis=1, kind="stable")
            if kk > 0:
                sel = order[:, :kk]
                nbr[s:e, :kk] = sel + s
                d2o[s:e, :kk] = np.take_along_axis(d2, sel, axis=1)
            continue
        if kk <= 0:
            continue
        for r0 in range(0, m, rows_per_chunk):
            r1 = min(r0 + rows_per_chunk, m)
            d2 = _sq_dist(p[r0:r1], p)
            rows = np.arange(r1 - r0)
            d2[rows, rows + r0] = np.inf
            kth = np.partition(d2, kk - 1, axis=1)[:, kk - 1:kk]
            row, col = np.nonzero(d2 <= kth)                 # row-major: ids ascend inside every row
            val = d2[row, col]
            order = np.lexsort((col, val, row))             # by row, then distance, then id
            first = np.concatenate([[0], np.cumsum(np.bincount(row, minlength=r1 - r0))[:-1]])
            pick = order[(first[:, None] + np.arange(kk)[None, :]).reshape(-1)].reshape(r1 - r0, kk)
            nbr[s + r0:s + r1, :kk] = col[pick] + s
            d2o[s + r0:s + r1, :kk] = val[pick]
    return nbr, d2o


def knn_edges(nbr: np.ndarray) -> np.ndarray:
    """nbr[n,k] -> edge_index[2,E] int64 (row0 = neighbour, row1 = centre), -1 slots dropped."""
    n, k = nbr.shape
    centre = np.repeat(np.arange(n, dtype=np.int64), k)
    flat = nbr.reshape(-1)
    keep = flat >= 0
    return np.stack([flat[keep], centre[keep]])


def gaussian_edge_weights(features: np.ndarray, edges: np.ndarray, eps: float = 1e-6) -> np.ndarray:
    """data.py:835-845 restated for ONE graph (positions = features[:,1:4])."""
    positions = features[:, 1:4]
    d = np.linalg.norm(positions[edges[0]] - positions[edges[1]], axis=1)
    sigma = np.median(d) + eps
    return np.exp(-(d ** 2) / (2 * sigma ** 2)).astype(np.float32)
