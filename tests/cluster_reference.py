"""TEST INFRASTRUCTURE ONLY — CPU restatement of the cluster analysis (ljmd_clusters): the links of
tests/cluster_reference.c (the fp32 pair rule of the library), their connected components through
scipy.sparse.csgraph, and the library's labels (smallest index of the cluster, -1 for an inactive particle) and
sizes.

The C file is compiled on first use (tests/cref.py).  The product package never imports this module.
"""
from __future__ import annotations

import ctypes

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

import cref

def _mask(mask, N):
    return None if mask is None else np.ascontiguousarray(np.broadcast_to(np.asarray(mask) != 0, (N,)), np.uint8)


def links(R, box, r_link, mask=None):
    """(L, 2) int32 pairs (i, j), i < j, of one snapshot R (N, 2): both active, r_ij <= r_link in fp32."""
    R = np.ascontiguousarray(R, dtype=np.float32)
    N = R.shape[0]
    m = _mask(mask, N)
    mp = None if m is None else m.ctypes.data
    lib = cref.load("cluster_reference", {"bref_links": ([ctypes.c_int64, ctypes.c_void_p, ctypes.c_float,
                                                          ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p],
                                                         ctypes.c_int64)})
    args = (N, R.ctypes.data, float(np.float32(box)), float(np.float32(r_link)), mp)
    n = lib.bref_links(*args, None)
    pairs = np.zeros((max(n, 1), 2), np.int32)
    assert lib.bref_links(*args, pairs.ctypes.data) == n
    return pairs[:n]


def active(R, mask=None):
    R = np.asarray(R, np.float32)
    a = np.isfinite(R).all(axis=1)
    return a if mask is None else a & (_mask(mask, R.shape[0]) != 0)


def labels_from_links(pairs, act):
    """(labels, sizes) int32 (N,) in the library's convention from the links and the active flags."""
    N = act.shape[0]
    g = coo_matrix((np.ones(len(pairs), np.int8), (pairs[:, 0], pairs[:, 1])), shape=(N, N))
    _, comp = connected_components(g, directed=False)
    first = np.full(comp.max() + 1 if N else 0, N, np.int64)
    np.minimum.at(first, comp, np.arange(N))                  # smallest index of every component
    labels = np.where(act, first[comp], -1).astype(np.int32)
    sizes = np.bincount(labels[act], minlength=N).astype(np.int32)
    return labels, sizes


def clusters(R, box, r_link, mask=None):
    """(labels, sizes) int32 (N,) of one snapshot, as ljmd_clusters."""
    return labels_from_links(links(R, box, r_link, mask), active(R, mask))


def brute_force(R, box, r_link):
    """(labels, sizes) by a plain Python union-find over all pairs (every particle active), with numpy's fp32
    minimum image (d - box rint(d / box), as the C reference)."""
    R = np.asarray(R, np.float32)
    N = R.shape[0]
    box = np.float32(box)
    parent = list(range(N))

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    for i in range(N):
        d = R[i + 1:] - R[i]
        d = (d - box * np.rint(d / box)).astype(np.float32)
        r = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]).astype(np.float32))
        for j in np.nonzero(r <= np.float32(r_link))[0] + i + 1:
            a, b = find(i), find(int(j))
            if a != b:
                parent[max(a, b)] = min(a, b)
    labels = np.array([find(i) for i in range(N)], np.int32)
    return labels, np.bincount(labels, minlength=N).astype(np.int32)
