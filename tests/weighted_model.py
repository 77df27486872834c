"""A plain numpy restatement of the arithmetic of the weighted FP32 pair tiles (k_weighted_tiles, csrc/weighted.cu).

Given the fp64 embedding of a few samples it computes, for chosen pairs, the fp32 value the kernel stores, rounding
by rounding:
  - the operand as k_weighted_operand_panels forms it: float(len * a) (pre-scaled) or float(a) with the length
    float(len) applied by an FFMA (negative lengths; fmaf is emulated in fp64, which may differ from the device in the
    last bit: compare that form within a tolerance only);
  - the nodes in column order (pre-order id), fp32 running sums flushed every FLUSH nodes into the per-pair total;
  - the epilogue in fp64 and the final fp32 store.

`scheme` selects the arithmetic:
  "f64tot" (the kernel as built): the total is fp64, and the keyed variant sums len * (match ? |a - b| : a + b)
           directly (the non-cancelling numerator, as the unkeyed one sums len * |a - b|);
  "f32tot" (the kernel before that change, kept to show why the accuracy tests use the inputs they do): the total is
           fp32, and the keyed variant sums S = sum over matched nodes of len * min(a, b) and forms
           numer = W_i + W_j - 2 S, a cancellation that multiplies the error of S by about (1 - d) / d.
"""
from __future__ import annotations

import numpy as np

FLUSH = 256            # nodes between two flushes of the running sums (weighted.cu: KT * FLUSH slabs)
SCHEME = "f64tot"      # the kernel as built
F32 = np.float32


def operands(E, length, total=None, prescaled=True):
    """fp32 operand rows [n_samples][B] and fp64 denominators W[n_samples] of k_weighted_operand_panels.

    E: fp64 subtree sums [n_samples][B]; total: the normalisers (normalize = 1) or None (raw values)."""
    E = np.asarray(E, np.float64)
    length = np.asarray(length, np.float64)
    if total is None:
        a = E
    else:
        t = np.asarray(total, np.float64)
        inv = np.where(t > 0, 1.0 / np.where(t > 0, t, 1.0), 0.0)
        a = E * inv[:, None]
    la = length[None, :] * a
    return (la if prescaled else a).astype(F32), la.sum(axis=1)


def _fma(l, x, acc):
    return (np.float64(l) * x.astype(np.float64) + acc.astype(np.float64)).astype(F32)


def terms(ai, aj, match=None, keyed_scheme=SCHEME):
    """fp32 per-node terms [B][P] of pairs with operand rows ai, aj [P][B] (match: keyed panels agree, [P][B])."""
    ai, aj = np.asarray(ai, F32).T, np.asarray(aj, F32).T
    if match is None:
        return np.abs(ai - aj)
    match = np.asarray(match).T
    if keyed_scheme == "f32tot":
        return np.where(match, np.minimum(ai, aj), F32(0))
    return np.abs(ai - np.where(match, aj, -aj))


def accumulate(t, lenf=None, scheme=SCHEME):
    """The kernel's two-level sum of the terms t [B][P] in node order: (tot, acc) after the last node.

    lenf (FFMA form): the fp32 lengths, acc = fmaf(len, term, acc)."""
    t = np.asarray(t, F32)
    P = t.shape[1]
    acc = np.zeros(P, F32)
    tot = np.zeros(P, np.float64 if scheme == "f64tot" else F32)
    for v in range(t.shape[0]):
        if lenf is None:
            acc = acc + t[v]
        else:
            acc = _fma(lenf[v], t[v], acc)
        if v % FLUSH == FLUSH - 1:
            tot = tot + (acc.astype(np.float64) if scheme == "f64tot" else acc)
            acc = np.zeros(P, F32)
    return tot, acc


def epilogue(tot, acc, wi, wj, keyed=False, scheme=SCHEME):
    """The fp32 distances the kernel stores from the accumulators and the fp64 denominators."""
    wi, wj = np.asarray(wi, np.float64), np.asarray(wj, np.float64)
    if scheme == "f64tot":
        num = tot + acc.astype(np.float64)
    else:
        s = (tot + acc).astype(np.float64)
        num = (wi + wj) - 2.0 * s if keyed else s
    return (num / (wi + wj)).astype(F32)


def distances(A, W, pairs, keys=None, lenf=None, scheme=SCHEME):
    """Model of the fp32 distances of `pairs` (list of (i, j)) from operand rows A [n][B] (operands()), W [n] and, for
    the keyed -l tiles, the key rows [n][B] (the largest present leaf id under each node, -1 when absent)."""
    i = np.array([p[0] for p in pairs])
    j = np.array([p[1] for p in pairs])
    match = None if keys is None else keys[i] == keys[j]
    t = terms(A[i], A[j], match, scheme)
    tot, acc = accumulate(t, lenf, scheme)
    return epilogue(tot, acc, W[i], W[j], keys is not None, scheme)


def constant_sum(c, n, lead=0, scheme=SCHEME):
    """The accumulated numerator (fp64) of `lead` zero terms followed by n equal fp32 terms c, for a vector of
    constants c: the unkeyed worst case (a star tree's root, then its leaves), vectorised over c."""
    c = np.asarray(c, F32)
    counts = []                      # terms c in each flush block, in order
    pos, end = lead, lead + n
    while pos < end:
        nxt = min(end, (pos // FLUSH + 1) * FLUSH)
        counts.append((nxt - pos, nxt % FLUSH == 0))
        pos = nxt
    folds = {}
    for m, _ in counts:
        if m not in folds:
            s = np.zeros_like(c)
            for _ in range(m):
                s = s + c
            folds[m] = s
    tot = np.zeros(c.shape, np.float64 if scheme == "f64tot" else F32)
    acc = np.zeros_like(c)
    for m, flushed in counts:
        if flushed:
            tot = tot + (folds[m].astype(np.float64) if scheme == "f64tot" else folds[m])
        else:
            acc = folds[m]
    if scheme == "f64tot":
        return tot + acc.astype(np.float64)
    return (tot + acc).astype(np.float64)


# ------------------------------------------------------------------ inputs and their fp64 distances
def embed(parent, rp, col, val, rows=None):
    """Subtree sums E [n][B] and keys K [n][B] of the CSR rows `rows` (default all), pre-order ids (parent < child)."""
    parent = np.asarray(parent)
    B = len(parent)
    rows = range(len(rp) - 1) if rows is None else rows
    E = np.zeros((len(rows), B))
    K = np.full((len(rows), B), -1, np.int64)
    for r, s in enumerate(rows):
        c = col[rp[s]:rp[s + 1]]
        E[r, c] = val[rp[s]:rp[s + 1]]
        K[r, c] = c
    for v in range(B - 1, 0, -1):
        p = parent[v]
        E[:, p] += E[:, v]
        K[:, p] = np.maximum(K[:, p], K[:, v])
    return E, K


def exact(E, K, length, pairs, keyed):
    """fp64 distances of the pairs from the embedding (normalised or raw as E is given)."""
    out = []
    for i, j in pairs:
        a, b = E[i], E[j]
        t = np.where(K[i] == K[j], np.abs(a - b), a + b) if keyed else np.abs(a - b)
        out.append(np.dot(length, t) / np.dot(length, a + b))
    return np.array(out)


def star(n_leaves, length):
    """Star tree: root 0 (length 0) and leaves 1..n_leaves of the given length."""
    parent = np.zeros(n_leaves + 1, np.int32)
    parent[0] = -1
    L = np.full(n_leaves + 1, length, np.float64)
    L[0] = 0.0
    return parent, L


def csr(rows):
    """CSR (row_ptr, col, val) from a list of (leaf ids, values)."""
    rp = np.concatenate([[0], np.cumsum([len(c) for c, _ in rows])]).astype(np.int64)
    col = np.concatenate([np.asarray(c, np.int32) for c, _ in rows])
    val = np.concatenate([np.asarray(v, np.float64) for _, v in rows])
    return rp, col, val


def length_for_operand(bits, scale=1.0):
    """The fp64 branch length whose pre-scaled operand len * scale rounds to the fp32 with these bits exactly
    (scale a power of two)."""
    return float(np.array([bits], np.uint32).view(F32)[0]) / scale
