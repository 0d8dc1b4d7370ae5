"""Vectorised NumPy restatement of how NumPy reduces a 1-D column: the pairwise float64 sum behind np.sum / np.mean
(numpy/_core/src/umath/loops_utils.h.src, pairwise_sum), the chunked cast of an int64 / bool mean through the ufunc
buffer, and np.var / np.std (numpy/_core/_methods.py, _var).  The device kernels of probabilit_b200/csrc/stats.cu
follow exactly this order; tests/test_stats_cpu.py pins it against NumPy itself.

pw(a, m): m < 8 -> a sequential sum; m <= 128 -> eight accumulators r[j] = a[j], r[j] += a[i + j] for
i = 8, 16, ... below m - m % 8, then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) and the m % 8 tail in order;
otherwise n2 = m/2 - (m/2) % 8 and pw(a, n2) + pw(a + n2, m - n2).  The reduction adds the tree to its initial 0.0.
"""
import numpy as np

LEAF = 128


def _leaf_sums(rows, off, size):
    """Leaf sums of every row of `rows` (r, L) for the leaves (off, size): -> (r, len(off))."""
    out = np.empty((rows.shape[0], len(off)))
    for m in np.unique(size):
        sel = np.flatnonzero(size == m)
        block = rows[:, off[sel][:, None] + np.arange(m)]  # (r, leaves, m)
        if m < 8:
            res = np.full(block.shape[:2], -0.0)
            for i in range(m):
                res = res + block[:, :, i]
        else:
            r = block[:, :, 0:8].copy()
            i = 8
            while i < m - m % 8:
                r = r + block[:, :, i:i + 8]
                i += 8
            res = ((r[..., 0] + r[..., 1]) + (r[..., 2] + r[..., 3])) + ((r[..., 4] + r[..., 5]) + (r[..., 6] + r[..., 7]))
            for k in range(i, m):
                res = res + block[:, :, k]
        out[:, sel] = res
    return out


def pairwise_rows(rows):
    """NumPy's pairwise tree over each row of a float64 (r, L) array (without the reduction's initial 0.0)."""
    rows = np.asarray(rows, dtype=np.float64)
    L = rows.shape[1]
    if L == 0:
        return np.full(rows.shape[0], -0.0)
    levels = []
    off, size = np.zeros(1, dtype=np.int64), np.array([L], dtype=np.int64)
    while True:  # the tree level by level: each internal node's children are a (left, right) pair of the next level
        leaf = size <= LEAF
        levels.append((off, size, leaf))
        inner = ~leaf
        if not inner.any():
            break
        h = size[inner] // 2
        n2 = h - h % 8
        off = np.stack([off[inner], off[inner] + n2], axis=1).ravel()
        size = np.stack([n2, size[inner] - n2], axis=1).ravel()
    below = None
    for off, size, leaf in reversed(levels):
        val = np.empty((rows.shape[0], len(off)))
        if leaf.any():
            val[:, leaf] = _leaf_sums(rows, off[leaf], size[leaf])
        if below is not None:
            val[:, ~leaf] = below[:, 0::2] + below[:, 1::2]
        below = val
    return below[:, 0]


def pairwise_sum(a):
    """np.add.reduce of a float64 column: 0.0 + the pairwise tree."""
    return np.float64(0.0) + pairwise_rows(np.asarray(a, dtype=np.float64)[None, :])[0]


def chunked_sum(a, chunk=None):
    """np.add.reduce(a, dtype=float64) of an int64 / bool column: the cast runs through the ufunc buffer, so the
    pairwise tree covers one chunk of np.getbufsize() elements, and the chunk sums are added in order."""
    chunk = int(np.getbufsize()) if chunk is None else int(chunk)
    x = np.asarray(a).astype(np.float64)
    n = x.size
    full = n // chunk
    sums = list(pairwise_rows(x[:full * chunk].reshape(full, chunk))) if full else []
    if n % chunk:
        sums.append(pairwise_rows(x[full * chunk:][None, :])[0])
    total = np.float64(0.0)
    for s in sums:
        total = total + s
    return total


def mean(a):
    a = np.asarray(a)
    s = pairwise_sum(a) if a.dtype == np.float64 else chunked_sum(a)
    with np.errstate(all="ignore"):
        return s / np.float64(a.size)


def var(a, ddof=0):
    a = np.asarray(a)
    m = mean(a)
    x = a.astype(np.float64) - m
    x = x * x
    with np.errstate(all="ignore"):
        return pairwise_sum(x) / np.float64(max(a.size - ddof, 0))


def std(a, ddof=0):
    with np.errstate(all="ignore"):
        return np.sqrt(var(a, ddof))
