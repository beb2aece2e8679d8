"""Numpy restatement of the k-NN contract of include/irt_b200.h (irt_nnset_knn): the distance summed left to right
with every operation rounded on its own, and the k nearest by (distance, index).  Used as the reference of
tests/test_gpu_knn.py and as the device stand-in of tests/test_knn_host_logic.py."""
import numpy as np


def metric_tuple(m):
    """(n_euclid, so2_col, lin_col, w_so2, w_lin) of an irt_b200.Metric or a tuple"""
    if isinstance(m, tuple):
        return m
    return (m.n_euclid, m.so2_col, m.lin_col, m.w_so2, m.w_lin)


def distances(rows, q, metric):
    """d(q, row) for every row, in the contract's order of operations"""
    ne, so2, lin, w_so2, w_lin = metric_tuple(metric)
    rows = np.asarray(rows, dtype=np.float64).reshape(len(rows), -1)
    s = np.zeros(len(rows))
    for j in range(ne):
        t = q[j] - rows[:, j]
        s = s + t * t
    d = np.sqrt(s)
    if so2 != -1:
        dr = np.abs(q[so2] - rows[:, so2])
        d = d + w_so2 * np.where(dr > np.pi, 2.0 * np.pi - dr, dr)
    if lin != -1:
        d = d + w_lin * np.abs(q[lin] - rows[:, lin])
    return d


def knn(rows, queries, metric, k, bound=np.inf, exclude=None):
    """(idx int64[m][k], dist float64[m][k]) with -1 / inf past the last hit; exclude: None or bool[n]"""
    rows = np.asarray(rows, dtype=np.float64)
    queries = np.asarray(queries, dtype=np.float64)
    queries = queries.reshape(-1, queries.shape[-1])
    m, n = len(queries), len(rows)
    idx = np.full((m, k), -1, dtype=np.int64)
    dist = np.full((m, k), np.inf)
    if n == 0:
        return idx, dist
    keep = np.ones(n, dtype=bool) if exclude is None else ~np.asarray(exclude, dtype=bool)[:n]
    for i, q in enumerate(queries):
        d = distances(rows, q, metric)
        with np.errstate(invalid="ignore"):
            ok = keep & np.isfinite(d) & (d <= bound)
        ids = np.nonzero(ok)[0]
        if len(ids) > k:      # every item at or below the k-th smallest distance, ties included
            ids = ids[d[ids] <= np.partition(d[ids], k - 1)[k - 1]]
        order = ids[np.lexsort((ids, d[ids]))][:k]
        idx[i, :len(order)] = order
        dist[i, :len(order)] = d[order]
    return idx, dist


class NumpyNearestSet:
    """host stand-in of irt_b200.NearestSet with the same methods; counts what reaches the "device" """

    def __init__(self, ctx, dim, metric):
        self.dim, self.metric = int(dim), metric_tuple(metric)
        self.rows = np.zeros((0, self.dim))
        self.appended = self.clears = self.queries = 0

    def size(self):
        return len(self.rows)

    def append(self, rows):
        rows = np.ascontiguousarray(rows, dtype=np.float64).reshape(-1, self.dim)
        self.rows = np.concatenate([self.rows, rows])
        self.appended += len(rows)

    def clear(self):
        self.rows = np.zeros((0, self.dim))
        self.clears += 1

    def knn(self, queries, k, bound=np.inf, exclude=None):
        self.queries += len(np.asarray(queries).reshape(-1, self.dim))
        if exclude is not None:
            exclude = np.asarray(exclude)
            assert exclude.dtype == bool and len(exclude) == len(self.rows), "mask must cover the set exactly"
        return knn(self.rows, queries, self.metric, k, bound, exclude)
