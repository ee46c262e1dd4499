"""numpy / scipy restatement of the chain agreement metrics (bisbm_chain_agreement), used by the agreement tests."""
import numpy as np
from scipy.optimize import linear_sum_assignment


def table(x, y):
    """contingency table n_ij of two label vectors (any non-negative ids)"""
    x = np.asarray(x, dtype=np.int64)
    y = np.asarray(y, dtype=np.int64)
    _, xi = np.unique(x, return_inverse=True)
    _, yi = np.unique(y, return_inverse=True)
    t = np.zeros((xi.max(initial=-1) + 1, yi.max(initial=-1) + 1), dtype=np.int64)
    np.add.at(t, (xi, yi), 1)
    return t


def metrics(x, y):
    """{"vi", "nmi", "ari", "overlap"} of two partitions of the same n nodes; overlap = maximal matched nodes / n"""
    t = table(x, y)
    n = int(t.sum())
    a, b = t.sum(1), t.sum(0)

    def xlogx(v):
        v = v[v > 0].astype(np.float64)
        return float((v * np.log(v)).sum())

    def pairs(v):
        v = v.astype(np.int64)
        return int((v * (v - 1) // 2).sum())

    s_xy, s_x, s_y = xlogx(t.ravel()), xlogx(a), xlogx(b)
    ln = np.log(n)
    hx = 0.0 if len(a) <= 1 else ln - s_x / n
    hy = 0.0 if len(b) <= 1 else ln - s_y / n
    mi = 0.0 if len(a) <= 1 or len(b) <= 1 else ln + (s_xy - s_x - s_y) / n
    nmi = 1.0 if hx + hy == 0 else 2 * mi / (hx + hy)
    p_xy, p_x, p_y, n2 = pairs(t.ravel()), pairs(a), pairs(b), n * (n - 1) // 2
    expected = p_x * p_y / n2 if n2 else 0.0
    denom = 0.5 * (p_x + p_y) - expected
    ari = 1.0 if denom == 0 else (p_xy - expected) / denom
    r, c = linear_sum_assignment(-t)
    return {"vi": (s_x + s_y - 2 * s_xy) / n, "nmi": nmi, "ari": ari, "overlap": int(t[r, c].sum()) / n,
            "matched": int(t[r, c].sum())}


def slots(x, y, na):
    """metrics of two global-id label vectors per slot: type a, type b, and the whole partition (type b ids offset so
    the two types never share an id)"""
    x = np.asarray(x, dtype=np.int64)
    y = np.asarray(y, dtype=np.int64)
    big = int(max(x.max(), y.max())) + 1
    xw = np.where(np.arange(len(x)) < na, x, x + big)
    yw = np.where(np.arange(len(y)) < na, y, y + big)
    return [metrics(x[:na], y[:na]), metrics(x[na:], y[na:]), metrics(xw, yw)]
