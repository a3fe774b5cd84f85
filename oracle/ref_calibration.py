"""numpy restatement of the calibration table of stag_calibration (csrc/mc_predictive.cu, include/stag_b200.h).

Every entry is an integer: a count, or a sum of fx(x) = rint(x * 2^32) (half to even).  The one float sum, the
Categorical row sum s, is taken in the kernel's order: lane l of a warp adds classes l, l+32, ... in order, then an xor
butterfly over offsets 16, 8, 4, 2, 1.  Bin edges are the doubles i * (1.0 / B), the values np.linspace(0, 1, B + 1)
produces (not i / B), and bin(x) is the number of interior edges strictly below x: sklearn's
calibration_curve(strategy="uniform").  ``table_fn`` has the signature of ``stag_b200.ops.calibration_table`` so tests can
put it in place of the kernel.
"""
import numpy as np
import torch

ONE = 2.0 ** 32
HEAD = 6
KINDS = {"categorical": 0, "bernoulli": 1}


def table_len(C, B):
    return HEAD + 3 * B + 3 * C * B


def edges(B):
    """All B + 1 bin edges."""
    return np.linspace(0.0, 1.0, B + 1)


def bin_of(x, B):
    return np.searchsorted(np.arange(1, B) * (1.0 / B), x, side="left")


def fx(x):
    return np.rint(np.asarray(x, dtype=np.float64) * ONE).astype(np.int64)


def row_sum(m):
    """Row sums of m [N, C] float64 in the kernel's order."""
    N, C = m.shape
    K = (C + 31) // 32
    lanes = np.zeros((N, K * 32))
    lanes[:, :C] = m
    lanes = lanes.reshape(N, K, 32)
    acc = np.zeros((N, 32))
    for k in range(K):
        acc = acc + lanes[:, k, :]
    for o in (16, 8, 4, 2, 1):
        acc = acc + acc[:, np.arange(32) ^ o]
    return acc[:, 0]


def table(probs, y, kind="categorical", n_bins=15, mask=None):
    """int64 numpy table of float32 probs [N, C] with labels y (int [N] or float32 [N, C]) and an optional mask [N]."""
    kind = KINDS.get(kind, kind)
    m = np.asarray(probs, dtype=np.float32).astype(np.float64)
    N, C = m.shape
    B = int(n_bins)
    t = np.zeros(table_len(C, B), dtype=np.int64)
    top = t[HEAD:HEAD + 3 * B].reshape(3, B)
    cls = t[HEAD + 3 * B:].reshape(3, C, B)
    rows = np.ones(N, bool) if mask is None else np.asarray(mask).astype(bool)
    m = m[rows]
    cc = np.broadcast_to(np.arange(C), m.shape)
    if kind == 0:
        yy = np.asarray(y, dtype=np.int64)[rows]
        s = row_sum(m)
        bad = (~np.isfinite(m) | (m < 0)).any(1) | (s == 0) | (yy < 0) | (yy >= C)
        m, s, yy, cc = m[~bad], s[~bad], yy[~bad], cc[~bad]
        q = m / s[:, None]
        k = np.argmax(m, axis=1)
        conf = q[np.arange(len(q)), k]
        ok = (k == yy).astype(np.int64)
        onehot = cc == yy[:, None]
        t[:3] = [len(q), int(bad.sum()), ok.sum()]
        t[5] = fx((q - onehot) ** 2).sum()
        b = bin_of(conf, B)
        np.add.at(top[0], b, 1)
        np.add.at(top[1], b, fx(conf))
        np.add.at(top[2], b, ok)
        label = onehot.astype(np.int64)
        val = q
    else:
        yv = np.asarray(y, dtype=np.float32).astype(np.float64)[rows]
        bad = ((np.isnan(m) | (m < 0) | (m > 1)) | (np.isnan(yv) | (yv < 0) | (yv > 1))).any(1)
        m, yv, cc = m[~bad], yv[~bad], cc[~bad]
        pos, tru = m > 0.5, yv > 0.5
        t[:6] = [len(m), int(bad.sum()), (pos & tru).sum(), (pos & ~tru).sum(), (~pos & tru).sum(),
                 fx((m - yv) ** 2).sum()]
        label = fx(yv)
        val = m
    b = bin_of(val, B)
    np.add.at(cls[0], (cc, b), 1)
    np.add.at(cls[1], (cc, b), fx(val))
    np.add.at(cls[2], (cc, b), label)
    return t


def table_fn(probs, y, kind="categorical", n_bins=15, mask=None, out=None):
    """``ops.calibration_table`` in numpy: an int64 torch tensor (CPU, or ``out``'s device when it adds into ``out``)."""
    def host(a):
        return None if a is None else (a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a))
    t = torch.from_numpy(table(host(probs), host(y), kind, n_bins, host(mask)))
    if out is None:
        return t
    out += t.to(out.device)
    return out
