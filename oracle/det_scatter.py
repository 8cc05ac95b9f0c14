"""numpy restatement of the deterministic hash-grid gradient (mipsfusion_b200/csrc/det_kernels.cu).

Every contribution c = fl(w * dy) (w the trilinear corner weight of oracle.hashgrid.grid_corners, dy a feature gradient) to the
gradient float e is rounded to the integer round(c * 2^s), s = 188 - h - E[e], where E[e] is the largest effective binary
exponent max(biased exponent, 1) among e's non-zero contributions and h = ceil(log2(8 n + 1)) (n the points of the launch).
The int64 sums are converted to fp32 once (the integer rounded to fp32, then scaled by 2^-s in fp64 and rounded to fp32, which
only rounds again for a subnormal result) and added to the incoming gradient with one fp32 addition.  Non-finite contributions
make the sum +Inf, -Inf or NaN as fp32 arithmetic would.  Zero contributions are skipped."""
import numpy as np
import torch

from . import hashgrid as hg

MAX_H = 35          # det_kernels.cu MF_DET_MAX_H: at most 2^32 - 1 points per launch


def headroom(n):
    """h = ceil(log2(8 n + 1)); raises for more points than one launch accepts."""
    h = int(8 * n).bit_length()
    if n < 1 or n >= 1 << 32 or h > MAX_H:
        raise ValueError(f"{n} points exceed the fixed-point headroom")
    return h


def contributions(x, dy, table):
    """(e, c): flat gradient index and fp32 contribution of every (point, level, corner, feature), zeros included."""
    x = np.ascontiguousarray(x, dtype=np.float32); dy = np.ascontiguousarray(dy, dtype=np.float32)
    idx, w, _ = hg.grid_corners(torch.from_numpy(x), table)
    idx = idx.numpy(); w = w.numpy().astype(np.float32)
    L = table["n_levels"]
    es, cs = [], []
    for l in range(L):
        off = int(table["offset"][l])
        for c in range(8):
            for k in range(2):
                es.append(2 * (off + idx[:, l, c]) + k)
                cs.append((w[:, l, c] * dy[:, 2 * l + k]).astype(np.float32))
    return np.concatenate(es).astype(np.int64), np.concatenate(cs).astype(np.float32)


def fixed_point_sum(e, c, h, grad):
    """grad (fp32, modified copy returned) += the pre-rounded fixed-point sums of the contributions (e, c); also returns the
    int64 accumulators and exponents of the touched entries (for the accuracy checks)."""
    grad = np.array(grad, dtype=np.float32, copy=True)
    P = grad.shape[0]
    keep = c != 0
    e, c = e[keep], c[keep]
    bits = c.view(np.uint32)
    be = ((bits >> 23) & 0xFF).astype(np.int64)
    nonfinite = be == 255
    pinf = np.zeros(P, bool); ninf = np.zeros(P, bool); nan = np.zeros(P, bool)
    np.logical_or.at(nan, e[nonfinite], np.isnan(c[nonfinite]))
    np.logical_or.at(pinf, e[nonfinite], c[nonfinite] == np.inf)
    np.logical_or.at(ninf, e[nonfinite], c[nonfinite] == -np.inf)
    fin = ~nonfinite
    E = np.zeros(P, np.int64)
    np.maximum.at(E, e[fin], np.maximum(be[fin], 1))
    s = 188 - h - E[e[fin]]
    q = np.rint(c[fin].astype(np.float64) * np.exp2(s.astype(np.float64))).astype(np.int64)
    acc = np.zeros(P, np.int64)
    np.add.at(acc, e[fin], q)
    touched = np.unique(e)
    flagged = pinf | ninf | nan
    t = touched[~flagged[touched]]
    st = (188 - h - E[t]).astype(np.float64)
    v = (acc[t].astype(np.float32).astype(np.float64) * np.exp2(-st)).astype(np.float32)
    grad[t] = (grad[t] + v).astype(np.float32)
    tf = touched[flagged[touched]]
    vf = np.where(nan[tf] | (pinf[tf] & ninf[tf]), np.float32(np.nan), np.where(pinf[tf], np.float32(np.inf), np.float32(-np.inf)))
    with np.errstate(invalid="ignore"):
        grad[tf] = (grad[tf] + vf.astype(np.float32)).astype(np.float32)
    return grad, acc, E


def det_hashgrid_bwd(x, dy, table, grad=None):
    """grad_grid of mf_hashgrid_bwd in deterministic mode: x (N, 3), dy (N, 2 L) fp32."""
    if grad is None:
        grad = np.zeros(table["n_params"], np.float32)
    e, c = contributions(x, dy, table)
    return fixed_point_sum(e, c, headroom(x.shape[0]), grad)[0]
