"""CPU checks of the deterministic hash-grid gradient's arithmetic (oracle/det_scatter.py, restating det_kernels.cu):
order independence, the accuracy bound of DESIGN §4 (Deterministic mode), the special values and the headroom."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import det_scatter as ds
from oracle import hashgrid as hg


def _batch(n, seed, T=12):
    rng = np.random.default_rng(seed)
    table = hg.level_table(T)
    x = rng.uniform(-0.05, 1.05, size=(n, 3)).astype(np.float32)            # also outside [0, 1]: wrapping cells
    dy = (rng.standard_normal((n, 32)) * np.exp2(rng.integers(-12, 6, size=(n, 32)))).astype(np.float32)
    dy[rng.random((n, 32)) < 0.1] = 0.0
    return table, x, dy


def test_shuffled_contributions_give_identical_bits():
    table, x, dy = _batch(600, 1)
    e, c = ds.contributions(x, dy, table)
    h = ds.headroom(600)
    g0 = np.random.default_rng(2).standard_normal(table["n_params"]).astype(np.float32)
    ref = ds.fixed_point_sum(e, c, h, g0)[0]
    rng = np.random.default_rng(3)
    for _ in range(3):
        p = rng.permutation(e.shape[0])
        assert np.array_equal(ds.fixed_point_sum(e[p], c[p], h, g0)[0].view(np.uint32), ref.view(np.uint32))
    perm = rng.permutation(600)                                              # point order, end to end
    assert np.array_equal(ds.det_hashgrid_bwd(x[perm], dy[perm], table).view(np.uint32),
                          ds.det_hashgrid_bwd(x, dy, table).view(np.uint32))


def test_error_against_exact_sum_within_bound():
    """|acc 2^-s - exact| <= n_e 2^(-s-1) <= n_e 2^(h-62) max|c|, then one fp32 rounding of the sum (DESIGN §4)."""
    table, x, dy = _batch(300, 4)
    e, c = ds.contributions(x, dy, table)
    h = ds.headroom(300)
    zero = np.zeros(table["n_params"], np.float32)
    got, acc, E = ds.fixed_point_sum(e, c, h, zero)
    keep = c != 0
    e, c = e[keep], c[keep]
    order = np.argsort(e, kind="stable")
    e, c = e[order], c[order]
    starts = np.flatnonzero(np.r_[True, e[1:] != e[:-1]])
    ends = np.r_[starts[1:], e.shape[0]]
    err_fixed = err_fp32 = 0.0
    for a, b in zip(starts, ends):
        k = int(e[a])
        exact = sum((Fraction(float(v)) for v in c[a:b]), Fraction(0))
        s = 188 - h - int(E[k])
        fixed = Fraction(int(acc[k])) / Fraction(2) ** s if s >= 0 else Fraction(int(acc[k])) * Fraction(2) ** (-s)
        n_e = b - a
        quantum_err = abs(fixed - exact)
        assert quantum_err <= Fraction(n_e, 2) / (Fraction(2) ** s if s >= 0 else Fraction(1, 2 ** (-s)))
        assert quantum_err <= n_e * Fraction(2) ** (h - 62) * Fraction(float(np.max(np.abs(c[a:b]))))
        tol = float(quantum_err) + abs(float(exact)) * 2.0 ** -24 + 2.0 ** -150
        assert abs(float(got[k]) - float(exact)) <= tol * (1 + 1e-12), (k, float(got[k]), float(exact))
        if n_e >= 3:                 # the fp32 sum of the same contributions in index order, over the entries where order matters
            naive = np.float32(0)
            for v in c[a:b]:
                naive = np.float32(naive + v)
            err_fp32 += abs(Fraction(float(naive)) - exact)
            err_fixed += abs(Fraction(float(got[k])) - exact)
    # summed over those entries the fixed-point result is at least as close to the exact sums as a sequential fp32 sum
    assert 0 < err_fp32 and err_fixed <= err_fp32, (float(err_fixed), float(err_fp32))


def test_special_values():
    P = 8
    h = ds.headroom(10)
    g = np.zeros(P, np.float32)
    g[5] = np.float32(-0.0)
    e = np.array([0, 0, 1, 1, 2, 2, 3, 4, 4, 6, 6, 7], np.int64)
    tiny = np.float32(1e-45)                                                 # the smallest subnormal
    c = np.array([np.inf, 1.0, -np.inf, 2.0, np.inf, -np.inf, np.nan, tiny, tiny, 3.0, -3.0, 0.0], np.float32)
    out = ds.fixed_point_sum(e, c, h, g)[0]
    assert out[0] == np.inf and out[1] == -np.inf and np.isnan(out[2]) and np.isnan(out[3])
    assert out[4] == np.float32(2 * tiny)                                     # subnormals are summed exactly
    assert out[5].view(np.uint32) == np.float32(-0.0).view(np.uint32)        # untouched: stays -0
    assert out[6] == 0.0                                                     # exact cancellation
    assert out[7] == 0.0                                                     # zero contributions are skipped
    # subnormal and normal contributions to one entry: the result is the correctly rounded exact sum here
    e2 = np.zeros(3, np.int64)
    c2 = np.array([np.float32(2.0 ** -130), np.float32(1.5 * 2 ** -140), np.float32(-2.0 ** -131)], np.float32)
    out2 = ds.fixed_point_sum(e2, c2, h, np.zeros(1, np.float32))[0]
    assert out2[0] == np.float32(2.0 ** -131 + 1.5 * 2 ** -140)


def test_headroom_has_no_overflow_at_the_largest_accepted_n():
    n_max = (1 << 32) - 1
    h = ds.headroom(n_max)
    assert h <= ds.MAX_H
    # every contribution of an entry is below 2^(62 - h) after scaling; at most 8 n of them reach one entry
    assert 8 * n_max * 2 ** (62 - h) < 2 ** 63
    with pytest.raises(ValueError):
        ds.headroom(n_max + 1)
    for n in (1, 2, 87_000, 1 << 20, (1 << 31) - 1):
        h = ds.headroom(n)
        assert 2 ** h >= 8 * n + 1 > 2 ** (h - 1)
        assert 8 * n * 2 ** (62 - h) < 2 ** 63
