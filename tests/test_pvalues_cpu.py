"""Exact p-values of the scan's Float16 score, host side: the forward-DP oracle against enumeration of every window, the
Benjamini-Hochberg q-values and the Sidak form of records.py, and the default background."""
import decimal

import numpy as np
import pytest
import scipy.stats

from motifs_jl_b200 import records
from oracle import pvalue_oracle as po

UNIFORM = np.full(4, 0.25)
SKEWED = np.array([0.35, 0.1, 0.2, 0.35])


def _edge_pwms():
    rng = np.random.default_rng(3)
    out = {"m1": rng.normal(0, 2, (4, 1)), "random7": rng.normal(0, 2, (4, 7)), "zero_col": rng.normal(0, 1, (4, 6))}
    out["zero_col"][:, 2] = 0
    ninf = rng.normal(0, 1, (4, 5))
    ninf[1, 3] = -np.inf                                      # the rest of column 3 becomes NaN (Inf * 0)
    out["neg_inf"] = ninf
    big = rng.normal(0, 1, (4, 6))
    big[0, 1], big[3, 2], big[2, 4], big[1, 0] = 60000, 60000, -60000, -60000   # sums overflow to +-Inf, Inf + -Inf = NaN
    out["overflow"] = big
    out["fine8"] = np.round(rng.normal(0, 1, (4, 8)) * 8) / 8   # many ties
    return {k: v.astype(np.float16) for k, v in out.items()}


@pytest.mark.parametrize("bg", [UNIFORM, SKEWED], ids=["uniform", "skewed"])
@pytest.mark.parametrize("name", sorted(_edge_pwms()))
def test_oracle_equals_enumeration(name, bg):
    pwm = _edge_pwms()[name]
    for tab in po.eff_tables(pwm):
        S, B = po.survival(tab, bg), po.brute_survival(tab, bg)
        nan = np.isnan(B)
        assert np.array_equal(np.isnan(S), nan)
        assert np.all(S[~nan][B[~nan] == 0] == 0)
        pos = ~nan & (B > 0)
        assert np.max(np.abs(S[pos] - B[pos]) / B[pos]) <= 1e-13
        # -0 and +0 share their value; S is non-increasing in value order
        assert S[0x8000] == S[0]
        order = np.argsort(po.rank(np.arange(65536)[~nan]), kind="stable")
        assert np.all(np.diff(S[~nan][order]) <= 0)


def test_nan_mass_is_excluded():
    pwm = _edge_pwms()["neg_inf"]
    tab, _ = po.eff_tables(pwm)
    S = po.survival(tab, UNIFORM)
    assert np.isclose(S[0xFC00], 0.25)                         # only base C of column 3 is not NaN; it gives -Inf
    assert S[0x0000] == 0.0


@pytest.mark.parametrize("n_tests,n", [(1000, 0), (1000, 1), (5000, 40), (200, 200)])
def test_bh_qvalues_equal_scipy(n_tests, n):
    rng = np.random.default_rng(n_tests + n)
    p = np.sort(rng.uniform(0, 1e-3, n))[rng.permutation(n)]
    p[: n // 4] = p[n // 4: 2 * (n // 4)]                       # ties
    q = records.bh_qvalues(p, n_tests)
    full = scipy.stats.false_discovery_control(np.concatenate([p, np.ones(n_tests - n)]))[:n]
    assert np.allclose(q, full, rtol=1e-12, atol=0)


def test_sidak():
    p = np.array([1e-12, 1e-6, 1e-3, 0.1, 0.5, 1.0, 0.0])
    n = np.array([10, 1000, 500, 3, 7, 4, 9])
    got = records.sidak(p, n)
    direct = 1 - (1 - p) ** n
    ok = p >= 1e-3                                             # where 1 - (1 - p)^n is stable
    assert np.allclose(got[ok], direct[ok], rtol=1e-12)
    with decimal.localcontext() as c:                          # everywhere: against 50-digit arithmetic
        c.prec = 50
        exact = np.array([float(1 - (1 - decimal.Decimal(float(x))) ** int(k)) for x, k in zip(p, n)])
    assert np.allclose(got, exact, rtol=1e-14, atol=0)
    assert got[-1] == 0.0 and got[-2] == 1.0


def test_base_background():
    bases = np.frombuffer(b"AAAACCGT" + b"ACGTTT", np.uint8).copy()
    rec = records.Records(["a", "b"], np.array([8, 6]), np.array([0, 1]), np.array([0, 0]), np.array([8, 6]), bases)
    bg = records.base_background(rec)
    n = np.array([5, 3, 2, 4], float)                          # A C G T
    n = n + n[::-1]
    assert np.allclose(bg, n / n.sum()) and bg[0] == bg[3] and bg[1] == bg[2] and np.isclose(bg.sum(), 1)
    empty = records.Records([], np.zeros(0, np.int64), *(np.zeros(0, np.int64),) * 3, np.zeros(0, np.uint8))
    with pytest.raises(ValueError):
        records.base_background(empty)
