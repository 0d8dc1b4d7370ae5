"""NumPy's reduction order that the device statistics (probabilit_b200/csrc/stats.cu) reproduce, pinned against
NumPy itself through the restatement in oracle/reductions.py, and the argument checks of probabilit_b200.stats,
which raise NumPy's exception types before any device call (no GPU needed)."""
import warnings

import numpy as np
import pytest

from oracle import reductions as red
from probabilit_b200 import stats
from probabilit_b200.modeling import Distribution

SIZES = list(range(0, 301)) + [8191, 8192, 8193, 1_000_003, 10_000_007]


def _column(dtype, n, rng):
    if dtype == "f8":
        return rng.lognormal(size=n) * 1e3 - rng.normal(size=n) * 1e6
    if dtype == "i8":  # values beyond 2^53, both signs
        return rng.integers(-(2 ** 62), 2 ** 62, size=n, dtype=np.int64)
    return rng.random(n) < 0.3


def _bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


@pytest.mark.parametrize("dtype", ["f8", "i8", "bool"])
def test_restatement_equals_numpy_moments(dtype):
    rng = np.random.default_rng(7)
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        for n in SIZES:
            a = _column(dtype, n, rng)
            assert _bits(red.mean(a)) == _bits(np.mean(a)), (dtype, n)
            ddofs = (0, 1, 2.5) if n <= 300 or n == 8193 or n == 10_000_007 else (0,)
            for ddof in ddofs:
                assert _bits(red.var(a, ddof)) == _bits(np.var(a, ddof=ddof)), (dtype, n, ddof)
                assert _bits(red.std(a, ddof)) == _bits(np.std(a, ddof=ddof)), (dtype, n, ddof)


@pytest.mark.parametrize("n", [1, 5, 8, 200, 8193])
def test_restatement_negative_zero_column(n):
    a = np.full(n, -0.0)
    assert _bits(red.mean(a)) == _bits(np.mean(a))  # +0.0: the reduction starts from 0.0
    assert _bits(red.var(a)) == _bits(np.var(a))


def test_chunk_length_is_a_parameter():
    a = np.arange(20_000, dtype=np.int64) * (2 ** 40 + 3)
    old = np.getbufsize()
    try:
        np.setbufsize(4096)
        assert _bits(red.chunked_sum(a, 4096) / a.size) == _bits(np.mean(a))
    finally:
        np.setbufsize(old)


def _host_node(values):
    node = Distribution("norm")
    node.samples_ = values
    return node


def test_invalid_arguments_raise_numpy_types_without_gpu():
    x = _host_node(np.arange(10.0))
    b = _host_node(np.arange(10) % 2 == 0)
    with pytest.raises(ValueError, match=r"Quantiles must be in the range \[0, 1\]"):
        stats.quantile(x, 1.5)
    with pytest.raises(ValueError, match=r"Quantiles must be in the range \[0, 1\]"):
        stats.quantile(x, [0.5, -0.1])
    with pytest.raises(ValueError, match=r"Percentiles must be in the range \[0, 100\]"):
        stats.percentile(x, 101)
    for method in ("linear", "midpoint"):
        with pytest.raises(TypeError):
            np.quantile(np.arange(10) % 2 == 0, 0.5, method=method)
        with pytest.raises(TypeError):
            stats.quantile(b, 0.5, method=method)
        with pytest.raises(TypeError):
            stats.percentile(b, [10, 90], method=method)
    with pytest.raises(TypeError):
        stats.mean(_host_node(None))
    with pytest.raises(TypeError):
        stats.quantile(_host_node(None), 0.5)
    with pytest.raises(TypeError):
        stats.mean(_host_node(np.array(["a", "b"])))
    with pytest.raises(ValueError):  # not a method NumPy knows
        stats.quantile(x, 0.5, method="bogus")
    with pytest.raises(NotImplementedError):
        stats.quantile(x, 0.5, method="hazen")
    with pytest.raises(NotImplementedError):
        stats.quantile(x, 0.5, weights=np.ones(10))
    with pytest.raises(NotImplementedError):
        stats.percentile(x, 50, axis=0)
    with pytest.raises(NotImplementedError):
        stats.quantile(x, 0.5, out=np.empty(()))
    with pytest.raises(NotImplementedError):
        stats.quantile(x, 0.5, keepdims=True)
    for fn in (stats.mean, stats.var, stats.std):
        with pytest.raises(NotImplementedError):
            fn(x, axis=0)
        with pytest.raises(NotImplementedError):
            fn(x, out=np.empty(()))
        with pytest.raises(NotImplementedError):
            fn(x, keepdims=True)
    with pytest.raises(AttributeError):
        stats.mean(Distribution("norm"))  # never sampled
    with pytest.raises(TypeError):
        stats.mean(np.arange(3.0))  # host arrays are NumPy's job
