"""The host half of probabilit_b200.stats.histogram / histogram_bin_edges / min / max / ptp (no GPU): NumPy's bin-edge
logic restated in stats._edges_plan, run with the device primitives replaced by their NumPy equivalents, equals
np.histogram_bin_edges; the edge-array counts rebuilt from cell counts equal np.histogram; and every invalid argument
raises NumPy's exception before any library call."""
import warnings

import numpy as np
import pytest

from probabilit_b200 import _lib, stats
from probabilit_b200.modeling import Distribution

ESTIMATORS = ["auto", "fd", "rice", "scott", "sqrt", "sturges"]
SIZES = list(range(1, 41)) + list(range(41, 320, 23)) + [1_000_000]


def _keep(a, keep):
    """The kernels' keep_value: each edge compared in its own type."""
    lo_cmp, hi_cmp, lo_f, hi_f, lo_i, hi_i = keep
    lo = a.astype(np.int64) >= lo_i if lo_cmp == stats._CMP_I64 else a.astype(np.float64) >= lo_f
    hi = a.astype(np.int64) <= hi_i if hi_cmp == stats._CMP_I64 else a.astype(np.float64) <= hi_f
    return lo & hi


class HostPrims:
    """stats._Device's primitives on host arrays (bool data already cast to uint8, as NumPy bins it)."""

    def minmax(self, cols):
        return [(a.min().item(), a.max().item()) for a in cols]

    def compact(self, cols, keeps):
        out = [a[_keep(a, keep)] for a, keep in zip(cols, keeps)]
        return out, [a.size for a in out]

    def std(self, cols):
        return [np.std(a) for a in cols]

    def iqr(self, cols):
        return [np.subtract(*np.percentile(a, [75, 25])) for a in cols]


def _data(dtype, n, rng):
    if dtype == "f8":
        return rng.lognormal(size=n) * 1e3 - rng.normal(size=n) * 1e5
    if dtype == "i8":  # values beyond 2^53, both signs, with ties
        a = rng.integers(-(2 ** 62), 2 ** 62, size=n, dtype=np.int64)
        a[::3] = 2 ** 53 + 1
        return a
    if dtype == "i8small":
        return rng.integers(-20, 20, size=n, dtype=np.int64)
    if dtype == "i8near":  # spaced by 1 around 2^53, where float64 rounds to even
        return 2 ** 53 + rng.integers(-12, 12, size=n, dtype=np.int64)
    return rng.random(n) < 0.3


def _ranges(a):
    if a.dtype == np.bool_:
        return [None, (0, 1), (0.5, 1.0), (1, 1), (-2, 0)]
    lo, q1, q3, hi = np.quantile(a.astype(np.float64), [0, 0.25, 0.75, 1])
    out = [None, (float(lo) - 1.0, float(hi) + 1.0), (float(q1), float(q3)), (int(q1), int(q3)), (int(hi) + 5, int(hi) + 9)]
    if a.dtype == np.int64:
        out.append((int(a.min()), int(a.max())))  # Python ints: exact int64 comparisons
        out.append((np.int64(a.min()), float(q3)))
        out += _mixed_ranges(a)
    return out


def _mixed_ranges(a):
    """An int edge and a float edge, each cutting the data (the int edge odd: above 2^53 float64 rounds it away)."""
    lo, hi = int(np.quantile(a, 0.3)) | 1, int(np.quantile(a, 0.8)) | 1
    return [(lo, float(hi)), (float(lo), hi), (np.int64(lo), float(hi)), (float(lo), np.int64(hi))]


def _plan_edges(a, bins, range):
    host = a.astype(np.uint8) if a.dtype == np.bool_ else a
    (edges, _), = stats._edges_plan(HostPrims(), [host], [host.dtype], a.size, bins, range)
    return edges


def _check_edges(a, bins, range):
    try:
        want = np.histogram_bin_edges(a, bins, range)
    except ValueError as e:
        with pytest.raises(ValueError) as got:  # NumPy's checks on a prototype first, as stats does
            np.histogram_bin_edges(np.zeros(2, a.dtype), bins, range)
            _plan_edges(a, bins, range)
        assert str(got.value) == str(e)
        return
    got = _plan_edges(a, bins, range)
    assert got.dtype == want.dtype and got.shape == want.shape, (a.dtype, a.size, range, bins)
    np.testing.assert_array_equal(got, want, err_msg=f"{a.dtype} n={a.size} range={range} bins={bins}")


@pytest.mark.parametrize("dtype", ["f8", "i8", "i8small", "i8near", "bool"])
def test_bin_edges_restatement_equals_numpy(dtype):
    rng = np.random.default_rng(5)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for n in SIZES:
            a = _data(dtype, n, rng)
            for range in _ranges(a) if n < 1_000_000 else [None, _ranges(a)[2]]:
                for bins in ESTIMATORS + [1, 10, 257]:
                    _check_edges(a, bins, range)


def test_constant_columns_and_ties():
    for a in (np.full(50, 3.25), np.full(7, -(2 ** 62), dtype=np.int64), np.ones(9, dtype=bool),
              np.array([2 ** 53 + 1, 2 ** 53 + 3], dtype=np.int64)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for bins in ESTIMATORS + [1, 3]:
                _check_edges(a, bins, None)


def _uniform_counts(a, edges, uniform):
    """The equal-bin kernel (histogram_kernel, PBL_HIST_UNIFORM) in NumPy, from the spec the host builds."""
    keep, first, denom, nbins, table = stats._uniform_spec(a.dtype, edges, uniform)
    x = a[_keep(a, keep)].astype(np.float64)
    i = (((x - first) / denom) * nbins).astype(np.intp)
    i[i == nbins] -= 1
    assert i.min(initial=0) >= 0 and i.max(initial=0) < nbins  # (no case here leaves the table)
    i[x < table[i]] -= 1
    i[(x >= table[i + 1]) & (i != nbins - 1)] += 1
    return np.bincount(i, minlength=nbins)


@pytest.mark.parametrize("dtype", ["f8", "i8", "i8near"])
def test_uniform_counts_emulation_equals_numpy(dtype):
    rng = np.random.default_rng(8)
    for n in (1, 7, 300, 5000):
        a = _data(dtype, n, rng)
        for range in _ranges(a):
            for bins in (1, 3, 10, 257, "auto", "fd"):
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    try:
                        want, want_edges = np.histogram(a, bins, range)
                    except ValueError:
                        continue
                    (edges, uniform), = stats._edges_plan(HostPrims(), [a], [a.dtype], n, bins, range)
                np.testing.assert_array_equal(edges, want_edges)
                np.testing.assert_array_equal(_uniform_counts(a, edges, uniform), want,
                                              err_msg=f"{dtype} n={n} range={range} bins={bins}")


def test_mixed_int_float_range_beyond_2_53():
    """NumPy compares an int64 array with an int edge exactly and with a float edge in float64, one edge at a time."""
    a = np.array([2 ** 53, 2 ** 53 + 2, 2 ** 53 + 6], dtype=np.int64)
    for range in ((2 ** 53 + 1, 2.0 ** 53 + 8), (np.int64(2 ** 53 + 1), 2.0 ** 53 + 8)):
        want, want_edges = np.histogram(a, bins=2, range=range)
        (edges, uniform), = stats._edges_plan(HostPrims(), [a], [a.dtype], a.size, 2, range)
        np.testing.assert_array_equal(_uniform_counts(a, edges, uniform), want)  # [1, 1]: 2^53 is not kept
        for bins in ("sqrt", "auto"):
            _check_edges(a, bins, range)


def _cells(a, table, common):
    """The device's cell counts (PBL_HIST_EDGES) of `a`, in NumPy."""
    v = a.astype(common)
    m = table.size
    cells = np.zeros(2 * m + 2, dtype=np.intp)
    nan = np.isnan(v) if common == np.float64 else np.zeros(v.size, bool)
    lo = np.searchsorted(table, v[~nan], side="left")
    eq = (lo < m) & (table[np.minimum(lo, m - 1)] == v[~nan])
    np.add.at(cells, 2 * lo + eq, 1)
    cells[-1] = nan.sum()
    return cells


@pytest.mark.parametrize("edges", [[0.0, 1.0, 2.5, 7.0], [0, np.nan, 3], [np.nan, 1.0], [1.0, np.nan], [-1, 0, 0, 5],
                                   [np.nan, np.nan], [-0.0, 0.0, 1.0], np.array([2 ** 53 + 2, 2 ** 53 + 4], np.int64),
                                   [2.0 ** 53, 2.0 ** 53 + 4]])
def test_edge_array_counts_from_cells(edges):
    rng = np.random.default_rng(1)
    data = [np.array([1.0, 2, 3]), np.concatenate([rng.normal(size=200), [np.nan, -0.0, 0.0, 1.0, 2.5, np.inf]]),
            np.array([2 ** 53 + 1, 2 ** 53 + 3, 2 ** 53 + 4, -5, 0], dtype=np.int64)]
    edges = np.asarray(edges)
    for a in data:
        common, table = stats._edge_table(a.dtype, edges)
        cum = stats._cumulative(_cells(a, table, common), table, edges, common, a.size)
        want, _ = np.histogram(a, bins=edges)
        got = np.diff(cum)
        assert got.dtype == want.dtype
        np.testing.assert_array_equal(got, want, err_msg=f"{a} {edges}")


def _host_node(values):
    node = Distribution("norm")
    node.samples_ = values
    return node


def test_invalid_arguments_raise_numpy_types_without_gpu(monkeypatch):
    def no_gpu():
        raise AssertionError("a library call before the arguments were checked")

    monkeypatch.setattr(_lib, "require_gpu", no_gpu)
    x = _host_node(np.arange(10.0))
    i = _host_node(np.arange(10))
    b = _host_node(np.arange(10) % 2 == 0)
    for fn in (stats.histogram, stats.histogram_bin_edges):
        with pytest.raises(ValueError, match="is not a valid estimator"):
            fn(x, bins="bogus")
        with pytest.raises(ValueError, match="must increase monotonically"):
            fn(x, bins=[0, 2, 1])
        with pytest.raises(ValueError, match="must be 1d"):
            fn(x, bins=[[0, 1], [2, 3]])
        with pytest.raises(ValueError, match="must be positive"):
            fn(x, bins=0)
        with pytest.raises(TypeError, match="must be an integer, a string, or an array"):
            fn(x, bins=2.5)
        with pytest.raises(ValueError, match="max must be larger than min"):
            fn(x, range=(3, 1))
        with pytest.raises(ValueError, match="is not finite"):
            fn(x, range=(0, np.inf))
        with pytest.raises(ValueError, match="is not finite"):
            fn(i, bins="auto", range=(np.nan, 1))
        with pytest.raises(NotImplementedError):
            fn(x, weights=np.ones(10))
        for name in ("doane", "stone"):
            with pytest.raises(NotImplementedError):
                fn(x, bins=name)
        with pytest.raises(NotImplementedError):  # float16 edges: NumPy bins in float16
            fn(b, range=(np.float16(0), np.float16(1)))
        with pytest.raises(NotImplementedError):  # uint8 data, uint8 edges: compared as uint8
            fn(b, bins=np.array([0, 1], dtype=np.uint8))
        with pytest.warns(RuntimeWarning, match="Converting input from bool"):
            with pytest.raises(NotImplementedError):
                fn(b, weights=None, bins="stone")
        with pytest.raises(TypeError):
            fn(_host_node(None))
    with pytest.raises(TypeError):
        stats.ptp(b)
    for fn in (stats.min, stats.max):
        for kw in ({"axis": 0}, {"out": np.empty(())}, {"keepdims": True}, {"initial": 0}, {"where": True}):
            with pytest.raises(NotImplementedError):
                fn(x, **kw)
    for kw in ({"axis": 0}, {"out": np.empty(())}, {"keepdims": False}):
        with pytest.raises(NotImplementedError):
            stats.ptp(x, **kw)


def test_empty_columns_follow_numpy(monkeypatch):
    def no_gpu():
        raise AssertionError("an empty column needs no device")

    monkeypatch.setattr(_lib, "require_gpu", no_gpu)
    for values in (np.empty(0), np.empty(0, dtype=np.int64)):
        x = _host_node(values)
        for fn, npfn in ((stats.min, np.min), (stats.max, np.max), (stats.ptp, np.ptp)):
            with pytest.raises(ValueError) as got:
                fn(x)
            with pytest.raises(ValueError) as want:
                npfn(values)
            assert str(got.value) == str(want.value)
        for bins in (10, "auto", [0, 1, 2]):
            h, e = stats.histogram(x, bins=bins)
            wh, we = np.histogram(values, bins=bins)
            assert h.dtype == wh.dtype and e.dtype == we.dtype
            np.testing.assert_array_equal(h, wh)
            np.testing.assert_array_equal(e, we)
