"""The host half of probabilit_b200.stats.unique / bincount (no GPU): the assembly of NumPy's results from what the
device returns (runs, first rows, counts, NaN rows and the inverse), fed with a NumPy restatement of those outputs,
equals np.unique / np.bincount; and every invalid argument raises NumPy's exception before any library call."""
import numpy as np
import pytest

from probabilit_b200 import _lib, stats
from probabilit_b200.modeling import Distribution, _Samples


def _device_outputs(a, equal_nan):
    """pbl_stats_unique restated: a stable sort of the values with -0.0 and +0.0 as one key and the NaNs left out;
    per run of equal keys the first element's value (its own sign) and row, and the run length; the NaN rows in row
    order with their bits; the inverse (run ids, NaN rows after them)."""
    f = np.asarray(a).astype(np.float64)
    nan = np.isnan(f)
    rows = np.flatnonzero(~nan)
    order = np.argsort(f[rows], kind="stable")
    srows = rows[order]
    keys = f[srows]
    start = np.ones(keys.size, dtype=bool)
    start[1:] = keys[1:] != keys[:-1]
    first = srows[start]
    counts = np.diff(np.append(np.flatnonzero(start), keys.size))
    nan_rows = np.flatnonzero(nan)
    inverse = np.empty(f.size, dtype=np.int64)
    inverse[srows] = np.cumsum(start) - 1
    inverse[nan_rows] = first.size + (0 if equal_nan else np.arange(nan_rows.size))
    return f[first], first, counts, nan_rows, f[nan_rows].view(np.uint64), inverse


def _host_unique(a, equal_nan, categories=None):
    """stats.unique's host steps on the restated device outputs -> (values, index, inverse, counts)."""
    values, first, counts, nan_rows, nan_bits, inverse = _device_outputs(a, equal_nan)
    if categories is not None:
        values, first, counts, table = stats._merge_categories(categories, values, first, counts, len(a))
        inverse = table[inverse]  # pbl_stats_remap
    dtype = np.asarray(a).dtype if categories is None else categories.dtype
    values, first, counts = stats._assemble(dtype, values, first, counts, nan_rows, nan_bits, equal_nan)
    return values, first, inverse, counts


def _check_unique(a, equal_nan, categories=None):
    got = _host_unique(a, equal_nan, categories)
    data = a if categories is None else categories[a]
    want = np.unique(data, return_index=True, return_inverse=True, return_counts=True, equal_nan=equal_nan)
    assert got[0].dtype == want[0].dtype
    if want[0].dtype == np.float64:  # bit for bit: the sign of zero and the NaN payloads
        np.testing.assert_array_equal(got[0].view(np.int64), want[0].view(np.int64))
    else:
        np.testing.assert_array_equal(got[0], want[0])
    for g, w in zip(got[1:], want[1:]):
        assert g.dtype == np.intp and g.shape == w.shape
        np.testing.assert_array_equal(g, w)


def _nan(sign, payload):
    return np.array([(0xFFF0000000000000 if sign else 0x7FF0000000000000) | payload], dtype=np.uint64).view(np.float64)[0]


def _float_cases(rng):
    special = np.array([0.0, -0.0, np.inf, -np.inf, _nan(0, 1), _nan(1, 2), _nan(0, 1 << 51), _nan(1, 3), 1.5, -1.5])
    return [
        rng.normal(size=1000),
        np.round(rng.normal(size=3000), 1),
        np.where(rng.random(500) < 0.5, -0.0, 0.0),
        np.concatenate([[0.0], np.where(rng.random(200) < 0.5, -0.0, 0.0)]),
        special[rng.integers(0, special.size, 400)],
        np.full(17, np.nan),
        np.full(9, 2.5),
        np.array([3.0]),
    ]


@pytest.mark.parametrize("equal_nan", [True, False])
def test_assembly_equals_numpy_floats(equal_nan):
    for a in _float_cases(np.random.default_rng(1)):
        _check_unique(a, equal_nan)


@pytest.mark.parametrize("equal_nan", [True, False])
def test_assembly_equals_numpy_ints_and_bools(equal_nan):
    rng = np.random.default_rng(2)
    for a in (rng.poisson(3.0, 2000), rng.integers(-2 ** 53, 2 ** 53, 500, dtype=np.int64),
              np.array([-(2 ** 53), 2 ** 53, 0, 2 ** 53], dtype=np.int64), rng.random(300) < 0.3,
              np.ones(5, dtype=bool), np.zeros(1, dtype=np.int64)):
        _check_unique(a, equal_nan)


def test_category_merging():
    rng = np.random.default_rng(3)
    for categories in (np.array(["b", "a", "b", "c"]), np.array(["x", "yy", "x", "x", "a"], dtype=object),
                       np.array([2, 1, 2, 5], dtype=object), np.array(["only"])):
        for n in (1, 7, 1000):
            idx = rng.integers(0, categories.size, n)
            _check_unique(idx, True, categories)
    # a category never sampled is never compared: mixed types fail only if both occur, as in NumPy
    mixed = np.array([1, "a", 2], dtype=object)
    _check_unique(np.array([0, 2, 2, 0]), True, mixed)
    with pytest.raises(TypeError):
        np.unique(mixed[[0, 1]])
    with pytest.raises(TypeError):
        _host_unique(np.array([0, 1, 2]), True, mixed)


def test_bincount_from_runs():
    rng = np.random.default_rng(4)
    for a in (rng.poisson(2.0, 1000), np.array([5]), rng.random(50) < 0.5, np.array([0, 0, 0]),
              np.array([7, 3, 3, 10 ** 6], dtype=np.int64)):
        values, _, _, counts = _host_unique(a, True)
        for minlength in (0, 1, 3, 20, np.int64(12)):
            got = stats._bincount(values, counts, minlength)
            want = np.bincount(a, minlength=minlength)
            assert got.dtype == want.dtype
            np.testing.assert_array_equal(got, want)
    values, _, _, counts = _host_unique(np.array([3, -2, 5]), True)
    with pytest.raises(ValueError) as got:
        stats._bincount(values, counts, 0)
    with pytest.raises(ValueError) as want:
        np.bincount(np.array([3, -2, 5]))
    assert str(got.value) == str(want.value)


def _host_node(values):
    node = Distribution("norm")
    node.samples_ = values
    return node


class _FakeColumns:
    """A device column that is never touched (the calls must fail before any library call)."""

    def __init__(self, n):
        self.n = n

    def column_ptr(self, j):
        return 1 << 40


def _category_node(n, categories):
    node = Distribution("norm")
    node.__dict__["_store"] = _Samples(columns=_FakeColumns(n), index=0, dtype=categories.dtype, categories=categories)
    return node


class _HugeArray:
    def __init__(self, typestr):
        self.__cuda_array_interface__ = {"shape": (2 ** 31,), "typestr": typestr, "data": (1 << 40, False),
                                         "version": 3}


def _no_gpu(monkeypatch):
    def no_gpu():
        raise AssertionError("a library call before the arguments were checked")

    monkeypatch.setattr(_lib, "require_gpu", no_gpu)


def test_invalid_arguments_raise_numpy_types_without_gpu(monkeypatch):
    _no_gpu(monkeypatch)
    x = _host_node(np.arange(10.0))
    i = _host_node(np.arange(10))
    b = _host_node(np.arange(10) % 2 == 0)
    cat = _category_node(10, np.array(["a", "b"]))
    for bad in (dict(axis=0), dict(axis=None, sorted=False)):
        for node in (x, i, cat):
            with pytest.raises(NotImplementedError):
                stats.unique(node, **bad)
    with pytest.raises(NotImplementedError):
        stats.unique(_HugeArray("<f8"), return_counts=True)
    with pytest.raises(NotImplementedError):
        stats.bincount(_HugeArray("<i8"))
    with pytest.raises(NotImplementedError):
        stats.bincount(i, weights=np.ones(10))
    for node in (x, cat):  # float64 and strings cannot be cast to intp safely
        with pytest.raises(TypeError):
            stats.bincount(node)
    for node in (i, b):
        with pytest.raises(ValueError):
            stats.bincount(node, minlength=-1)
        for minlength in (1.5, None):
            with pytest.raises(TypeError):
                stats.bincount(node, minlength=minlength)
    for fn in (stats.mean, stats.quantile, stats.min, stats.histogram):  # categories stay refused elsewhere
        with pytest.raises(TypeError):
            fn(cat, 0.5) if fn is stats.quantile else fn(cat)
    with pytest.raises(TypeError):
        stats.unique([x, 3])


def test_empty_columns_follow_numpy(monkeypatch):
    _no_gpu(monkeypatch)
    cat = np.array(["a", "b"])
    for node, values in ((_host_node(np.empty(0)), np.empty(0)), (_host_node(np.empty(0, np.int64)), np.empty(0, np.int64)),
                         (_host_node(np.empty(0, bool)), np.empty(0, bool)), (_category_node(0, cat), cat[:0])):
        for flags in ((False, False, False), (True, True, True), (False, True, False)):
            got = stats.unique(node, *flags)
            want = np.unique(values, *flags)
            for g, w in zip(got if isinstance(got, tuple) else (got,), want if isinstance(want, tuple) else (want,)):
                assert g.dtype == w.dtype and g.shape == w.shape
        if values.dtype != np.float64 and node.__dict__["_store"].categories is None:
            for minlength in (0, 4):
                got = stats.bincount(node, minlength=minlength)
                np.testing.assert_array_equal(got, np.bincount(values, minlength=minlength))
                assert got.dtype == np.intp
