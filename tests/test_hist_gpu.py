"""probabilit_b200.stats on the GPU: min / max / ptp / histogram / histogram_bin_edges of device columns equal NumPy
on the host copy, with NumPy's dtype, shape and bits (and its exceptions), without downloading the column."""
import warnings

import numpy as np
import pytest

from test_stats_gpu import SIZES, _device, _graph, _refuse_downloads

pytestmark = pytest.mark.gpu

ESTIMATORS = ["auto", "fd", "rice", "scott", "sqrt", "sturges"]
BINS = [1, 10, 20_000] + ESTIMATORS  # 20 000 bins: above the shared-memory arm (16 384 counts)


def _same(got, want):
    """Equal values, dtype and shape; a zero's sign is free (min / max, and edges taken from them)."""
    if isinstance(want, tuple):
        assert isinstance(got, tuple) and len(got) == len(want)
        for g, w in zip(got, want):
            _same(g, w)
        return
    assert type(got) is type(want), (type(got), type(want))
    assert np.asarray(got).dtype == np.asarray(want).dtype
    assert np.shape(got) == np.shape(want)
    np.testing.assert_array_equal(got, want)


def _check(fn, npfn, x, host, *args, **kw):
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        try:
            want = npfn(host, *args, **kw)
        except Exception as e:  # noqa: BLE001 -- NumPy's exception type is the expected result
            with pytest.raises(type(e)):
                fn(x, *args, **kw)
            return
        got = fn(x, *args, **kw)
    _same(got, want)


def _ranges(h):
    if h.dtype == np.bool_:
        return [None, (0, 1), (0.5, 2.0)]
    finite = h[np.isfinite(h)].astype(np.float64)
    if finite.size == 0:
        return [None, (-1.0, 1.0)]
    lo, q1, q3, hi = np.quantile(finite, [0, 0.2, 0.7, 1])
    return [None, (float(lo) - 1, float(hi) + 1), (float(q1), float(q3)), (int(q1), int(q3) + 1)]


def _check_all(x, h, bins_list=BINS, edges=True):
    from probabilit_b200 import stats

    for fn, npfn in ((stats.min, np.min), (stats.max, np.max), (stats.ptp, np.ptp)):
        _check(fn, npfn, x, h)
    arrays = [np.array([-1.0, 0.5, 2.0, 3.5, 7.0]), np.array([-3, 0, 2, 5]), np.array([0.0, np.nan, 3.0])] if edges else []
    for rng in _ranges(h):
        for bins in bins_list + arrays:
            _check(stats.histogram_bin_edges, np.histogram_bin_edges, x, h, bins, rng)
            _check(stats.histogram, np.histogram, x, h, bins, rng)
        _check(stats.histogram, np.histogram, x, h, "auto", rng, density=True)
        _check(stats.histogram, np.histogram, x, h, 7, rng, density=True)


@pytest.mark.parametrize("n", SIZES)
def test_node_encodings_equal_numpy(n, monkeypatch):
    nodes = _graph(n, seed=n + 3)
    hosts = [v.samples_ for v in nodes]
    _refuse_downloads(monkeypatch)
    for node, h in zip(nodes, hosts):
        _check_all(node, h)


@pytest.mark.parametrize("case", ["nan", "inf", "constant", "zeros", "int_2_53", "int_2_62", "int_small"])
@pytest.mark.parametrize("n", [1, 2, 1000, 100_003])
def test_device_arrays(case, n):
    from probabilit_b200 import stats

    rng = np.random.default_rng(n)
    if case == "nan":
        a = rng.normal(size=n)
        a[n // 2] = np.nan
    elif case == "inf":
        a = rng.normal(size=n)
        a[rng.random(n) < 0.2] = np.inf
        a[0] = -np.inf
    elif case == "constant":
        a = np.full(n, 2.5)
    elif case == "zeros":
        a = np.where(rng.random(n) < 0.5, -0.0, 0.0)
    elif case == "int_2_53":
        a = 2 ** 53 + rng.integers(-40, 40, size=n, dtype=np.int64)
    elif case == "int_2_62":
        a = rng.integers(-(2 ** 62), 2 ** 62, size=n, dtype=np.int64)
        a[::5] = 2 ** 53 + 1
    else:
        a = rng.integers(-7, 9, size=n, dtype=np.int64)
    x = _device(a)
    _check_all(x, a, bins_list=[1, 10, 20_000, "auto", "fd", "sqrt"])
    if a.dtype == np.int64:
        lo, hi = int(a.min()), int(a.max())
        q3, q8 = int(np.quantile(a, 0.3)) | 1, int(np.quantile(a, 0.8)) | 1  # odd: float64 rounds them away
        mixed = [(q3, float(q8)), (float(q3), q8), (np.int64(q3), float(q8)), (float(q3), np.int64(q8))]
        for rng_ in [(lo, hi), (lo + 1, hi - 1), (float(lo), float(hi)), (np.int64(lo), float(hi) - 1e3)] + mixed:
            for bins in (3, 257, "auto", "sturges", np.array([lo, lo + 2, hi], dtype=np.int64),
                         np.array([lo, lo + 2, hi], dtype=np.float64)):
                _check(stats.histogram, np.histogram, x, a, bins, rng_)


def test_mixed_int_float_range_beyond_2_53():
    """NumPy compares int64 data with an int edge exactly and with a float edge in float64, one edge at a time."""
    from probabilit_b200 import stats

    a = np.array([2 ** 53, 2 ** 53 + 2, 2 ** 53 + 6], dtype=np.int64)
    x = _device(a)
    for rng_ in ((2 ** 53 + 1, 2.0 ** 53 + 8), (np.int64(2 ** 53 + 1), 2.0 ** 53 + 8)):
        for bins in (2, 5, "auto", "sqrt", "sturges"):
            _check(stats.histogram, np.histogram, x, a, bins, rng_)
            _check(stats.histogram_bin_edges, np.histogram_bin_edges, x, a, bins, rng_)
    b = 2 ** 53 + np.random.default_rng(4).integers(-30, 30, size=100_003, dtype=np.int64)
    for rng_ in ((2 ** 53 - 9, 2.0 ** 53 + 11), (2.0 ** 53 - 9, 2 ** 53 + 11)):
        for bins in (7, "auto", "fd", "scott"):
            _check(stats.histogram, np.histogram, _device(b), b, bins, rng_)


def test_large_edge_array():
    from probabilit_b200 import stats

    a = np.random.default_rng(6).normal(size=1_000_003)
    edges = np.linspace(-4, 4, 100_001)
    edges[500] = np.nan
    _check(stats.histogram, np.histogram, _device(a), a, edges)


def test_index_outside_the_edges_raises_numpy_error():
    from probabilit_b200 import stats

    a = np.array([2 ** 53 + 1, 2 ** 53 + 3], dtype=np.int64)
    with pytest.raises(Exception) as want:
        np.histogram(a, bins=2)
    with pytest.raises(type(want.value)) as got:
        stats.histogram(_device(a), bins=2)
    assert str(got.value) == str(want.value)


def test_bool_warns_like_numpy(monkeypatch):
    nodes = _graph(1000, seed=2)
    from probabilit_b200 import stats

    with pytest.warns(RuntimeWarning, match="Converting input from bool"):
        stats.histogram(nodes[3], bins="auto")
    with pytest.warns(RuntimeWarning, match="Converting input from bool"):
        stats.histogram_bin_edges(nodes[3])


def test_batch_equals_single_calls_with_fewer_launches(monkeypatch):
    import probabilit_b200.modeling as m
    from probabilit_b200 import _lib, stats

    n = 100_003
    nodes = [m.Distribution("norm", loc=i, scale=1 + i) for i in range(12)] + _graph(n, seed=9)
    m.NoOp(*nodes).sample(n, random_state=5)
    _refuse_downloads(monkeypatch)
    cases = [(stats.min, ()), (stats.max, ()), (stats.histogram, (10,)), (stats.histogram, ("auto", (2.0, 6.0))),
             (stats.histogram, ("fd",)), (stats.histogram, (np.array([0.0, 1.0, 5.0, 9.0]),)),
             (stats.histogram_bin_edges, ("scott", (0, 4)))]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for fn, args in cases:
            before = _lib.kernel_launches()
            batch = fn(nodes, *args)
            batch_launches = _lib.kernel_launches() - before
            before = _lib.kernel_launches()
            singles = [fn(v, *args) for v in nodes]
            single_launches = _lib.kernel_launches() - before
            assert batch_launches < single_launches, (fn.__name__, args)
            for g, w in zip(batch, singles):
                _same(g, w)


def test_host_only_samples_are_uploaded():
    import probabilit_b200.modeling as m
    from probabilit_b200 import stats

    node = m.Distribution("norm")
    node.samples_ = np.random.default_rng(0).normal(size=777)
    _check_all(node, node.samples_, bins_list=[10, "auto"], edges=False)
    const = m.Constant(3) + m.Constant(4)
    m.NoOp(const, m.Distribution("norm")).sample(10, random_state=0)
    _same(stats.histogram(const), np.histogram(const.samples_))
    _same(stats.max(const), np.max(const.samples_))


def test_mutual_fund_1e7(monkeypatch):
    import graph_recipes
    import probabilit_b200.modeling as m

    sink, _ = graph_recipes.mutual_fund(m)
    sink.sample(10_000_000, random_state=0, gc_strategy=[])
    h = sink.samples_
    _refuse_downloads(monkeypatch)
    _check_all(sink, h, bins_list=[10, 20_000, "auto", "sqrt", "fd"], edges=True)
