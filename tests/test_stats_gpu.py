"""probabilit_b200.stats on the GPU: mean / var / std / quantile / percentile of device columns equal NumPy on the
host copy bit for bit, with NumPy's dtype and shape, without downloading the column."""
import numpy as np
import pytest

import graph_recipes
import int_graphs

pytestmark = pytest.mark.gpu

SIZES = [1, 2, 7, 8, 9, 127, 128, 129, 255, 8191, 8192, 8193, 1_000_003]
METHODS = ["linear", "lower", "higher", "nearest", "midpoint", "closest_observation"]
QS = [0.5, 0.0, 1.0, [0.3, 0.3, 0.9, 0.1], np.linspace(0, 1, 101), np.array([[0.25, 0.75], [1.0, 0.0]]), 1, [0, 1]]


def _graph(n, seed=0):
    """A float64 node, an int64-bits node (two dice), an int64 table node (one die) and a bool node, sampled."""
    import probabilit_b200.modeling as m

    x = m.Distribution("norm", loc=3, scale=2)
    d1 = int_graphs.die(m)
    dice = d1 + int_graphs.die(m)
    b = x > 4
    m.NoOp(x * 1.0, dice, d1, b).sample(n, random_state=seed)
    return [x, dice, d1, b]


def _same_bits(got, want):
    assert np.asarray(got).dtype == np.asarray(want).dtype
    assert np.asarray(got, dtype=np.float64).view(np.int64) == np.asarray(want, dtype=np.float64).view(np.int64)


def _refuse_downloads(monkeypatch):
    from probabilit_b200._device import DeviceColumns

    def refuse(self, j):
        raise AssertionError("the column was copied to the host")

    monkeypatch.setattr(DeviceColumns, "column_to_host", refuse)


class _quiet:
    """NumPy's warnings for n <= ddof and for inf - inf in the interpolation."""

    def __enter__(self):
        import warnings

        self.w = warnings.catch_warnings()
        self.w.__enter__()
        warnings.simplefilter("ignore")

    def __exit__(self, *exc):
        return self.w.__exit__(*exc)


@pytest.mark.parametrize("n", SIZES)
def test_moments_equal_numpy(n, monkeypatch):
    from probabilit_b200 import stats

    nodes = _graph(n, seed=n)
    host = [v.samples_ for v in nodes]
    assert [h.dtype for h in host] == [np.float64, np.int64, np.int64, np.bool_]
    assert [v.__dict__["_store"].ibits for v in nodes] == [False, True, False, False]
    _refuse_downloads(monkeypatch)
    with np.errstate(all="ignore"), _quiet():
        for node, h in zip(nodes, host):
            _same_bits(stats.mean(node), np.mean(h))
            for ddof in (0, 1, 2.5):
                _same_bits(stats.var(node, ddof=ddof), np.var(h, ddof=ddof))
                _same_bits(stats.std(node, ddof=ddof), np.std(h, ddof=ddof))


def _check_quantiles(x, host, qs=QS, methods=METHODS):
    from probabilit_b200 import stats

    for method in methods:
        for q in qs:
            for fn, npfn, scale in ((stats.quantile, np.quantile, 1), (stats.percentile, np.percentile, 100)):
                qq = q if isinstance(q, int) and scale == 1 else np.multiply(q, scale)
                if isinstance(q, float):
                    qq = float(qq)
                try:
                    want = npfn(host, qq, method=method)
                except TypeError:
                    with pytest.raises(TypeError):
                        fn(x, qq, method=method)
                    continue
                got = fn(x, qq, method=method)
                assert type(got) is type(want), (method, q)
                assert np.asarray(got).dtype == np.asarray(want).dtype, (method, q)
                np.testing.assert_array_equal(got, want, err_msg=f"{method} {q}")


@pytest.mark.parametrize("n", [1, 2, 1001, 1000, 1_000_003])
def test_quantiles_equal_numpy(n, monkeypatch):
    nodes = _graph(n, seed=n + 1)
    hosts = [v.samples_ for v in nodes]
    _refuse_downloads(monkeypatch)
    for node, h in zip(nodes, hosts):
        _check_quantiles(node, h)


def _device(arr):
    import torch

    return torch.as_tensor(arr, device="cuda")


@pytest.mark.parametrize("case", ["normal", "lognorm3", "constant", "two_valued", "poisson", "int_big", "inf",
                                  "nan", "zeros"])
@pytest.mark.parametrize("n", [1, 2, 999, 1000, 1_000_003])
def test_quantiles_of_device_arrays(case, n):
    rng = np.random.default_rng(n)
    if case == "normal":
        a = rng.normal(size=n)
    elif case == "lognorm3":
        a = np.exp(3 * rng.normal(size=n))
    elif case == "constant":
        a = np.full(n, 2.5)
    elif case == "two_valued":
        a = np.where(rng.random(n) < 0.4, -1.0, 7.0)
    elif case == "poisson":
        a = rng.poisson(0.7, n).astype(np.float64)
    elif case == "int_big":
        a = rng.integers(-(2 ** 62), 2 ** 62, size=n, dtype=np.int64)
        a[::7] = np.int64(2 ** 53 + 1)
    elif case == "inf":
        a = rng.normal(size=n)
        a[rng.random(n) < 0.3] = np.inf
        a[rng.random(n) < 0.3] = -np.inf
    elif case == "nan":
        a = rng.normal(size=n)
        a[n // 2] = np.nan
    else:
        a = np.where(rng.random(n) < 0.5, -0.0, 0.0)
    qs = [0.5, [0.0, 1.0, 0.37], np.linspace(0, 1, 101)]
    with _quiet():
        _check_quantiles(_device(a), a, qs=qs)


def test_moments_of_device_arrays_and_int_beyond_2_53():
    from probabilit_b200 import stats

    rng = np.random.default_rng(3)
    for n in (5, 300, 8193, 100_003):
        for a in (rng.normal(size=n) * 1e6, rng.integers(-(2 ** 62), 2 ** 62, size=n, dtype=np.int64)):
            t = _device(a)
            _same_bits(stats.mean(t), np.mean(a))
            _same_bits(stats.var(t, ddof=1), np.var(a, ddof=1))
            _same_bits(stats.std(t), np.std(a))


def test_batch_launches_and_no_download(monkeypatch):
    import probabilit_b200.modeling as m
    from probabilit_b200 import _lib, stats

    n = 100_003
    nodes = [m.Distribution("norm", loc=i, scale=1 + i) for i in range(20)]
    m.NoOp(*nodes).sample(n, random_state=5)
    hosts = [v.samples_ for v in nodes]
    _refuse_downloads(monkeypatch)
    q = np.linspace(0, 100, 101)
    before = _lib.kernel_launches()
    means = stats.mean(nodes)
    stds = stats.std(nodes, ddof=1)
    pct = stats.percentile(nodes, q)
    launches = _lib.kernel_launches() - before
    assert launches <= 2 + 4 + 18  # no sort, no n-sized copy: a fixed number of launches per statistic
    for h, mu, sd, p in zip(hosts, means, stds, pct):
        _same_bits(mu, np.mean(h))
        _same_bits(sd, np.std(h, ddof=1))
        np.testing.assert_array_equal(p, np.percentile(h, q))


def test_input_forms():
    import probabilit_b200.modeling as m
    from probabilit_b200 import stats
    from probabilit_b200._device import DeviceColumns

    rng = np.random.default_rng(11)
    a = rng.normal(size=(5000, 2))
    cols = DeviceColumns.from_host(a)
    _same_bits(stats.mean((cols, 1)), np.mean(a[:, 1]))
    np.testing.assert_array_equal(stats.quantile((cols, 0), [0.1, 0.9]), np.quantile(a[:, 0], [0.1, 0.9]))
    node = m.Distribution("norm")
    node.samples_ = a[:, 0].copy()  # host only: uploaded
    _same_bits(stats.var(node), np.var(a[:, 0]))
    ints = rng.integers(-50, 50, size=777)
    node.samples_ = ints
    _same_bits(stats.mean(node), np.mean(ints))
    np.testing.assert_array_equal(stats.quantile(node, [0.2, 0.5], method="nearest"),
                                  np.quantile(ints, [0.2, 0.5], method="nearest"))
    const = m.Constant(3) + m.Constant(4)  # folded: no device column
    m.NoOp(const, m.Distribution("norm")).sample(10, random_state=0)
    _same_bits(stats.mean(const), np.mean(const.samples_))
    noop = m.NoOp(m.Distribution("norm"))
    noop.sample(10, random_state=0)
    with pytest.raises(TypeError):
        stats.mean(noop)


def test_mutual_fund_1e8():
    import probabilit_b200.modeling as m
    from probabilit_b200 import stats

    sink, _ = graph_recipes.mutual_fund(m)
    sink.sample(100_000_000, random_state=0, gc_strategy=[])
    h = sink.samples_
    _same_bits(stats.mean(sink), np.mean(h))
    _same_bits(stats.std(sink), np.std(h))
    _same_bits(stats.var(sink, ddof=1), np.var(h, ddof=1))
    q = [10, 50, 90]
    for method in ("linear", "nearest"):
        np.testing.assert_array_equal(stats.percentile(sink, q, method=method), np.percentile(h, q, method=method))


def _pw_arange(off, size):
    """NumPy's pairwise tree over arange(off, off + size) as doubles: exact below 2^53."""
    exact = size * off + size * (size - 1) // 2
    if exact < 2 ** 53:
        return float(exact)
    h = size // 2
    n2 = h - h % 8
    return _pw_arange(off, n2) + _pw_arange(off + n2, size - n2)


def test_64bit_counts():
    import torch

    from probabilit_b200 import stats

    n = 2 ** 31 + 5
    if torch.cuda.mem_get_info()[0] < n * 8 + (4 << 30):
        pytest.skip("not enough device memory for 2^31 + 5 doubles")
    x = torch.arange(n, dtype=torch.float64, device="cuda")
    _same_bits(stats.mean(x), np.float64(0.0 + _pw_arange(0, n)) / np.float64(n))
    q = np.array([0.0, 0.1, 0.5, 0.9, 1.0])
    vi = np.float64(n - 1) * q  # sorted values are their own ranks
    lo = np.floor(vi)
    hi = np.minimum(lo + 1, n - 1)
    g = vi - lo
    want = np.where(g >= 0.5, hi - (hi - lo) * (1 - g), lo + (hi - lo) * g)  # numpy's _lerp
    np.testing.assert_array_equal(stats.quantile(x, q), want)
    np.testing.assert_array_equal(stats.quantile(x, q, method="higher"), np.ceil(vi))
    del x
    torch.cuda.empty_cache()
