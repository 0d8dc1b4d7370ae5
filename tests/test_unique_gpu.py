"""probabilit_b200.stats.unique / bincount on the GPU: equal np.unique / np.bincount on the host copy (value bits, dtype
and shape) for every column encoding, category nodes included, without downloading the column."""
import itertools

import numpy as np
import pytest

import int_graphs
from test_stats_gpu import SIZES, _refuse_downloads

pytestmark = pytest.mark.gpu

FLAGS = list(itertools.product([False, True], repeat=3))  # return_index, return_inverse, return_counts


def _nodes(n, seed):
    """float64, int64 bits (two dice), int64 table (one die), bool, poisson and a category node with a repeated
    category value, sampled."""
    import probabilit_b200.modeling as m

    x = m.Distribution("norm", loc=3, scale=2)
    d1 = int_graphs.die(m)
    dice = d1 + int_graphs.die(m)
    b = x > 4
    p = m.Distribution("poisson", mu=2.5)
    cat = m.DiscreteDistribution(["b", "a", "b", "c"], [0.1, 0.2, 0.3, 0.4])
    m.NoOp(x * 1.0, dice, d1, b, p, cat).sample(n, random_state=seed)
    return [x, dice, d1, b, p, cat]


def _tuple(r):
    return r if isinstance(r, tuple) else (r,)


def _check(x, host, flags, equal_nan=True):
    from probabilit_b200 import stats

    got, want = _tuple(stats.unique(x, *flags, equal_nan=equal_nan)), _tuple(np.unique(host, *flags, equal_nan=equal_nan))
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert type(g) is np.ndarray and g.dtype == w.dtype and g.shape == w.shape, (flags, equal_nan)
    if want[0].dtype == np.float64 and flags[0]:  # the sign of zero and the NaN payloads are NumPy's here
        np.testing.assert_array_equal(got[0].view(np.int64), want[0].view(np.int64))
    else:
        np.testing.assert_array_equal(got[0], want[0])
    got, want = list(got), list(want)
    if flags[1] and not flags[0] and not equal_nan:
        # one entry per NaN, ordered by NumPy's quicksort: the NaN rows map to those entries in some order
        at = 1
        nan = np.isnan(host)
        np.testing.assert_array_equal(np.sort(got[at][nan]), np.sort(want[at][nan]))
        got[at], want[at] = got[at][~nan], want[at][~nan]
    for g, w in zip(got[1:], want[1:]):
        np.testing.assert_array_equal(g, w, err_msg=f"{flags} {equal_nan}")


@pytest.mark.parametrize("n", SIZES)
def test_unique_of_nodes_equals_numpy(n, monkeypatch):
    nodes = _nodes(n, seed=n)
    hosts = [v.samples_ for v in nodes]
    assert [h.dtype for h in hosts[:5]] == [np.float64, np.int64, np.int64, np.bool_, np.float64]
    assert hosts[5].dtype.kind == "U" and nodes[5].__dict__["_store"].categories is not None
    assert nodes[1].__dict__["_store"].ibits
    _refuse_downloads(monkeypatch)
    for node, h in zip(nodes, hosts):
        for flags in FLAGS:
            for equal_nan in ((True, False) if h.dtype == np.float64 else (True,)):
                _check(node, h, flags, equal_nan)


@pytest.mark.parametrize("n", SIZES)
def test_bincount_of_nodes_equals_numpy(n, monkeypatch):
    from probabilit_b200 import stats

    nodes = _nodes(n, seed=n + 1)
    hosts = [v.samples_ for v in nodes]
    _refuse_downloads(monkeypatch)
    for node, h in zip(nodes, hosts):
        if h.dtype in (np.int64, np.bool_):
            for minlength in (0, 10):
                got, want = stats.bincount(node, minlength=minlength), np.bincount(h, minlength=minlength)
                assert got.dtype == want.dtype
                np.testing.assert_array_equal(got, want)
        else:
            with pytest.raises(TypeError):
                np.bincount(h)
            with pytest.raises(TypeError):
                stats.bincount(node)


def _nan(sign, payload):
    return np.array([(0xFFF0000000000000 if sign else 0x7FF0000000000000) | payload], dtype=np.uint64).view(np.float64)[0]


@pytest.mark.parametrize("n", [1, 2, 9, 8193, 100_003])
def test_special_values_of_device_arrays(n):
    import torch

    rng = np.random.default_rng(n)
    special = np.array([0.0, -0.0, np.inf, -np.inf, _nan(0, 1), _nan(1, 2), _nan(0, 1 << 51), _nan(1, 3), 1.5, -1.5,
                        5e-324, -5e-324])
    cases = [special[rng.integers(0, special.size, n)], np.where(rng.random(n) < 0.5, -0.0, 0.0),
             np.full(n, _nan(1, 7)), np.round(rng.normal(size=n), 2)]
    cases[3][rng.random(n) < 0.1] = np.nan
    for a in cases:
        t = torch.as_tensor(a, device="cuda")
        for flags in FLAGS:
            for equal_nan in (True, False):
                _check(t, a, flags, equal_nan)
    ints = rng.integers(-(2 ** 53), 2 ** 53 + 1, n, dtype=np.int64)  # int64 bit patterns within +-2^53, with ties
    ints[::3] %= 5
    ints[:3] = np.array([2 ** 53, -(2 ** 53), 2 ** 53 - 1])[:n]
    for flags in FLAGS:
        _check(torch.as_tensor(ints, device="cuda"), ints, flags)


def test_int64_beyond_2_53_and_negative_bincount():
    import torch

    from probabilit_b200 import stats

    for v in (2 ** 53 + 1, -(2 ** 53) - 1, 2 ** 62):
        a = np.array([0, 5, v, 5], dtype=np.int64)
        with pytest.raises(NotImplementedError):
            stats.unique(torch.as_tensor(a, device="cuda"), return_counts=True)
        with pytest.raises(NotImplementedError):
            stats.bincount(torch.as_tensor(a, device="cuda"))
    a = np.array([4, 2, -3, 2], dtype=np.int64)
    with pytest.raises(ValueError) as got:
        stats.bincount(torch.as_tensor(a, device="cuda"))
    with pytest.raises(ValueError) as want:
        np.bincount(a)
    assert str(got.value) == str(want.value)
    np.testing.assert_array_equal(stats.bincount(torch.as_tensor(a + 3, device="cuda"), minlength=9),
                                  np.bincount(a + 3, minlength=9))


def test_constant_columns_batches_and_host_samples(monkeypatch):
    import torch

    import probabilit_b200.modeling as m
    from probabilit_b200 import stats

    n = 1_000_003
    for a in (np.full(n, 2.5), np.full(n, -0.0), np.full(n, 7, dtype=np.int64)):
        for flags in FLAGS:
            _check(torch.as_tensor(a, device="cuda"), a, flags)
    nodes = _nodes(10_007, seed=3)
    hosts = [v.samples_ for v in nodes]
    _refuse_downloads(monkeypatch)
    got = stats.unique(nodes, return_index=True, return_inverse=True, return_counts=True)
    assert isinstance(got, list) and len(got) == len(nodes)
    for g, h in zip(got, hosts):
        want = np.unique(h, return_index=True, return_inverse=True, return_counts=True)
        for u, w in zip(g, want):
            assert u.dtype == w.dtype
            np.testing.assert_array_equal(u, w)
    ints = [v for v, h in zip(nodes, hosts) if h.dtype != np.float64 and h.dtype.kind != "U"]
    for g, v in zip(stats.bincount(ints, minlength=3), ints):
        np.testing.assert_array_equal(g, np.bincount(v.samples_, minlength=3))
    node = m.Distribution("norm")
    for values in (np.array([3.0, -0.0, 0.0, np.nan, 3.0]), np.array([9, -4, 9], dtype=np.int64),
                   np.array([True, True])):
        node.samples_ = values  # host only: uploaded
        for flags in FLAGS:
            _check(node, values, flags)
    const = m.Constant(3) + m.Constant(4)  # folded: no device column
    m.NoOp(const, m.Distribution("norm")).sample(10, random_state=0)
    _check(const, const.samples_, (True, True, True))
    np.testing.assert_array_equal(stats.bincount(const), np.bincount(const.samples_))


def test_continuous_column_runs_all_passes():
    import torch

    a = np.random.default_rng(7).normal(size=10_000_019)
    a[::1000] = 0.25  # ties
    t = torch.as_tensor(a, device="cuda")
    _check(t, a, (True, True, True))
    _check(t, a, (False, False, True))


def test_one_tile_per_block_digit_pass(monkeypatch):
    """Columns longer than PBL_CLASSIC_ABOVE rows are sorted by the one-tile-per-block digit pass."""
    import torch

    monkeypatch.setenv("PBL_CLASSIC_ABOVE", "1000")
    rng = np.random.default_rng(9)
    for a in (np.round(rng.normal(size=300_007), 3), rng.normal(size=70_001)):
        t = torch.as_tensor(a, device="cuda")
        _check(t, a, (True, True, True))
    nodes = _nodes(50_001, seed=4)
    for node in nodes:
        _check(node, node.samples_, (True, True, True))
