"""Parity of the fused graph kernel (csrc/graph.cu through pbl_graph_eval_f64 / pbl_ppf_f64)
against the unmodified reference's golden vectors, SciPy and the oracle.

Bar (north_star): ppf within 4 ulp of scipy for norm / triang / uniform / expon / lognorm;
poisson / binom exact integers; gamma reported as a ulp distribution (scipy's own gammaincinv is
up to 18 ulp from the truth, SURVEY.md section 7) and bounded here; arithmetic nodes equal to NumPy
where the ufunc is correctly rounded (+ - * / sqrt floor ...) and within a few ulp for libm-backed
ones; booleans / dtypes / NoOp / gc semantics identical to the reference."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import scipy.stats as st

import graph_recipes
import gpu_util
from probabilit_b200 import _lib

pytestmark = pytest.mark.gpu

GOLDEN = np.load(os.path.join(os.path.dirname(__file__), "golden", "graph_reference.npz"))

EXACT = {"stat", "lt", "le", "gt", "ge", "eq", "ne", "all", "any", "bool_add", "bool_mul", "floor", "ceil", "sign",
         "eggs", "survived", "p_small", "p_big", "discrete:b", "b_big", "be", "shifted", "counts", "hits", "u",
         "sigma", "shape", "mode", "emp", "dice", "low", "mid", "near", "cum", "disc", "discf", "cat"}
# libm-backed transforms: CUDA's implementations are <= 2 ulp, the inputs themselves carry <= 4 ulp
LOOSE = {"pow", "rpow", "exp", "tan", "sin", "cos", "sinh", "cosh", "tanh", "arctanh", "arccosh", "arcsinh",
         "arcsin", "arccos", "arctan", "arctan2", "log", "log10", "mod", "rmod", "floordiv", "g", "g1", "total",
         "result", "t", "x", "returns", "expr", "d", "avg", "pow2", "square", "div", "rdiv", "rate",
         "correlated:b", "correlated:a", "correlated:c", "noisy"}


def ppf_device(what, q, p0=0.0, p1=0.0, p2=0.0):
    lib = _lib.require_gpu()
    q = np.ascontiguousarray(q, dtype=np.float64)
    dq = gpu_util.DeviceArray(q)
    dout = gpu_util.DeviceArray(np.empty_like(q))
    st_ = _lib.check(lib.pbl_ppf_f64(what, dq.ptr, q.size, p0, p1, p2, dout.ptr, None))
    assert st_ == 0
    out = gpu_util.read_device(dout.ptr.value, q.shape)
    dq.free()
    dout.free()
    return out


def grid(n=200_000, seed=0):
    rng = np.random.default_rng(seed)
    q = rng.random(n)
    tails = np.concatenate([10.0 ** -rng.uniform(1, 300, 2000), 1 - 10.0 ** -rng.uniform(1, 15.9, 2000)])
    return np.concatenate([q, tails, [0.5, 0.25, 0.75, 1e-320, 1 - 2.0 ** -53]])


def test_norm_triang_uniform_expon_lognorm_within_4_ulp():
    from probabilit_b200.modeling import OP

    q = grid()
    cases = [
        (OP["PPF_NORM"], (1.0, 2.0, 0.0), st.norm(loc=1.0, scale=2.0)),
        (OP["PPF_NORM"], (0.0, 1.0, 0.0), st.norm()),
        (OP["PPF_UNIFORM"], (2.0, 3.0, 0.0), st.uniform(loc=2.0, scale=3.0)),
        (OP["PPF_EXPON"], (0.0, 1 / 3, 0.0), st.expon(scale=1 / 3)),
        (OP["PPF_TRIANG"], (0.5, 0.0, 1.0), st.triang(0.5)),
        (OP["PPF_TRIANG"], (0.3, -1.0, 4.0), st.triang(0.3, loc=-1, scale=4)),
        (OP["PPF_LOGNORM"], (0.7, 0.0, 2.0), st.lognorm(0.7, scale=2.0)),
    ]
    for what, p, dist in cases:
        got, want = ppf_device(what, q, *p), dist.ppf(q)
        # 4 ulp of the standardised ppf; `* scale + loc` can cancel, so the unit is the spacing of the
        # larger of |result| and |loc| (for loc = 0 this is plain ulps of the result)
        loc, scale = (p[0], p[1]) if what in (OP["PPF_NORM"], OP["PPF_UNIFORM"], OP["PPF_EXPON"]) else (p[1], p[2])
        z = (want - loc) / scale  # the standardised ppf: 4 ulp of it, scaled, plus the final rounding
        limit = 4 if what != OP["PPF_LOGNORM"] else 8  # exp() amplifies the <= 4 ulp of s * ndtri(q)
        tol = limit * scale * np.spacing(np.abs(z)) + np.spacing(np.abs(want))
        err = np.abs(got - want) / tol
        assert err.max() <= 1.0, (what, p, float(err.max()), q[np.argmax(err)])
    # edge semantics of the scipy wrapper: q = 0 / 1 -> support bounds, invalid -> nan
    e = np.array([0.0, 1.0, -0.1, 1.1, np.nan])
    np.testing.assert_array_equal(ppf_device(OP["PPF_NORM"], e, 1.0, 2.0), st.norm(1.0, 2.0).ppf(e))
    np.testing.assert_array_equal(ppf_device(OP["PPF_TRIANG"], e, 0.3, -1.0, 4.0), st.triang(0.3, -1, 4).ppf(e))
    np.testing.assert_array_equal(ppf_device(OP["PPF_NORM"], e, 0.0, -1.0), st.norm(0, -1).ppf(e))
    np.testing.assert_array_equal(ppf_device(OP["PPF_TRIANG"], e, 1.5, 0.0, 1.0), st.triang(1.5).ppf(e))


@pytest.mark.parametrize("mu", [0.0, 0.7, 3.0, 31.5, 250.5, 12345.6])
def test_poisson_exact(mu):
    from probabilit_b200.modeling import OP

    q = grid(100_000, seed=1)
    q = q[(q < 1 - 1e-13) & (q > 1e-290)]
    got, want = ppf_device(OP["PPF_POISSON"], q, mu, 0.0), st.poisson(mu).ppf(q)
    assert np.count_nonzero(got != want) == 0, (mu, q[got != want][:5], got[got != want][:5], want[got != want][:5])
    e = np.array([0.0, 1.0, np.nan, 2.0])
    np.testing.assert_array_equal(ppf_device(OP["PPF_POISSON"], e, mu, 3.0), st.poisson(mu, loc=3).ppf(e))


@pytest.mark.parametrize("n,p", [(0, 0.4), (1, 0.25), (7, 0.4), (40, 0.3), (5000, 0.6), (100000, 0.001), (30, 0.0),
                                 (30, 1.0), (2000, 0.999)])
def test_binom_exact(n, p):
    from probabilit_b200.modeling import OP

    q = grid(100_000, seed=2)
    q = q[(q < 1 - 1e-13) & (q > 1e-290)]  # the tail walk stops at pmf < 1e-300 (special.cuh)
    got, want = ppf_device(OP["PPF_BINOM"], q, float(n), p, 0.0), st.binom(n, p).ppf(q)
    assert np.count_nonzero(got != want) == 0, (n, p, q[got != want][:5], got[got != want][:5], want[got != want][:5])
    if n == 1:
        np.testing.assert_array_equal(ppf_device(OP["PPF_BERNOULLI"], q, p, 0.0), st.bernoulli(p).ppf(q))


def test_beta_truncnorm_against_scipy():
    """beta.ppf (PERT) and truncnorm.ppf: relative agreement with scipy + the ulp distribution."""
    from probabilit_b200.modeling import OP

    rng = np.random.default_rng(8)
    q = np.concatenate([rng.random(100_000), 10.0 ** -rng.uniform(1, 12, 500), 1 - 10.0 ** -rng.uniform(1, 12, 500)])
    report = {}
    for a, b in ((3.4, 2.6), (7.0, 5.0), (0.6, 0.8), (1.0, 1.0), (0.2, 30.0), (120.0, 45.0), (1.0, 3.0)):
        got, want = ppf_device(OP["PPF_BETA"], q, a, b, 1.0), st.beta(a, b).ppf(q)
        rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
        ulp = gpu_util.ulp_diff(got, want)
        report[f"beta({a},{b})"] = {"max_rel": float(rel.max()), "p99_ulp": float(np.percentile(ulp, 99))}
        assert rel.max() < 1e-10, (a, b, rel.max(), q[np.argmax(rel)])
    for a, b in ((-1.5, 2.0), (2.5, 6.0), (-8.0, -3.0), (-0.1, 0.1), (5.0, 40.0), (-30.0, 30.0)):
        got, want = ppf_device(OP["PPF_TRUNCNORM"], q, a, b, 1.0), st.truncnorm(a, b).ppf(q)
        err = np.abs(got - want) / np.maximum(np.abs(want), 1e-3)
        report[f"truncnorm({a},{b})"] = {"max_rel": float(err.max())}
        assert err.max() < 1e-9, (a, b, err.max(), q[np.argmax(err)])
    print("beta / truncnorm vs scipy:", json.dumps(report))


def test_gamma_ulp_distribution():
    """gamma.ppf = gammaincinv: report the ulp distribution against scipy (stdout)."""
    from probabilit_b200.modeling import OP

    rng = np.random.default_rng(3)
    q = rng.random(200_000)
    report = {}
    for a in (0.05, 0.5, 1.0, 2.0, 2.5, 9.0, 30.0, 150.0, 1000.0):
        got, want = ppf_device(OP["PPF_GAMMA"], q, a, 0.0, 1.0), st.gamma(a).ppf(q)
        ulp = gpu_util.ulp_diff(got, want)
        report[str(a)] = {"max": int(ulp.max()), "p99": float(np.percentile(ulp, 99)),
                          "frac_le_4": float(np.mean(ulp <= 4)), "median": float(np.median(ulp))}
        rel = np.abs(got - want) / np.abs(want)
        assert rel.max() < 1e-13, (a, rel.max(), q[np.argmax(rel)])
    print("gamma ppf ulp vs scipy:", json.dumps(report))
    # The device restates SciPy's own algorithm (Cephes / xsf igami: DiDonato-Morris start, exactly three
    # Halley steps, no FMA contraction), so the bar of 4 ulp of SciPy holds for the bulk wherever the
    # problem does not amplify the last-place differences between CUDA's and glibc's log / exp / lgamma:
    for a in ("1.0", "2.0", "2.5", "9.0", "30.0", "1000.0"):
        assert report[a]["frac_le_4"] > 0.98, (a, report[a])
    # a < 1: P(a, x) ~ x^a / Gamma(a+1), so dx/x = (1/a) dP/P, and P itself comes from
    # exp(a log x - x - lgamma a), whose argument carries ~1e-16 ABSOLUTE error from each libm call: two
    # implementations scatter by 2-3 ulp in P and 1/a times that in x whatever the algorithm.  SciPy is itself
    # 2.4 ulp (a = 0.5) / 34 ulp (a = 0.05) in the median from the mpmath truth, the device 2.4 / 19
    # (tools/gamma_truth.py -> profiles/r2_gamma_truth.json).  a = 150: the same through x^a (a ulp of log x is
    # a ulp of the result).  Those shapes are bounded, not held to 4 ulp:
    assert report["0.5"]["frac_le_4"] > 0.7 and report["0.5"]["p99"] <= 128, report["0.5"]
    assert report["0.05"]["p99"] < 400, report["0.05"]
    assert report["150.0"]["frac_le_4"] > 0.9 and report["150.0"]["max"] <= 32, report["150.0"]


@pytest.mark.parametrize("name", list(graph_recipes.RECIPES))
def test_graph_matches_reference_golden(name):
    import probabilit_b200.modeling as m

    recipe, n = graph_recipes.RECIPES[name]
    sink, named = recipe(m)
    sink.sample_from_quantiles(GOLDEN[f"{name}__quantiles"])
    worst = {}
    for label, node in named:
        want, got = GOLDEN[f"{name}__{label}"], node.samples_
        assert got.dtype == want.dtype and got.shape == want.shape, (label, got.dtype, want.dtype)
        if want.dtype == np.bool_ or label in EXACT or f"{name}:{label}" in EXACT:
            mism = np.count_nonzero(got != want)
            # a comparison can flip only where its float operands differ by ulps *and* nearly tie
            assert mism == 0, (name, label, mism)
        else:
            ulp = gpu_util.ulp_diff(got, want)
            worst[label] = int(ulp.max())
            if name == "four_param":  # betaincinv / truncnorm restated from the published algorithms
                np.testing.assert_allclose(got, want, rtol=5e-12, atol=1e-300, err_msg=f"{name}:{label}")
            elif label in LOOSE or f"{name}:{label}" in LOOSE:
                np.testing.assert_allclose(got, want, rtol=2e-13, atol=1e-300, err_msg=f"{name}:{label}")
            else:
                assert ulp.max() <= 4, (name, label, int(ulp.max()))
    print(name, "max ulp per node:", worst)


def test_readme_examples_with_reference_stream():
    """README.md:21-76 through the public sample() with the reference's own quantile draw."""
    import probabilit_b200.modeling as m

    s, _ = graph_recipes.height(m)
    out = s.sample(999, random_state=0, quantile_source="numpy")
    assert out.mean() == 0.9039039039039038
    np.testing.assert_array_equal(out, GOLDEN["readme__height"])
    s, _ = graph_recipes.birds(m)
    np.testing.assert_array_equal(s.sample(9, random_state=0, quantile_source="numpy"),
                                  np.array([2., 1., 1., 2., 2., 2., 2., 0., 0.]))
    s, _ = graph_recipes.mutual_fund(m)
    out = s.sample(999, random_state=42, quantile_source="numpy")
    np.testing.assert_allclose(out, GOLDEN["readme__mutual_fund"], rtol=1e-13)
    np.testing.assert_allclose([out.mean(), out.std()], [76583.58738496085, 33483.2245611436], rtol=1e-12)


@pytest.mark.parametrize("method", [None, "lhs", "sobol", "halton"])
def test_device_generated_quantiles(method):
    """GPU-native streams: KS and moment tests against the exact marginals (north_star)."""
    import probabilit_b200.modeling as m

    a = m.Distribution("norm", loc=176, scale=7.1)
    b = m.Distribution("gamma", a=2.0, scale=3.0)
    expr = a + b
    n = 200_000 if method != "halton" else 50_000
    out = expr.sample(n, random_state=7, method=method)
    assert out.shape == (n,) and np.all(np.isfinite(out))
    assert st.kstest(a.samples_, st.norm(176, 7.1).cdf).pvalue > 1e-3
    assert st.kstest(b.samples_, st.gamma(2.0, scale=3.0).cdf).pvalue > 1e-3
    assert abs(a.samples_.mean() - 176) < 0.1 and abs(b.samples_.mean() - 6.0) < 0.05
    assert abs(np.corrcoef(a.samples_, b.samples_)[0, 1]) < 0.02
    np.testing.assert_array_equal(out, a.samples_ + b.samples_)
    # reproducible
    np.testing.assert_array_equal(out, expr.sample(n, random_state=7, method=method))


def test_isclose_intended_semantics_and_gc():
    import probabilit_b200.modeling as m

    a, b = m.Distribution("norm"), m.Distribution("norm", scale=1e-9)
    node = m.IsClose(a, a + b)
    q = np.random.default_rng(0).random((1000, 2))
    got = node.sample_from_quantiles(q, gc_strategy=[])
    want = np.isclose(st.norm().ppf(q[:, 0]), st.norm().ppf(q[:, 0]) + st.norm(scale=1e-9).ppf(q[:, 1]))
    assert got.dtype == np.bool_ and np.count_nonzero(got != want) <= 2
    assert not hasattr(a, "samples_")


def test_correlated_graph_on_device():
    """`.correlate()` graph end to end on the GPU (ppf -> Iman-Conover -> rest of the graph)."""
    import probabilit_b200.modeling as m

    recipe, n = graph_recipes.RECIPES["correlated"]
    sink, named = recipe(m)
    nodes = dict(named)
    sink.sample_from_quantiles(GOLDEN["correlated__quantiles"], correlator="imanconover")
    for label in ("a", "b", "c"):
        # Iman-Conover output = a re-ordering of the marginal: same multiset, same order as the reference
        np.testing.assert_allclose(nodes[label].samples_, GOLDEN[f"correlated__{label}"], rtol=1e-14)
    r = np.corrcoef(nodes["a"].samples_, nodes["b"].samples_)[0, 1]
    assert abs(r - np.corrcoef(GOLDEN["correlated__a"], GOLDEN["correlated__b"])[0, 1]) < 1e-12
    # the Cholesky correlator through the same seam (modeling.py:505)
    sink.sample_from_quantiles(GOLDEN["correlated__quantiles"], correlator="cholesky")
    r = np.corrcoef(nodes["b"].samples_, nodes["c"].samples_)[0, 1]
    assert abs(r - (-0.4)) < 1e-10


def test_large_graph_in_one_launch():
    """Mutual-fund graph at n = 2e6 with in-kernel Philox: one kernel launch for 81 nodes."""
    import probabilit_b200.modeling as m

    s, _ = graph_recipes.mutual_fund(m)
    before = _lib.kernel_launches()
    out = s.sample(2_000_000, random_state=1, gc_strategy=[])
    assert _lib.kernel_launches() - before == 1
    assert abs(out.mean() / 76583.6 - 1) < 0.01


@pytest.mark.parametrize("rows,program", [("2", ""), ("4", ""), ("4", "global"), ("2", "global")])
def test_kernel_variants_agree(monkeypatch, rows, program):
    """graph_eval_kernel<2> / <4> (rows per thread, chosen by the shared-memory budget) and the decode-from-global
    path (programs that do not fit beside the slots) are selected by size; forced here on a small graph: all of
    them must give the values of the default configuration, bit for bit -- in-kernel Philox, supplied quantiles,
    an odd number of rows (pairs straddle the end) and all nodes retained."""
    import probabilit_b200.modeling as m

    def run():
        s, named = graph_recipes.mutual_fund(m)
        a = s.sample(100_001, random_state=3)  # all nodes retained, odd n
        kept = [np.array(node.samples_) for _, node in named]
        s2, _ = graph_recipes.mutual_fund(m)
        q = np.random.default_rng(5).random((4097, 20))
        b = s2.sample_from_quantiles(q, gc_strategy=[])
        return [np.array(a), np.array(b)] + kept

    want = run()
    monkeypatch.setenv("PBL_GRAPH_ROWS", rows)
    if program:
        monkeypatch.setenv("PBL_GRAPH_PROGRAM", program)
    got = run()
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w)
