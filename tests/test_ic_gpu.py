"""Parity of the CUDA Iman-Conover path (through the C ABI) against the CPU oracle and the
reference's golden vectors.  Bar: output bit-exact (it is a per-column re-ordering of the input),
rank indices identical, scores within 4 ulp of scipy's norm.ppf, R/T to 1e-12."""
import numpy as np
import pytest
import scipy as sp
import scipy.stats

from conftest import random_target
from oracle import iman_conover as oic

import gpu_util

pytestmark = pytest.mark.gpu

CASES = ["readme_lhs", "toy_ties", "normal_1000x2", "lognormal_1000x2", "sobol_mixed_4096x16",
         "poisson_2000x3", "specials_500x4", "wide_700x64"]


@pytest.mark.parametrize("name", CASES)
def test_output_equals_reference_golden(ic_golden, name):
    from probabilit_b200 import ImanConover

    X, C, Y = ic_golden[name]
    got = ImanConover().set_target(C)(X)
    assert got.dtype == Y.dtype and got.shape == Y.shape
    assert got.flags.f_contiguous == Y.flags.f_contiguous
    np.testing.assert_array_equal(got, Y)


@pytest.mark.parametrize("name", CASES)
def test_stages_against_oracle(ic_golden, name):
    X, C, Y = ic_golden[name]
    ref = oic.iman_conover_stages(X, C)
    got = gpu_util.run_stages(X, C)
    assert got["status"] == 0
    np.testing.assert_array_equal(got["sortedX"], ref["sortedX"])
    ulp = gpu_util.ulp_diff(got["scores"], ref["scores"])
    assert ulp.max() <= 4, f"scores differ by {ulp.max()} ulp"
    N = X.shape[0]
    np.testing.assert_allclose(got["gram"], ref["scores"].T @ ref["scores"], rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(got["colsum"], ref["scores"].sum(axis=0), rtol=0, atol=1e-9 * N ** 0.5)
    np.testing.assert_allclose(got["Q"], ref["Q"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got["T"], ref["T"], rtol=0, atol=1e-10)
    np.testing.assert_allclose(got["correlated"], ref["correlated"], rtol=0, atol=1e-10)
    np.testing.assert_array_equal(got["result"], Y)


@pytest.mark.parametrize("consumer", ["tma", "classic"])
@pytest.mark.parametrize("n,k,seed", [(100_000, 5, 0), (300_001, 3, 1), (4097, 7, 2), (65_536, 16, 3),
                                      (700_001, 3, 4)])
def test_random_problems_bit_exact(monkeypatch, n, k, seed, consumer):
    """Multi-tile sorts (look-back across tiles), finished by either consumer kernel: "classic" moves the
    long-column rule (PBL_CLASSIC_ABOVE) below these sizes, so that post_sort_kernel finishes batches of 3-16
    columns, as it does for columns of more than 3e8 rows; the digit pass of such batches stays pass_tma_kernel."""
    from probabilit_b200 import ImanConover

    if consumer == "classic":
        monkeypatch.setenv("PBL_CLASSIC_ABOVE", "1000")
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.normal(size=(n, k)) * rng.lognormal(size=k) + rng.normal(size=k))
    C = random_target(rng, k)
    want = oic.iman_conover(X, C)
    got = ImanConover().set_target(C)(X)
    np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("n,k,seed,ties", [(300_001, 3, 11, False), (1_200_000, 2, 12, False), (500_000, 3, 13, True),
                                           (700_000, 2, 14, True)])
def test_one_tile_per_block_consumer_is_bit_exact(monkeypatch, n, k, seed, ties):
    """Columns longer than PBL_CLASSIC_ABOVE rows (default 3e8: the multi-GPU shapes) are finished by
    post_sort_kernel instead of the persistent post_tma_kernel, and launches on one or two such columns use the
    one-tile-per-block digit pass instead of pass_tma_kernel (sort.cu: sort_classic_consumer / sort_classic_pass);
    the threshold is moved below these sizes, so that the path the 8-GPU runs take is pinned against the oracle.
    The 3-column cases run post_sort_kernel on unpartitioned pairs (fewer than 2^19 rows), as columns of more than
    3e8 rows written with a row stride other than 1 do."""
    from probabilit_b200 import ImanConover

    monkeypatch.setenv("PBL_CLASSIC_ABOVE", "1000")
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, k)) * rng.lognormal(size=k) + rng.normal(size=k)
    if ties:
        X = np.round(X, 3)
    X = np.asfortranarray(X)
    C = random_target(rng, k)
    want = oic.iman_conover(X, C)
    got = ImanConover().set_target(C)(X)
    np.testing.assert_array_equal(got, want)


def test_heavy_ties_multi_tile():
    """Tie runs that span many tiles (binary-search path of the post-sort kernel)."""
    from probabilit_b200 import ImanConover

    rng = np.random.default_rng(7)
    n, k = 50_000, 4
    X = np.empty((n, k), order="F")
    X[:, 0] = rng.poisson(2.0, n)
    X[:, 1] = rng.integers(0, 3, n)
    X[:, 2] = np.round(rng.normal(size=n), 2)
    X[:, 3] = rng.normal(size=n)
    C = random_target(rng, k)
    want = oic.iman_conover(X, C)
    got = ImanConover().set_target(C)(X)
    np.testing.assert_array_equal(got, want)


def test_heavy_ties_partitioned_scatter():
    """n > 2^19 rows: the scatter runs as window partition + window-local scatter; discrete data
    makes every tile take the tie-run path and skips most digit passes."""
    from probabilit_b200 import ImanConover

    rng = np.random.default_rng(8)
    n, k = 1_200_000, 3
    X = np.empty((n, k), order="F")
    X[:, 0] = rng.poisson(3.0, n)
    X[:, 1] = rng.normal(size=n)
    X[:, 2] = rng.binomial(10, 0.4, n)
    C = random_target(rng, k)
    want = oic.iman_conover(X, C)
    got = ImanConover().set_target(C)(X)
    np.testing.assert_array_equal(got, want)


def test_dense_cluster_falls_back_to_full_sort():
    """Distinct values packed more densely than the 32-bit sort window resolves (here 2^-52 apart in a
    column spanning ~2000 binades): the window
    cannot separate them, the post-sort kernel raises the retry flag and the plan repeats the
    transform with the exact 64-bit sort.  Output must still be bit-exact."""
    from probabilit_b200 import ImanConover

    rng = np.random.default_rng(12)
    n, k = 40_000, 3
    X = np.asfortranarray(rng.normal(size=(n, k)))
    X[: n // 2, 1] = 1.0 + rng.permutation(n // 2) * 2.0 ** -52  # n/2 distinct neighbours of 1.0
    X[n // 2:, 1] = np.exp(rng.uniform(-600, 600, n - n // 2))   # huge dynamic range
    C = random_target(rng, k)
    want = oic.iman_conover(X, C)
    got_stages = gpu_util.run_stages(X, C)
    assert got_stages["attempts"] == 2 and got_stages["status"] == 0
    np.testing.assert_array_equal(got_stages["result"], want)
    np.testing.assert_array_equal(ImanConover().set_target(C)(X), want)


def test_window_collisions_are_completed_in_tile():
    """Many short runs of distinct keys sharing a window value (no fallback needed)."""
    rng = np.random.default_rng(13)
    n, k = 150_000, 2
    X = np.asfortranarray(rng.normal(size=(n, k)))
    base = np.exp(rng.uniform(-300, 300, n // 8))
    # groups of 8 distinct neighbours (1 ulp apart) around values spread over a huge range
    X[: (n // 8) * 8, 0] = (base[:, None] * (1.0 + np.arange(8)[None, :] * 2.0 ** -52)).ravel()
    C = random_target(rng, k)
    want = oic.iman_conover(X, C)
    got = gpu_util.run_stages(X, C)
    assert got["attempts"] == 1 and got["status"] == 0
    np.testing.assert_array_equal(got["result"], want)


@pytest.mark.parametrize("group,attempts", [(31, 1), (32, 1), (33, 2), (48, 2)])
def test_window_runs_around_the_in_tile_limit(group, attempts):
    """Runs of `group` distinct keys that share one window value: up to 32 keys are re-ordered inside the
    post-sort tile, longer ones raise the retry flag (exact 64-bit sort).  Bit-exact either way."""
    rng = np.random.default_rng(14)
    n, k = 120_000, 2
    X = np.asfortranarray(rng.normal(size=(n, k)))
    m = n // (2 * group)
    base = np.exp(rng.uniform(-300, 300, m))
    vals = (base[:, None] * (1.0 + np.arange(group)[None, :] * 2.0 ** -52)).ravel()
    X[: m * group, 1] = rng.permutation(vals)
    C = random_target(rng, k)
    want = oic.iman_conover(X, C)
    got = gpu_util.run_stages(X, C)
    assert got["attempts"] == attempts and got["status"] == 0
    np.testing.assert_array_equal(got["result"], want)


def test_row_chunk_hook_delivers_the_same_scores_chunk_by_chunk():
    """pbl_ic_plan_set_chunk_hook (the multi-GPU driver's hook): the scatter by row is enqueued per row
    chunk, first_chunk first, the callback fires once per (column, chunk), results are unchanged."""
    import ctypes as C_
    from probabilit_b200 import _lib
    from probabilit_b200.correlation import _IcPlan

    lib = _lib.require_gpu()
    rng = np.random.default_rng(15)
    n, k, chunks = 1_500_000, 2, 4  # > 2^19 rows: grouped pairs, chunked delivery
    X = np.asfortranarray(rng.normal(size=(n, k)))
    plan = _IcPlan(n, k, 0)
    plan.set_target(np.eye(k))
    dX = gpu_util.DeviceArray(X)
    chunk_rows = (n + chunks - 1) // chunks
    try:
        _lib.check(lib.pbl_ic_stage_begin(plan.handle, None))
        _lib.check(lib.pbl_ic_stage_rank_scores(plan.handle, dX.ptr, 1, n, 0, k, None))
        want = gpu_util.read_device(plan.buffer(0)[0], (n, k), order="F")
        zeros = np.zeros((n, k), order="F")  # so that a row the chunked delivery missed would show
        _lib.check(lib.pbl_memcpy_h2d(C_.c_void_p(plan.buffer(0)[0]), zeros.ctypes.data, zeros.nbytes, None))
        _lib.check(lib.pbl_stream_synchronize(None))
        seen = []
        cb = _lib.CHUNK_FN(lambda col, g, user: seen.append((col, g)))
        _lib.check(lib.pbl_ic_plan_set_chunk_hook(plan.handle, chunk_rows, 2, cb, None))
        _lib.check(lib.pbl_ic_stage_begin(plan.handle, None))
        for c in range(k):
            _lib.check(lib.pbl_ic_stage_rank_scores(plan.handle, dX.ptr, 1, n, c, 1, None))
        _lib.check(lib.pbl_ic_plan_set_chunk_hook(plan.handle, 0, 0, None, None))
        got = gpu_util.read_device(plan.buffer(0)[0], (n, k), order="F")
        assert _lib.check(lib.pbl_ic_stage_status(plan.handle, None)) == 0
    finally:
        dX.free()
        plan.close()
    assert seen == [(c, g) for c in range(k) for g in (2, 3, 0, 1)]
    np.testing.assert_array_equal(got, want)


def test_c_order_and_column_batches():
    from probabilit_b200 import ImanConover

    rng = np.random.default_rng(11)
    X = np.ascontiguousarray(rng.normal(size=(20_000, 6)))
    C = random_target(rng, 6)
    want = oic.iman_conover(X, C)
    got = ImanConover(col_batch=4).set_target(C)(X)
    assert got.flags.c_contiguous
    np.testing.assert_array_equal(got, want)


def test_one_shot_c_entry_point(ic_golden):
    """pbl_iman_conover_f64: the single C call a foreign host would bind."""
    from probabilit_b200 import _lib

    lib = _lib.require_gpu()
    X, C, Y = ic_golden["sobol_mixed_4096x16"]
    P = np.ascontiguousarray(np.linalg.cholesky(C))
    out = np.empty_like(X)
    rs, cs = (s // 8 for s in X.strides)
    st = lib.pbl_iman_conover_f64(X.ctypes.data, X.shape[0], X.shape[1], rs, cs, P.ctypes.data,
                                  out.ctypes.data, rs, cs)
    assert st == 0, _lib.last_error()
    np.testing.assert_array_equal(out, Y)


def test_error_conventions():
    """Same exception types as the reference (tests/test_iman_conover.py:49-109, :200-210)."""
    from probabilit_b200 import CorrelatorError, ImanConover

    rng = np.random.default_rng(0)
    X = rng.normal(size=(100, 3))
    with pytest.raises(ValueError):
        ImanConover().set_target(np.array([[1.0, 0.7, -0.3], [0.8, 1.0, 0.5], [-0.3, 0.5, 1.0]]))(X)
    with pytest.raises(ValueError):
        ImanConover().set_target(np.array([[1.0, 2.0, 0.3], [2.0, 1.0, 0.2], [0.3, 0.2, 1.0]]))(X)
    with pytest.raises(ValueError):
        ImanConover().set_target(np.array([[1.0, 0.5], [0.5, 1.0]]))(X)
    with pytest.raises(ValueError, match="not positive definite"):
        ImanConover().set_target(np.identity(2))(np.array([[1.0, 1], [2.0, 1.1], [2.1, 3]]))
    with pytest.raises(CorrelatorError):
        ImanConover()(X)
    with pytest.raises(TypeError):
        ImanConover().set_target(np.identity(3))([[1.0, 2.0, 3.0]])
    Xn = X.copy()
    Xn[3, 1] = np.nan
    with pytest.raises(ValueError, match="infs or NaNs"):
        ImanConover().set_target(np.identity(3))(Xn)
    with pytest.raises(ValueError):  # rows <= columns
        ImanConover().set_target(np.identity(3))(X[:3])


def test_reference_property_tests():
    """Ports of tests/test_iman_conover.py:33-46 and :146-176 (marginals, Spearman, distance)."""
    from probabilit_b200 import ImanConover

    for seed in range(10):
        rng = np.random.default_rng(seed)
        n_variables = int(rng.integers(2, 100))
        n_observations = n_variables * 10
        desired = random_target(rng, n_variables)
        X = rng.normal(size=(n_observations, n_variables))
        Xt = ImanConover().set_target(desired)(X)
        for j in range(n_variables):
            np.testing.assert_array_equal(np.sort(X[:, j]), np.sort(Xt[:, j]))
        before = sp.linalg.norm(np.corrcoef(X, rowvar=False) - desired, ord="fro")
        after = sp.linalg.norm(np.corrcoef(Xt, rowvar=False) - desired, ord="fro")
        assert after <= before


def test_device_resident_tensor_path():
    torch = pytest.importorskip("torch")
    from probabilit_b200 import ImanConover

    rng = np.random.default_rng(3)
    X = np.asfortranarray(rng.normal(size=(30_000, 8)))
    C = random_target(rng, 8)
    want = oic.iman_conover(X, C)
    Xd = torch.from_numpy(np.ascontiguousarray(X.T)).cuda().T  # (n, k) view, column-major
    assert Xd.stride() == (1, X.shape[0])
    Yd = ImanConover().set_target(C)(Xd)
    assert Yd.is_cuda and Yd.stride() == Xd.stride()
    np.testing.assert_array_equal(Yd.cpu().numpy(), want)


def test_large_n_invariants():
    """N = 2^24 rows, d = 4: too big for the oracle in seconds on every column, so check the
    size-independent properties: per-column permutation (sorted columns identical), column 0
    unchanged (T[0,0] > 0), Spearman close to target, and the oracle on one column."""
    torch = pytest.importorskip("torch")
    from probabilit_b200 import ImanConover

    n, k = 1 << 24, 4
    g = torch.Generator(device="cuda").manual_seed(0)
    Xd = torch.randn((k, n), generator=g, device="cuda", dtype=torch.float64).T
    rng = np.random.default_rng(0)
    C = random_target(rng, k)
    Yd = ImanConover().set_target(C)(Xd)
    assert torch.equal(torch.sort(Xd, dim=0).values, torch.sort(Yd, dim=0).values)
    assert torch.equal(Xd[:, 0], Yd[:, 0])
    R = torch.corrcoef(Yd.T).cpu().numpy()
    assert np.abs(R - C).max() < 0.01


@pytest.mark.parametrize("shape", [(9, 2), (5000, 6), (20000, 40)])
def test_cholesky_correlator_matches_oracle(shape):
    """Cholesky().set_target(C)(X) (reference correlation.py:205-285): float output, 1e-12."""
    from probabilit_b200 import Cholesky

    rng = np.random.default_rng(4)
    N, K = shape
    X = rng.normal(size=shape) * rng.uniform(0.5, 3, K) + rng.uniform(-5, 200, K)
    C = random_target(rng, K) if K > 2 else np.array([[1, 0.7], [0.7, 1]])
    want = oic.cholesky_correlator(X, C)
    got = Cholesky().set_target(C)(X)
    assert got.shape == want.shape and got.dtype == np.float64
    np.testing.assert_allclose(got, want, rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(np.corrcoef(got, rowvar=False), C, atol=1e-10)


def test_full_size_properties():
    """BASELINE.json configs[2] at full size (N = 1e8, d = 16; PBL_TEST_FULL_ROWS overrides): the
    reference cannot run this (~150 GB of host RAM), so the size-independent properties are checked
    on the device: every output column is a permutation of its input column, column 0 is unchanged
    (T[0,0] = 1), and the rank correlation of the result equals the target's to sampling accuracy."""
    import os

    import torch

    from bench import make_workload_device, target_matrix
    from probabilit_b200 import ImanConover

    n = int(float(os.environ.get("PBL_TEST_FULL_ROWS", "1e8")))
    d = 16
    free, _ = torch.cuda.mem_get_info()
    if free < n * d * 8 * 9:
        pytest.skip("not enough free device memory for the full-size case")
    X = make_workload_device(n, d, seed=99, torch=torch)
    Ct = target_matrix(d)
    Y = ImanConover().set_target(Ct)(X)
    assert Y.shape == X.shape and Y.stride() == X.stride()
    assert torch.equal(X[:, 0], Y[:, 0])
    # Exact fp64 ties between two of the 1e8 correlated scores of a column are expected about once per
    # column (birthday bound: N^2/2 * integral(pdf^2) * ulp ~ 0.5); the reference then gives both rows the
    # tie-run's midpoint value (correlation.py:422), so a column may differ from a permutation in a
    # handful of entries -- never more.
    mismatches = []
    for c in range(d):
        a, b = torch.sort(X[:, c]).values, torch.sort(Y[:, c]).values
        mismatches.append(int((a != b).sum().item()))
        del a, b
    print("entries per column that differ from a permutation (tie-runs of the correlated scores):", mismatches)
    assert max(mismatches) <= 16 and sum(mismatches) <= 64, mismatches
    # Spearman matrix of the result, on the device (pbl_corrcoef_f64)
    from probabilit_b200.correlation import corrcoef

    spearman = corrcoef(Y, spearman=True)
    # the induced rank correlation matches the target's rank correlation: for normal scores
    # rho_s = 6/pi * asin(rho/2)
    want = 6.0 / np.pi * np.arcsin(Ct / 2.0)
    assert np.max(np.abs(spearman - want)) < 5e-3, np.max(np.abs(spearman - want))


def config3_inputs(n, d, seed=0):
    """BASELINE.json configs[2] as SURVEY.md section 8(d) C3 spells it out: scrambled Sobol' quantiles
    (SciPy, `seed`) pushed through marginals cycling norm(1, 2) / triang(0.5) / gamma(a=2) by column."""
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # "balance properties of Sobol' points require n to be a power of 2"
        q = sp.stats.qmc.Sobol(d, seed=seed, scramble=True).random(n)
    X = np.empty((n, d), order="F")
    for c in range(d):
        dist = (sp.stats.norm(loc=1, scale=2), sp.stats.triang(0.5), sp.stats.gamma(a=2))[c % 3]
        X[:, c] = dist.ppf(q[:, c])
    return X


def test_config3_at_1e7_rows_is_bit_exact():
    """The headline configuration at the largest size the CPU oracle finishes in about a minute
    (N = 1e7, d = 16; SURVEY.md section 7, hard part 1: exact equality is expected up to N = 1e7):
    reference generator + SciPy ppfs on the host, output compared entry for entry."""
    import os

    from bench import target_matrix
    from probabilit_b200 import ImanConover

    n = int(float(os.environ.get("PBL_TEST_EXACT_ROWS", "1e7")))
    d = 16
    X = config3_inputs(n, d)
    assert np.isfinite(X).all()
    Ct = target_matrix(d)
    got = ImanConover().set_target(Ct)(X)
    want = oic.iman_conover(X, Ct)
    assert got.flags.f_contiguous and got.dtype == want.dtype
    np.testing.assert_array_equal(got, want)


def test_full_size_strided_columns_against_numpy():
    """N = 1e8, d = 16 (PBL_TEST_FULL_ROWS overrides), stage by stage on the device, two columns downloaded
    and re-derived on the host with NumPy (SURVEY.md section 7, hard part 1):  sortedX == np.sort(X[:, c]);
    scores within 4 ulp of ndtri(rankdata / (N + 1)); and the final index is exactly the reference's
    `rankdata(correlated).astype(int) - 1` of the DEVICE's correlated scores, i.e.
    Y[:, c] == np.sort(X[:, c])[midpoint_index(correlated[:, c])]  (correlation.py:419-423)."""
    import ctypes as C
    import os

    import torch
    from scipy.special import ndtri

    from bench import make_workload_device, target_matrix
    from probabilit_b200 import _lib
    from probabilit_b200.correlation import _IcPlan

    n = int(float(os.environ.get("PBL_TEST_FULL_ROWS", "1e8")))
    d = 16
    free, _ = torch.cuda.mem_get_info()
    if free < n * d * 8 * 9:
        pytest.skip("not enough free device memory for the full-size case")
    lib = _lib.require_gpu()
    X = make_workload_device(n, d, seed=7, torch=torch)
    Y = torch.empty_strided(X.shape, X.stride(), dtype=X.dtype, device=X.device)
    plan = _IcPlan(n, d, torch.cuda.current_device())
    plan.set_target(np.linalg.cholesky(target_matrix(d)))
    h, sp_ = plan.handle, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cols = (4, 11)  # a triang and a gamma marginal (column 0 takes the T[0,0] == 1 shortcut elsewhere)

    def grab(buffer_index):
        base = plan.buffer(buffer_index)[0]
        return [gpu_util.read_device(base + c * n * 8, (n,)) for c in cols]

    chk = _lib.check
    chk(lib.pbl_ic_stage_begin(h, sp_))
    chk(lib.pbl_ic_stage_rank_scores(h, X.data_ptr(), 1, n, 0, d, sp_))
    scores, sorted_x = grab(0), grab(1)
    chk(lib.pbl_ic_stage_gram(h, sp_))
    chk(lib.pbl_ic_stage_solve(h, n, sp_))
    chk(lib.pbl_ic_stage_transform(h, sp_))
    correlated = grab(0)
    chk(lib.pbl_ic_stage_rank_gather(h, Y.data_ptr(), 1, n, 0, d, sp_))
    assert chk(lib.pbl_ic_stage_status(h, sp_)) == 0
    for i, c in enumerate(cols):
        x = X[:, c].cpu().numpy()
        ranks, order = oic.average_ranks(x)
        np.testing.assert_array_equal(sorted_x[i], x[order])
        want_scores = ndtri(ranks / (n + 1))
        ulp = gpu_util.ulp_diff(scores[i], want_scores)
        # the bar is 4 ulp of SciPy's ndtri; over 1e8 points a handful land at 5 (CUDA's log and glibc's differ
        # in the last place for ~1e-3 of the tail-branch inputs, and x0 - x1 amplifies that by up to ~2):
        # the count is printed, bounded, and the maximum may not exceed 6
        over = int((ulp > 4.0).sum())
        print(f"column {c}: max {ulp.max():.1f} ulp vs scipy.special.ndtri, {over} of {n} scores beyond 4 ulp")
        assert ulp.max() <= 6.0 and over <= max(1, n // 1_000_000)
        del ranks, order, want_scores, ulp
        idx = oic.midpoint_index(correlated[i])
        np.testing.assert_array_equal(Y[:, c].cpu().numpy(), sorted_x[i][idx])
        del idx, x
    plan.close()


def test_column_longer_than_2_to_the_30_rows():
    """Columns of more than 2^30 rows (the previous limit of the look-back words; the 8-GPU weak-scaling run
    sorts 8e8-row columns): one column of 2^30 + 4099 doubles through the rank_scores stage.  Checked on the
    device: sortedX == torch.sort(X), and for a million sampled rows the score is ndtri(rank / (N + 1))."""
    import ctypes as C

    import torch
    from scipy.special import ndtri

    from probabilit_b200 import _lib
    from probabilit_b200.correlation import _IcPlan

    n = (1 << 30) + 4099
    free, _ = torch.cuda.mem_get_info()
    if free < n * 8 * 12:
        pytest.skip("not enough free device memory")
    lib = _lib.require_gpu()
    g = torch.Generator(device="cuda").manual_seed(5)
    X = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    plan = _IcPlan(n, 1, torch.cuda.current_device())
    plan.set_target(np.eye(1))
    h, sp_ = plan.handle, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.pbl_ic_stage_begin(h, sp_))
    _lib.check(lib.pbl_ic_stage_rank_scores(h, X.data_ptr(), 1, n, 0, 1, sp_))
    assert _lib.check(lib.pbl_ic_stage_status(h, sp_)) == 0
    from probabilit_b200.distributed import _DevBuf

    scores = torch.as_tensor(_DevBuf(plan.buffer(0)[0], (n,)), device="cuda")
    sorted_x = torch.as_tensor(_DevBuf(plan.buffer(1)[0], (n,)), device="cuda")
    want_sorted = torch.sort(X).values
    assert torch.equal(sorted_x, want_sorted)
    del want_sorted
    idx = torch.randint(0, n, (1_000_000,), generator=g, device="cuda")
    rank = torch.searchsorted(sorted_x, X[idx]) + 1  # untied: 1-based rank
    got = scores[idx].cpu().numpy()
    want = ndtri(rank.cpu().numpy() / (n + 1.0))
    assert gpu_util.ulp_diff(got, want).max() <= 6.0
    plan.close()


@pytest.mark.parametrize("n,k", [(3000, 100), (2500, 257)])
def test_wide_problem_uses_grid_cholesky(n, k):
    """k > 64: correlation / Cholesky / T are computed by the cooperative multi-block kernel."""
    from probabilit_b200 import Cholesky, ImanConover

    rng = np.random.default_rng(21)
    X = np.asfortranarray(rng.normal(size=(n, k)))
    C = random_target(rng, k)
    ref = oic.iman_conover_stages(X, C)
    got = gpu_util.run_stages(X, C)
    assert got["status"] == 0
    np.testing.assert_allclose(got["T"], ref["T"], rtol=0, atol=1e-10)
    np.testing.assert_array_equal(got["result"], ref["result"])
    np.testing.assert_array_equal(ImanConover().set_target(C)(X), oic.iman_conover(X, C))
    np.testing.assert_allclose(Cholesky().set_target(C)(X), oic.cholesky_correlator(X, C), rtol=1e-10, atol=1e-10)
    # perfectly collinear scores -> not positive definite, detected consistently by every block
    Xd = X.copy()
    Xd[:, 1] = Xd[:, 0]
    with pytest.raises(ValueError, match="not positive definite"):
        ImanConover().set_target(C)(Xd)


def test_device_corrcoef_pearson_and_spearman():
    """pbl_corrcoef_f64 against np.corrcoef / scipy.stats.spearmanr (1e-12), incl. ties."""
    from probabilit_b200.correlation import corrcoef

    rng = np.random.default_rng(30)
    X = rng.normal(size=(20_000, 5)) @ rng.normal(size=(5, 5))
    X[:, 2] = rng.poisson(4.0, 20_000)
    np.testing.assert_allclose(corrcoef(X), np.corrcoef(X, rowvar=False), rtol=0, atol=1e-12)
    np.testing.assert_allclose(corrcoef(X, spearman=True), sp.stats.spearmanr(X).statistic, rtol=0, atol=1e-12)
