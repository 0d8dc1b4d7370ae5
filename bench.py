#!/usr/bin/env python
"""Headline benchmark: Iman-Conover samples*vars/s (fp64, N=1e8 rows per GPU, d=16).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --gpus N --scaling strong  # N=1e8 rows in total, 1e8 / N per GPU
    python bench.py --impl reference          # the reference's CPU path (oracle port) on the host
    python bench.py --dump-outputs DIR        # also write the last timed step's result as DIR/Y.npy

A step = one ImanConover.__call__-equivalent over one (N, d) batch of synthetic input:
  value  device-resident (inputs already in HBM), CUDA events on the launching stream
  e2e    the public API call ImanConover().set_target(C)(X) with HOST (pinned) buffers, the
         host->device and device->host copies inside the timed region
Prints ONE JSON line (rank 0).  The inputs depend on the arguments only (seeded), so the Y.npy of two
builds of the project can be compared entry for entry.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "iman_conover_samples_vars_per_s"
UNIT = "samples*vars/s"
IC_BYTES_PER_SAMPLE_VAR = 456.0  # SURVEY.md section 8(d): fixed algorithmic accounting
# one digit pass moves 12 B in + 12 B out per key (u64 key + u32 row); the first of the 4 passes of the
# 32-bit window reads the 8 B double instead of 12 B
PASS_BYTES_PER_KEY = (3 * 24.0 + 20.0) / 4.0
# measured DRAM traffic of one digit pass, dram__bytes_read.sum + dram__bytes_write.sum per key, from the
# `ncu --set full` capture of the bench-size launches (N=1e8 x 16 = 1.6e9 keys per launch; raw CSV and
# summary: profiles/r2_ncu_n1e8_*): see PASS_DRAM_BYTES_NCU_SOURCE
PASS_DRAM_BYTES_PER_KEY_NCU = 23.7
PASS_DRAM_BYTES_NCU_SOURCE = ("ncu --set full capture AT THE BENCH SIZE (N=1e8 x 16 = 1.6e9 keys per launch; "
                              "profiles/r2_ncu_full_n1e8_summary.txt + _raw.csv): 13.10 GB read + 20.05 GB written by "
                              "the pass that reads the raw doubles, 19.42 + 20.05 GB by each of the other three -> "
                              "23.7 B/key on average (23 algorithmic), scaled to this launch's keys")


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def target_matrix(d):
    """Recipe of the reference's tests/test_iman_conover.py:154-155, seed 0."""
    rng = np.random.default_rng(0)
    A = rng.normal(size=(2 * d, d))
    return 0.9 * np.corrcoef(A, rowvar=False) + 0.1 * np.eye(d)


MARGINALS = ("norm(loc=1, scale=2)", "triang(c=0.5)", "gamma(a=2)")  # cycling by column (SURVEY.md 8d, C3)


def make_workload_device(n, d, seed, torch, skip=0, timings=None):
    """(n, d) fp64, column-major on the device, BASELINE.json configs[2] as SURVEY.md section 8(d) C3 states
    it: scrambled Sobol' quantiles (probabilit_b200.qmc.Sobol, bit-identical with SciPy's for the seed) pushed
    through the marginals norm(1, 2) / triang(0.5) / gamma(a=2) cycling by column with the library's ppf
    kernels (pbl_ppf_f64, in place).  `skip`: rows of the sequence to skip (rank r of a multi-GPU run takes
    rows [r*n, (r+1)*n)).  `timings`: dict that receives the device times of the two kernels."""
    import warnings

    from probabilit_b200 import _lib, qmc

    lib = _lib.require_gpu()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    eng = qmc.Sobol(d, seed=seed, scramble=True)
    eng.fast_forward(skip)
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # "balance properties of Sobol' points require n to be a power of 2"
        X = eng.random(n, device=True)  # (n, d) view with strides (1, n)
    e1.record()
    # 30-bit Sobol' points are multiples of 2^-30 and a scrambled point can be exactly 0 (once in 1.6e9 values
    # for this seed); norm.ppf(0) = -inf would leave the column with an infinite value, so such a point is
    # moved to 2^-31 (a user of Node.sample has to do the same to keep the model finite)
    X.clamp_(min=2.0 ** -31)
    e1b = torch.cuda.Event(enable_timing=True)
    e1b.record()
    PPF = {0: (16, 1.0, 2.0, 0.0), 1: (19, 0.5, 0.0, 1.0), 2: (20, 2.0, 0.0, 1.0)}  # PBL_PPF_NORM / TRIANG / GAMMA
    for c in range(d):
        what, p0, p1, p2 = PPF[c % 3]
        ptr = C.c_void_p(X.data_ptr() + c * n * 8)
        _lib.check(lib.pbl_ppf_f64(what, ptr, n, p0, p1, p2, ptr, stream), "pbl_ppf_f64")
    e2.record()
    torch.cuda.synchronize()
    if timings is not None:
        t_gen, t_ppf = e0.elapsed_time(e1) * 1e-3, e1b.elapsed_time(e2) * 1e-3
        timings.update({
            "sobol": {"ms": t_gen * 1e3, "samples_vars_per_s": n * d / t_gen, "bytes_per_sample_var": 8,
                      "GB_per_s": 8.0 * n * d / t_gen / 1e9},
            "ppf": {"ms": t_ppf * 1e3, "samples_vars_per_s": n * d / t_ppf, "bytes_per_sample_var": 16,
                    "GB_per_s": 16.0 * n * d / t_ppf / 1e9, "marginals": list(MARGINALS)}})
    return X


def make_workload_host(n, d, seed):
    """The same workload from the reference stack on the host (scipy.stats.qmc.Sobol + scipy ppfs)."""
    import warnings

    import scipy.stats as st

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        q = st.qmc.Sobol(d, seed=seed, scramble=True).random(n)
    X = np.empty((n, d), order="F")
    for c in range(d):
        u = q[:, c]
        if c % 3 == 0:
            X[:, c] = st.norm(loc=1, scale=2).ppf(u)
        elif c % 3 == 1:
            X[:, c] = st.triang(0.5).ppf(u)
        else:
            X[:, c] = st.gamma(a=2).ppf(u)
    return X


class ClockSampler:
    """nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "200", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smmax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smmax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val == "Active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smmax)) if smmax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_BYTES = 48 << 20  # below the 64 MB a dump may take, .npy header included


def dump_rows(n, d):
    """Rows of the (n, d) fp64 result that --dump-outputs writes: all of them if they fit in DUMP_BYTES, else
    a sample drawn with a fixed seed (the same rows for the same n and d), in ascending order."""
    m = DUMP_BYTES // (8 * d)
    if n <= m:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=m, replace=False))


def dump_outputs(out_dir, Y):
    """out_dir/Y.npy: the rows dump_rows() picks of the result Y (NumPy array or CUDA tensor), float64."""
    rows = dump_rows(*Y.shape)
    if isinstance(Y, np.ndarray):
        sample = Y[rows]
    else:
        import torch

        sample = Y[torch.from_numpy(rows).to(Y.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "Y.npy"), np.ascontiguousarray(sample, dtype=np.float64))


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([i.get("num_threads", 1) for i in threadpool_info()] or [1])
    except Exception:
        return os.cpu_count() or 1


def time_cpu_port(n_rows, d, reps=1):
    """The reference's CPU path (oracle port: same SciPy/NumPy calls, oracle/iman_conover.py)."""
    from oracle import iman_conover as oic

    X = make_workload_host(n_rows, d, seed=1)
    Ct = target_matrix(d)
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        oic.iman_conover(X, Ct)
        best = min(best, time.perf_counter() - t0)
    return n_rows * d / best, best


def time_graph(n, lib):
    """Secondary line (BASELINE.json configs[1]): the README mutual-fund graph (20 norm ppf + 40
    arithmetic nodes) evaluated by the fused graph kernel, quantiles generated in-kernel (Philox),
    only the sink retained.  Host wall time of the synchronous evaluation, best of 3."""
    import probabilit_b200.modeling as m

    returns = 0
    for _ in range(20):
        returns = returns * m.Distribution("norm", loc=1.11, scale=0.15) + 1200
    best = float("inf")
    for rep in range(6):
        run = m._GraphRun(returns, m._PhiloxSource(rep, n, 20), "imanconover", [])
        lib.pbl_stream_synchronize(None)
        t0 = time.perf_counter()
        run.execute()
        lib.pbl_stream_synchronize(None)
        if rep:
            best = min(best, time.perf_counter() - t0)
    return {"workload": f"README mutual-fund graph, n={n}, 20 norm ppf + 40 arithmetic nodes, in-kernel Philox, "
                        "sink retained", "ms": best * 1e3, "samples_per_s": n / best,
            "distribution_samples_per_s": 20 * n / best, "bound": "fp64/integer ALU (20 ndtri per 8 B written)",
            "hbm_bytes_per_sample": 8}


# ------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    d = args.d
    n_ref = args.ref_rows
    if n_ref <= 0:
        # as many rows per step as keep the whole --steps/--warmup run within ~4 minutes (the CPU path
        # takes ~5.5 us per row at d=16 around 1e6-1e7 rows), at most 1e7 (15 GB of host RAM)
        n_ref = int(min(1e7, max(2e5, 240.0 / ((args.steps + args.warmup) * 5.5e-6))))
    from oracle import iman_conover as oic

    X = make_workload_host(n_ref, d, seed=0)
    Ct = target_matrix(d)
    for _ in range(args.warmup):
        oic.iman_conover(X, Ct)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        Y = oic.iman_conover(X, Ct)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, Y)
    value = n_ref * d * args.steps / dt
    sample = (f"{n_ref} of the {args.n} rows x d={d} per step (the full N needs ~150 GB of host RAM in "
              "the reference); same marginals and target as the GPU arm")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"Iman-Conover fp64 N={args.n} rows per GPU, d={d}, mixed norm/triang/gamma "
                               "marginals on scrambled Sobol' quantiles (BASELINE.json configs[2])",
                   "rows_per_gpu": args.n, "d": d, "cpu_rows_per_step": n_ref,
                   "note": "the reference's NumPy/SciPy path (oracle port) on the host cores; each step is a "
                           "bounded row sample of the workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": blas_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def multi_gpu_parity_check(n_small, d, Ct, rank, world, local_rank, dist, torch, lib):
    """G-GPU == 1-GPU, bit for bit, before anything is timed (the driver's pytest box has one GPU, so this
    is where the multi-GPU path is checked at round end): the same workload at n_small rows per GPU through
    DistributedImanConover, gathered on rank 0 and compared with the single-plan result of the whole matrix."""
    from probabilit_b200 import _lib
    from probabilit_b200.correlation import _IcPlan
    from probabilit_b200.distributed import DistributedImanConover

    Xs = make_workload_device(n_small, d, seed=0, torch=torch, skip=rank * n_small)
    Ys = torch.empty_strided(Xs.shape, Xs.stride(), dtype=Xs.dtype, device=Xs.device)
    small = DistributedImanConover(n_small, d, Ct, dist)
    small.run(Xs, Ys)
    small.close()
    # shards as [d][n_small] blocks; rank 0 stitches the (world * n_small, d) matrices together column-major
    xs = [torch.empty((d, n_small), dtype=torch.float64, device="cuda") for _ in range(world)]
    ys = [torch.empty((d, n_small), dtype=torch.float64, device="cuda") for _ in range(world)]
    dist.all_gather(xs, Xs.T.contiguous())
    dist.all_gather(ys, Ys.T.contiguous())
    verdict = torch.zeros(2, dtype=torch.int64, device="cuda")
    if rank == 0:
        nt = n_small * world
        Xf = torch.cat(xs, dim=1).contiguous()  # [d][nt]
        Yf = torch.empty_like(Xf)
        plan = _IcPlan(nt, d, local_rank)
        plan.set_target(np.linalg.cholesky(Ct))
        st = lib.pbl_ic_plan_run(plan.handle, Xf.data_ptr(), 1, nt, Yf.data_ptr(), 1, nt,
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
        plan.close()
        if st != 0:
            raise RuntimeError(f"parity check: pbl_ic_plan_run status {st}: {_lib.last_error()}")
        got = torch.cat(ys, dim=1)
        verdict[0] = int(torch.equal(got, Yf))
        verdict[1] = int((got != Yf).sum().item())
        del Xf, Yf, got
    dist.broadcast(verdict, 0)
    del xs, ys, Xs, Ys
    torch.cuda.empty_cache()
    if not int(verdict[0].item()):
        raise RuntimeError(f"bench: the {world}-GPU result differs from the single-GPU result in "
                           f"{int(verdict[1].item())} entries")
    return {"what": f"{world}-GPU DistributedImanConover == single-GPU plan, bit for bit",
            "rows_per_gpu": n_small, "rows_total": n_small * world, "d": d, "equal": True}


# ------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch

    from probabilit_b200 import ImanConover, _lib
    from probabilit_b200.correlation import _IcPlan

    lib = _lib.require_gpu()  # raises without the CUDA library / a GPU: no fallback
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    d = args.d
    n = args.n // world if args.scaling == "strong" else args.n  # rows on this GPU
    Ct = target_matrix(d)
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)

    parity = None
    if world > 1 and args.parity_rows > 0:
        parity = multi_gpu_parity_check(args.parity_rows, d, Ct, rank, world, local_rank, dist, torch, lib)

    gen = {}
    # one Sobol' sequence for the whole job: rank r holds its rows [r*n, (r+1)*n)
    X = make_workload_device(n, d, seed=0, torch=torch, skip=rank * n, timings=gen)
    Y = torch.empty_strided(X.shape, X.stride(), dtype=X.dtype, device=X.device)

    if world > 1:
        from probabilit_b200.distributed import DistributedImanConover
        runner = DistributedImanConover(n, d, Ct, dist)
        step = lambda: runner.run(X, Y)  # noqa: E731
    else:
        plan = _IcPlan(n, d, local_rank, args.col_batch)
        plan.set_target(np.linalg.cholesky(Ct))

        def step():
            st = lib.pbl_ic_plan_run(plan.handle, X.data_ptr(), X.stride(0), X.stride(1),
                                     Y.data_ptr(), Y.stride(0), Y.stride(1), sp)
            if st != 0:
                raise RuntimeError(f"pbl_ic_plan_run status {st}: {_lib.last_error()}")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    lib.pbl_sort_profile_enable(1)
    launches0 = _lib.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.kernel_launches() - launches0
    nl, pms, nkeys = C.c_int64(), C.c_double(), C.c_int64()
    lib.pbl_sort_profile_read(C.byref(nl), C.byref(pms), C.byref(nkeys))
    lib.pbl_sort_profile_enable(0)
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = float(n) * d * world * args.steps / (ms * 1e-3)

    # parity guard inside the bench: Y is a per-column permutation of X (column 0 untouched)
    if not torch.equal(X[:, 0], Y[:, 0]):
        raise RuntimeError("bench: column 0 changed -- the transform is broken")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, Y)

    # ---- e2e through the public API with host (pinned) buffers ----
    e2e = None
    if world == 1 and args.e2e_steps > 0:
        nbytes = n * d * 8
        hx, hy = C.c_void_p(), C.c_void_p()
        _lib.check(lib.pbl_host_malloc_pinned(C.byref(hx), nbytes))
        _lib.check(lib.pbl_host_malloc_pinned(C.byref(hy), nbytes))
        Xh = np.ctypeslib.as_array(C.cast(hx, C.POINTER(C.c_double)), shape=(d, n)).T
        Yh = np.ctypeslib.as_array(C.cast(hy, C.POINTER(C.c_double)), shape=(d, n)).T
        _lib.check(lib.pbl_memcpy_d2h(hx, C.c_void_p(X.data_ptr()), nbytes, None))
        _lib.check(lib.pbl_stream_synchronize(None))
        plan.close()  # the public-API object below owns its own workspace
        torch.cuda.synchronize()
        ic = ImanConover(device=local_rank, col_batch=args.col_batch).set_target(Ct)
        ic(Xh, out=Yh)  # warm-up (allocates the device workspace)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            ic(Xh, out=Yh)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if not np.array_equal(Xh[:1000, 0], Yh[:1000, 0]):
            raise RuntimeError("bench e2e: column 0 changed")
        e2e = {"value": float(n) * d * args.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
               "steps": args.e2e_steps, "ms_per_step": dt / args.e2e_steps * 1e3,
               "api": "probabilit_b200.ImanConover().set_target(C)(X_host, out=Y_host_pinned)"}
        ic.close()
        lib.pbl_host_free_pinned(hx)
        lib.pbl_host_free_pinned(hy)

    if world > 1 and args.e2e_steps > 0:
        # every rank's row shard starts and ends in pinned HOST memory: H2D of the shard, the multi-GPU call,
        # D2H of the result, all inside the timed region (wall clock, max over ranks)
        nbytes = n * d * 8
        hx, hy = C.c_void_p(), C.c_void_p()
        ok = lib.pbl_host_malloc_pinned(C.byref(hx), nbytes) == 0 and lib.pbl_host_malloc_pinned(C.byref(hy), nbytes) == 0
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)  # every rank takes the same branch
        ok = bool(flag.item())
    if world > 1 and args.e2e_steps > 0 and not ok:
        for h in (hx, hy):
            if h.value:
                lib.pbl_host_free_pinned(h)
        e2e = {"value": None, "unit": UNIT, "note": "pinned host buffers could not be allocated on every rank"}
    if world > 1 and args.e2e_steps > 0 and ok:
        Xh = np.ctypeslib.as_array(C.cast(hx, C.POINTER(C.c_double)), shape=(d, n)).T
        Yh = np.ctypeslib.as_array(C.cast(hy, C.POINTER(C.c_double)), shape=(d, n)).T
        _lib.check(lib.pbl_memcpy_d2h(hx, C.c_void_p(X.data_ptr()), nbytes, sp))
        torch.cuda.synchronize()

        def e2e_step():
            runner.run_host(Xh, Yh)  # H2D / D2H per exchange round, overlapped with the sorts
            torch.cuda.synchronize()

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        if not np.array_equal(Xh[:1000, 0], Yh[:1000, 0]):
            raise RuntimeError("bench e2e: column 0 changed")
        e2e = {"value": float(n) * d * world * args.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": nbytes * world, "d2h_bytes_per_step": nbytes * world,
               "steps": args.e2e_steps, "ms_per_step": dt / args.e2e_steps * 1e3,
               "api": "probabilit_b200.distributed.DistributedImanConover.run_host: every rank's row shard starts "
                      "and ends in pinned host memory (one PCIe link per GPU); the copies go column by column, "
                      "overlapped with the exchange rounds and the sorts"}
        lib.pbl_host_free_pinned(hx)
        lib.pbl_host_free_pinned(hy)

    graph = None
    if world == 1 and args.graph_rows > 0:
        graph = time_graph(args.graph_rows, lib)

    if world > 1:
        runner.close()  # collective: unmaps the peers' buffers before anybody frees them
    if rank != 0:
        dist.destroy_process_group()
        return
    peak, peak_src = hbm_peak()
    pass_gbs = PASS_BYTES_PER_KEY * nkeys.value / (pms.value * 1e-3) / 1e9 if pms.value > 0 else None
    roofline = {
        "kernel": "pass_tma_kernel (one onesweep radix digit pass over all columns of a batch; persistent, "
                  "cp.async.bulk + mbarrier double-buffered tiles)",
        "bound": "hbm", "achieved": pass_gbs, "peak": peak, "unit": "GB/s",
        "frac": (pass_gbs / peak) if pass_gbs else None,
        "traffic": PASS_DRAM_BYTES_PER_KEY_NCU * nkeys.value / max(nl.value, 1),
        "traffic_source": PASS_DRAM_BYTES_NCU_SOURCE,
        "peak_source": peak_src,
        "launches_timed": nl.value, "avg_launch_ms": (pms.value / nl.value) if nl.value else None,
        "algorithmic_bytes_per_launch": PASS_BYTES_PER_KEY * nkeys.value / max(nl.value, 1),
        "share_of_step": pms.value / ms if ms > 0 else None,
        "pipeline": {"algorithmic_bytes_per_sample_var": IC_BYTES_PER_SAMPLE_VAR,
                     "achieved": IC_BYTES_PER_SAMPLE_VAR * value / world / 1e9,
                     "frac": IC_BYTES_PER_SAMPLE_VAR * value / world / 1e9 / peak},
    }
    cpu = None
    if world == 1 and args.cpu_rows > 0:
        v, secs = time_cpu_port(args.cpu_rows, d)
        cpu = {"value": v, "unit": UNIT, "cores": blas_threads(), "kind": "port",
               "seconds": secs,
               "sample": f"first-principles same workload at {args.cpu_rows} rows x d={d} (1 run); "
                         "sorts/ndtri are single-threaded NumPy/SciPy, only BLAS uses the threads"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"Iman-Conover fp64 N={n} rows per GPU ({n * world} in total), d={d}, marginals "
                               "norm(1,2) / triang(0.5) / gamma(2) cycling by column on scrambled Sobol' "
                               "quantiles (seed 0), generated on the device by the library's own Sobol' and "
                               "ppf kernels (BASELINE.json configs[2], SURVEY.md 8d C3)",
                   "rows_per_gpu": n, "rows_total": n * world, "d": d,
                   "l2": f"inputs ({n * d * 8 / 1e9:.1f} GB per GPU) far exceed the 126 MB L2",
                   "col_batch": args.col_batch,
                   **({"transport": "row <-> column transposes by copy engines over CUDA-IPC peer mappings "
                                    "(NVLink), NCCL for the Gram all-reduce and the barriers"} if world > 1 else {})},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
        "clocks": clocks, "generator": gen, "parity_check": parity, "graph": graph,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", dest="n", type=lambda s: int(float(s)), default=100_000_000)
    ap.add_argument("--d", type=int, default=16)
    ap.add_argument("--col-batch", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-rows", type=lambda s: int(float(s)), default=3_000_000)
    ap.add_argument("--ref-rows", type=lambda s: int(float(s)), default=0,
                    help="rows per step of the reference arm (0: sized to the --steps/--warmup budget)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --rows per GPU; strong: --rows in total, split over the GPUs")
    ap.add_argument("--parity-rows", type=lambda s: int(float(s)), default=1_000_000,
                    help="rows per GPU of the multi-GPU == single-GPU check that precedes the timing (0: skip)")
    ap.add_argument("--graph-rows", type=lambda s: int(float(s)), default=100_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/Y.npy (float64; a seeded sample of "
                         "whole rows when it exceeds 48 MB; rank 0's rows in a multi-GPU run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the ONE JSON line only: whatever a library writes to file descriptor 1 meanwhile
    # (NCCL prints its version banner there) goes to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
