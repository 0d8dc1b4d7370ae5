"""Statistics of sampled nodes on the device, bit-identical to NumPy on the host copy.

    from probabilit_b200 import stats
    stats.mean(x); stats.var(x, ddof=0); stats.std(x, ddof=0)
    stats.quantile(x, q, method="linear"); stats.percentile(x, q, method="linear")
    stats.min(x); stats.max(x); stats.ptp(x)
    stats.histogram(x, bins=10, range=None, density=None); stats.histogram_bin_edges(x, bins=10, range=None)

``x`` is a sampled ``Node``, a column ``(DeviceColumns, j)``, a 1-D contiguous CUDA array (``<f8`` or ``<i8``,
``__cuda_array_interface__``: torch tensors included), or a list of ``Node``s of one ``n`` (then the result is a
list, computed in one pass over all columns).  The result equals ``np.mean(node.samples_)`` ... ``np.percentile``,
``np.min`` ... ``np.histogram`` bit for bit, with NumPy's dtype and shape; the column is never copied to the host.
Samples that only exist on the host (folded constants, ``samples_`` set by the caller) are uploaded and reduced by the
same kernels (csrc/stats.cu).  Arguments are checked before any device call, with NumPy's exception types.
"""
import builtins
import ctypes as C
import operator
import warnings

import numpy as np

from . import _lib
from ._device import DeviceColumns

F64, I64_BITS, I64_AS_F64, BOOL_AS_F64 = range(4)  # pbl_stats_kind
MEAN, VAR, STD = range(3)  # pbl_stats_moment
METHODS = {"linear": 0, "lower": 1, "higher": 2, "nearest": 3, "midpoint": 4, "closest_observation": 5}
# the other methods np.quantile knows (NotImplementedError here; an unknown name is NumPy's ValueError)
_NUMPY_ONLY_METHODS = {"inverted_cdf", "averaged_inverted_cdf", "interpolated_inverted_cdf", "hazen", "weibull",
                       "median_unbiased", "normal_unbiased"}
_F64, _I64, _BOOL = np.dtype(np.float64), np.dtype(np.int64), np.dtype(np.bool_)


class _Column:
    """One input column: a device address and its encoding, or host values still to upload."""

    def __init__(self, dtype, n, ptr=None, kind=None, keep=None, host=None):
        self.dtype, self.n, self.ptr, self.kind, self.keep, self.host = dtype, n, ptr, kind, keep, host

    def upload(self):
        """Host values -> a device column (kept alive by this object)."""
        if self.ptr is None:
            if self.dtype == _I64:
                bits, self.kind = self.host.view(np.float64), I64_BITS
            else:
                bits, self.kind = self.host.astype(np.float64), (F64 if self.dtype == _F64 else BOOL_AS_F64)
            self.keep = DeviceColumns.from_host(bits.reshape(-1, 1))
            self.ptr = self.keep.column_ptr(0)


def _host_column(values):
    if values is None:
        raise TypeError("the node's samples_ is None (a NoOp has no samples)")
    arr = np.asarray(values)
    if arr.dtype.kind in "OUSV":
        raise TypeError(f"statistics of non-numeric samples (dtype {arr.dtype}) are not defined")
    if arr.ndim != 1:
        raise NotImplementedError("statistics of samples_ that are not 1-D")
    if arr.dtype not in (_F64, _I64, _BOOL):
        raise NotImplementedError(f"statistics of {arr.dtype} samples")
    return _Column(arr.dtype, arr.shape[0], host=np.ascontiguousarray(arr))


def _node_column(node):
    store = node.__dict__.get("_store")
    if store is None:
        raise AttributeError(f"{type(node).__name__!r} object has no attribute 'samples_'")
    if store.none:
        return _host_column(None)
    if store.columns is None:  # folded constant, or samples_ set on the host
        return _host_column(store._host if store.const is None else store.host())
    if store.categories is not None:
        raise TypeError(f"statistics of non-numeric samples (dtype {store.categories.dtype}) are not defined")
    dtype = np.dtype(store.dtype)
    if store.ibits:
        kind = I64_BITS
    elif dtype == _F64:
        kind = F64
    elif dtype == _BOOL:
        kind = BOOL_AS_F64
    elif dtype == _I64:
        kind = I64_AS_F64
    else:
        raise NotImplementedError(f"statistics of {dtype} samples")
    return _Column(dtype, store.columns.n, ptr=store.columns.column_ptr(store.index), kind=kind, keep=store.columns)


def _cuda_column(x, cai):
    shape, strides = tuple(cai["shape"]), cai.get("strides")
    if len(shape) != 1:
        raise NotImplementedError("statistics of device arrays that are not 1-D (axis= is not supported)")
    if cai["typestr"] not in ("<f8", "<i8"):
        raise TypeError(f"device arrays must be <f8 or <i8, not {cai['typestr']}")
    if strides is not None and shape[0] > 1 and tuple(strides) != (8,):
        raise ValueError("device arrays must be contiguous")
    if type(x).__module__.startswith("torch"):  # the library runs on the default stream
        import torch

        torch.cuda.current_stream(x.device).synchronize()
    dtype = _F64 if cai["typestr"] == "<f8" else _I64
    return _Column(dtype, int(shape[0]), ptr=int(cai["data"][0]), kind=F64 if dtype == _F64 else I64_BITS, keep=x)


def _columns(x):
    """-> (list of _Column, batched).  No device call."""
    from .modeling import Node

    if isinstance(x, (list, tuple)) and not (len(x) == 2 and isinstance(x[0], DeviceColumns)):
        if not x or not all(isinstance(v, Node) for v in x):
            raise TypeError("a batch of statistics is a non-empty list of sampled Nodes")
        cols = [_node_column(v) for v in x]
        if len({c.n for c in cols}) != 1:
            raise ValueError("every node of a batch must have the same number of samples")
        return cols, True
    if isinstance(x, Node):
        return [_node_column(x)], False
    if isinstance(x, tuple):
        cols, j = x
        return [_Column(_F64, cols.n, ptr=cols.column_ptr(int(j)), kind=F64, keep=cols)], False
    cai = getattr(x, "__cuda_array_interface__", None)
    if cai is not None and not isinstance(x, np.ndarray):
        return [_cuda_column(x, cai)], False
    raise TypeError(f"expected a sampled Node, (DeviceColumns, j), a CUDA array or a list of Nodes, not {type(x)!r}")


def _no_extras(**kwargs):
    for name, (value, default) in kwargs.items():
        if value is not default:
            raise NotImplementedError(f"stats: {name}= is not supported")


def _pointers(cols):
    for c in cols:
        c.upload()
    ptrs = (C.c_void_p * len(cols))(*[c.ptr for c in cols])
    kinds = (C.c_int32 * len(cols))(*[c.kind for c in cols])
    return ptrs, kinds


def _moment(x, what, ddof):
    cols, batched = _columns(x)
    n = cols[0].n
    if n == 0:  # nothing to reduce: NumPy's own result (nan) and warning
        out = [np.float64((np.mean, np.var, np.std)[what](np.empty(0, c.dtype), **({} if what == MEAN else {"ddof": ddof})))
               for c in cols]
        return out if batched else out[0]
    divisor = 0.0
    if what != MEAN:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            divisor = float(np.maximum(n - ddof, 0))  # numpy/_core/_methods.py:_var, rcount = max(n - ddof, 0)
    lib = _lib.require_gpu()
    ptrs, kinds = _pointers(cols)
    res = np.empty(len(cols), dtype=np.float64)
    _lib.check(lib.pbl_stats_moments(ptrs, kinds, len(cols), n, int(np.getbufsize()), what, divisor,
                                     res.ctypes.data, None), "pbl_stats_moments")
    if what != MEAN and n - ddof <= 0:
        warnings.warn("Degrees of freedom <= 0 for slice", RuntimeWarning, stacklevel=3)
    out = [np.float64(v) for v in res]
    return out if batched else out[0]


def mean(x, axis=None, dtype=None, out=None, keepdims=False):
    """``np.mean(x.samples_)``, computed on the device."""
    _no_extras(axis=(axis, None), dtype=(dtype, None), out=(out, None), keepdims=(keepdims, False))
    return _moment(x, MEAN, 0)


def var(x, axis=None, dtype=None, out=None, ddof=0, keepdims=False):
    """``np.var(x.samples_, ddof=ddof)``, computed on the device."""
    _no_extras(axis=(axis, None), dtype=(dtype, None), out=(out, None), keepdims=(keepdims, False))
    return _moment(x, VAR, ddof)


def std(x, axis=None, dtype=None, out=None, ddof=0, keepdims=False):
    """``np.std(x.samples_, ddof=ddof)``, computed on the device."""
    _no_extras(axis=(axis, None), dtype=(dtype, None), out=(out, None), keepdims=(keepdims, False))
    return _moment(x, STD, ddof)


def _quantiles(x, q, method, percent):
    cols, batched = _columns(x)
    n = cols[0].n
    numpy_fn = np.percentile if percent else np.quantile
    # NumPy itself on two values of each dtype: its range check, its TypeError for interpolating bool, and the
    # dtype and shape of the result
    protos = [numpy_fn(np.zeros(2, dtype=c.dtype), q, method=method) for c in cols]
    if method not in METHODS:
        raise NotImplementedError(f"method={method!r} is not supported on the device: use one of {list(METHODS)}")
    if n == 0:
        out = [numpy_fn(np.empty(0, dtype=c.dtype), q, method=method) for c in cols]
        return out if batched else out[0]
    code = METHODS[method]
    per_col = []  # (q as NumPy uses it, method) per column: it depends on the column's dtype
    for c in cols:
        if percent:
            qa = np.true_divide(q, c.dtype.type(100) if c.dtype.kind == "f" else 100)
        elif isinstance(q, (int, float)) and c.dtype.kind == "f":
            qa = np.asanyarray(q, dtype=c.dtype)
        else:
            qa = np.asanyarray(q)
        if qa.dtype.kind in "biu":
            # integer q: (n - 1) * q is an integer index and "linear" takes that element (no interpolation)
            per_col.append((qa.astype(np.float64), METHODS["lower"] if code == METHODS["linear"] else code))
        elif qa.dtype == _F64:
            per_col.append((qa, code))
        else:
            raise NotImplementedError(f"q of dtype {qa.dtype} (NumPy computes its indices in that precision)")
    lib = _lib.require_gpu()
    results = [None] * len(cols)
    # one call per distinct (q, method): a batch of one dtype is one call
    todo = list(range(len(cols)))
    while todo:
        qa, m = per_col[todo[0]]
        same = [i for i in todo if per_col[i][1] == m and np.array_equal(per_col[i][0], qa)]
        todo = [i for i in todo if i not in same]
        sub = [cols[i] for i in same]
        ptrs, kinds = _pointers(sub)
        qf = np.ascontiguousarray(qa, dtype=np.float64).ravel()
        raw = np.empty((len(sub), qf.size), dtype=np.int64)
        _lib.check(lib.pbl_stats_quantiles(ptrs, kinds, len(sub), n, qf.ctypes.data_as(C.POINTER(C.c_double)),
                                           qf.size, m, raw.ctypes.data, None), "pbl_stats_quantiles")
        for row, i in enumerate(same):
            c, proto = cols[i], protos[i]
            vals = raw[row]
            if m in (METHODS["linear"], METHODS["midpoint"]) or c.kind == F64 or c.dtype == _F64:
                vals = vals.view(np.float64)
            elif c.dtype == _BOOL:
                vals = vals != 0
            arr = vals.astype(np.asarray(proto).dtype, copy=False).reshape(np.shape(proto))
            results[i] = arr if isinstance(proto, np.ndarray) else arr[()]
    return results if batched else results[0]


def quantile(x, q, method="linear", axis=None, out=None, keepdims=False, *, weights=None):
    """``np.quantile(x.samples_, q, method=method)``, computed on the device."""
    _no_extras(axis=(axis, None), out=(out, None), keepdims=(keepdims, False), weights=(weights, None))
    return _quantiles(x, q, method, percent=False)


def percentile(x, q, method="linear", axis=None, out=None, keepdims=False, *, weights=None):
    """``np.percentile(x.samples_, q, method=method)``, computed on the device."""
    _no_extras(axis=(axis, None), out=(out, None), keepdims=(keepdims, False), weights=(weights, None))
    return _quantiles(x, q, method, percent=True)


# ---------------------------------------------------------------------------------------------------------------
# min / max / ptp and histograms (numpy/lib/_histograms_impl.py of NumPy 2.3 restated on the host; the device
# supplies min / max, the ordered subset a range keeps, std, the two percentiles and the counts)
_NO_VALUE = np._NoValue
_U8 = np.dtype(np.uint8)
_CMP_F64, _CMP_I64 = range(2)  # pbl_hist_cmp
_UNIFORM, _EDGES = range(2)  # pbl_hist_mode
_INT64_MIN, _INT64_MAX = -(2 ** 63), 2 ** 63 - 1
# Estimators restated here.  'doane' cubes with np.power, a SIMD routine whose last bit depends on the host CPU;
# 'stone' evaluates up to max(100, sqrt(n)) full histograms.
_ESTIMATORS = ("auto", "fd", "rice", "scott", "sqrt", "sturges")


def _minmax_values(cols):
    """[(min, max)] of device columns as Python floats / ints (a float column with a NaN gives NaN for both)."""
    lib = _lib.require_gpu()
    ptrs, kinds = _pointers(cols)
    raw = np.empty((len(cols), 2), dtype=np.int64)
    _lib.check(lib.pbl_stats_minmax(ptrs, kinds, len(cols), cols[0].n, raw.ctypes.data, None), "pbl_stats_minmax")
    return [tuple(r.view(np.float64)) if c.kind == F64 else tuple(int(v) for v in r) for r, c in zip(raw, cols)]


def _extremum(x, which, numpy_fn, extras):
    _no_extras(**extras)
    cols, batched = _columns(x)
    if cols[0].n == 0:  # NumPy's own ValueError for an empty array
        out = [numpy_fn(np.empty(0, dtype=c.dtype)) for c in cols]
    else:
        out = [c.dtype.type(v[which]) for c, v in zip(cols, _minmax_values(cols))]
    return out if batched else out[0]


def min(x, axis=None, out=None, keepdims=_NO_VALUE, initial=_NO_VALUE, where=_NO_VALUE):  # noqa: A001
    """``np.min(x.samples_)``, computed on the device."""
    extras = dict(axis=(axis, None), out=(out, None), keepdims=(keepdims, _NO_VALUE), initial=(initial, _NO_VALUE),
                  where=(where, _NO_VALUE))
    return _extremum(x, 0, np.min, extras)


def max(x, axis=None, out=None, keepdims=_NO_VALUE, initial=_NO_VALUE, where=_NO_VALUE):  # noqa: A001
    """``np.max(x.samples_)``, computed on the device."""
    extras = dict(axis=(axis, None), out=(out, None), keepdims=(keepdims, _NO_VALUE), initial=(initial, _NO_VALUE),
                  where=(where, _NO_VALUE))
    return _extremum(x, 1, np.max, extras)


def ptp(x, axis=None, out=None, keepdims=_NO_VALUE):
    """``np.ptp(x.samples_)``, computed on the device (an int64 range wraps, as in NumPy)."""
    _no_extras(axis=(axis, None), out=(out, None), keepdims=(keepdims, _NO_VALUE))
    cols, batched = _columns(x)
    for c in cols:
        np.ptp(np.zeros(2, dtype=c.dtype))  # NumPy's TypeError for bool
    if cols[0].n == 0:
        out = [np.ptp(np.empty(0, dtype=c.dtype)) for c in cols]
    else:  # max - min of the two values is the column's ptp, with NumPy's type, wrap-around and warnings
        out = [np.ptp(np.array(v, dtype=c.dtype)) for c, v in zip(cols, _minmax_values(cols))]
    return out if batched else out[0]


def _unsigned_subtract(a, b):
    """numpy/lib/_histograms_impl.py:_unsigned_subtract: a - b, unsigned for signed integers."""
    dt = np.result_type(a, b)
    if dt.kind == "i":
        unsigned = np.dtype(dt.str.replace("i", "u"))
        return np.subtract(np.asarray(a, dtype=dt), np.asarray(b, dtype=dt), casting="unsafe", dtype=unsigned)
    return np.subtract(a, b, dtype=dt)


def _outer_edges(mn, mx, range):
    """numpy/lib/_histograms_impl.py:_get_outer_edges, with the data's min and max given (NumPy scalars)."""
    if range is not None:
        first_edge, last_edge = range  # (validated by NumPy on the prototype)
    else:
        first_edge, last_edge = mn, mx
        if not (np.isfinite(first_edge) and np.isfinite(last_edge)):
            raise ValueError(f"autodetected range of [{first_edge}, {last_edge}] is not finite")
    if first_edge == last_edge:
        first_edge = first_edge - 0.5
        last_edge = last_edge + 0.5
    return first_edge, last_edge


def _keep_range(dtype, first_edge, last_edge):
    """``(a >= first) & (a <= last)`` -> (lo_cmp, hi_cmp, lo_f, hi_f, lo_i, hi_i).  NumPy compares each edge in its
    own result type with the data: integer data against an integer edge exactly (an edge beyond int64 clamped, which
    keeps the answer), against a float edge in float64."""
    out = []
    for e in (first_edge, last_edge):
        if dtype.kind in "iu" and isinstance(e, (int, np.integer)) and not isinstance(e, (bool, np.bool_)):
            out.append((_CMP_I64, 0.0, int(np.clip(int(e), _INT64_MIN, _INT64_MAX))))
        else:
            out.append((_CMP_F64, float(e), 0))
    (lo_cmp, lo_f, lo_i), (hi_cmp, hi_f, hi_i) = out
    return lo_cmp, hi_cmp, lo_f, hi_f, lo_i, hi_i


def _width(name, size, ptp, std, iqr):
    """The bin width of estimator `name` (numpy/lib/_histograms_impl.py:_hist_bin_*) from the kept data's size,
    ptp (_unsigned_subtract(max, min)), np.std and np.subtract(*np.percentile(x, [75, 25]))."""
    def sqrt():
        return ptp / np.sqrt(size)

    def sturges():
        return ptp / (np.log2(size) + 1.0)

    def fd():
        return 2.0 * iqr * size ** (-1.0 / 3.0)

    if name == "sqrt":
        return sqrt()
    if name == "sturges":
        return sturges()
    if name == "rice":
        return ptp / (2.0 * size ** (1.0 / 3))
    if name == "scott":
        return (24.0 * np.pi ** 0.5 / size) ** (1.0 / 3.0) * std
    if name == "fd":
        return fd()
    fd_bw_corrected = builtins.max(fd(), sqrt() / 2)  # auto
    return builtins.min(fd_bw_corrected, sturges())


def _by_size(fn, which, cols, sizes):
    """{c: fn result} for the columns `which`, one batched call per column length."""
    out = {}
    for size in sorted({sizes[c] for c in which}):
        group = [c for c in which if sizes[c] == size]
        out.update(zip(group, fn([cols[c] for c in group])))
    return out


def _edges_plan(dev, cols, dtypes, n, bins, range):
    """numpy/lib/_histograms_impl.py:_get_bin_edges for every column (n >= 1, arguments validated), with the data
    reached through `dev` (minmax / compact / std / iqr over lists of columns, each one batched call).  dtypes[c]
    is the dtype NumPy bins (uint8 for bool).  -> [(bin_edges, (first_edge, last_edge, nbins) or None)]."""
    k = len(cols)
    if not isinstance(bins, str) and np.ndim(bins) == 1:
        edges = np.asarray(bins)
        return [(edges, None)] * k
    scalar = [lambda v, d=d: d.type(v) for d in dtypes]
    if isinstance(bins, str) or range is None:
        mm = [(s(a), s(b)) for s, (a, b) in zip(scalar, dev.minmax(cols))]
    outer = [_outer_edges(*(mm[c] if range is None else (None, None)), range) for c in builtins.range(k)]
    if isinstance(bins, str):
        sub, sizes, sub_mm = list(cols), [n] * k, list(mm)
        if range is not None:  # the estimator sees a[(a >= first) & (a <= last)], in order
            keeps = [_keep_range(d, *outer[c]) for c, d in enumerate(dtypes)]
            cut = [c for c in builtins.range(k) if not (mm[c][0] >= outer[c][0] and mm[c][1] <= outer[c][1])]
            if cut:
                kept_cols, kept = dev.compact([cols[c] for c in cut], [keeps[c] for c in cut])
                for c, col, size in zip(cut, kept_cols, kept):
                    sub[c], sizes[c] = col, size
                for c, v in _by_size(dev.minmax, [c for c in cut if sizes[c] > 0], sub, sizes).items():
                    sub_mm[c] = (scalar[c](v[0]), scalar[c](v[1]))
        live = [c for c in builtins.range(k) if sizes[c] > 0]
        std = _by_size(dev.std, live, sub, sizes) if bins == "scott" else {}
        iqr = _by_size(dev.iqr, live, sub, sizes) if bins in ("fd", "auto") else {}
        plan = []
        for c in builtins.range(k):
            nbins = 1
            if sizes[c] > 0:
                width = _width(bins, sizes[c], _unsigned_subtract(sub_mm[c][1], sub_mm[c][0]), std.get(c), iqr.get(c))
                if width:
                    if dtypes[c].kind in "iu" and width < 1:
                        width = 1
                    nbins = int(np.ceil(_unsigned_subtract(outer[c][1], outer[c][0]) / width))
            plan.append(nbins)
    else:
        plan = [operator.index(bins)] * k
    out = []
    for c in builtins.range(k):
        first_edge, last_edge = outer[c]
        bin_type = np.result_type(first_edge, last_edge, np.empty(0, dtypes[c]))
        if np.issubdtype(bin_type, np.integer):
            bin_type = np.result_type(bin_type, float)
        edges = np.linspace(first_edge, last_edge, plan[c] + 1, endpoint=True, dtype=bin_type)
        if np.any(edges[:-1] >= edges[1:]):
            raise ValueError(f"Too many bins for data range. Cannot create {plan[c]} finite-sized bins.")
        out.append((edges, (first_edge, last_edge, plan[c])))
    return out


class _Device:
    """The device primitives of _edges_plan, over lists of _Column."""

    def __init__(self):
        self.owned = []  # scratch columns of compact(), freed when the call returns

    def minmax(self, cols):
        return _minmax_values(cols)

    def compact(self, cols, keeps):
        """The kept values of every column, in order, in one scratch buffer sized by a counting pass first."""
        lib = _lib.require_gpu()
        ptrs, kinds = _pointers(cols)
        ranges = (_lib.StatsRange * len(cols))(*[_lib.StatsRange(*k) for k in keeps])
        kept = np.empty(len(cols), dtype=np.int64)
        _lib.check(lib.pbl_stats_compact(ptrs, kinds, len(cols), cols[0].n, ranges, None, kept.ctypes.data, None),
                   "pbl_stats_compact")
        sizes = [int(m) for m in kept]
        at = np.concatenate(([0], np.cumsum(sizes)))
        if at[-1] == 0:
            return [None] * len(cols), sizes
        scratch = DeviceColumns(int(at[-1]), 1)
        self.owned.append(scratch)
        base = scratch.column_ptr(0)
        outs = (C.c_void_p * len(cols))(*[base + 8 * int(a) for a in at[:-1]])
        _lib.check(lib.pbl_stats_compact(ptrs, kinds, len(cols), cols[0].n, ranges, outs, kept.ctypes.data, None),
                   "pbl_stats_compact")
        return ([_Column(c.dtype, m, ptr=base + 8 * int(a), kind=c.kind, keep=scratch)
                 for c, m, a in zip(cols, sizes, at)], sizes)

    def std(self, cols):  # np.std(x), ddof 0
        lib = _lib.require_gpu()
        ptrs, kinds = _pointers(cols)
        res = np.empty(len(cols), dtype=np.float64)
        _lib.check(lib.pbl_stats_moments(ptrs, kinds, len(cols), cols[0].n, int(np.getbufsize()), STD,
                                         float(cols[0].n), res.ctypes.data, None), "pbl_stats_moments")
        return [np.float64(v) for v in res]

    def iqr(self, cols):  # np.subtract(*np.percentile(x, [75, 25])): linear, on the 0 / 1 integers of bool data too
        lib = _lib.require_gpu()
        ptrs, _ = _pointers(cols)
        kinds = (C.c_int32 * len(cols))(*[I64_AS_F64 if c.kind == BOOL_AS_F64 else c.kind for c in cols])
        q = np.true_divide([75, 25], 100)
        raw = np.empty((len(cols), 2), dtype=np.float64)
        _lib.check(lib.pbl_stats_quantiles(ptrs, kinds, len(cols), cols[0].n, q.ctypes.data_as(C.POINTER(C.c_double)),
                                           2, METHODS["linear"], raw.ctypes.data, None), "pbl_stats_quantiles")
        return [np.subtract(*r) for r in raw]

    def free(self):
        for s in self.owned:
            s.free()


def _histogram_args(x, bins, range, weights):
    """Columns, batch flag and the dtype NumPy bins (uint8 for bool), every argument checked by NumPy itself on a
    prototype of each column's dtype.  No device call."""
    if weights is not None:
        raise NotImplementedError("stats: weights= is not supported")
    cols, batched = _columns(x)
    dtypes = []
    for c in cols:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")  # (the bool warning is raised once, below)
            proto = np.histogram_bin_edges(np.zeros(2, dtype=c.dtype), bins, range)
        if c.dtype == _BOOL:
            warnings.warn(f"Converting input from {c.dtype} to {np.uint8} for compatibility.", RuntimeWarning,
                          stacklevel=4)
        d = _U8 if c.dtype == _BOOL else c.dtype
        if isinstance(bins, str):
            if bins not in _ESTIMATORS:
                raise NotImplementedError(f"bins={bins!r} is not supported on the device: use one of {_ESTIMATORS}")
        if not isinstance(bins, str) and np.ndim(bins) == 1:
            common = np.result_type(d, proto.dtype)
            if common not in (_F64, _I64):
                raise NotImplementedError(f"bins of dtype {proto.dtype} (compared with {d} data as {common})")
        elif proto.dtype != _F64:
            raise NotImplementedError(f"bin edges of dtype {proto.dtype}")
        dtypes.append(d)
    return cols, batched, dtypes


def _plan(x, bins, range, weights, dev):
    cols, batched, dtypes = _histogram_args(x, bins, range, weights)
    if cols[0].n == 0:
        return cols, batched, dtypes, None
    return cols, batched, dtypes, _edges_plan(dev, cols, dtypes, cols[0].n, bins, range)


def histogram_bin_edges(x, bins=10, range=None, weights=None):
    """``np.histogram_bin_edges(x.samples_, bins, range)``, with the data's statistics computed on the device."""
    dev = _Device()
    try:
        cols, batched, dtypes, plan = _plan(x, bins, range, weights, dev)
    finally:
        dev.free()
    if plan is None:
        out = [np.histogram_bin_edges(np.empty(0, d), bins, range) for d in dtypes]
    else:
        out = [edges for edges, _ in plan]
    return out if batched else out[0]


def _read_value(col, row):
    raw = np.empty(1, dtype=np.int64)
    _lib.check(_lib.load().pbl_memcpy_d2h(raw.ctypes.data, C.c_void_p(col.ptr + 8 * row), 8, None), "pbl_memcpy_d2h")
    _lib.check(_lib.load().pbl_stream_synchronize(None))
    if col.kind == I64_BITS:
        return raw
    return raw.view(np.float64)


def _uniform_spec(dtype, edges, uniform):
    """numpy/lib/_histograms_impl.py:816-873 as the kernel runs it -> (keep, first, denom, nbins, float64 table):
    keep = (a >= first_edge) & (a <= last_edge) on the uncast data, x = float64(a),
    i = intp(((x - first) / denom) * nbins), then the fix-ups against the table."""
    first_edge, last_edge, nbins = uniform
    return (_keep_range(dtype, first_edge, last_edge), float(np.float64(first_edge)),
            float(np.float64(_unsigned_subtract(last_edge, first_edge))), nbins,
            np.ascontiguousarray(edges, dtype=np.float64))


def _edge_table(dtype, edges):
    """numpy/lib/_histograms_impl.py:874-893 (searchsorted in np.result_type(data, edges)) -> (that type, the distinct
    non-NaN edge values ascending; a single placeholder when every edge is NaN, whose counts come from the NaN rule)."""
    common = np.result_type(dtype, edges.dtype)
    values = edges.astype(common)
    table = np.unique(values[~np.isnan(values)] if common == _F64 else values)
    return common, (table if table.size else np.zeros(1, dtype=common))


def histogram(x, bins=10, range=None, density=None, weights=None):
    """``np.histogram(x.samples_, bins, range, density)``, computed on the device."""
    dev = _Device()
    try:
        cols, batched, dtypes, plan = _plan(x, bins, range, weights, dev)
    finally:
        dev.free()
    if plan is None:
        out = [np.histogram(np.empty(0, d), bins, range, density) for d in dtypes]
        return out if batched else out[0]
    specs = (_lib.HistSpec * len(cols))()
    tables, total = [], 0
    for c, (d, (edges, uniform)) in enumerate(zip(dtypes, plan)):
        s = specs[c]
        s.offset = total
        if uniform is not None:
            keep, s.first, s.denom, s.nbins, table = _uniform_spec(d, edges, uniform)
            s.mode, s.keep = _UNIFORM, _lib.StatsRange(*keep)
            total += s.nbins
        else:
            common, table = _edge_table(d, edges)
            s.mode, s.cmp, s.nbins = _EDGES, (_CMP_F64 if common == _F64 else _CMP_I64), table.size
            total += 2 * s.nbins + 2
        tables.append(table)
        s.table = table.ctypes.data
    lib = _lib.require_gpu()
    ptrs, kinds = _pointers(cols)
    counts = np.empty(total, dtype=np.uint64)
    bad = np.empty(len(cols), dtype=np.int64)
    status = _lib.check(lib.pbl_stats_histogram(ptrs, kinds, len(cols), cols[0].n, specs, counts.ctypes.data, total,
                                                bad.ctypes.data, None), "pbl_stats_histogram")
    if status == _lib.STATUS_OUT_OF_TABLE:  # NumPy fails inside its index arithmetic: let it raise on that value
        for c, row in enumerate(bad):
            if row >= 0:
                first_edge, last_edge, nbins = plan[c][1]
                value = _read_value(cols[c], int(row)).astype(dtypes[c])
                np.histogram(value, bins=nbins, range=(first_edge, last_edge))
        raise _lib.PblError("pbl_stats_histogram reported an index outside the edges that NumPy accepts")
    if status != _lib.STATUS_OK:
        raise _lib.PblError(f"pbl_stats_histogram failed: {_lib.last_error()}")
    out = []
    for c, (d, (edges, uniform)) in enumerate(zip(dtypes, plan)):
        s = specs[c]
        if uniform is not None:
            hist = counts[s.offset:s.offset + s.nbins].astype(np.intp)
        else:
            hist = np.diff(_cumulative(counts[s.offset:s.offset + 2 * s.nbins + 2].astype(np.intp), tables[c], edges,
                                       np.result_type(d, edges.dtype), cols[c].n))
        if density:
            db = np.array(np.diff(edges), float)
            hist = hist / db / hist.sum()
        out.append((hist, edges))
    return out if batched else out[0]


def _cumulative(cells, table, edges, common, n):
    """np.histogram's cum_n (searchsorted 'left' of every edge but the last, 'right' of the last; NaN sorts last)
    from the device's cell counts over the distinct edge values `table`."""
    below = np.concatenate(([0], np.cumsum(cells)))  # below[j]: values in cells < j
    values = edges.astype(common)
    nan = np.isnan(values) if common == _F64 else np.zeros(values.size, dtype=bool)
    k = np.searchsorted(table, np.where(nan, table[0], values))  # a non-NaN edge is table[k]
    cum = below[2 * k + 1]  # 'left': the values below table[k]
    cum[-1] = below[2 * k[-1] + 2]  # 'right': and those equal to it
    cum[nan] = n - cells[-1]  # every value but a NaN is below a NaN edge
    if nan[-1]:
        cum[-1] = n  # NaN <= NaN
    return cum.astype(np.intp)
