"""Statistics of sampled nodes on the device, bit-identical to NumPy on the host copy.

    from probabilit_b200 import stats
    stats.mean(x); stats.var(x, ddof=0); stats.std(x, ddof=0)
    stats.quantile(x, q, method="linear"); stats.percentile(x, q, method="linear")

``x`` is a sampled ``Node``, a column ``(DeviceColumns, j)``, a 1-D contiguous CUDA array (``<f8`` or ``<i8``,
``__cuda_array_interface__``: torch tensors included), or a list of ``Node``s of one ``n`` (then the result is a
list, computed in one pass over all columns).  The result equals ``np.mean(node.samples_)`` ... ``np.percentile``
bit for bit, with NumPy's dtype and shape; the column is never copied to the host.  Samples that only exist on the
host (folded constants, ``samples_`` set by the caller) are uploaded and reduced by the same kernels
(csrc/stats.cu).  Arguments are checked before any device call, with NumPy's exception types.
"""
import ctypes as C
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
