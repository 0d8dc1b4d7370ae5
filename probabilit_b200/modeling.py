"""Modeling graph with the reference's API, evaluated by ONE fused CUDA kernel.

Host mirror of src/probabilit/modeling.py of the reference: the same node classes
(``Distribution``, ``Constant``, ``Add`` ... ``Arctanh``), operator overloads (:674-747), and
``Node.sample(size, random_state, method, correlator, gc_strategy)`` (:431-493) /
``Node.sample_from_quantiles(quantiles, correlator, gc_strategy)`` (:495-614) / ``correlate``
(:628-661) with the reference's column assignment, evaluation order, dtype rules and errors.

What differs is the execution: instead of one NumPy temporary per node, the graph is compiled
(here, on the host: control plane, ~100 nodes) into the bytecode of ``pbl_graph_eval_f64``
(include/probabilit_b200.h) and evaluated per sample in a single pass on the GPU
(csrc/graph.cu).  Sub-graphs without any distribution are folded on the host at compile time.
``node.samples_`` stays device resident and is copied to the host on first access.

There is no CPU fallback: a node type or dtype combination the device program cannot express
raises ``NotImplementedError`` at compile time.

Quantile source of ``sample``: by default the unit-cube draw is generated on the GPU
(``quantile_source="device"``: in-kernel Philox for ``method=None``, probabilit_b200.qmc engines
for "sobol"/"halton" (bit-exact with SciPy) and "lhs").  ``quantile_source="numpy"`` draws the
quantiles exactly like the reference (NumPy/SciPy on the host, modeling.py:479-489) and uploads
them -- bit-for-bit the reference's stream, used for parity checks.
"""
import abc
import copy
import ctypes as C
import functools
import heapq
import itertools
import numbers
import operator

import networkx as nx
import numpy as np

from . import _lib
from ._device import DeviceColumns, as_device_columns
from .correlation import Cholesky, ImanConover, nearest_correlation_matrix

OP = dict(
    NOP=0, LOAD=1, STORE=2, CHECK=3, MOV=4, UNIFORM=5, SPILL=6, FILL=7,
    PPF_NORM=16, PPF_UNIFORM=17, PPF_EXPON=18, PPF_TRIANG=19, PPF_GAMMA=20, PPF_LOGNORM=21,
    PPF_POISSON=22, PPF_BINOM=23, PPF_BERNOULLI=24, TABLE_INTERP=25, TABLE_SEARCH=26, TABLE_QUANTILE=27,
    PPF_BETA=28, PPF_TRUNCNORM=29,
    ADD=32, MUL=33, SUB=34, DIV=35, POW=36, FLOORDIV=37, MOD=38, MAX=39, MIN=40, ATAN2=41, LT=42, LE=43,
    GT=44, GE=45, EQ=46, NE=47, AND=48, OR=49, ISCLOSE=50,
    I_ADD=51, I_SUB=52, I_MUL=53, I_FLOORDIV=54, I_MOD=55, I_POW=56, I_MAX=57, I_MIN=58, I_LT=59, I_LE=60, I_EQ=61,
    I_NE=62,
    NEG=64, ABS=65, LOG=66, EXP=67, FLOOR=68, CEIL=69, SIGN=70, SQRT=71, SQUARE=72, LOG10=73, SIN=74,
    COS=75, TAN=76, ASIN=77, ACOS=78, ATAN=79, SINH=80, COSH=81, TANH=82, ASINH=83, ACOSH=84, ATANH=85,
    NOT=86, LOOKUP=87, I_NEG=88, I_ABS=89, I_SIGN=90, I_SQUARE=91, I2F=92, F2I=93,
)
QUANTILE_METHODS = {"linear": 0, "lower": 1, "higher": 2, "nearest": 3, "midpoint": 4, "closest_observation": 5}
MAX_SLOTS = 96
MAX_INSTR = 4096
MAX_SPILLS = 1024
MAX_TAGS = 0xFFF + 1  # a fused CHECK carries a 12-bit node tag
MAX_OUTPUTS = 1 << 11  # a fused STORE carries its output index in bits 20-30 of the (non-negative) dst word

_F64 = np.dtype(np.float64)
_BOOL = np.dtype(np.bool_)
_I64 = np.dtype(np.int64)

# integer instructions: operands are int64 bit patterns; all but the comparisons (booleans) and I2F (a double)
# produce one
_INT_IN = {OP[k] for k in ("I_ADD", "I_SUB", "I_MUL", "I_FLOORDIV", "I_MOD", "I_POW", "I_MAX", "I_MIN", "I_LT",
                           "I_LE", "I_EQ", "I_NE", "I_NEG", "I_ABS", "I_SIGN", "I_SQUARE", "I2F")}
_INT_OUT = (_INT_IN - {OP[k] for k in ("I_LT", "I_LE", "I_EQ", "I_NE", "I2F")}) | {OP["F2I"]}
_INT_CMP = {"LT": ("I_LT", False), "LE": ("I_LE", False), "GT": ("I_LT", True), "GE": ("I_LE", True),
            "EQ": ("I_EQ", False), "NE": ("I_NE", False)}  # GT / GE: the operands swapped
_EXACT_INT = 2 ** 53  # integers up to this magnitude are exact doubles


def _beyond_exact(values):
    """Integer table values that a double does not hold exactly."""
    return values.dtype.kind in "iu" and values.size > 0 and max(int(values.max()), -int(values.min())) > _EXACT_INT


def _integral(val):
    """An int64 / bool value, or an immediate that NumPy casts to int64 exactly."""
    if val.is_imm:
        return val.dtype.kind in "bi" or (val.dtype.kind == "u" and val.dtype.itemsize < 8)
    return val.dtype in (_I64, _BOOL)


def python_to_prob(argument):
    """Numbers become Constant nodes (reference modeling.py:289-296)."""
    if isinstance(argument, numbers.Number):
        return Constant(argument)
    if isinstance(argument, Node):
        return argument
    raise ValueError(f"Type not compatible with probabilit: {argument}")


def build_corrmat(correlations):
    """[(indices, corrmat), ...] -> one correlation matrix (reference utils.py:92-115)."""
    k = 1 + max(max(idx) for idx, _ in correlations)
    out = np.eye(k, dtype=float)
    for idx, block in correlations:
        out[np.ix_(idx, idx)] = block
    return out


# ==========================================================================================
# storage of node.samples_
# ==========================================================================================
class _Samples:
    """Where a node's samples live: a device column, a host array, or a folded constant."""

    def __init__(self, *, host=None, columns=None, index=None, dtype=None, const=None, size=None, none=False,
                 categories=None, ibits=False):
        self._host, self.columns, self.index, self.dtype = host, columns, index, dtype
        self.const, self.size, self.none, self.categories = const, size, none, categories
        self.ibits = ibits  # the column holds int64 bit patterns (the result of an integer instruction)

    def host(self):
        if self._host is None and not self.none:
            if self.columns is not None:
                raw = self.columns.column_to_host(self.index)
                if self.categories is not None:  # the device holds indices into non-numeric values
                    self._host = self.categories[raw.astype(np.intp)]
                elif self.ibits:
                    self._host = raw.view(np.int64)
                else:
                    self._host = raw if self.dtype == _F64 else (raw != 0 if self.dtype == _BOOL else raw.astype(self.dtype))
            else:
                self._host = np.ones(self.size, dtype=self.const.dtype) * self.const[0]
        return self._host

    def device_ptr(self):
        return None if self.columns is None else self.columns.column_ptr(self.index)


# ==========================================================================================
# nodes
# ==========================================================================================
class Node(abc.ABC):
    """A node in the computational graph (reference modeling.py:335-672)."""

    id_iter = itertools.count()

    def __init__(self):
        self._id = next(self.id_iter)
        self._correlations = []

    def __eq__(self, other):
        if not isinstance(other, Node):
            return NotImplemented
        return self._id == other._id

    def __hash__(self):
        return self._id

    # -- samples_ : device resident, host copy on first access ---------------------------------
    @property
    def samples_(self):
        store = self.__dict__.get("_store")
        if store is None:
            raise AttributeError(f"{type(self).__name__!r} object has no attribute 'samples_'")
        return store.host()

    @samples_.setter
    def samples_(self, value):
        self.__dict__["_store"] = _Samples(host=value)

    @samples_.deleter
    def samples_(self):
        if self.__dict__.pop("_store", None) is None:
            raise AttributeError("samples_")

    def samples_device_ptr(self):
        """Device address of this node's samples (n fp64), or None if they only exist on the host."""
        store = self.__dict__.get("_store")
        return None if store is None else store.device_ptr()

    # -- graph walking ---------------------------------------------------------------------------
    def nodes(self):
        """self and all ancestors, depth first, in the reference's order (:403-420)."""
        stack = [self]
        while stack:
            node = stack.pop()
            yield node
            stack.extend(node.get_parents())

    def num_distribution_nodes(self):
        return sum(1 for node in set(self.nodes()) if isinstance(node, AbstractDistribution))

    def _is_initial_sampling_node(self):
        if not isinstance(self, AbstractDistribution):
            return False
        return not any(isinstance(n, AbstractDistribution) for n in set(self.nodes()) - {self})

    def to_graph(self):
        """networkx MultiDiGraph built exactly like the reference's (:663-683), so that
        nx.topological_sort -- which fixes the quantile column of every non-initial distribution
        -- visits the nodes in the same order."""
        nodes = list(self.nodes())
        if len(nodes) == 1:
            G = nx.MultiDiGraph()
            G.add_node(self)
            return G
        edges = [(parent, node) for node in nodes for parent in node.get_parents() if not node.is_leaf]
        return nx.MultiDiGraph(edges)

    def copy(self):
        """Copy the node including the graph above it (:352-401)."""
        fresh = {}

        def remap(item):
            return fresh[item._id] if isinstance(item, Node) else copy.deepcopy(item)

        for node in nx.topological_sort(self.to_graph()):
            dup = copy.copy(node)
            fresh[dup._id] = dup
            dup._correlations = copy.deepcopy(dup._correlations)
            if isinstance(dup, (AbstractDistribution, ScalarFunctionTransform)) and hasattr(dup, "args"):
                dup.args = tuple(remap(a) for a in dup.args)
                dup.kwargs = {k: remap(v) for k, v in dup.kwargs.items()}
            elif isinstance(dup, (VariadicTransform, BinaryTransform)):
                dup.parents = tuple(remap(p) for p in dup.parents)
            elif isinstance(dup, UnaryTransform):
                dup.parent = remap(dup.parent)
            elif isinstance(dup, Constant):
                dup.value = remap(dup.value)
        return fresh[self._id]

    def correlate(self, *variables, corr_mat):
        """Store correlations between ancestor variables (:628-661)."""
        assert corr_mat.ndim == 2
        assert corr_mat.shape[0] == corr_mat.shape[1]
        assert corr_mat.shape[0] == len(variables)
        assert len(variables) == len(set(variables))
        members = set(self.nodes())
        for var in variables:
            if var not in members:
                raise ValueError(f"{var} is not an ancestor of {self}")
        self._correlations.append((list(variables), np.copy(corr_mat)))
        return self

    # -- sampling ----------------------------------------------------------------------------------
    def sample(self, size=None, random_state=None, method=None, correlator="imanconover", gc_strategy=None, *,
               quantile_source="device"):
        """Sample this node and set ``samples_`` on the graph (reference :431-493)."""
        size = 1 if size is None else int(size)
        d = self.num_distribution_nodes()
        if quantile_source == "numpy":  # the reference's own draw, for bit parity
            import scipy.stats
            from scipy._lib._util import check_random_state

            engines = {"lhs": scipy.stats.qmc.LatinHypercube, "halton": scipy.stats.qmc.Halton,
                       "sobol": scipy.stats.qmc.Sobol}
            if method is None:
                quantiles = check_random_state(random_state).random((size, d))
            else:
                quantiles = engines[method.lower().strip()](d=d, rng=random_state).random(n=size)
        elif quantile_source == "device":
            from . import qmc

            if method is None:
                seed = int(qmc._rng_integers(qmc.check_random_state(_as_seed(random_state)), 2 ** 62, None, np.int64))
                quantiles = _PhiloxSource(seed, size, d)
            else:
                engines = {"lhs": qmc.LatinHypercube, "halton": qmc.Halton, "sobol": qmc.Sobol}
                quantiles = engines[method.lower().strip()](d=d, rng=random_state).random(n=size, device="columns")
        else:
            raise ValueError("quantile_source must be 'device' or 'numpy'")
        return self.sample_from_quantiles(quantiles, correlator=correlator, gc_strategy=gc_strategy)

    def sample_from_quantiles(self, quantiles, correlator="imanconover", gc_strategy=None):
        """Evaluate the graph on an (n, d) array of quantiles in [0, 1] (reference :495-614).
        ``quantiles`` may be a host array, a CUDA tensor / DeviceColumns (no host traffic)."""
        _GraphRun(self, quantiles, correlator, gc_strategy).execute()
        return self.samples_


def _as_seed(random_state):
    if isinstance(random_state, np.random.RandomState):
        return int(random_state.randint(0, 2 ** 31 - 1))
    return random_state


class _PhiloxSource:
    """Quantiles generated inside the graph kernel (PBL_OP_UNIFORM): nothing to read from HBM."""

    def __init__(self, seed, n, d):
        self.seed, self.shape = int(seed), (int(n), int(d))


class OverloadMixin:
    """Operator overloads building Transform nodes (reference :686-747)."""

    def __add__(self, other): return Add(self, other)
    def __radd__(self, other): return Add(self, other)
    def __mul__(self, other): return Multiply(self, other)
    def __rmul__(self, other): return Multiply(self, other)
    def __floordiv__(self, other): return FloorDivide(self, other)
    def __rfloordiv__(self, other): return FloorDivide(other, self)
    def __truediv__(self, other): return Divide(self, other)
    def __rtruediv__(self, other): return Divide(other, self)
    def __mod__(self, other): return Mod(self, other)
    def __rmod__(self, other): return Mod(other, self)
    def __sub__(self, other): return Subtract(self, other)
    def __rsub__(self, other): return Subtract(other, self)
    def __pow__(self, other): return Power(self, other)
    def __rpow__(self, other): return Power(other, self)
    def __neg__(self): return Negate(self)
    def __abs__(self): return Abs(self)
    def __lt__(self, other): return LessThan(self, other)
    def __le__(self, other): return LessThanOrEqual(self, other)
    def __gt__(self, other): return GreaterThan(self, other)
    def __ge__(self, other): return GreaterThanOrEqual(self, other)


class Constant(Node, OverloadMixin):
    """A number (reference :750-770)."""

    is_leaf = True

    def __init__(self, value):
        self.value = value.value if isinstance(value, Constant) else value
        super().__init__()

    def _fold(self):
        return np.ones(1, dtype=type(self.value)) * self.value  # :763, one element

    def get_parents(self):
        yield from ()

    def __repr__(self):
        return f"{type(self).__name__}({self.value})"


class AbstractDistribution(Node, OverloadMixin, abc.ABC):
    pass


# scipy.stats name -> (device op, shape parameter names in scipy's positional order, has scale)
_DISTRIBUTIONS = {
    "norm": ("PPF_NORM", (), True),
    "uniform": ("PPF_UNIFORM", (), True),
    "expon": ("PPF_EXPON", (), True),
    "triang": ("PPF_TRIANG", ("c",), True),
    "gamma": ("PPF_GAMMA", ("a",), True),
    "lognorm": ("PPF_LOGNORM", ("s",), True),
    "poisson": ("PPF_POISSON", ("mu",), False),
    "binom": ("PPF_BINOM", ("n", "p"), False),
    "bernoulli": ("PPF_BERNOULLI", ("p",), False),
    # four-parameter ones: the device op takes (q, a, b, scale); loc is added by a separate ADD
    "beta": ("PPF_BETA", ("a", "b"), True),
    "truncnorm": ("PPF_TRUNCNORM", ("a", "b"), True),
}


class Distribution(AbstractDistribution):
    """``Distribution("norm", loc=0, scale=1)``: a scipy.stats distribution by name, sampled by
    inverse CDF (reference :773-819).  Parameters may be numbers or Nodes (composite)."""

    def __init__(self, distr, *args, **kwargs):
        self.distr = distr
        self.args = args
        self.kwargs = kwargs
        super().__init__()

    def __repr__(self):
        parts = [f'"{self.distr}"'] + [repr(a) for a in self.args]
        parts += [f"{k}={v!r}" for k, v in self.kwargs.items()]
        return f"{type(self).__name__}({', '.join(parts)})"

    def get_parents(self):
        for arg in self.args + tuple(self.kwargs.values()):
            if isinstance(arg, Node):
                yield arg

    @property
    def is_leaf(self):
        return list(self.get_parents()) == []

    def _bound_parameters(self):
        """(device op, [shape..., loc(, scale)]) with scipy's argument parsing: positional
        arguments are shapes, then loc, then scale; everything may also be a keyword."""
        if self.distr not in _DISTRIBUTIONS:
            raise NotImplementedError(
                f"scipy.stats.{self.distr} has no device inverse CDF (available: {sorted(_DISTRIBUTIONS)})")
        op, shapes, has_scale = _DISTRIBUTIONS[self.distr]
        names = list(shapes) + ["loc"] + (["scale"] if has_scale else [])
        if len(self.args) > len(names):
            raise TypeError(f"{self.distr}: too many positional arguments")
        bound = dict(zip(names, self.args))
        for key, val in self.kwargs.items():
            if key not in names:
                raise TypeError(f"{self.distr}: unexpected keyword argument {key!r}")
            if key in bound:
                raise TypeError(f"{self.distr}: got multiple values for argument {key!r}")
            bound[key] = val
        missing = [s for s in shapes if s not in bound]
        if missing:
            raise TypeError(f"_parse_args() missing required positional argument(s): {missing}")
        bound.setdefault("loc", 0)
        if has_scale:
            bound.setdefault("scale", 1)
        return OP[op], [bound[name] for name in names]


class EmpiricalDistribution(AbstractDistribution):
    """Inverse-CDF sampling of observed data: ``np.quantile(data, q, **kwargs)`` (reference :825-845).
    On the device: a binary-search-free index computation on the sorted data (NumPy's quantile
    methods linear / lower / higher / nearest / midpoint / closest_observation)."""

    is_leaf = True

    def __init__(self, data, **kwargs):
        self.data = np.array(data)
        self.kwargs = kwargs
        super().__init__()

    def __repr__(self):
        return f"{type(self).__name__}()"

    def get_parents(self):
        yield from ()

    def _table(self):
        extra = set(self.kwargs) - {"method"}
        method = self.kwargs.get("method", "linear")
        if extra or method not in QUANTILE_METHODS:
            raise NotImplementedError(f"np.quantile(**{self.kwargs}) has no device implementation "
                                      f"(methods: {sorted(QUANTILE_METHODS)})")
        if not np.issubdtype(self.data.dtype, np.number) or self.data.ndim != 1 or self.data.size == 0:
            raise NotImplementedError("EmpiricalDistribution needs a non-empty 1-D numeric data array")
        # methods without interpolation take an element of the data and keep its dtype; the others are float64
        dtype = self.data.dtype if method in ("lower", "higher", "nearest", "closest_observation") else _F64
        return np.sort(self.data.astype(np.float64)), QUANTILE_METHODS[method], np.dtype(dtype)


class CumulativeDistribution(AbstractDistribution):
    """A distribution given by points of its CDF: ``np.interp(q, quantiles, cumulatives)`` (reference :848-884)."""

    is_leaf = True

    def __init__(self, quantiles, cumulatives):
        self.q = np.array(quantiles)
        self.cumulatives = np.array(cumulatives)
        if not np.all(np.diff(self.q) > 0):
            raise ValueError("The quantiles must be strictly increasing.")
        if not np.all(np.diff(self.cumulatives) > 0):
            raise ValueError("The cumulatives must be strictly increasing.")
        if not (np.isclose(np.min(self.q), 0) and np.isclose(np.max(self.q), 1)):
            raise ValueError("Lowest quantile must be 0 and highest must be 1.")
        super().__init__()

    def __repr__(self):
        return f"{type(self).__name__}(quantiles={repr(self.q)}, cumulatives={repr(self.cumulatives)})"

    def get_parents(self):
        yield from ()


class DiscreteDistribution(AbstractDistribution):
    """Categorical distribution: ``values[np.searchsorted(np.cumsum(p), q, side="right")]`` (reference :887-927).
    Non-numeric values stay on the host; the device computes the category index."""

    is_leaf = True

    def __init__(self, values, probabilities=None):
        self.values = np.array(values)
        if probabilities is None:
            self.probabilities = np.ones(len(self.values), dtype=float)
            self.probabilities = self.probabilities / np.sum(self.probabilities)
        else:
            self.probabilities = np.array(probabilities)
        if not len(self.values) == len(self.probabilities):
            raise ValueError(f"Length mismatch: {len(self.values)=}  {len(self.probabilities)=}")
        if not np.isclose(np.sum(self.probabilities), 1.0):
            raise ValueError(f"Probabilities must sum to 1. {sum(self.probabilities)=}")
        if np.any(self.probabilities < 0):
            raise ValueError("Probabilities are not non-negative.")
        super().__init__()

    def __repr__(self):
        return f"{type(self).__name__}(values={repr(self.values)}, probabilities={repr(self.probabilities)})"

    def get_parents(self):
        yield from ()


class Transform(Node, OverloadMixin, abc.ABC):
    """Arithmetic on nodes (reference :933-940)."""

    is_leaf = False

    def __repr__(self):
        return f"{type(self).__name__}({', '.join(repr(p) for p in self.get_parents())})"


class VariadicTransform(Transform):
    """Add(a, b, c, ...) = reduce(op, parents) (reference :943-959)."""

    def __init__(self, *args):
        self.parents = tuple(python_to_prob(arg) for arg in args)
        super().__init__()

    def get_parents(self):
        yield from self.parents

    def _numpy(self, arrays):
        return functools.reduce(self.op, arrays)

    def _emit(self, em, vals):
        acc = vals[0]
        for nxt in vals[1:]:
            acc = em.binary(self, acc, nxt)
        return acc


class BinaryTransform(Transform):
    def __init__(self, *args):
        self.parents = tuple(python_to_prob(arg) for arg in args)
        super().__init__()

    def get_parents(self):
        yield from self.parents

    def _numpy(self, arrays):
        return self.op(*arrays)

    def _emit(self, em, vals):
        if len(vals) != 2:
            raise TypeError(f"{type(self).__name__} takes two arguments")
        return em.binary(self, vals[0], vals[1])


class UnaryTransform(Transform):
    def __init__(self, arg):
        self.parent = python_to_prob(arg)
        super().__init__()

    def get_parents(self):
        yield self.parent

    def _numpy(self, arrays):
        return self.op(arrays[0])

    def _emit(self, em, vals):
        return em.unary(self, vals[0])


def _variadic(name, op, dev, dev_bool=None):
    return type(name, (VariadicTransform,), {"op": staticmethod(op), "dev": dev, "dev_bool": dev_bool or dev})


def _binary(name, op, dev):
    return type(name, (BinaryTransform,), {"op": staticmethod(op), "dev": dev, "dev_bool": dev})


def _unary(name, op, dev):
    return type(name, (UnaryTransform,), {"op": staticmethod(op), "dev": dev})


# op table of reference modeling.py:962-1169 (class -> NumPy callable) + the device opcode
Add = _variadic("Add", operator.add, "ADD", "OR")  # bool + bool is logical or in NumPy
Multiply = _variadic("Multiply", operator.mul, "MUL", "AND")
Max = _variadic("Max", np.maximum, "MAX")
Min = _variadic("Min", np.minimum, "MIN")
All = _variadic("All", np.logical_and, "AND")
Any = _variadic("Any", np.logical_or, "OR")


class Avg(VariadicTransform):
    """np.average(np.vstack(samples), axis=0) (reference :986-990): row-by-row sum, then / count."""

    def _numpy(self, arrays):
        return np.average(np.vstack(arrays), axis=0)

    def _emit(self, em, vals):
        acc = vals[0]
        for nxt in vals[1:]:
            acc = em.raw_binary("ADD", acc, nxt, _F64)
        return em.raw_binary("DIV", acc, em.imm(float(len(vals)), _F64), _F64)


class NoOp(VariadicTransform):
    """Samples all ancestors, yields nothing (reference :993-997)."""

    def _numpy(self, arrays):
        return None

    def _emit(self, em, vals):
        return None


FloorDivide = _binary("FloorDivide", np.floor_divide, "FLOORDIV")
Mod = _binary("Mod", np.mod, "MOD")
Divide = _binary("Divide", operator.truediv, "DIV")
Power = _binary("Power", operator.pow, "POW")
Subtract = _binary("Subtract", operator.sub, "SUB")
Equal = _binary("Equal", np.equal, "EQ")
NotEqual = _binary("NotEqual", np.not_equal, "NE")
LessThan = _binary("LessThan", operator.lt, "LT")
LessThanOrEqual = _binary("LessThanOrEqual", operator.le, "LE")
GreaterThan = _binary("GreaterThan", operator.gt, "GT")
GreaterThanOrEqual = _binary("GreaterThanOrEqual", operator.ge, "GE")
IsClose = _binary("IsClose", np.isclose, "ISCLOSE")
Arctan2 = _binary("Arctan2", np.arctan2, "ATAN2")

Negate = _unary("Negate", operator.neg, "NEG")
Abs = _unary("Abs", operator.abs, "ABS")
Log = _unary("Log", np.log, "LOG")
Exp = _unary("Exp", np.exp, "EXP")
Floor = _unary("Floor", np.floor, "FLOOR")
Ceil = _unary("Ceil", np.ceil, "CEIL")
Sign = _unary("Sign", np.sign, "SIGN")
Sqrt = _unary("Sqrt", np.sqrt, "SQRT")
Square = _unary("Square", np.square, "SQUARE")
Log10 = _unary("Log10", np.log10, "LOG10")
Sin = _unary("Sin", np.sin, "SIN")
Cos = _unary("Cos", np.cos, "COS")
Tan = _unary("Tan", np.tan, "TAN")
Arcsin = _unary("Arcsin", np.arcsin, "ASIN")
Arccos = _unary("Arccos", np.arccos, "ACOS")
Arctan = _unary("Arctan", np.arctan, "ATAN")
Sinh = _unary("Sinh", np.sinh, "SINH")
Cosh = _unary("Cosh", np.cosh, "COSH")
Tanh = _unary("Tanh", np.tanh, "TANH")
Arcsinh = _unary("Arcsinh", np.arcsinh, "ASINH")
Arccosh = _unary("Arccosh", np.arccosh, "ACOSH")
Arctanh = _unary("Arctanh", np.arctanh, "ATANH")


class ScalarFunctionTransform(Transform):
    """Arbitrary Python callables per sample (reference :1172-1204) cannot run on the device."""

    def __init__(self, func, args, kwargs):
        self.func, self.args, self.kwargs = func, args, kwargs
        super().__init__()

    def get_parents(self):
        for arg in self.args + tuple(self.kwargs.values()):
            if isinstance(arg, Node):
                yield arg


# ==========================================================================================
# compiler: graph -> bytecode
# ==========================================================================================
class _Val:
    """A node's value while compiling: an immediate (folded, 1-element array) or a virtual register.

    An int64 register lives in one of two lanes: ``ibits`` (the int64 bit pattern, computed by an integer
    instruction) or, like every table output, an exact double.  ``big``: a table value of this register may
    exceed 2^53 in magnitude, so the double is not exact.  ``conv``: the register converted to the other lane."""

    __slots__ = ("arr", "vreg", "dtype", "ibits", "big", "conv")

    def __init__(self, arr=None, vreg=None, dtype=None, ibits=False, big=False):
        self.arr, self.vreg = arr, vreg
        self.dtype = np.dtype(dtype if dtype is not None else arr.dtype)
        self.ibits, self.big, self.conv = ibits, big, None

    @property
    def is_imm(self):
        return self.vreg is None


class _Emitter:
    def __init__(self):
        self.instrs = []  # [op, dst_vreg or None, [src vreg or None]*4, [imm]*4]
        self.nv = 0
        self.table_base = 0  # index of the first lookup table in the kernel's input pointer list

    def imm(self, value, dtype):
        return _Val(arr=np.array([value], dtype=dtype))

    def _new(self):
        self.nv += 1
        return self.nv - 1

    def _push(self, op, operands, dst=True, aux=None):
        op = OP[op] if isinstance(op, str) else op
        srcs, imms = [None] * 4, [0.0] * 4
        for i, o in enumerate(operands):
            if isinstance(o, _Val):
                if o.is_imm:
                    # an integer instruction takes the int64 bit pattern (NumPy casts a bool / smaller int to int64)
                    imms[i] = float(np.int64(o.arr[0]).view(np.float64)) if op in _INT_IN else float(o.arr[0])
                else:
                    srcs[i] = self._lane(o, op in _INT_IN).vreg
            else:
                imms[i] = float(o)
        d = self._new() if dst else None
        self.instrs.append([op, d, srcs, imms, aux])
        return d

    def _lane(self, val, ibits):
        """``val`` as an instruction operand that holds int64 bits (ibits) or a double: inserts F2I / I2F."""
        if val.ibits == ibits:
            return val
        if val.conv is None:
            if ibits and val.big:
                raise NotImplementedError(
                    "an integer table with values beyond 2^53 feeds integer arithmetic; the device holds table "
                    "values as doubles, which are not exact there")
            d = self._push("F2I" if ibits else "I2F", [val])
            val.conv = _Val(vreg=d, dtype=val.dtype, ibits=ibits)
        return val.conv

    def load(self, input_index):
        d = self._push("LOAD", [], aux=("in", input_index))
        return _Val(vreg=d, dtype=_F64)

    def uniform(self, seed, col):
        d = self._push("UNIFORM", [np.frombuffer(np.uint64(seed).tobytes(), dtype=np.float64)[0]], aux=("col", col))
        return _Val(vreg=d, dtype=_F64)

    def store(self, val, out_index):
        self._push("STORE", [], dst=False, aux=("store", val.vreg, out_index))

    def check(self, val, tag):
        self._push("CHECK", [], dst=False, aux=("check", val.vreg, tag))

    def materialise(self, val):
        """An immediate that must live in a slot (to be stored)."""
        if not val.is_imm:
            return val
        d = self._push("MOV", [val])
        return _Val(vreg=d, dtype=val.dtype)

    def ppf(self, op, q, params):
        d = self._push(op, [q] + list(params))
        return _Val(vreg=d, dtype=_F64)

    def table(self, op, q, table_index, length, method=0, dtype=_F64, big=False):
        d = self._push(op, [q, 0.0, 0.0], aux=("table", table_index))
        self.instrs[-1][3][1] = float(length)
        self.instrs[-1][3][2] = float(method)
        return _Val(vreg=d, dtype=dtype, big=big)

    def lookup(self, idx, table_index, length, dtype, big=False):
        d = self._push("LOOKUP", [idx, 0.0], aux=("table", table_index))
        self.instrs[-1][3][1] = float(length)
        return _Val(vreg=d, dtype=dtype, big=big)

    def raw_binary(self, dev, a, b, dtype):
        if a.is_imm and b.is_imm:
            raise AssertionError("constant sub-graphs are folded before emission")
        d = self._push(dev, [a, b])
        return _Val(vreg=d, dtype=dtype, ibits=OP[dev] in _INT_OUT)

    def _result_dtype(self, node, vals):
        with np.errstate(all="ignore"):
            out = node._numpy([np.empty(0, dtype=v.dtype) for v in vals])
        return np.dtype(out.dtype)

    def _require(self, node, dtype, vals):
        ok = (_F64, _BOOL, _I64)
        if dtype not in ok or any(v.dtype not in ok and not v.is_imm for v in vals):
            raise NotImplementedError(
                f"{node}: NumPy would compute this node in {dtype} from {[str(v.dtype) for v in vals]}; "
                "the device program handles float64, int64 and bool values")

    def binary(self, node, a, b):
        dtype = self._result_dtype(node, [a, b])
        self._require(node, dtype, [a, b])
        if dtype == _I64:  # + - * // % ** max min of int64 / bool operands
            return self.raw_binary("I_" + node.dev, a, b, dtype)
        if node.dev in _INT_CMP and (a.ibits or b.ibits) and _integral(a) and _integral(b):
            op, swap = _INT_CMP[node.dev]  # exact also beyond 2^53
            return self.raw_binary(op, b, a, dtype) if swap else self.raw_binary(op, a, b, dtype)
        both_bool = a.dtype == _BOOL and b.dtype == _BOOL
        return self.raw_binary(node.dev_bool if both_bool else node.dev, a, b, dtype)

    def unary(self, node, a):
        dtype = self._result_dtype(node, [a])
        self._require(node, dtype, [a])
        if dtype == _I64:
            if node.dev in ("FLOOR", "CEIL"):  # the identity on int64
                return a
            return _Val(vreg=self._push("I_" + node.dev, [a]), dtype=dtype, ibits=True)
        d = self._push(node.dev, [a])
        return _Val(vreg=d, dtype=dtype)

    # -- register allocation: virtual registers -> shared-memory slots -------------------------
    def fuse(self):
        """Peephole pass: fold LOAD / UNIFORM into the ppf that consumes the quantile, and CHECK / STORE
        into the instruction that produced the value (flags of include/probabilit_b200.h), so that one
        node costs one interpreted instruction."""
        readers, definer = {}, {}
        for i, (op, d, srcs, imms, aux, *_) in enumerate(self.instrs):
            if d is not None:
                definer[d] = i
            for v in [x for x in srcs if x is not None] + ([aux[1]] if aux and aux[0] in ("store", "check") else []):
                readers.setdefault(v, []).append(i)
        drop = set()
        for i, ins in enumerate(self.instrs):
            op, d, srcs, imms, aux = ins[:5]
            if op in (OP["LOAD"], OP["UNIFORM"]) and len(readers.get(d, [])) == 1:
                j = readers[d][0]
                tgt = self.instrs[j]
                if 16 <= (tgt[0] & 0xFF) < 32 and tgt[2][0] == d and d not in tgt[2][1:]:
                    tgt[0] |= 0x100 if op == OP["LOAD"] else 0x200
                    tgt[2][0] = None
                    tgt[3][0] = imms[0]
                    tgt.append(("q", aux[1]))  # column index, resolved in assemble()
                    drop.add(i)
            elif aux and aux[0] in ("store", "check"):
                j = definer.get(aux[1])
                if j is None:
                    continue
                tgt = self.instrs[j]
                base = tgt[0] & 0xFF
                flag = 0x800 if aux[0] == "store" else 0x400
                if (base >= 16 or (base == OP["MOV"] and aux[0] == "store")) and not (tgt[0] & flag):
                    tgt[0] |= flag
                    tgt.append((aux[0], aux[2]))
                    drop.add(i)
        self.instrs = [ins for i, ins in enumerate(self.instrs) if i not in drop]

    def assemble(self):
        """The program in emission order (the reference's topological order) as ONE launch.  Raises
        ``_GraphTooLarge`` when it needs more slots, instructions, check tags or stored nodes than one launch
        holds."""
        self.fuse()
        return _allocate(self.instrs, self.table_base)

    # -- models larger than one launch ------------------------------------------------------------
    def schedule(self):
        """Leaf chains -- pure instructions that read no value from outside the chain: a ppf of a quantile with
        immediate parameters, a table search and its lookup, a beta / truncnorm core and its ``+ loc``, the LOAD of
        a correlated column, the F2I of a table value -- move to just before their first reader.  A sum of any
        length then keeps 1-2 values live.  Tags stay with their instructions, so the smallest failing tag is the
        same node in any order."""
        n_readers = {}
        for ins in self.instrs:
            for v in set(_reads(ins)):
                n_readers[v] = n_readers.get(v, 0) + 1
        pending, out = {}, []  # defined value -> its chain, not placed yet
        for ins in self.instrs:
            reads = list(dict.fromkeys(_reads(ins)))
            if ins[1] is not None and all(v in pending and n_readers[v] == 1 for v in reads):
                pending[ins[1]] = [x for v in reads for x in pending.pop(v)] + [ins]
                continue
            for v in reads:
                out.extend(pending.pop(v, ()))
            out.append(ins)
        for chain in pending.values():  # values only retained: in emission order
            out.extend(chain)
        return out

    def spill(self, prog):
        """Belady's rule on one launch: when more than MAX_SLOTS values would be live, the one read again furthest
        away is copied to a spill slot (SPILL, unless an earlier copy is still valid), and a FILL into a fresh
        register brings it back just before its next reader.  Returns (program, number of spill slots)."""
        uses = {}
        for i, ins in enumerate(prog):
            for v in set(_reads(ins)):
                uses.setdefault(v, []).append(i)
        nxt = {v: 0 for v in uses}  # index into uses[v] of the next read

        def next_use(v):
            k = nxt[v]
            return uses[v][k] if k < len(uses[v]) else len(prog)

        name, resident, spill_of, free_spills, out = {}, set(), {}, [], []
        n_spills = 0

        def evict(keep):
            nonlocal n_spills
            victim = max((v for v in resident if v not in keep), key=next_use)
            resident.discard(victim)
            if victim not in spill_of:
                if free_spills:
                    spill_of[victim] = heapq.heappop(free_spills)
                else:
                    spill_of[victim], n_spills = n_spills, n_spills + 1
                out.append([OP["SPILL"], None, [name.get(victim, victim), None, None, None], [0.0] * 4,
                            ("spill", spill_of[victim])])

        for ins in prog:
            reads = list(dict.fromkeys(_reads(ins)))
            for v in reads:
                if v not in resident and v in spill_of:
                    if len(resident) >= MAX_SLOTS:
                        evict(set(reads))
                    name[v] = self._new()
                    out.append([OP["FILL"], name[v], [None] * 4, [0.0] * 4, ("fill", spill_of[v])])
                    resident.add(v)
            ins = _renamed(ins, name)
            for v in reads:
                nxt[v] += 1
                if nxt[v] == len(uses[v]):  # last read: the slot (and the spill slot) is free again
                    resident.discard(v)
                    if v in spill_of:
                        heapq.heappush(free_spills, spill_of.pop(v))
            d = ins[1]
            if d is not None and len(resident) >= MAX_SLOTS:
                evict(set(reads))
            out.append(ins)
            if d is not None and d in uses:
                resident.add(d)
        return out, n_spills

    def split(self, n_in, n_out):
        """The scheduled program cut into launches that each fit the kernel (instructions, slots after spills,
        spill slots, check tags).  Cuts go where few values are live.  A value live across a cut goes through an
        n-row column: a retained node's own output column, the input column of a LOAD, or a carry column that
        the defining launch stores.  Each launch gets inputs = caller's inputs + caller's outputs + carry columns.

        Returns (launches, number of carry columns); a launch is (program, slots, tags, outs): ``tags[t]`` is the
        node tag of local CHECK tag t (tags are dense per launch, in increasing order), ``outs`` the indices into
        caller's outputs + carry columns of its output list."""
        order = self.schedule()
        n = len(order)
        pos = {ins[1]: i for i, ins in enumerate(order) if ins[1] is not None}
        last = {}
        for i, ins in enumerate(order):
            for v in _reads(ins):
                last[v] = i
        delta = [0] * (n + 2)
        for v, i in last.items():
            delta[pos[v] + 1] += 1
            delta[i + 1] -= 1
        live = list(itertools.accumulate(delta))  # live[p]: values defined before p and read at p or later
        carry = {}  # value -> input index of the column it travels in
        launches, n_carry, start = [], 0, 0
        while start < n:
            size = MAX_INSTR * 3 // 4
            while True:
                end = n if n - start <= size else \
                    min(range(start + (size + 1) // 2, start + size + 1), key=lambda p: (live[p], -p))
                try:
                    launch, new_carry = self._one_launch(order, start, end, last, carry, n_in, n_out, n_carry)
                    break
                except _GraphTooLarge:
                    if size == 1:
                        raise
                    size //= 2
            launches.append(launch)
            for v, idx in new_carry.items():
                carry[v] = idx
                n_carry += idx >= n_in + n_out
            start = end
        return launches, n_carry

    def _one_launch(self, order, start, end, last, carry, n_in, n_out, n_carry):
        seg, loaded, new_carry = [], set(), {}
        for i in range(start, end):
            ins = order[i]
            for v in _reads(ins):
                if v in carry and v not in loaded:  # defined by an earlier launch
                    seg.append([OP["LOAD"], v, [None] * 4, [0.0] * 4, ("in", carry[v])])
                    loaded.add(v)
            ins = [ins[0], ins[1], list(ins[2]), list(ins[3]), ins[4], *ins[5:]]
            v = ins[1]
            if v is not None and last.get(v, -1) >= end:  # read by a later launch
                stored = [o for kind, o in ins[5:] if kind == "store"]
                if stored:
                    new_carry[v] = n_in + stored[0]
                elif ins[0] == OP["LOAD"]:
                    new_carry[v] = ins[4][1]
                else:
                    new_carry[v] = n_in + n_out + n_carry + sum(i >= n_in + n_out for i in new_carry.values())
                    if (ins[0] & 0xFF) >= 16 or (ins[0] & 0xFF) == OP["MOV"]:
                        ins[0] |= 0x800
                        ins.append(("store", new_carry[v] - n_in))
                    else:
                        seg.append(ins)
                        ins = [OP["STORE"], None, [None] * 4, [0.0] * 4, ("store", v, new_carry[v] - n_in)]
            seg.append(ins)
        prog, n_spills = self.spill(seg)
        if n_spills > MAX_SPILLS:
            raise _GraphTooLarge(f"a launch needs {n_spills} spill slots (max {MAX_SPILLS})")
        tags = sorted({_tag(ins) for ins in prog} - {None})
        outs = sorted({_out(ins) for ins in prog} - {None})
        local_tag, local_out = {t: k for k, t in enumerate(tags)}, {o: k for k, o in enumerate(outs)}
        for k, ins in enumerate(prog):
            aux = ins[4]
            if aux and aux[0] == "check":
                aux = ("check", aux[1], local_tag[aux[2]])
            elif aux and aux[0] == "store":
                aux = ("store", aux[1], local_out[aux[2]])
            extra = [(kind, local_tag[x] if kind == "check" else local_out[x] if kind == "store" else x)
                     for kind, x in ins[5:]]
            prog[k] = [ins[0], ins[1], ins[2], ins[3], aux, *extra]
        return (*_allocate(prog, self.table_base), tags, outs), new_carry


class _GraphTooLarge(NotImplementedError):
    """A program needs more slots, instructions or check tags than one launch of the kernel holds."""


def _reads(ins):
    """The values an instruction [op, dst, srcs, imms, aux, *fused] reads."""
    aux = ins[4]
    return [s for s in ins[2] if s is not None] + ([aux[1]] if aux and aux[0] in ("store", "check") else [])


def _renamed(ins, name):
    if not any(v in name for v in _reads(ins)):
        return ins
    aux = ins[4]
    if aux and aux[0] in ("store", "check"):
        aux = (aux[0], name.get(aux[1], aux[1]), aux[2])
    return [ins[0], ins[1], [name.get(s, s) for s in ins[2]], ins[3], aux, *ins[5:]]


def _tag(ins):
    aux = ins[4]
    if aux and aux[0] == "check":
        return aux[2]
    return next((x for kind, x in ins[5:] if kind == "check"), None)


def _out(ins):
    aux = ins[4]
    if aux and aux[0] == "store":
        return aux[2]
    return next((x for kind, x in ins[5:] if kind == "store"), None)


def _allocate(instrs, table_base):
    """Virtual registers -> slots (linear scan, a slot is reused after the last read of its value) and the
    pbl_graph_instr records of one launch."""
    reads = [_reads(ins) for ins in instrs]
    last = {}
    for i, r in enumerate(reads):
        for v in r:
            last[v] = i
    free, slot_of, n_slots = [], {}, 0
    prog = (_lib.GraphInstr * len(instrs))()
    for i, (op, d, srcs, imms, aux, *extra) in enumerate(instrs):
        ins = prog[i]
        ins.op = op
        for j in range(4):
            ins.src[j] = -1 if srcs[j] is None else slot_of[srcs[j]]
            ins.imm[j] = imms[j]
        if aux:
            if aux[0] in ("in", "col", "fill"):
                ins.src[0] = aux[1]
            elif aux[0] == "table":
                ins.src[1] = table_base + aux[1]
            elif aux[0] in ("store", "check"):
                ins.src[0], ins.src[1] = slot_of[aux[1]], aux[2]
            elif aux[0] == "spill":
                ins.src[1] = aux[1]
        for v in set(reads[i]):
            if last[v] == i:
                free.append(slot_of[v])
        ins.dst = 0
        if d is not None:
            if free:
                s = free.pop()
            else:
                s, n_slots = n_slots, n_slots + 1
            slot_of[d] = s
            ins.dst = s
            if d not in last:  # never read: the slot is free again right away
                free.append(s)
        for kind, value in extra:  # fused flags
            if kind == "q":
                ins.src[0] = value
            elif kind == "check":
                if value >= MAX_TAGS:
                    raise _GraphTooLarge(f"graph has more than {MAX_TAGS} checked nodes")
                ins.dst |= (value & 0xFFF) << 8
            elif kind == "store":
                if value >= MAX_OUTPUTS:
                    raise _GraphTooLarge(f"graph stores more than {MAX_OUTPUTS} nodes")
                ins.dst |= value << 20
    if n_slots > MAX_SLOTS:
        raise _GraphTooLarge(f"graph needs {n_slots} live values per sample; the kernel holds {MAX_SLOTS}")
    if len(instrs) > MAX_INSTR:
        raise _GraphTooLarge(f"graph compiles to {len(instrs)} instructions (max {MAX_INSTR})")
    return prog, max(n_slots, 1)


def _launch(prog, n_slots, n, row0, inputs, outputs):
    """One pbl_graph_eval_f64 call.  Returns the smallest failing CHECK tag of the program or -1."""
    lib = _lib.require_gpu()
    if len(prog) == 0:
        return -1
    in_arr = (C.c_void_p * max(len(inputs), 1))(*inputs)
    out_arr = (C.c_void_p * max(len(outputs), 1))(*outputs)
    bad = C.c_int32(-1)
    st = _lib.check(lib.pbl_graph_eval_f64(prog, len(prog), n_slots, n, row0, in_arr, len(inputs), out_arr,
                                           len(outputs), C.byref(bad), None), "pbl_graph_eval_f64")
    if st != _lib.STATUS_OK:
        raise ValueError(_lib.last_error())
    return bad.value


def _run_program(em, n, row0, inputs, outputs):
    """inputs / outputs: lists of device column addresses.  Returns the smallest failing node tag or -1.

    A program that fits one launch in emission order runs as it is.  A larger one is scheduled, spilled and cut
    into several launches (``_Emitter.split``).  Every launch runs even after one has failed: scheduling can
    move a node with a smaller tag into a later launch, and the smallest failing tag over all launches is the
    node the reference reports first."""
    try:
        prog, n_slots = em.assemble()
    except _GraphTooLarge:
        pass
    else:
        return _launch(prog, n_slots, n, row0, inputs, outputs)
    launches, n_carry = em.split(len(inputs), len(outputs))
    carry = DeviceColumns(n, n_carry) if n_carry else None  # freed when the call returns
    columns = list(outputs) + [carry.column_ptr(j) for j in range(n_carry)]
    bad = -1
    for prog, n_slots, tags, outs in launches:
        b = _launch(prog, n_slots, n, row0, list(inputs) + columns, [columns[o] for o in outs])
        if b >= 0 and (bad < 0 or tags[b] < bad):
            bad = tags[b]
    return bad


class _GraphRun:
    """One call of sample_from_quantiles: compile, run, attach ``samples_``."""

    def __init__(self, sink, quantiles, correlator, gc_strategy):
        self.sink = sink
        self.G = sink.to_graph()
        assert nx.is_directed_acyclic_graph(self.G)
        if isinstance(quantiles, _PhiloxSource):
            self.philox, self.qcols, self._keep = quantiles, None, None
            self.size, n_dim = quantiles.shape
        else:
            self.philox = None
            self.qcols, self._keep = as_device_columns(quantiles)
            self.size, n_dim = self.qcols.n, self.qcols.k
        assert n_dim == sink.num_distribution_nodes()
        table = {"imanconover": ImanConover, "cholesky": Cholesky}  # reference :505-507
        self.correlator = table[correlator.lower()] if isinstance(correlator, str) else correlator
        if not (gc_strategy is None or hasattr(gc_strategy, "__contains__")):
            raise TypeError(f"`strategy` must be None or a collection, got: {gc_strategy}")
        self.gc_strategy = gc_strategy

    # -- which nodes keep samples_ (reference garbage_collector.py:24-71) -----------------------
    def retained(self, node):
        return self.gc_strategy is None or node is self.sink or node == self.sink or node in self.gc_strategy

    def quantile(self, em, col):
        return em.uniform(self.philox.seed, col) if self.philox else em.load(col)

    def parameters(self, node, value_of):
        op, params = node._bound_parameters()
        vals = []
        for p in params:
            if isinstance(p, Node):
                vals.append(value_of[p])
            elif isinstance(p, numbers.Number):
                vals.append(_Val(arr=np.array([float(p)])))
            else:
                raise NotImplementedError(f"{node}: parameter {p!r} is neither a number nor a Node")
        return op, vals

    def add_table(self, array):
        self.tables.append(np.ascontiguousarray(array, dtype=np.float64))
        return len(self.tables) - 1

    def emit_distribution(self, em, node, value_of, column):
        """One distribution node: quantile column -> inverse CDF (scipy ppf or a table lookup)."""
        q = self.quantile(em, column[node])
        if isinstance(node, Distribution):
            op, params = self.parameters(node, value_of)
            if op in (OP["PPF_BETA"], OP["PPF_TRUNCNORM"]):  # (a, b, loc, scale) -> op(q, a, b, scale) + loc
                a, b, loc, scale = params
                core = em.ppf(op, q, [a, b, scale])
                return em.raw_binary("ADD", core, loc, _F64)
            return em.ppf(op, q, params)
        if isinstance(node, CumulativeDistribution):  # np.interp(q, self.q, self.cumulatives), reference :880-882
            t = self.add_table(np.concatenate([node.q.astype(np.float64), node.cumulatives.astype(np.float64)]))
            return em.table("TABLE_INTERP", q, t, len(node.q))
        if isinstance(node, EmpiricalDistribution):  # np.quantile(self.data, q, **kwargs), reference :841-842
            data, method, dtype = node._table()
            return em.table("TABLE_QUANTILE", q, self.add_table(data), len(data), method, dtype=dtype,
                            big=_beyond_exact(node.data))
        # DiscreteDistribution: values[searchsorted(cumsum(p), q, "right")], reference :910-913
        cum = np.cumsum(node.probabilities)
        idx = em.table("TABLE_SEARCH", q, self.add_table(cum), len(cum))
        values = node.values
        if np.issubdtype(values.dtype, np.number) or values.dtype == np.bool_:
            return em.lookup(idx, self.add_table(values.astype(np.float64)), len(values), values.dtype,
                             big=_beyond_exact(values))
        self.categories[node] = values  # non-numeric categories: the device keeps the index
        return _Val(vreg=idx.vreg, dtype=values.dtype)

    def upload_tables(self):
        cols = [DeviceColumns.from_host(t.reshape(-1, 1)) for t in self.tables]
        return cols, [c.column_ptr(0) for c in cols]

    def execute(self):
        sink, G, n = self.sink, self.G, self.size
        self.tables, self.categories = [], {}
        members = set(sink.nodes())
        for node in members:
            node.__dict__.pop("_store", None)
        table_kinds = (EmpiricalDistribution, CumulativeDistribution, DiscreteDistribution)
        unsupported = [m for m in members if isinstance(m, ScalarFunctionTransform) or
                       (isinstance(m, AbstractDistribution) and not isinstance(m, (Distribution,) + table_kinds))]
        if unsupported:
            raise NotImplementedError(f"no device implementation for {unsupported[0]!r}")

        # quantile columns: initial sampling nodes by _id, then the rest in topological order
        topo = list(nx.topological_sort(G))
        isns = sorted((m for m in members if m._is_initial_sampling_node()), key=lambda m: m._id)
        column = {node: i for i, node in enumerate(isns)}
        for node in topo:
            if isinstance(node, AbstractDistribution) and node not in column:
                column[node] = len(column)

        # correlations to induce (reference :540-569)
        correlations = []
        for node in members:
            correlations.extend(node._correlations)
        for variables, _ in correlations:
            for variable in variables:
                if variable not in isns:
                    raise ValueError(f"Cannot correlate variable: {variable}")
        var_sets = [set(variables) for variables, _ in correlations]
        for s1, s2 in itertools.combinations(var_sets, 2):
            common = s1 & s2
            if len(common) > 1:
                raise ValueError(f"Correlations specified more than once: {common}")
        corr_vars = sorted(functools.reduce(set.union, var_sets, set()), key=lambda m: m._id)
        corr_index = {v: i for i, v in enumerate(corr_vars)}

        # constant folding: nodes without any distribution above them
        folded = {}
        for node in topo:
            if isinstance(node, Constant):
                folded[node] = node._fold()
            elif isinstance(node, Transform) and all(p in folded for p in node.get_parents()):
                with np.errstate(all="ignore"):
                    folded[node] = node._numpy([folded[p] for p in node.get_parents()])

        corr_cols = None
        if correlations:
            corr_cols = self.run_correlation(corr_vars, corr_index, correlations, column, folded)

        # main program, nodes in topological order (reference :586-612)
        em = _Emitter()
        value_of = {node: _Val(arr=arr) for node, arr in folded.items() if arr is not None}
        keep, const_fail, n_stored = [], None, 0
        int_pow = set()  # tags of int64 Power nodes: their CHECK reports a negative exponent
        for tag, node in enumerate(topo):
            if node in folded:
                arr = folded[node]
                val = None if arr is None else value_of[node]
            elif node in corr_index:
                val = em.load(("corr", corr_index[node]))
            elif isinstance(node, AbstractDistribution):
                val = self.emit_distribution(em, node, value_of, column)
            else:
                val = node._emit(em, [value_of[p] for p in node.get_parents()])
            if val is None:  # NoOp: `samples_` is None (reference :993-997)
                if self.retained(node):
                    node.__dict__["_store"] = _Samples(none=True)
                continue
            value_of[node] = val
            numeric = np.issubdtype(val.dtype, np.number)
            if val.is_imm:
                if numeric and not np.all(np.isfinite(val.arr)) and const_fail is None:
                    const_fail = tag
            elif isinstance(node, Power) and val.ibits:
                em.check(val, tag)
                int_pow.add(tag)
            elif numeric and not val.ibits:
                em.check(val, tag)
            if self.retained(node):
                keep.append((node, val))
                if not val.is_imm and node not in corr_index:
                    em.store(val, n_stored)  # right away: the slot is free again after its last use
                    n_stored += 1

        # inputs: quantile columns first, then the correlated columns
        nq = 0 if self.qcols is None else self.qcols.k
        inputs = [] if self.qcols is None else [self.qcols.column_ptr(j) for j in range(nq)]
        for ins in em.instrs:
            aux = ins[4]
            if aux and aux[0] == "in" and isinstance(aux[1], tuple):
                ins[4] = ("in", nq + aux[1][1])
        if corr_cols is not None:
            inputs += [corr_cols.column_ptr(j) for j in range(corr_cols.k)]
        em.table_base = len(inputs)
        table_cols, table_ptrs = self.upload_tables()
        inputs += table_ptrs

        stored = [(node, val) for node, val in keep if not val.is_imm and node not in corr_index]
        assert len(stored) == n_stored
        out_cols = DeviceColumns(n, len(stored)) if stored else None
        outputs = [out_cols.column_ptr(j) for j in range(len(stored))]
        bad = _run_program(em, n, 0, inputs, outputs)
        if const_fail is not None and (bad < 0 or const_fail < bad):
            bad = const_fail
        if bad in int_pow:
            raise ValueError("Integers to negative integer powers are not allowed.")  # NumPy's message
        if bad >= 0:
            raise ValueError(f"Sampling this node gave non-finite values: {topo[bad]}")

        for node, val in keep:
            if val.is_imm:
                node.__dict__["_store"] = _Samples(const=val.arr, size=n)
            elif node in corr_index:
                node.__dict__["_store"] = _Samples(columns=corr_cols, index=corr_index[node], dtype=val.dtype)
        for j, (node, val) in enumerate(stored):
            node.__dict__["_store"] = _Samples(columns=out_cols, index=j, dtype=val.dtype,
                                               categories=self.categories.get(node), ibits=val.ibits)

    def run_correlation(self, corr_vars, corr_index, correlations, column, folded):
        """Sample the correlated initial sampling nodes, induce the correlations
        (reference :571-583) and return the correlated (n, k) device columns."""
        n = self.size
        em = _Emitter()
        value_of = {node: _Val(arr=arr) for node, arr in folded.items() if arr is not None}
        X = DeviceColumns(n, len(corr_vars))
        first_table = len(self.tables)
        for j, node in enumerate(corr_vars):
            if node in self.categories or (isinstance(node, DiscreteDistribution)
                                           and not np.issubdtype(node.values.dtype, np.number)):
                raise ValueError(f"Cannot correlate non-numeric variable: {node}")
            em.store(self.emit_distribution(em, node, value_of, column), j)
        inputs = [] if self.qcols is None else [self.qcols.column_ptr(j) for j in range(self.qcols.k)]
        em.table_base = len(inputs)
        table_cols, table_ptrs = self.upload_tables()
        _run_program(em, n, 0, inputs + table_ptrs, [X.column_ptr(j) for j in range(X.k)])
        del self.tables[first_table:]  # the main program registers its own tables

        indexed = [(tuple(corr_index[v] for v in variables), mat) for variables, mat in correlations]
        target = nearest_correlation_matrix(build_corrmat(indexed))
        instance = self.correlator().set_target(target)
        if hasattr(instance, "correlate_device"):
            return instance.correlate_device(X)
        out = instance(X.to_host())  # a foreign correlator: the reference's NumPy protocol
        return DeviceColumns.from_host(out)


def scalar_transform(func):
    @functools.wraps(func)
    def wrapped(*args, **kwargs):
        return ScalarFunctionTransform(func, args, kwargs)

    return wrapped
