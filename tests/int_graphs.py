"""Modeling graphs whose nodes NumPy computes in int64, shared by tests/test_graph_int_cpu.py (compiler + bytecode VM)
and tests/test_graph_int_gpu.py (the kernel).  Each graph builder takes the module of node classes and returns the
sink; every node of the graph is compared with oracle.modeling.evaluate, dtype and bits.

Not in graph_recipes.RECIPES: those recipes are pinned to golden vectors of the unmodified reference."""
import numpy as np

I64MIN = int(np.iinfo(np.int64).min)
SNAN = 0x7FF0000000000001  # an int64 whose bit pattern is a signalling NaN


def die(m):
    return m.DiscreteDistribution([1, 2, 3, 4, 5, 6])


def two_dice(m):
    return die(m) + die(m)


def counting_events(m):
    x, y, u = m.Distribution("norm"), m.Distribution("norm"), m.Distribution("uniform")
    return m.NoOp(3 * (x > 0), (u < 0.3) + 0, m.Add(x > 0, y > 1) * 1)


def scenarios(m):
    d1, d2 = die(m), die(m)
    return m.NoOp(m.DiscreteDistribution([100, 200, 500]) * 4, m.Max(d1, d2), m.Min(d1, 4), -d1, abs(d1 - 4))


def integer_ufuncs(m):
    d = die(m)
    return m.NoOp(d // 2, m.Equal(d % 2, 0), d ** 2, m.Sign(d - 3), m.Square(d), m.Floor(d), m.Ceil(d - 2), 7 // d,
                  7 % (d - 3), -7 % (d - 3))


def empirical(m):
    lower = m.EmpiricalDistribution([1, 5, 9], method="lower")
    near = m.EmpiricalDistribution([-4, 5, 9, 12], method="closest_observation")
    return m.NoOp(lower * 2, near - lower, m.EmpiricalDistribution([3, 1, 2], method="nearest") ** 3)


def works_before(m):
    d = die(m)
    return m.NoOp(d / 2, m.Equal(d, 3), d)


def wrap_around(m):
    d1, d2 = die(m), die(m)
    big = d1 * 2 ** 62
    return m.NoOp(big * 4, (d1 + 2 ** 62) * 4, d1 * 3 ** 39, 2 ** (d1 + 60), (d2 + 1) ** 40, -(big - I64MIN),
                  abs(d1 * 0 + I64MIN), m.Square(d1 * 2 ** 31 + 7), d1 - I64MIN, d1 * -1, d1 + SNAN,
                  (d1 - d1) ** (d2 - d2), m.Sign(big))


def division_edges(m):
    d = m.DiscreteDistribution([-3, -2, -1, 0, 1, 2, 3])
    lo = d * 0 + I64MIN
    return m.NoOp(lo // d, lo % d, I64MIN // d, I64MIN % d, (lo + 5) // (d - d - 1), (d - 4) // d, (d + 7) % d,
                  lo // -1, lo % -1, d // 0, d % 0)


def big_comparisons(m):
    d1, d2 = die(m), die(m)
    a, b = d1 + 2 ** 53, d2 + 2 ** 53
    return m.NoOp(a > b, a >= b, a < b, a <= b, m.Equal(a, b), m.NotEqual(a, b), m.Equal(a, 2 ** 53 + 1),
                  d1 * 2 ** 60 < d2 * 2 ** 60, m.GreaterThan(d1 + SNAN, d2 + SNAN), m.Equal(d1 % 2, True))


def int_to_float(m):
    d1, d2 = die(m), die(m)
    a = d1 + 2 ** 53
    x = m.Distribution("norm")
    return m.NoOp(a + 0.5, a * 1.0, m.Equal(a, 2.0 ** 53), a > 2.0 ** 53, (d1 + d2) / 2, m.Sqrt(d1 * d2), a + x,
                  m.Max(d1 + d2, x), m.Log(d1 * 3), m.Arctan2(d1 - 3, d2 + 0), (d1 + d2) ** 0.5, 2.5 ** (d1 - 3),
                  m.IsClose(d1 + d2, 7), d1 * 2 // 1.5)


def bool_int_mixing(m):
    d1, d2 = die(m), die(m)
    x, y = m.Distribution("norm"), m.Distribution("norm")
    lo = d1 * 0 + I64MIN
    return m.NoOp((x > 0) + d1, (x > 0) * (d1 + d2), m.Max(x > 0, d1 - 3), d1 ** (y > 0), (d1 - 3) // (x > 0),
                  m.All(d1 % 2, x > 0), m.Any(d1 % 3, d2 % 3), m.All(lo, lo), m.Equal((x > 0) + 0, 1),
                  m.DiscreteDistribution([True, False]) + d1, m.Avg(d1, d2, x), m.Avg(d1 + d2, d1 - 1),
                  m.Avg(d1 + d2, x > y))


def composite(m):
    d1, d2 = die(m), die(m)
    n = d1 + d2
    b = m.Distribution("binom", n=n, p=0.4)
    p = m.Distribution("poisson", mu=d1 * 2)
    g = m.Distribution("norm", loc=d1 + d2, scale=abs(d1 - 3) + 1)
    return m.NoOp(b, b + n, p - d2, g * (d1 % 2))


GRAPHS = {f.__name__: f for f in (two_dice, counting_events, scenarios, integer_ufuncs, empirical, works_before,
                                  wrap_around, division_edges, big_comparisons, int_to_float, bool_int_mixing,
                                  composite)}


def random_graph(m, seed):
    """Dice, integer tables and events combined by random integer (and some float) ufuncs.  A combination NumPy
    rejects or computes in another dtype is skipped, and so is a float // % or ** (it can be non-finite)."""
    r = np.random.default_rng(4000 + seed)
    pool = [die(m), m.DiscreteDistribution([-5, 0, 7, 1000], [0.1, 0.2, 0.3, 0.4]),
            m.EmpiricalDistribution([2, 3, 5, 7, 11], method="higher"), m.Distribution("norm") > 0.3,
            m.Distribution("poisson", mu=4.5)]
    probe = {id(n): np.ones(1, dtype=t) for n, t in zip(pool, (np.int64, np.int64, np.int64, np.bool_, np.float64))}

    def dtype_of(node):  # NumPy's result dtype, from one-element arrays
        if id(node) not in probe:
            with np.errstate(all="ignore"):
                probe[id(node)] = (node._fold() if isinstance(node, m.Constant)
                                   else node._numpy([dtype_of(p) for p in node.get_parents()]))
        return probe[id(node)]

    ops = {
        "add": lambda a, b: a + b, "sub": lambda a, b: a - b, "mul": lambda a, b: a * b,
        "floordiv": lambda a, b: a // b, "mod": lambda a, b: a % b, "pow": lambda a, b: a ** (abs(b) % 4),
        "max": m.Max, "min": m.Min, "gt": lambda a, b: a > b, "le": lambda a, b: a <= b, "eq": m.Equal,
        "ne": m.NotEqual, "neg": lambda a, b: -a, "abs": lambda a, b: abs(a), "sign": lambda a, b: m.Sign(a),
        "square": lambda a, b: m.Square(a), "avg": m.Avg, "all": m.All, "any": m.Any,
    }
    for _ in range(int(r.integers(8, 18))):
        a = pool[int(r.integers(len(pool)))]
        b = pool[int(r.integers(len(pool)))] if r.random() < 0.7 else \
            [int(r.integers(-9, 10)), 2 ** int(r.integers(40, 63)), True, float(r.normal())][int(r.integers(4))]
        op = str(r.choice(list(ops)))
        try:
            node = ops[op](a, b)
            dtype = dtype_of(node).dtype
        except TypeError:
            continue
        if dtype in (np.int64, np.bool_) or (dtype == np.float64 and op not in ("floordiv", "mod", "pow")):
            pool.append(node)
    return m.NoOp(*pool[-6:])
