"""Models larger than one launch of the graph kernel holds in the reference's evaluation order: more than 96 live
values, more than 4096 instructions or more than 4096 checked nodes.  Shared by tests/test_graph_large_cpu.py
(compiler + bytecode VM) and tests/test_graph_large_gpu.py (the kernel).  Each builder takes the module of node
classes and returns the sink.

Not in graph_recipes.RECIPES: those recipes are pinned to golden vectors of the unmodified reference."""
import numpy as np


def triang_clt(m, k=562):
    """The central-limit example of the reference's tests: a sum of k triangular distributions."""
    c = np.linspace(0.05, 0.95, k)
    return m.Add(*[m.Distribution("triang", c=float(ci), loc=i % 7, scale=1 + i % 3) for i, ci in enumerate(c)])


def items(m, k, seed=0):
    """k mixed cost items: norm, gamma, beta (PERT), truncnorm and empirical."""
    rng = np.random.default_rng(seed)
    data = rng.lognormal(size=101)
    out = []
    for i in range(k):
        kind = i % 5
        if kind == 0:
            out.append(m.Distribution("norm", loc=10 + i % 9, scale=1 + i % 4))
        elif kind == 1:
            out.append(m.Distribution("gamma", a=1.5 + i % 3, scale=2.0))
        elif kind == 2:
            out.append(m.Distribution("beta", a=2.0 + i % 5, b=3.0, loc=i % 11, scale=5.0))
        elif kind == 3:
            out.append(m.Distribution("truncnorm", a=-1.0, b=2.5, loc=3.0, scale=0.5 + i % 2))
        else:
            out.append(m.EmpiricalDistribution(data * (1 + i % 3)))
    return out


def fanout(m, k=200):
    """A sum and a maximum over the same k items: every item stays live from the sum to the maximum, so the
    program needs about k values at once and spills."""
    xs = items(m, k)
    return m.Add(*xs) - m.Max(*xs)


def dice(m, k=150):
    """int64 arithmetic over k dice that are all live at once: the spilled values are int64 bit patterns."""
    ds = [m.DiscreteDistribution([1, 2, 3, 4, 5, 6]) for _ in range(k)]
    return m.Add(*ds) * 1000 + m.Max(*ds) - m.Min(*ds)


def pert_items(m, k=1500):
    """k PERT line items (beta core, + loc, + to the sum: 3 instructions each): several launches."""
    rng = np.random.default_rng(7)
    lo = rng.uniform(1, 10, k)
    mode = lo + rng.uniform(0, 5, k)
    hi = mode + rng.uniform(1, 10, k)
    a = 1 + 4 * (mode - lo) / (hi - lo)
    b = 1 + 4 * (hi - mode) / (hi - lo)
    return m.Add(*[m.Distribution("beta", a=float(a[i]), b=float(b[i]), loc=float(lo[i]), scale=float(hi[i] - lo[i]))
                   for i in range(k)])


def long_chain(m, k=2100):
    """A chain of 2k + 3 nodes, constants included: node tags beyond the 12 bits of one launch."""
    x = m.Distribution("norm", loc=5, scale=1)
    for i in range(k):
        x = x * 0.999 if i % 2 else x + 0.25
    return x + m.Distribution("uniform")


def correlated(m, k=120):
    """k correlated initial sampling nodes summed."""
    xs = [m.Distribution("norm", loc=i % 5, scale=1) if i % 2 else m.Distribution("expon", scale=1 + i % 3)
          for i in range(k)]
    corr = np.full((k, k), 0.2) + 0.8 * np.eye(k)
    return m.Add(*xs).correlate(*xs, corr_mat=corr)


def boundary(m, k):
    """A sum of k triangular distributions: 96 fit one launch in the reference's order, 97 do not."""
    return m.Add(*[m.Distribution("triang", c=0.25 + 0.5 * (i % 2), loc=i, scale=2) for i in range(k)])


GRAPHS = {"triang_clt": triang_clt, "fanout": fanout, "dice": dice, "pert_items": pert_items,
          "long_chain": long_chain, "correlated": correlated, "boundary96": lambda m: boundary(m, 96),
          "boundary97": lambda m: boundary(m, 97)}
