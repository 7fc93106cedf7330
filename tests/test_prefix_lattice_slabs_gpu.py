"""Register patterns that stress the lattice level pass (-m gpu): values above the shared table's V (the spill
rows), the full-set cells counted per thread, small per-CTA register ranges and the largest V.  Every case
compares histograms (==) and cardinalities (==) with the planes path, and a few cells with the oracle."""
import numpy as np
import pytest
import torch

from tests.test_prefix_lattice_gpu import both, oracle_cells, orderings, random_regs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    return Engine(0)


def check(eng, regs_np, p, n_ord=6, seed=0):
    n, nk, _ = regs_np.shape
    orders = orderings(np.random.default_rng(seed), n, n_ord, n)
    for final_only in (False, True):
        hist, cards, differ = both(eng, torch.from_numpy(regs_np).cuda(), orders, p, final_only)
        assert differ
        oracle_cells(regs_np, orders, p, final_only, hist, cards, [(o, n - 1, k) for o in range(2) for k in (0, nk - 1)] +
                     ([] if final_only else [(0, st, 0) for st in range(n)]))


@pytest.mark.parametrize("n", [12, 10])
def test_values_above_table(eng, n):
    """Most registers >= 15 (V = 14 at n = 12, 56 at n = 10): most updates take the spill rows."""
    rng = np.random.default_rng(21 + n)
    p, nk = 12, 3
    top = 64 - p + 1
    base = rng.integers(10, top + 1, size=(1, nk, 1 << p))
    regs = np.repeat(base, n, axis=0)
    own = rng.random((n, nk, 1 << p)) > 0.5
    regs[own] = rng.integers(0, top + 1, size=int(own.sum()))
    check(eng, regs.astype(np.uint8), p)


@pytest.mark.parametrize("values", [(1, 2, 3), (4, 5, 6)])
def test_equal_sketches_small_values(eng, values):
    """Every sketch equal, values from a short range: each register is one full-set level, at the minima counted
    per thread (1..4) or in the shared table (5, 6)."""
    rng = np.random.default_rng(values[0])
    n, nk, p = 12, 2, 16
    one = rng.choice(np.array(values, np.uint8), size=(1, nk, 1 << p))
    check(eng, np.repeat(one, n, axis=0), p)


def test_many_k_small_p(eng):
    """p = 12 with 23 k: a few CTAs per k, each with a short register range."""
    rng = np.random.default_rng(12)
    regs = random_regs(rng, 12, 23, 12)
    check(eng, regs, 12)


@pytest.mark.parametrize("n", [1, 3, 7])
def test_few_genomes(eng, n):
    """n = 3 holds the whole value range in shared memory (V = 63); n = 1 and 7 cover the other word counts,
    n = 1 with minima far above the per-thread counters."""
    rng = np.random.default_rng(30 + n)
    p, nk = 16, 4
    regs = random_regs(rng, n, nk, p)
    if n == 1:
        regs = np.minimum(regs.astype(np.int32) + 10, 64 - p + 1).astype(np.uint8)
    check(eng, regs, p)
