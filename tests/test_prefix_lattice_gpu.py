"""Prefix unions from the per-k subset table (-m gpu): dd_prefix_union_card takes the lattice path for index-mode jobs
of n_genomes <= 12 and p >= 12.  Every case compares histograms (==) and cardinalities (==) with the planes path
(dd_set_option("prefix_lattice", 0)), and a few cells with the oracle."""
import numpy as np
import pytest
import torch

import bench
from oracle import pyoracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    return Engine(0)


def run(eng, regs, orders, p, final_only, lattice):
    """(hist [n_ord, steps, nk, 64], cards [n_ord, steps, nk], kernel launches) of one dd_prefix_union_card call."""
    from dandd_b200._lib import check
    n_g, nk, _ = regs.shape
    order = torch.as_tensor(np.asarray(orders, dtype=np.int32)).cuda().contiguous()
    n_ord, n_steps = order.shape
    osteps = 1 if final_only else n_steps
    hist = torch.full((n_ord, osteps, nk, 64), 0x5A5A5A5A, dtype=torch.int32, device="cuda")   # every bin must be written
    cards = torch.empty((n_ord, osteps, nk), dtype=torch.float64, device="cuda")
    ws = torch.empty(eng.lib.dd_prefix_union_workspace_bytes(n_ord, n_steps, n_g, nk, p), dtype=torch.uint8, device="cuda")
    check(eng.lib.dd_set_option(b"prefix_lattice", int(lattice)), "dd_set_option")
    try:
        torch.cuda.synchronize()
        l0 = eng.lib.dd_kernel_launches()
        check(eng.lib.dd_prefix_union_card(regs.data_ptr(), order.data_ptr(), n_ord, n_steps, n_g, nk, p, int(final_only),
                                           cards.data_ptr(), hist.data_ptr(), None, ws.data_ptr(), ws.numel(), None),
              "dd_prefix_union_card")
        torch.cuda.synchronize()
        launches = eng.lib.dd_kernel_launches() - l0
    finally:
        check(eng.lib.dd_set_option(b"prefix_lattice", 1), "dd_set_option")
    return hist.cpu().numpy(), cards.cpu().numpy(), launches


def both(eng, regs, orders, p, final_only):
    h1, c1, l1 = run(eng, regs, orders, p, final_only, True)
    h0, c0, l0 = run(eng, regs, orders, p, final_only, False)
    assert np.array_equal(h1, h0)
    assert np.array_equal(c1, c0)
    assert (h1.astype(np.int64).sum(-1) == 1 << p).all()
    return h1, c1, l1 != l0


def oracle_cells(regs_np, orders, p, final_only, hist, cards, cells):
    for o, st, k in cells:
        members = [g for g in orders[o][:st + 1] if 0 <= g < regs_np.shape[0]]
        u = orc.union_max([regs_np[g, k] for g in members]) if members else np.zeros(1 << p, np.uint8)
        row = 0 if final_only else st
        assert np.array_equal(hist[o, row, k], orc.hist(u, p)[:64].astype(np.int32))
        want = orc.card(u, p)
        assert abs(cards[o, row, k] - want) <= 1e-9 * max(want, 1.0)


def random_regs(rng, n, nk, p, shared=0.7):
    """Related sketches: a common base, each genome replacing a share of the registers with its own values."""
    top = 64 - p + 1
    base = np.minimum(rng.geometric(0.5, size=(nk, 1 << p)), top)
    regs = np.repeat(base[None], n, axis=0)
    own = rng.random((n, nk, 1 << p)) > shared
    regs[own] = np.minimum(rng.geometric(0.5, size=int(own.sum())), top)
    regs[:, :, :64] = 0   # a run of registers that are empty in every sketch
    return regs.astype(np.uint8)


def orderings(rng, n, n_ord, n_steps):
    return np.stack([rng.permutation(n)[:n_steps] if n_steps <= n else rng.integers(0, n, n_steps)
                     for _ in range(n_ord)]).astype(np.int32)


@pytest.mark.parametrize("n", [1, 2, 11, 12, 13])
@pytest.mark.parametrize("p", [12, 16, 20])
@pytest.mark.parametrize("nk", [1, 23])
@pytest.mark.parametrize("final_only", [False, True])
def test_random_sketches(eng, n, p, nk, final_only):
    if p == 20 and nk == 23:
        pytest.skip("p = 20 with 23 k is the bench-shape case")
    rng = np.random.default_rng(1000 * n + 10 * p + nk + final_only)
    regs_np = random_regs(rng, n, nk, p)
    orders = orderings(rng, n, 7, n)
    regs = torch.from_numpy(regs_np).cuda()
    hist, cards, differ = both(eng, regs, orders, p, final_only)
    assert differ == (n <= 12 and not (final_only and n == 2))   # n = 13 and pairs take the planes path
    last = n - 1
    oracle_cells(regs_np, orders, p, final_only, hist, cards, [(0, last, 0), (6, last, nk - 1)] +
                 ([] if final_only else [(1, 0, nk // 2), (3, n // 2, 0)]))


def test_repeats_and_skipped_members(eng):
    """Orderings that name a genome twice inside a prefix, entries < 0 or >= n_genomes, an all-skipped ordering."""
    rng = np.random.default_rng(5)
    n, nk, p = 6, 3, 14
    regs_np = random_regs(rng, n, nk, p)
    orders = np.array([[0, 0, 3, 3, 5, 0, 1, 2],
                       [-1, 4, 4, 99, 2, -7, 2, 1],
                       [-1, -1, -1, -1, -1, -1, -1, -1],
                       [5, 4, 3, 2, 1, 0, 5, 4]], dtype=np.int32)
    for final_only in (False, True):
        hist, cards, differ = both(eng, torch.from_numpy(regs_np).cuda(), orders, p, final_only)
        assert differ
        cells = [(o, 7, k) for o in range(4) for k in range(nk)]
        if not final_only:
            cells += [(o, st, 1) for o in range(4) for st in range(7)]
        oracle_cells(regs_np, orders, p, final_only, hist, cards, cells)


@pytest.mark.parametrize("case", ["zero", "equal", "one_on_top", "extremes"])
def test_crafted_registers(eng, case):
    rng = np.random.default_rng(9)
    n, nk, p = 12, 2, 12
    top = 64 - p + 1
    m = 1 << p
    if case == "zero":
        regs_np = np.zeros((n, nk, m), np.uint8)
    elif case == "equal":
        regs_np = np.repeat(rng.integers(0, top + 1, size=(1, nk, m)), n, axis=0).astype(np.uint8)
    elif case == "one_on_top":
        regs_np = np.repeat(rng.integers(0, top, size=(1, nk, m)), n, axis=0).astype(np.uint8)
        g = rng.integers(0, n, size=(nk, m))
        for kk in range(nk):
            regs_np[g[kk], kk, np.arange(m)] += 1
    else:   # every value 0..top in every genome, independently
        regs_np = rng.integers(0, top + 1, size=(n, nk, m)).astype(np.uint8)
        regs_np[:, :, :top + 1] = np.arange(top + 1, dtype=np.uint8)
    orders = orderings(rng, n, 5, n)
    for final_only in (False, True):
        hist, cards, differ = both(eng, torch.from_numpy(regs_np).cuda(), orders, p, final_only)
        assert differ
        oracle_cells(regs_np, orders, p, final_only, hist, cards, [(o, n - 1, k) for o in range(5) for k in range(nk)] +
                     ([] if final_only else [(o, st, 0) for o in range(2) for st in range(n)]))


def test_bench_shape(eng):
    """12 x 5 Mbp bench genomes, k = 10..32, p = 20, the bench's 30 orderings."""
    regs = torch.empty((bench.N_GENOMES, len(bench.KS), 1 << bench.P), dtype=torch.uint8, device="cuda")
    for g, (text, _) in enumerate(bench.make_genomes(seed=2)):
        eng.sketch(eng.pack(text), bench.KS, p=bench.P, out=regs[g])
    orders = bench.make_orderings(bench.N_GENOMES, bench.N_ORDERINGS, seed=2)
    hist, cards, differ = both(eng, regs, orders, bench.P, False)
    assert differ
    regs_np = regs.cpu().numpy()
    oracle_cells(regs_np, orders, bench.P, False, hist, cards, [(0, 0, 0), (3, 5, 11), (29, 11, 22), (17, 8, 6)])
