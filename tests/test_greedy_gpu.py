"""K11 (dd_greedy_dense_hist, dd_greedy_compact, dd_greedy_sparse_hist) on the device: histograms and live counts
against torch brute force bit for bit, sparse steps against dense ones over successive union updates, the whole
greedy order against per-candidate K3 unions, refusals, and the greedy command line on the real engine against the
`dandd progressive -r ordering.pickle --ksweep` replay."""
import csv
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
BINS = 64


@pytest.fixture(scope="module")
def eng():
    from dandd_b200.engine import get_engine
    return get_engine()


def make_regs(n, nk, p, seed, dev, clusters=None):
    """HLL-like registers, values 1 .. 64 - p + 1, in clusters of near-copies, with an exact duplicate and a zero
    genome when n > 2."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    m = 1 << p
    top = 64 - p + 1
    geo = lambda *shape: torch.clamp(torch.distributions.Geometric(0.5).sample(shape).to(torch.int64) + 1, max=top)  # noqa: E731
    torch.manual_seed(seed)
    roots = geo(clusters or max(1, n // 8), nk, m)
    regs = roots[torch.randint(0, roots.shape[0], (n,), generator=g)].clone()
    change = torch.rand((n, nk, m), generator=g) < 0.1
    regs[change] = geo(int(change.sum()))
    if n > 2:
        regs[n - 1] = regs[0]
        regs[n // 2] = 0
    return regs.to(torch.uint8).to(dev).contiguous()


def brute(regs, union, cand):
    """(hist int32 [C, nk, 64], live int32 [C, nk]) by explicit maxima."""
    nk = union.shape[0]
    rowid = torch.arange(nk, device=regs.device)[:, None] * BINS
    hist = torch.stack([torch.bincount((rowid + torch.maximum(union, regs[g]).long()).flatten(), minlength=nk * BINS)
                        .view(nk, BINS) for g in cand])
    live = torch.stack([(regs[g] > union).sum(dim=1) for g in cand])
    return hist.int(), live.int()


def union_case(case, regs, p, seed):
    nk, m = regs.shape[1:]
    if case == "zero":
        return torch.zeros((nk, m), dtype=torch.uint8, device=regs.device)
    if case == "equal":
        return regs[0].clone()
    if case == "maximal":
        return torch.full((nk, m), 64 - p + 1, dtype=torch.uint8, device=regs.device)
    idx = np.random.default_rng(seed).choice(regs.shape[0], min(3, regs.shape[0]), replace=False)
    return regs[torch.as_tensor(idx, device=regs.device)].amax(dim=0)


def cand_case(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "all":
        return list(range(n))
    if kind == "one":
        return [int(rng.integers(n))]
    return sorted(rng.choice(n, max(1, n // 3), replace=False).tolist())


def offsets(live, cand, n, nk):
    counts = np.zeros((n, nk), dtype=np.int64)
    counts[cand] = live.cpu().numpy()
    return np.concatenate([[0], np.cumsum(counts.reshape(-1))])


SHAPES = [(2, 31, 20), (3, 23, 18), (3, 1, 10), (40, 23, 14), (40, 1, 20), (400, 1, 18), (400, 31, 10), (400, 7, 14)]


@pytest.mark.parametrize("kind", ["all", "subset", "one"])
@pytest.mark.parametrize("case", ["zero", "equal", "maximal", "grown"])
@pytest.mark.parametrize("n,nk,p", SHAPES)
def test_dense_and_sparse_equal_brute_force(eng, n, nk, p, case, kind):
    regs = make_regs(n, nk, p, seed=n * 1000 + nk * 10 + p, dev=eng.device)
    union = union_case(case, regs, p, seed=n + p)
    cand = cand_case(kind, n, seed=nk + p)
    _, uh = eng.cards_hist(union, p)
    want = brute(regs, union, cand)
    got = eng.greedy_dense_hist(regs, union, uh, cand, p)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    state = eng.greedy_compact(regs, union, cand, offsets(want[1], cand, n, nk), p)
    assert torch.equal(state["seg_len"].view(n, nk)[cand], want[1])
    got = eng.greedy_sparse_hist(state, union, uh, cand, p)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


@pytest.mark.parametrize("n,nk,p", [(40, 23, 14), (400, 7, 14), (3, 31, 20)])
def test_sparse_follows_union_updates(eng, n, nk, p):
    """Compact once at the empty union, then 1..5 union updates: sparse == dense == brute force every time,
    including segments that empty (the duplicate of genome 0, and the chosen genomes' near-copies)."""
    regs = make_regs(n, nk, p, seed=p + n, dev=eng.device)
    union = torch.zeros((nk, 1 << p), dtype=torch.uint8, device=eng.device)
    cand = list(range(n))
    _, uh = eng.cards_hist(union, p)
    _, live = eng.greedy_dense_hist(regs, union, uh, cand, p)
    state = eng.greedy_compact(regs, union, cand, offsets(live, cand, n, nk), p)
    for pick in [0, 1, 2, 3, 4][:min(5, n - 1)]:
        union = torch.maximum(union, regs[pick])
        cand.remove(pick)
        _, uh = eng.cards_hist(union, p)
        want = brute(regs, union, cand)
        dense = eng.greedy_dense_hist(regs, union, uh, cand, p)
        sparse = eng.greedy_sparse_hist(state, union, uh, cand, p)
        for got in (dense, sparse):
            assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), pick
    if n > 2:
        assert int(state["seg_len"].view(n, nk)[n - 1].sum()) == 0      # genome n - 1 == genome 0


def k3_greedy(eng, regs, ks, p, steps, order, first):
    """The greedy order from per-candidate K3 unions (Engine.union_sets over chosen + candidate, all k)."""
    n, nk, m = regs.shape
    base = regs.data_ptr()
    kdiv = np.asarray(ks, dtype=np.float64)
    picks, cards = [], []
    for t in range(steps):
        rest = [g for g in range(n) if g not in picks]
        table = np.array([[base + (i * nk + c) * m for i in picks + [g]] for g in rest for c in range(nk)], dtype=np.int64)
        got = eng.union_sets(table, p, final_only=True).cpu().numpy().reshape(len(rest), nk)
        if t < len(first):
            pick = first[t]
        else:
            d = (got / kdiv).max(axis=1)
            pick = rest[int(np.argmax(d) if order == "max" else np.argmin(d))]
        picks.append(pick)
        cards.append(got[rest.index(pick)])
    return picks, np.asarray(cards)


@pytest.mark.parametrize("budget", [None, 0], ids=["selected", "dense_only"])
@pytest.mark.parametrize("order,first", [("max", ()), ("min", ()), ("max", (7, 3))])
@pytest.mark.parametrize("n,clusters", [(40, 5), (200, 20)])
def test_order_equals_per_candidate_unions(eng, monkeypatch, n, clusters, order, first, budget):
    from dandd_b200 import store as ddstore
    ks, p = list(range(8, 13)), 12
    regs = make_regs(n, len(ks), p, seed=n + clusters, dev=eng.device, clusters=clusters)
    if budget is None:
        monkeypatch.setattr(ddstore, "SPARSE_CROSS", 0)            # the sparse phase from the first evaluated step
    st = ddstore.GpuSketchStore(engine=eng)
    steps = n if n == 40 else 60
    got, cards, stats = st.greedy_order(regs, ks, p, steps, order=order, first=first, budget=budget)
    want, want_cards = k3_greedy(eng, regs, ks, p, steps, order, first)
    assert got.tolist() == want and np.array_equal(cards, want_cards)
    assert (stats["sparse_steps"] > 0) == (budget is None)


def test_refusals_leave_the_outputs_alone(eng):
    from dandd_b200._lib import DandDError
    p, nk, n = 10, 2, 4
    regs = make_regs(n, nk, p, seed=4, dev=eng.device)
    union = torch.zeros((nk, 1 << p), dtype=torch.uint8, device=eng.device)
    _, uh = eng.cards_hist(union, p)
    before = eng.lib.dd_kernel_launches()
    for cand, match in [([0, 4], "outside"), ([-1], "outside"), ([1, 1], "listed twice")]:
        with pytest.raises(DandDError, match=match):
            eng.greedy_dense_hist(regs, union, uh, cand, p)
        with pytest.raises(DandDError, match=match):
            eng.greedy_compact(regs, union, cand, np.zeros(n * nk + 1, dtype=np.int64), p)
    with pytest.raises(DandDError, match="decrease"):
        eng.greedy_compact(regs, union, [0], np.array([0, 5, 3] + [3] * (n * nk - 2), dtype=np.int64), p)
    with pytest.raises(DandDError, match="16-byte"):
        eng.greedy_dense_hist(regs, torch.zeros(nk * (1 << p) + 1, dtype=torch.uint8, device=eng.device)[1:].view(nk, -1),
                              uh, [0], p)
    torch.cuda.synchronize()
    assert eng.lib.dd_kernel_launches() == before
    # a refused sparse call leaves the segments as they were
    _, live = eng.greedy_dense_hist(regs, union, uh, [0, 1], p)
    state = eng.greedy_compact(regs, union, [0, 1], offsets(live, [0, 1], n, nk), p)
    entries, seg_len = state["entries"].clone(), state["seg_len"].clone()
    with pytest.raises(DandDError, match="outside"):
        eng.greedy_sparse_hist(state, regs[2], uh, [0, 9], p)
    torch.cuda.synchronize()
    assert torch.equal(entries, state["entries"]) and torch.equal(seg_len, state["seg_len"])


def _read_tsv(path, delimiter="\t"):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter=delimiter))


def test_command_line_on_the_engine(tmp_path):
    """helpers/greedy.py on synthetic FASTAs; growth.tsv == the `dandd progressive -r ordering.pickle --ksweep` replay
    on the real store."""
    from dandd_b200 import store as ddstore
    from dandd_b200.helpers import greedy
    from tests.host_harness import run_dandd
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 8, 20000, seed=12)
    name, out = str(tmp_path / "run"), str(tmp_path / "out")
    lo, hi, p = 8, 15, 14
    ddstore.set_store(ddstore.GpuSketchStore())
    try:
        greedy.go(["-d", data, "--mink", str(lo), "--maxk", str(hi), "--registers", str(p), "--name", name])
        run_dandd(["tree", "-d", data, "-s", "gr", "-o", out, "-r", str(p)])
        run_dandd(["progressive", "-d", os.path.join(out, "gr_8_dashing_dtree.pickle"), "-o", out, "--ksweep",
                   "--mink", str(lo), "--maxk", str(hi), "-r", os.path.join(name, "ordering.pickle")])
    finally:
        ddstore.set_store(None)
    summary = [f for f in os.listdir(out) if f.endswith("summary.csv")]
    replay = {(int(r["ngen"]), int(r["kval"])): float(r["card"]) for r in _read_tsv(os.path.join(out, summary[0]), ",")}
    growth = _read_tsv(os.path.join(name, "growth.tsv"))
    assert len(growth) == len(replay) == 8 * (hi - lo + 1)
    for r in growth:
        assert float(r["card"]) == replay[(int(r["ngen"]), int(r["k"]))], r
