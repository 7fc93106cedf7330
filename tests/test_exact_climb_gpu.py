"""The family job on the device (dandd_b200.engine exact_family_counts): single counts from the K7 list-node counter and
first-rank histograms of set and prefix rows, against oracle k-mer sets; passes and shards; the length-sized plan;
and `tree --exact` / `progressive --exact` hill-climbs on the real engine against the per-union path, file for file."""
import os
import random

import numpy as np
import pytest

from tests.test_exact_climb import PROG, TREE, _assert_same, _snapshot
from tests.test_exact_pairs_gpu import _genomes
from tests.test_exact_sets_gpu import _holders, _want

pytestmark = pytest.mark.gpu

KS = [1, 7, 15, 16, 17, 31, 32, 33, 64, 65, 200]
NO = 0xFFFF


@pytest.fixture(scope="module")
def eng():
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    return Engine(0)


@pytest.fixture(scope="module")
def packed(eng):
    texts = _genomes()
    return texts, [eng.pack(t).check() for t in texts]


def _family_table(n, seed):
    """What a climb registers: set rows (tree nodes: zeros for the members) and prefix rows (orderings: positions),
    plus a partial ordering and a set holding only the genome without k-mers."""
    rng = np.random.default_rng(seed)
    rows = [np.where(rng.random(n) < 0.5, 0, NO) for _ in range(4)] + [np.zeros(n, dtype=np.int64)]
    rows += [np.argsort(rng.permutation(n)) for _ in range(4)]
    part = np.full(n, NO, dtype=np.int64)
    part[rng.permutation(n)[:3]] = [0, 1, 2]
    empty = np.full(n, NO, dtype=np.int64)
    empty[n - 2] = 0
    return np.array(rows + [part, empty], dtype=np.uint16)


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("k", KS)
def test_family_counts_equal_the_oracle_sets(eng, packed, k, canon):
    texts, seqs = packed
    held, singles = _holders(texts, k, canon)
    ranks = _family_table(len(seqs), k)
    got_singles, got = eng.exact_family_counts(seqs, k, canon, ranks)
    assert got_singles.dtype == np.uint64 and got.dtype == np.uint64 and got.shape == ranks.shape
    assert got_singles.astype(np.int64).tolist() == singles
    assert got.astype(np.int64).tolist() == _want(held, ranks).tolist()
    assert eng.last_pair_plan["path"] == "sparse"


@pytest.mark.parametrize("k", [12, 33, 99])
def test_passes_and_shards_add_up(eng, packed, k):
    texts, seqs = packed
    ranks = _family_table(len(seqs), 3)
    s1, h1 = eng.exact_family_counts(seqs, k, True, ranks, passes=1)
    for passes in (2, 3):
        s, h = eng.exact_family_counts(seqs, k, True, ranks, passes=passes)
        assert eng.last_pair_plan["passes"] == passes
        assert s.tolist() == s1.tolist() and h.tolist() == h1.tolist()
    parts = [eng.exact_family_counts(seqs, k, True, ranks, shard=(r, 2)) for r in range(2)]
    assert (parts[0][0] + parts[1][0]).tolist() == s1.tolist() and (parts[0][1] + parts[1][1]).tolist() == h1.tolist()
    assert all(p[0].sum() > 0 for p in parts)                     # both halves hold keys
    held, singles = _holders(texts, k, True)
    assert s1.astype(np.int64).tolist() == singles and h1.astype(np.int64).tolist() == _want(held, ranks).tolist()
    assert singles[len(seqs) - 2] == 0                             # the genome without k-mers


def test_no_rows_still_gives_singles(eng, packed):
    texts, seqs = packed
    s, h = eng.exact_family_counts(seqs, 21, True, np.zeros((0, len(seqs)), dtype=np.uint16))
    assert h.shape == (0, len(seqs)) and s.astype(np.int64).tolist() == _holders(texts, 21, True)[1]


@pytest.mark.parametrize("k", [3, 9, 21, 40, 120])
def test_length_sized_plan_covers_the_singles_sized_one(eng, packed, k):
    """The job sized from the lengths is never smaller than the one sized from the real counts, for one process and
    for each of two key-range shards, and it runs without overflow wherever the singles-sized job does."""
    from dandd_b200.engine import length_bounds, plan_pair_passes
    texts, seqs = packed
    n = len(seqs)
    ws = lambda c, m: int(eng.lib.dd_exact_pairs_workspace_bytes(k, c, m, n))    # noqa: E731
    for shard in (None, (0, 2), (1, 2)):
        singles = [eng.exact_counts([s], k, True, shard=shard)[0] for s in seqs]
        eng.exact_first_rank_hist(seqs, k, True, _family_table(n, 1), singles, shard=shard)   # the singles-sized job runs
        by_singles = eng.last_pair_plan
        eng.exact_family_counts(seqs, k, True, _family_table(n, 1), shard=shard)
        by_length = eng.last_pair_plan
        assert by_length["capacity"] >= by_singles["capacity"] and by_length["max_nodes"] >= by_singles["max_nodes"]
        bounds = length_bounds([s.nsym for s in seqs], k, shard[1] if shard else 1)
        if shard is None:
            assert all(b >= c for b, c in zip(bounds, singles))
        assert plan_pair_passes(bounds, k, ws, 1 << 40)["max_nodes"] >= sum(singles)


def test_overflow_raises(eng, packed):
    """A full node array still turns into DandDError (the forced plan here is far too small)."""
    from dandd_b200._lib import DandDError
    from dandd_b200 import engine as E
    _, seqs = packed
    real = E.length_bounds
    E.length_bounds = lambda nsyms, k, world=1: [1] * len(nsyms)
    try:
        with pytest.raises(DandDError, match="overflow"):
            eng.exact_family_counts(seqs, 21, True, _family_table(len(seqs), 1))
    finally:
        E.length_bounds = real


def _cli(tmp, argvs, batch):
    from dandd_b200 import store as ddstore
    from tests.host_harness import run_dandd
    from tests.util import make_dataset
    make_dataset(os.path.join(tmp, "data"), 5, 3000, seed=23)
    st = ddstore.GpuSketchStore()
    ddstore.set_store(st)
    os.environ["DANDD_B200_EXACT_SET_BATCH"] = "1" if batch else "0"
    try:
        for argv in argvs:
            random.seed(3)
            run_dandd([a.replace("<tmp>", tmp) for a in argv])
    finally:
        os.environ.pop("DANDD_B200_EXACT_SET_BATCH", None)
        ddstore.set_store(None)
    return _snapshot(tmp), st


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
def test_cli_hillclimb_equals_the_per_union_path(tmp_path, canon):
    argvs = [TREE + ["-n", "2", "-k", "6"] + ([] if canon else ["--no-canon"]), PROG + ["-n", "3", "--step", "2"]]
    a, st_a = _cli(str(tmp_path / "a"), argvs, True)
    b, st_b = _cli(str(tmp_path / "b"), argvs, False)
    _assert_same(a, b)
    assert any("progu" in f for f in a)
    assert st_a.stats["exact_family_jobs"] > 0 and st_b.stats["exact_family_jobs"] == 0
    assert st_a.stats["exact_calls"] == st_a.stats["exact_family_jobs"] < st_b.stats["exact_calls"]
