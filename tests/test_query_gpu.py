"""K13 on the device: query genomes against references over the K7 lists (dandd_b200.engine exact_query_counts) against
oracle k-mer sets, in one or several passes; both counter placements; more than 32 queries on one list; overflow; the
Q x R block and the set rows against K7 and K8 on the same genomes; the HLL path against K3 per-union cards and K6 pair
cards; and helpers/query.py end to end on the real engine against the CPU-double run."""
import csv
import os

import numpy as np
import pytest

from tests.test_exact_pairs_gpu import _genomes
from tests.test_exact_sets_gpu import _holders

pytestmark = pytest.mark.gpu

KS = [5, 12, 16, 17, 31, 32, 33, 64, 65, 127]
R = 3        # genomes 0..2 are the references, 3..6 the queries: genome 4 is a copy of genome 0, genome 5 holds no k-mer above k = 4


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


def _want(held, members, n_refs):
    """(singles, inter [Q, R], shared [Q], union) for genomes `members` (indices into the columns of held)."""
    h = held[:, members].astype(np.int64)
    ref, qry = h[:, :n_refs], h[:, n_refs:]
    has_ref = ref.any(axis=1)
    return h.sum(axis=0).tolist(), (qry.T @ ref).tolist(), qry[has_ref].sum(axis=0).tolist(), int(has_ref.sum())


def _got(res):
    singles, inter, shared, union = res
    assert singles.dtype == inter.dtype == shared.dtype == np.uint64
    return singles.astype(np.int64).tolist(), inter.astype(np.int64).tolist(), shared.astype(np.int64).tolist(), union


@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("k", KS)
def test_query_counts_equal_the_oracle_sets(eng, packed, k, canon, passes):
    """Queries sit on lists that hold references (a copy of reference 0 is a query): the walk relies on their order."""
    texts, seqs = packed
    held, _ = _holders(texts, k, canon)
    got = _got(eng.exact_query_counts(seqs, R, k, canon, passes=passes))
    assert eng.last_pair_plan["passes"] == passes
    want = _want(held, list(range(len(seqs))), R)
    assert got == want
    if k > 4:
        assert got[1][1][0] == got[2][1] == want[0][0]                  # the copy of reference 0 is all shared


@pytest.mark.parametrize("k", [21, 40])
@pytest.mark.parametrize("n_queries,n_refs", [(3, 40), (40, 700)])
def test_both_counter_placements(eng, packed, k, n_queries, n_refs):
    """Q = 3, R = 40: (QR + Q) u32 in shared memory; Q = 40, R = 700: 112 KiB, global atomics.  The genomes repeat the
    7 test genomes, so every list holds many references and queries."""
    texts, seqs = packed
    held, _ = _holders(texts, k, True)
    members = [(5 * i + 2) % len(seqs) for i in range(n_refs)] + [(3 * i + 1) % len(seqs) for i in range(n_queries)]
    got = _got(eng.exact_query_counts([seqs[g] for g in members], n_refs, k, True))
    assert got == _want(held, members, n_refs)


@pytest.mark.parametrize("k", [15, 31, 70])
def test_more_than_32_queries_on_one_list(eng, packed, k):
    """70 copies of genome 1 and a copy of reference 0 as queries: 71 query nodes precede the references on a list."""
    texts, seqs = packed
    held, _ = _holders(texts, k, True)
    members = [0, 2] + [1] * 70 + [4]
    got = _got(eng.exact_query_counts([seqs[g] for g in members], 2, k, True))
    want = _want(held, members, 2)
    assert got == want and got[2][0] > 0 and got[1][-1][0] == want[0][0]


def test_overflow_raises(eng, packed):
    from dandd_b200._lib import DandDError
    from dandd_b200 import engine as E
    _, seqs = packed
    real = E.length_bounds
    E.length_bounds = lambda nsyms, k, world=1: [1] * len(nsyms)
    try:
        with pytest.raises(DandDError, match="overflow"):
            eng.exact_query_counts(seqs, R, 21, True)
    finally:
        E.length_bounds = real


@pytest.mark.parametrize("k", [12, 25, 50, 90])
def test_equals_k7_and_k8_on_the_same_genomes(eng, packed, k):
    """The Q x R block of K7's all-pairs triangle over the R + Q genomes; K8 rows for U_R and every U_R + q."""
    texts, seqs = packed
    n = len(seqs)
    Q = n - R
    singles, inter, shared, union = eng.exact_query_counts(seqs, R, k, True)
    tri = eng.exact_pairs_sparse(seqs, k, True, singles.tolist()).astype(np.int64)
    row = lambda a, b: a * (2 * n - a - 1) // 2 + (b - a - 1)
    assert inter.astype(np.int64).tolist() == [[int(tri[row(r, R + q)]) for r in range(R)] for q in range(Q)]
    ranks = np.full((1 + Q, n), 0xFFFF, dtype=np.uint16)
    ranks[:, :R] = 0
    for q in range(Q):
        ranks[1 + q, R + q] = 0
    hist = eng.exact_first_rank_hist(seqs, k, True, ranks, singles=singles.tolist()).astype(np.int64)
    assert union == int(hist[0, 0])
    assert (union + singles[R:].astype(np.int64) - shared.astype(np.int64)).tolist() == hist[1:, 0].tolist()


@pytest.mark.parametrize("p", [10, 14])
def test_hll_cards_equal_k3_unions_and_pair_cards(eng, packed, p):
    import torch
    from dandd_b200.store import GpuSketchStore
    _, seqs = packed
    ks = list(range(9, 16))
    regs = torch.stack([eng.sketch(s, ks, p)[0] for s in seqs]).contiguous()
    st = GpuSketchStore(engine=eng)
    ref_single, query_single, union, with_q, pair = st.query_cards(regs, R, p)
    n, Q = len(seqs), len(seqs) - R
    single = eng.cards(regs, p).cpu().numpy()
    assert np.array_equal(ref_single, single[:R].T) and np.array_equal(query_single, single[R:].T)
    assert np.array_equal(union, eng.cards(eng.union([regs[r] for r in range(R)]), p).cpu().numpy())
    for q in range(Q):
        want = eng.cards(eng.union([regs[r] for r in range(R)] + [regs[R + q]]), p).cpu().numpy()
        assert np.array_equal(with_q[:, q], want), q
    pairs = [(r, R + q) for q in range(Q) for r in range(R)]
    want = st.pair_cards(regs, pairs, p)
    assert np.array_equal(pair.transpose(1, 2, 0).reshape(Q * R, len(ks)), want)
    assert np.array_equal(with_q[:, 1], union)                          # the copy of reference 0 adds nothing


def _tables(name):
    out = {}
    for fn in ("union.tsv", "collection.tsv", "with.tsv", "delta.tsv", "pairs.tsv", "kij.tsv"):
        with open(os.path.join(name, fn), newline="") as fh:
            out[fn] = list(csv.DictReader(fh, delimiter="\t"))
    return out


@pytest.mark.parametrize("tool", ["dashing", "kmc"])
def test_helper_matches_the_cpu_double(tmp_path, tool):
    """The helper on the real engine and on QueryFakeEngine: kmc files identical, dashing numbers within 1e-9."""
    import shutil
    from dandd_b200 import store as ddstore
    from dandd_b200.helpers import query
    from tests.query_engine import QueryFakeEngine
    from tests.util import make_dataset
    refs = make_dataset(str(tmp_path / "refs"), 4, 2500, seed=41, prefix="r")
    make_dataset(str(tmp_path / "queries"), 2, 2500, seed=41, sub=0.08, prefix="q")
    shutil.copy(refs[2], str(tmp_path / "queries" / "r2.fasta"))
    argv = ["-d", str(tmp_path / "refs"), "-q", str(tmp_path / "queries"), "--tool", tool, "--mink", "4", "--maxk", "12",
            "--registers", "12"]
    runs = {}
    for label, store in (("gpu", ddstore.GpuSketchStore()), ("cpu", ddstore.GpuSketchStore(engine=QueryFakeEngine()))):
        ddstore.set_store(store)
        try:
            query.go(argv + ["--name", str(tmp_path / label)])
        finally:
            ddstore.set_store(None)
        runs[label] = str(tmp_path / label)
    if tool == "kmc":
        for fn in ("union.tsv", "collection.tsv", "with.tsv", "delta.tsv", "pairs.tsv", "kij.tsv"):
            assert open(os.path.join(runs["gpu"], fn), "rb").read() == open(os.path.join(runs["cpu"], fn), "rb").read(), fn
        return
    gpu, cpu = _tables(runs["gpu"]), _tables(runs["cpu"])
    for fn in gpu:
        assert len(gpu[fn]) == len(cpu[fn]) > 0, fn
        for a, b in zip(gpu[fn], cpu[fn]):
            assert a.keys() == b.keys()
            for col in a:
                try:
                    x, y = float(a[col]), float(b[col])
                except ValueError:
                    assert a[col] == b[col], (fn, col)
                    continue
                if col in ("novel", "gain"):                            # differences of two estimates
                    assert x == pytest.approx(y, abs=1e-4), (fn, col)
                elif col in ("jaccard", "containment", "kij"):          # ratios of such differences
                    assert x == pytest.approx(y, abs=1e-6), (fn, col)
                else:
                    assert x == pytest.approx(y, rel=1e-9), (fn, col)
