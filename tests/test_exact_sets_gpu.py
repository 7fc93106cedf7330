"""K8 on the device: first-rank histograms over the K7 lists (dandd_b200.engine exact_first_rank_hist), against
histograms computed in Python from oracle k-mer sets, and the store's prefix counts against the per-ordering path."""
import numpy as np
import pytest

from tests.test_exact_pairs_gpu import _genomes, _kmer_set

pytestmark = pytest.mark.gpu

KS = [1, 5, 12, 16, 17, 31, 32, 33, 64, 65, 100, 256]
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


def _holders(texts, k, canon):
    """[n_keys, n] bool: which genome holds which distinct k-mer; and the single counts."""
    from oracle import pyoracle as orc
    sets = [_kmer_set(orc.fasta_symbols(t), k, canon) for t in texts]
    keys = list(set().union(*sets))
    return np.array([[x in s for s in sets] for x in keys], dtype=bool).reshape(len(keys), len(sets)), [len(s) for s in sets]


def _want(held, ranks):
    n = held.shape[1]
    out = np.zeros(ranks.shape, dtype=np.int64)
    for r, row in enumerate(ranks):
        first = np.where(held, row[None, :].astype(np.int64), NO).min(axis=1) if held.size else np.zeros(0, dtype=np.int64)
        out[r] = np.bincount(first[first < n], minlength=n)
    return out


def _rank_table(n, seed):
    """Random orderings, partial rows (genomes left out), rows with ties, set rows, an empty row."""
    rng = np.random.default_rng(seed)
    rows = [rng.permutation(n) for _ in range(5)]
    for _ in range(4):
        row = rng.permutation(n).astype(np.int64)
        row[rng.random(n) < 0.4] = NO
        rows.append(row)
    rows += [rng.integers(0, 3, n) for _ in range(4)]
    rows += [np.where(rng.random(n) < 0.5, 0, NO) for _ in range(4)]
    rows += [np.full(n, NO), np.zeros(n, dtype=np.int64)]
    return np.array(rows, dtype=np.uint16)


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("k", KS)
def test_hist_equals_the_oracle_sets(eng, packed, k, canon):
    """(k = 32 --no-canon: the poly-T runs of the genomes make the all-ones key, which lives in the extra slot.)"""
    texts, seqs = packed
    held, singles = _holders(texts, k, canon)
    ranks = _rank_table(len(seqs), k)
    got = eng.exact_first_rank_hist(seqs, k, canon, ranks, singles)
    assert got.dtype == np.uint64 and got.shape == ranks.shape
    assert got.astype(np.int64).tolist() == _want(held, ranks).tolist()


@pytest.mark.parametrize("rows", [40, 4000, 12000])
def test_shared_and_global_counters(eng, packed, rows):
    """R x n decides where counters and ranks live: 40 rows -- both in shared memory; 4000 -- counters in global
    memory (R x n x 4 > 96 KiB), ranks in shared memory; 12000 -- both global."""
    texts, seqs = packed
    held, singles = _holders(texts, 21, True)
    base = _rank_table(len(seqs), 9)
    reps = -(-rows // base.shape[0])
    ranks = np.tile(base, (reps, 1))[:rows]
    want = np.tile(_want(held, base), (reps, 1))[:rows]
    assert eng.exact_first_rank_hist(seqs, 21, True, ranks, singles).astype(np.int64).tolist() == want.tolist()


@pytest.mark.parametrize("k", [12, 21, 47, 99])
def test_passes_and_shards_add_up(eng, packed, k):
    texts, seqs = packed
    ranks = _rank_table(len(seqs), 3)
    one = eng.exact_first_rank_hist(seqs, k, True, ranks, passes=1)
    for passes in (2, 3):
        assert eng.exact_first_rank_hist(seqs, k, True, ranks, passes=passes).tolist() == one.tolist()
        assert eng.last_pair_plan["passes"] == passes
    world = 2
    parts = [eng.exact_first_rank_hist(seqs, k, True, ranks, shard=(r, world)) for r in range(world)]
    assert np.sum(parts, axis=0).tolist() == one.tolist()
    assert one.astype(np.int64).tolist() == _want(_holders(texts, k, True)[0], ranks).tolist()


@pytest.mark.parametrize("k", [13, 31, 64, 99])
def test_genome_inserted_in_two_ranges(eng, packed, k):
    """One genome's k-mers arriving in two overlapping ranges still count once."""
    import torch
    from dandd_b200._lib import check
    texts, seqs = packed
    ranks = _rank_table(3, 5)
    want = _want(_holders(texts[:3], k, True)[0], ranks)
    lib, st = eng.lib, eng.stream
    n, cap, nodes = 3, 1 << 16, 20000
    ws = torch.empty(lib.dd_exact_pairs_workspace_bytes(k, cap, nodes, n), dtype=torch.uint8, device=eng.device)
    d_ranks = torch.from_numpy(ranks.view(np.int16)).to(eng.device)
    out = torch.zeros(ranks.shape, dtype=torch.int64, device=eng.device)
    check(lib.dd_exact_pairs_begin(ws.data_ptr(), ws.numel(), k, cap, nodes, n, st))
    for g, s in enumerate(seqs[:3]):
        ns = s.nsym
        for b, e in ([(0, ns // 2 + 40), (ns // 2, ns)] if g == 1 else [(0, ns)]):
            check(lib.dd_exact_pairs_insert_shard(s.codes.data_ptr(), s.invalid.data_ptr(), b, e, k, 1, g, ws.data_ptr(),
                                                  ws.numel(), cap, nodes, n, 0, 1, st))
    check(lib.dd_exact_first_rank_hist(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, d_ranks.data_ptr(), ranks.shape[0],
                                       out.data_ptr(), st))
    assert out.cpu().tolist() == want.tolist()


def test_overflow_raises_and_bad_arguments_are_refused(eng, packed):
    from dandd_b200._lib import DandDError
    _, seqs = packed
    with pytest.raises(DandDError, match="overflow"):
        eng.exact_first_rank_hist(seqs, 21, True, _rank_table(len(seqs), 1), [1] * len(seqs))
    lib = eng.lib
    need = lib.dd_exact_pairs_workspace_bytes(21, 1024, 4096, 2)
    assert lib.dd_exact_first_rank_hist(1 << 20, need, 21, 1024, 4096, 2, 70000, 1 << 20, 1, 1 << 20, None) == -1
    assert b"n_genomes" in lib.dd_last_error()
    assert lib.dd_exact_first_rank_hist(1 << 20, need, 21, 1024, 4096, 2, 2, None, 1, 1 << 20, None) == -1
    assert lib.dd_exact_first_rank_hist(1 << 20, need - 1, 21, 1024, 4096, 2, 2, 1 << 20, 1, 1 << 20, None) == -3


def test_store_prefix_cards_equal_the_per_ordering_path(tmp_path):
    from dandd_b200 import build
    build.build()
    from dandd_b200 import store as ddstore
    st = ddstore.GpuSketchStore()
    files = []
    for i, t in enumerate(_genomes()):
        f = tmp_path / ("g%d.fasta" % i)
        f.write_bytes(t)
        files.append(str(f))
    rng = np.random.default_rng(4)
    orderings = [list(rng.permutation(len(files))) for _ in range(5)]
    ks = [7, 11, 20, 33, 70]
    got = st.exact_prefix_cards(files, orderings, ks, True)
    assert st.stats["exact_calls"] == len(ks)
    sets = [sorted(rng.choice(len(files), 3, replace=False).tolist()) for _ in range(4)]
    uni = st.exact_union_cards(files, sets, ks, True)
    for c, k in enumerate(ks):
        for o, order in enumerate(orderings):
            assert got[o, :, c].tolist() == st.exact_prefix_counts([files[g] for g in order], k, True)
        assert uni[:, c].tolist() == [st.exact_count([files[g] for g in s], k, True) for s in sets]
