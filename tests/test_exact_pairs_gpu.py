"""K7 on the device: |A n B| for every pair of genomes at one k (dandd_b200.engine exact_pair_intersections and
its two paths), against the intersection of k-mer sets built from the oracle's symbol streams."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KS = [1, 5, 9, 12, 13, 16, 17, 21, 31, 32, 33, 47, 64, 65, 99, 256]


@pytest.fixture(scope="module")
def eng():
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    return Engine(0)


def _fasta(records):
    return b"".join(b">r%d\n%s\n" % (i, r) for i, r in enumerate(records))


def _genomes():
    """Related genomes: shared blocks, substitutions, N runs, several records, an identical pair, a genome
    without any k-mer, and runs of T long enough for the all-ones key at k = 32 and k = 64 (--no-canon)."""
    rng = np.random.default_rng(7)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    base = acgt[rng.integers(0, 4, 3000)]

    def mutate(seq, rate):
        seq = seq.copy()
        pos = rng.random(seq.size) < rate
        seq[pos] = acgt[rng.integers(0, 4, int(pos.sum()))]
        return seq

    g0 = base.copy()
    g0[700:770] = ord("T")
    g1 = mutate(base, 0.01)
    g1[1200:1230] = ord("N")
    g1[2000:2080] = ord("T")
    g2 = np.concatenate([base[:1500], acgt[rng.integers(0, 4, 1500)]])
    g3 = acgt[rng.integers(0, 4, 2500)]
    texts = [
        _fasta([g0.tobytes()]),
        _fasta([g1[:1000].tobytes(), g1[1000:].tobytes().lower()]),      # two records, soft-masked
        _fasta([g2.tobytes()]),
        _fasta([g3.tobytes(), base[100:400].tobytes()]),
        _fasta([g0.tobytes()]),                                           # identical to genome 0
        _fasta([b"ACGTN", b"NNNN"]),                                      # no k-mer for k > 4
        _fasta([mutate(g3, 0.05)[::-1].tobytes()]),
    ]
    return texts


def _kmer_set(sym, k, canon):
    from oracle import pyoracle as orc
    if k <= 32:
        return set(orc.kmers(sym, k, canon).tolist())
    out, run = set(), 0
    for i, x in enumerate(sym.tolist()):
        run = 0 if x > 3 else run + 1
        if run >= k:
            s = bytes(sym[i - k + 1:i + 1])
            if canon:
                rc = bytes(3 - c for c in reversed(s))
                s = min(s, rc)
            out.add(s)
    return out


def _want(texts, k, canon):
    from oracle import pyoracle as orc
    sets = [_kmer_set(orc.fasta_symbols(t), k, canon) for t in texts]
    n = len(sets)
    return [len(sets[a] & sets[b]) for a in range(n) for b in range(a + 1, n)], [len(s) for s in sets]


@pytest.fixture(scope="module")
def packed(eng):
    texts = _genomes()
    return texts, [eng.pack(t).check() for t in texts]


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("k", KS)
def test_pairs_equal_the_oracle_sets(eng, packed, k, canon):
    from dandd_b200._lib import DD_EXACT_BITMAP_MAXK
    texts, seqs = packed
    want, singles = _want(texts, k, canon)
    assert eng.exact_counts(seqs[:1], k, canon) == singles[:1]
    got = eng.exact_pair_intersections(seqs, k, canon, singles)
    assert got.dtype == np.uint64 and got.tolist() == want
    assert eng.exact_pairs_sparse(seqs, k, canon, singles).tolist() == want
    if k <= DD_EXACT_BITMAP_MAXK:
        assert eng.exact_pairs_dense(seqs, k, canon).tolist() == want
        assert eng.exact_pairs_dense(seqs, k, canon, block=3).tolist() == want      # genome blocks that do not all fit


def test_one_genome_has_no_pairs(eng, packed):
    _, seqs = packed
    for k in (12, 21, 99):
        assert eng.exact_pair_intersections(seqs[:1], k, True, [1]).shape == (0,)
    assert eng.exact_pair_intersections([], 21, True, []).shape == (0,)


def test_dense_and_sparse_agree_at_the_crossover(eng):
    """The rule's crossover for genomes of 5000 k-mers sits between k = 8 (4^8/32 = 2048) and k = 9 (8192):
    both paths give the same counts on both sides of it."""
    from dandd_b200 import engine as E
    rng = np.random.default_rng(3)
    base = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 5000)]
    texts = [_fasta([np.roll(base, 97 * i)[:5000 - 300 * i].tobytes()]) for i in range(5)]
    seqs = [eng.pack(t).check() for t in texts]
    for k in (8, 9):
        singles = [eng.exact_counts([s], k)[0] for s in seqs]
        assert E.dense_pairs(k, singles) == (k == 8)
        want, _ = _want(texts, k, True)
        assert eng.exact_pairs_dense(seqs, k, True).tolist() == want
        assert eng.exact_pairs_sparse(seqs, k, True, singles).tolist() == want


@pytest.mark.parametrize("k", [12, 21, 47, 99])
def test_passes_and_shards_add_up(eng, packed, k):
    _, seqs = packed
    singles = [eng.exact_counts([s], k)[0] for s in seqs]
    one = eng.exact_pairs_sparse(seqs, k, True, singles, passes=1)
    assert eng.exact_pairs_sparse(seqs, k, True, singles, passes=3).tolist() == one.tolist()
    assert eng.last_pair_plan["passes"] == 3
    world = 3
    parts = []
    for r in range(world):
        mine = [eng.exact_counts([s], k, shard=(r, world))[0] for s in seqs]
        parts.append(eng.exact_pair_intersections(seqs, k, True, mine, shard=(r, world)))
    assert np.sum(parts, axis=0).tolist() == one.tolist()
    if k <= 16:
        assert np.sum([eng.exact_pairs_dense(seqs, k, True, shard=(r, world)) for r in range(world)], axis=0).tolist() == \
            eng.exact_pairs_dense(seqs, k, True).tolist() == one.tolist()


def test_undersized_workspace_raises(eng, packed):
    from dandd_b200._lib import DandDError
    _, seqs = packed
    with pytest.raises(DandDError, match="overflow"):
        eng.exact_pairs_sparse(seqs, 21, True, [1] * len(seqs))       # table and nodes sized for one k-mer each
    lib = eng.lib
    need = lib.dd_exact_pairs_workspace_bytes(21, 1024, 4096, 2)
    assert lib.dd_exact_pairs_begin(1 << 20, need - 1, 21, 1024, 4096, 2, None) == -3    # DD_ERR_WORKSPACE, nothing launched
    assert lib.dd_exact_pairs_begin(1 << 20, need, 21, 1000, 4096, 2, None) == -1       # capacity not a power of two


@pytest.mark.parametrize("k", [13, 31, 64, 99])
def test_genome_inserted_in_two_ranges(eng, packed, k):
    """One genome's k-mers arriving in two overlapping ranges still count once for each of its pairs."""
    import torch
    from dandd_b200._lib import check
    texts, seqs = packed
    want, _ = _want(texts[:3], k, True)
    lib, st = eng.lib, eng.stream
    n, cap, nodes = 3, 1 << 16, 20000
    ws = torch.empty(lib.dd_exact_pairs_workspace_bytes(k, cap, nodes, n), dtype=torch.uint8, device=eng.device)
    out = torch.zeros(3, dtype=torch.int64, device=eng.device)
    check(lib.dd_exact_pairs_begin(ws.data_ptr(), ws.numel(), k, cap, nodes, n, st))
    for g, s in enumerate(seqs[:3]):
        ns = s.nsym
        ranges = [(0, ns // 2 + 40), (ns // 2, ns)] if g == 1 else [(0, ns)]
        for b, e in ranges:
            check(lib.dd_exact_pairs_insert_shard(s.codes.data_ptr(), s.invalid.data_ptr(), b, e, k, 1, g, ws.data_ptr(),
                                                  ws.numel(), cap, nodes, n, 0, 1, st))
    check(lib.dd_exact_pairs_accumulate(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, out.data_ptr(), st))
    assert out.cpu().tolist() == want


def test_store_pair_cards_equal_the_per_pair_path(tmp_path):
    """GpuSketchStore.exact_pair_cards (one job per k) against exact_count of every single FASTA and pair."""
    from dandd_b200 import build
    build.build()
    from dandd_b200 import store as ddstore
    st = ddstore.GpuSketchStore()
    texts = _genomes()
    files = []
    for i, t in enumerate(texts):
        f = tmp_path / ("g%d.fasta" % i)
        f.write_bytes(t)
        files.append(str(f))
    ks = [7, 11, 20, 33, 70]
    single, union = st.exact_pair_cards(files, ks, True)
    assert st.stats["exact_calls"] == len(ks)
    n = len(files)
    for c, k in enumerate(ks):
        assert single[:, c].tolist() == [st.exact_count([f], k, True) for f in files]
        assert union[:, c].tolist() == [st.exact_count([files[a], files[b]], k, True) for a in range(n) for b in range(a + 1, n)]


def test_dense_path_beyond_one_launch_of_tiles(eng):
    """2100 genomes make 263 x 263 = 69 169 tiles of 8 x 8 genomes: more than one launch holds (grid.y <= 65 535)."""
    from oracle import pyoracle as orc
    rng = np.random.default_rng(11)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    texts = [_fasta([acgt[rng.integers(0, 4, int(rng.integers(1, 7)))].tobytes()]) for _ in range(2100)]
    seqs = [eng.pack(t).check() for t in texts]
    k = 2
    held = np.zeros((len(texts), 16), dtype=np.int64)
    for g, t in enumerate(texts):
        held[g, orc.kmers(orc.fasta_symbols(t), k, True).astype(np.int64)] = 1
    inter = held @ held.T
    want = inter[np.triu_indices(len(texts), 1)]
    got = eng.exact_pairs_dense(seqs, k, True)
    assert eng.last_pair_plan["block"] == len(texts)        # one block: the tile count alone exceeds a launch
    assert got.astype(np.int64).tolist() == want.tolist()


def test_abi_rejects_stream_indices_that_do_not_fit(eng):
    lib = eng.lib
    need = lib.dd_exact_pairs_workspace_bytes(99, 1024, 4096, 70000)
    assert lib.dd_exact_pairs_begin(1 << 20, need, 99, 1024, 4096, 70000, None) == -1      # 16-bit stream index
    assert b"max_streams" in lib.dd_last_error()
