"""Exact unions of many genome sets (K8) on the CPU: `progressive --exact` and `tree --exact --ksweep` through the
real store on an oracle-backed engine double that offers the first-rank histogram job, against the per-union
path (DANDD_B200_EXACT_SET_BATCH=0); the histogram -> prefix / set count arithmetic of the store; a cached re-run;
two gloo ranks."""
import os
import random
import socket

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from tests.fake_engine import FakeEngine, ListJobEngine

# the first-rank job alone: without the family job, a hill-climb's cells stay per union
SetFakeEngine = ListJobEngine.only("exact_first_rank_hist")


def _symbols_sets(fastas, k):
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    return [set(orc.kmers(orc.fasta_symbols(_read_fasta(f)), k, True).tolist()) for f in fastas]


def _dataset(tmp, n=6, length=3000, seed=5):
    from tests.util import make_dataset
    paths = make_dataset(os.path.join(tmp, "data"), n, length, seed=seed)
    empty = os.path.join(tmp, "data", "zz_empty.fasta")
    with open(empty, "wb") as fh:
        fh.write(b">nothing\nNNNN\n")
    return paths + [empty]


def test_histograms_give_prefix_and_set_counts(tmp_path):
    """Random memberships: partial orderings (absent genomes), a genome listed twice, sets with ties, a genome
    without k-mers; every count equals the union of the oracle k-mer sets, with one engine job per k."""
    fastas = _dataset(str(tmp_path))
    n = len(fastas)
    rng = np.random.default_rng(1)
    orderings = [list(rng.permutation(n)) for _ in range(4)] + [[3, 1], [n - 1, 0, 2], [2, 2, 4], []]
    sets = [sorted(rng.choice(n, int(rng.integers(1, n + 1)), replace=False).tolist()) for _ in range(6)] + [[n - 1], [0], []]
    ks = [5, 11, 21]
    st = ddstore.GpuSketchStore(engine=SetFakeEngine())
    pre = st.exact_prefix_cards(fastas, orderings, ks, True)
    uni = st.exact_union_cards(fastas, sets, ks, True)
    assert pre.shape == (len(orderings), n, len(ks)) and uni.shape == (len(sets), len(ks))
    assert st.stats["exact_calls"] == 2 * len(ks) and st.engine.calls["exact_first_rank_hist"] == 2 * len(ks)
    for c, k in enumerate(ks):
        kset = _symbols_sets(fastas, k)
        for o, order in enumerate(orderings):
            for i in range(n):
                want = len(set().union(*[kset[g] for g in order[:i + 1]])) if order else 0
                assert pre[o, i, c] == want, (o, i, k)
        for s, members in enumerate(sets):
            assert uni[s, c] == len(set().union(*[kset[g] for g in members])), (s, k)
    # an engine without the batched job: the same numbers, counted union by union
    plain = ddstore.GpuSketchStore(engine=FakeEngine())
    assert np.array_equal(plain.exact_prefix_cards(fastas, orderings, ks, True), pre)
    assert np.array_equal(plain.exact_union_cards(fastas, sets, ks, True), uni)
    # singles on record size the job (the double checks they are the exact leaf counts)
    singles = np.array([[len(s) for s in _symbols_sets(fastas, k)] for k in ks]).T
    assert np.array_equal(st.exact_union_cards(fastas, sets, ks, True, singles=singles), uni)


def _content(obj, path=()):
    """A tree object's content as plain data: which objects share identity (what pickle's memo records) is
    not part of it."""
    if isinstance(obj, dict):
        return {k: _content(v, path) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return [_content(v, path) for v in obj]
    if isinstance(obj, set):
        return sorted(_content(v, path) for v in obj)
    if hasattr(obj, "__dict__"):
        if id(obj) in path:
            return "<cycle>"
        return (type(obj).__name__, _content(vars(obj), path + (id(obj),)))
    return obj


def _snapshot(root):
    """Every file under root byte for byte, the root's own path replaced; a tree pickle by its content."""
    import pickle
    out = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            if "/data" in d or f.endswith(".bkp"):
                continue
            p = os.path.join(d, f)
            raw = open(p, "rb").read()
            if f.endswith("_dtree.pickle"):
                raw = repr(_content(pickle.loads(raw))).encode()
            out[os.path.relpath(p, root)] = raw.replace(root.encode(), b"<tmp>")
    return out


def _run(tmp, argvs, batch):
    """The dandd commands on a fresh dataset through the real store on SetFakeEngine; returns the files left behind
    and the exact store calls of each command."""
    from tests.host_harness import run_dandd
    from tests.util import make_dataset
    make_dataset(os.path.join(tmp, "data"), 5, 4000, seed=17)
    st = ddstore.GpuSketchStore(engine=SetFakeEngine())
    ddstore.set_store(st)
    os.environ["DANDD_B200_EXACT_SET_BATCH"] = "1" if batch else "0"
    calls = []
    try:
        for argv in argvs:
            random.seed(3)                    # the same orderings in both runs
            before = st.stats["exact_calls"]
            run_dandd([a.replace("<tmp>", tmp) for a in argv])
            calls.append(st.stats["exact_calls"] - before)
    finally:
        os.environ.pop("DANDD_B200_EXACT_SET_BATCH", None)
        ddstore.set_store(None)
    return _snapshot(tmp), calls, st


SWEEP = ["--ksweep", "--mink", "9", "--maxk", "12"]
TREE = ["tree", "-d", "<tmp>/data", "-s", "ex", "-k", "10", "-o", "<tmp>/out", "--exact"]
PROG = ["progressive", "-d", "<tmp>/out/ex_5_kmc_dtree.pickle", "-n", "3", "-o", "<tmp>/out", "--step", "2"]


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for key in a:
        assert a[key] == b[key], key


@pytest.mark.parametrize("mode", ["ksweep", "hillclimb"])
def test_progressive_exact_equals_the_per_union_path(tmp_path, mode):
    """`progressive --exact` (several orderings, --step 2) leaves every CSV, descriptor and pickle byte for byte as
    the per-union path does; with a sweep the prefix unions cost one store call per k."""
    tree = TREE + SWEEP
    prog = PROG + (SWEEP if mode == "ksweep" else ["-s", "hc"])
    a, calls_a, st = _run(str(tmp_path / "a"), [tree, prog], True)
    b, calls_b, _ = _run(str(tmp_path / "b"), [tree, prog], False)
    _assert_same(a, b)
    assert any("/ngen4/" in f and f.endswith(".kmc_pre") for f in a)            # prefix descriptors were written
    if mode == "ksweep":
        # 3 orderings x prefixes {2, 4} of 5 genomes x 4 k on the per-union path, 4 with one job per k
        assert calls_a[1] == 4 and calls_b[1] > 4 and st.engine.calls["exact_first_rank_hist"] == 4
    else:
        assert calls_a == calls_b                                                  # cells found by the hill-climb stay per union


@pytest.mark.parametrize("nchildren", ["2", "3"])
def test_tree_exact_ksweep_equals_the_per_union_path(tmp_path, nchildren):
    argv = TREE + SWEEP + ["-n", nchildren]
    a, calls_a, st = _run(str(tmp_path / "a"), [argv], True)
    b, calls_b, _ = _run(str(tmp_path / "b"), [argv], False)
    _assert_same(a, b)
    assert st.engine.calls["exact_first_rank_hist"] == 4
    assert calls_a[0] == 5 * 4 + 4 < calls_b[0]                               # leaves one by one, inner nodes one job per k


def test_cached_rerun_never_creates_the_store(tmp_path):
    from tests.host_harness import run_dandd
    tmp = str(tmp_path)
    _run(tmp, [TREE + SWEEP + ["-n", "2"], PROG + SWEEP], True)
    before = _snapshot(tmp)

    def trap(*a, **k):
        raise AssertionError("a fully cached re-run created the sketch store")
    real = ddstore.GpuSketchStore
    ddstore.GpuSketchStore = trap
    try:
        for argv in (TREE + SWEEP + ["-n", "2"], PROG + SWEEP):
            random.seed(3)
            run_dandd([x.replace("<tmp>", tmp) for x in argv])
    finally:
        ddstore.GpuSketchStore = real
        ddstore.set_store(None)
    after = _snapshot(tmp)
    assert {f for f in after if "kmc_" in f} == {f for f in before if "kmc_" in f}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _tree_worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from tests.host_harness import run_dandd
    st = ddstore.GpuSketchStore(engine=SetFakeEngine())
    ddstore.set_store(st)
    run_dandd([a.replace("<tmp>", tmp) for a in TREE + SWEEP + ["-n", "2"]])
    with open(os.path.join(tmp, "hist%d" % rank), "w") as fh:
        fh.write(str(st.engine.calls.get("exact_first_rank_hist", 0)))


def test_two_ranks(tmp_path):
    """`tree --exact --ksweep` under two gloo ranks: every rank runs its key range of each per-k job, the
    histograms are summed, and rank 0 leaves what one process leaves."""
    import torch.multiprocessing as mp
    from tests.util import make_dataset
    two = str(tmp_path / "a")
    make_dataset(os.path.join(two, "data"), 5, 4000, seed=17)
    mp.spawn(_tree_worker, args=(2, _free_port(), two), nprocs=2, join=True)
    assert [int(open(os.path.join(two, "hist%d" % r)).read()) for r in (0, 1)] == [4, 4]
    one, _, _ = _run(str(tmp_path / "b"), [TREE + SWEEP + ["-n", "2"]], True)
    got = {f: v for f, v in _snapshot(two).items() if not f.startswith("hist")}
    for snap in (got, one):       # rows of a set, in the order of the process's string hashes
        snap["out/ex_5_kmc_sketchdb.txt"] = sorted(snap["out/ex_5_kmc_sketchdb.txt"].split(b"\r\n"))
    _assert_same(got, one)
