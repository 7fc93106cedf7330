"""Exact all pairs (K7) on the CPU: the store's batched exact_pair_cards on the oracle-backed engine double and
`allpairs --tool kmc` against the per-pair path of the oracle store, and the key-range pass planner of the sparse
path."""
import os
import socket

import numpy as np
import pytest

from dandd_b200 import engine as E
from dandd_b200 import store as ddstore
from dandd_b200.helpers import allpairs
from tests import allpairs_cases as cases
from tests.fake_engine import FakeEngine
from tests.oracle_store import OracleStore

CASE = {"genomes": 5, "length": 2500, "seed": 31, "sub": 0.05, "klist": [9, 13, 21, 32], "nest": 4096, "extra": ""}


def _run_allpairs(tmp, st=None, case=CASE):
    """`allpairs --tool kmc` through `st` (default: the real store on the engine double)."""
    st = st or ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    try:
        _, dataset = cases.write_dataset(str(tmp), case)
        table = allpairs.go(cases.argv_for(str(tmp), case, dataset, tool="kmc"))
    finally:
        ddstore.set_store(None)
    files = {}
    for name in sorted(os.listdir(tmp)):
        path = os.path.join(tmp, name)
        if os.path.isfile(path) and name != "dataset.json":
            files[name] = open(path, "rb").read()
    return table, st, files


def test_allpairs_kmc_files_equal_the_per_pair_path(tmp_path):
    """The batched job writes the same bytes as one exact count per pair and k (the oracle store has no batched job), in
    O(k) store calls."""
    batched, st_b, files_b = _run_allpairs(tmp_path / "batched")
    per_pair, st_p, files_p = _run_allpairs(tmp_path / "per_pair", OracleStore())
    assert files_b == files_p and len(files_b) == 2 + 2 * (1 + len(CASE["klist"]))
    assert np.array_equal(batched.single, per_pair.single) and np.array_equal(batched.pair, per_pair.pair)
    n, nk = CASE["genomes"], len(CASE["klist"])
    assert st_b.stats["exact_calls"] == nk
    assert st_b.engine.calls["exact_pair_intersections"] == nk
    assert st_p.stats["exact_calls"] == nk * (n + n * (n - 1) // 2)


def test_store_remembers_the_table(tmp_path):
    eng = FakeEngine()
    st = ddstore.GpuSketchStore(engine=eng)
    inputs = cases.make_dataset(str(tmp_path), 4, 2000, seed=5, sub=0.1)
    single, union = st.exact_pair_cards(inputs, [11, 17], True, remember=True)
    before = eng.calls["exact_counts"]
    assert st.exact_count([inputs[2], inputs[0]], 17, True) == union[1, 1]
    assert st.exact_count([inputs[3]], 11, True) == single[3, 0]
    assert eng.calls["exact_counts"] == before                                   # answered from the table
    st.exact_count([inputs[0], inputs[1]], 12, True)                             # another k: counted
    assert eng.calls["exact_counts"] == before + 1


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, tmp):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    table, st, _ = _run_allpairs(os.path.join(tmp, "r%d" % rank))
    single, union = ddstore.GpuSketchStore(engine=FakeEngine()).exact_pair_cards(
        cases.make_dataset(os.path.join(tmp, "r%d" % rank, "data"), CASE["genomes"], CASE["length"], seed=CASE["seed"],
                           sub=CASE["sub"]), CASE["klist"], True)
    assert np.array_equal(table.single, single) and np.array_equal(table.pair, union)   # the ranks' shards summed
    assert st.engine.calls["exact_pair_intersections"] == len(CASE["klist"])            # every rank ran the whole job
    dist.barrier()
    dist.destroy_process_group()
    open(os.path.join(tmp, "ok%d" % rank), "w").close()


def test_two_ranks(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")
    assert open(tmp_path / "r0" / "card.tsv", "rb").read() == \
        _run_allpairs(tmp_path / "one")[2]["card.tsv"]


@pytest.mark.parametrize("passes,world", [(1, 1), (3, 1), (1, 4), (3, 2), (5, 3)])
def test_passes_times_ranks_cover_every_key_once(passes, world):
    """Pass p of rank r keeps the keys of shard pass_shard(r, world, p, passes) -- the device's test is
    (hash >> 40) % shard_world == shard_rank: every key lands in exactly one (rank, pass)."""
    rng = np.random.default_rng(passes * 7 + world)
    hashes = rng.integers(0, 2 ** 63, 20000, dtype=np.int64).astype(np.uint64) * np.uint64(2) + np.uint64(1)
    hits = np.zeros(hashes.size, dtype=np.int64)
    for r in range(world):
        for p in range(passes):
            srank, sworld = E.pass_shard(r, world, p, passes)
            mine = (hashes >> np.uint64(40)) % np.uint64(sworld) == np.uint64(srank)
            assert np.all((hashes[mine] >> np.uint64(40)) % np.uint64(world) == np.uint64(r))   # inside the rank's range
            hits += mine
    assert np.all(hits == 1)


def test_planner_fits_the_budget():
    ws = lambda cap, nodes: 256 + 16 * cap + 8 * (cap + 1) + 8 * nodes     # the k > 32 layout
    singles = [5_000_000] * 100
    one = E.plan_pair_passes(singles, 40, ws, 1 << 40)
    assert one["passes"] == 1 and one["capacity"] >= 2 * sum(singles) and one["max_nodes"] >= sum(singles)
    small = E.plan_pair_passes(singles, 40, ws, 4 << 30)
    assert small["passes"] > 1 and small["ws_bytes"] <= 4 << 30
    assert small["capacity"] * small["passes"] >= 2 * sum(singles) and small["max_nodes"] * small["passes"] >= sum(singles)
    assert E.plan_pair_passes(singles, 40, ws, 1, passes=3)["passes"] == 3
    assert E.plan_pair_passes([100] * 4, 3, ws, 1 << 30)["capacity"] == 2048     # 4^3 keys at most, not 400
    assert E.dense_pairs(13, [5_000_000]) and not E.dense_pairs(14, [5_000_000]) and not E.dense_pairs(17, [10 ** 12])
    assert E.dense_pairs(13, [2_500_000], world=2)                                   # shard counts stand for whole genomes


def _kij_exact_run(tmp, table):
    """`tree --exact`, then `kij --jaccard --afproject` (exact mode comes with the tree) on six genomes through the real store on
    the oracle-backed engine double; returns everything the run leaves behind (paths relative) and the
    number of exact store calls `kij` made."""
    import csv
    import pickle
    from tests.host_harness import run_dandd
    from tests.util import make_dataset
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    data = make_dataset(os.path.join(tmp, "data"), 6, 4000, seed=17)
    out = os.path.join(tmp, "out")
    os.environ["DANDD_B200_PAIR_TABLE"] = "1" if table else "0"
    try:
        run_dandd(["tree", "-d", os.path.dirname(data[0]), "-s", "kx", "-k", "12", "-o", out, "--exact"])
        before = st.stats["exact_calls"]
        run_dandd(["kij", "-d", os.path.join(out, "kx_6_kmc_dtree.pickle"), "-o", out, "--mink", "9", "--maxk", "14",
                   "--jaccard", "--afproject"])
        calls = st.stats["exact_calls"] - before
    finally:
        os.environ.pop("DANDD_B200_PAIR_TABLE", None)
        ddstore.set_store(None)
    db = os.path.join(out, "sketchdb")
    rel = lambda p: os.path.relpath(p, tmp)     # noqa: E731
    res = {"files": {rel(os.path.join(d, f)): open(os.path.join(d, f), "rb").read().replace(tmp.encode(), b"<tmp>")
                     for d, _, fs in os.walk(db) for f in fs if not f.endswith((".bkp", ".pickle"))}}
    for name in ("kx_6_kmc.kij.csv", "kx_6_kmc.j.csv"):
        res[name] = [{k: (rel(v) if k in ("A", "B") else v) for k, v in r.items()} for r in csv.DictReader(open(os.path.join(out, name)))]
    for f in os.listdir(db):
        if f.endswith(".pickle"):
            with open(os.path.join(db, f), "rb") as fh:
                obj = pickle.load(fh)
            res[f] = {(rel(k) if isinstance(k, str) and os.path.isabs(k) else k): v for k, v in obj.items()}
    with open(os.path.join(out, "kx_6_kmc_AFtuples.pickle"), "rb") as fh:
        res["af"] = sorted((t[0], os.path.basename(str(t[1])), os.path.basename(str(t[2])), t[3], t[4], t[5], t[6], t[7])
                           for t in pickle.load(fh))
    return res, calls


def test_kij_exact_from_the_pair_table_equals_one_spider_per_pair(tmp_path):
    """`kij --exact` replayed on the batched exact table (K7) leaves exactly what one SubSpider per pair leaves:
    the kij and Jaccard CSVs, the cardinality / fastahex / sketchinfo pickles, the AFproject tuples and every
    file of the sketch database byte for byte -- with one exact store call per k instead of per pair and k."""
    a, calls_a = _kij_exact_run(str(tmp_path / "table"), True)
    b, calls_b = _kij_exact_run(str(tmp_path / "spiders"), False)
    assert a.keys() == b.keys()
    for key in a:
        assert a[key] == b[key], key
    assert any(f.endswith(".kmc_pre") and "/ngen2/" in f for f in a["files"])     # pair descriptors were written
    # both runs make the same leaf counts (the leaves brought to the Jaccard range); the pairs then cost one call per
    # pair and k on the per-pair path (15 pairs x the 9 k the leaves hold) and one per k with the table
    assert calls_b - calls_a == 15 * 9 - 9 and calls_a <= 9 + 6 * 9
