"""Exact hill-climb unions from one family job per visited k, on the CPU: `tree --exact` and `progressive --exact`
without --ksweep through the real store on an oracle-backed engine double that offers Engine.exact_family_counts,
against the per-union path (DANDD_B200_EXACT_SET_BATCH=0) -- every file byte for byte, and the call accounting; the
paths that keep counting union by union; a cached re-run; two gloo ranks; the family's lifetime; the ABI entry."""
import os
import pickle
import random
import socket

import pytest

from dandd_b200 import store as ddstore
from tests.fake_engine import ListJobEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FamilyFakeEngine = ListJobEngine.only("exact_family_counts")
NoFamilyEngine = ListJobEngine.only()           # the same double without the family job


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


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for key in a:
        assert a[key] == b[key], key


def _run(tmp, argvs, batch, ngen=5, engine=FamilyFakeEngine, env=None):
    """The dandd commands on a fresh dataset through the real store on the double; returns the files left behind,
    per command (store exact calls, per-union engine counts by genome count, family-job ks), and the store."""
    from tests.host_harness import run_dandd
    from tests.util import make_dataset
    make_dataset(os.path.join(tmp, "data"), ngen, 3000, seed=23)
    st = ddstore.GpuSketchStore(engine=engine())
    ddstore.set_store(st)
    saved = {key: os.environ.get(key) for key in ["DANDD_B200_EXACT_SET_BATCH"] + list(env or {})}
    os.environ["DANDD_B200_EXACT_SET_BATCH"] = "1" if batch else "0"
    os.environ.update(env or {})
    calls = []
    try:
        for argv in argvs:
            random.seed(3)                    # the same orderings in both runs
            before = (st.stats["exact_calls"], len(st.engine.union_sizes), len(st.engine.family_ks))
            run_dandd([a.replace("<tmp>", tmp) for a in argv])
            calls.append({"exact_calls": st.stats["exact_calls"] - before[0],
                          "unions": st.engine.union_sizes[before[1]:],
                          "family_ks": st.engine.family_ks[before[2]:]})
    finally:
        for key, value in saved.items():
            if value is None:
                os.environ.pop(key, None)
            else:
                os.environ[key] = value
        ddstore.set_store(None)
    return _snapshot(tmp), calls, st


TREE = ["tree", "-d", "<tmp>/data", "-s", "ex", "-o", "<tmp>/out", "--exact"]


def _check_accounting(on, off):
    """Batched run `on` against the per-union run `off` of the same command."""
    assert on["unions"] == []                                           # no per-union count at all, singles included
    assert len(on["family_ks"]) == len(set(on["family_ks"]))            # one family job per k
    assert on["exact_calls"] == len(on["family_ks"])
    assert off["family_ks"] == [] and off["unions"]


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("kstart", ["4", "13"])
@pytest.mark.parametrize("nchildren", ["2", "3"])
@pytest.mark.parametrize("ngen", [2, 5, 7])
def test_tree_exact_hillclimb_equals_the_per_union_path(tmp_path, ngen, nchildren, kstart, canon):
    """`tree --exact -n c` hill-climb from below and from above the argmax k: every CSV, descriptor and pickle as the
    per-union path leaves it; one family job per distinct k the climb visited, no per-union count."""
    argv = TREE + ["-n", nchildren, "-k", kstart] + ([] if canon else ["--no-canon"])
    try:
        a, calls_a, _ = _run(str(tmp_path / "a"), [argv], True, ngen)
    except Exception as err:                                # a shape the reference cannot build: the same failure
        with pytest.raises(type(err)):
            _run(str(tmp_path / "b"), [argv], False, ngen)
        assert ngen == 2 and nchildren == "3"
        return
    b, calls_b, _ = _run(str(tmp_path / "b"), [argv], False, ngen)
    _assert_same(a, b)
    _check_accounting(calls_a[0], calls_b[0])
    assert {int(f.split("/k")[1].split("/")[0]) for f in a if f.endswith(".kmc_pre")} == set(calls_a[0]["family_ks"])
    assert calls_a[0]["exact_calls"] < calls_b[0]["exact_calls"]


def test_the_climb_goes_both_ways(tmp_path):
    """-k 4 climbs up to the argmax and -k 13 climbs down to it (the parametrised test above covers both)."""
    from tests.host_harness import read_csv
    for kstart in ("4", "13"):
        tmp = str(tmp_path / kstart)
        _run(tmp, [TREE + ["-n", "2", "-k", kstart]], True)
        ks = [int(r["k"]) for r in read_csv(os.path.join(tmp, "out", "ex_5_kmc_deltas.csv"))]
        assert (min(ks) > 4) if kstart == "4" else (max(ks) < 13), ks


PROG = ["progressive", "-d", "<tmp>/out/ex_5_kmc_dtree.pickle", "-o", "<tmp>/out"]


@pytest.mark.parametrize("variant", ["n3", "step2", "orderings_file", "subset"])
def test_progressive_exact_hillclimb_equals_the_per_union_path(tmp_path, variant):
    tree = TREE + ["-n", "2", "-k", "6"]

    def argvs(tmp):
        prog = PROG + {"n3": ["-n", "3"], "step2": ["-n", "3", "--step", "2"],
                       "orderings_file": ["-r", os.path.join(tmp, "orderings.pickle")],
                       "subset": ["-n", "2", "-f", os.path.join(tmp, "subset.txt")]}[variant]
        os.makedirs(tmp, exist_ok=True)
        with open(os.path.join(tmp, "orderings.pickle"), "wb") as fh:
            pickle.dump({(4, 0, 2, 1, 3), (1, 3, 0, 4, 2)}, fh)
        with open(os.path.join(tmp, "subset.txt"), "w") as fh:
            fh.write("".join(os.path.join(tmp, "data", "g%d.fasta" % g) + "\n" for g in (3, 0, 4)))
        return [tree, prog]

    ta, tb = str(tmp_path / "a"), str(tmp_path / "b")
    a, calls_a, _ = _run(ta, argvs(ta), True)
    b, calls_b, _ = _run(tb, argvs(tb), False)
    _assert_same(a, b)
    assert any("progu" in f for f in a)
    for on, off in zip(calls_a, calls_b):
        _check_accounting(on, off)


@pytest.mark.parametrize("how", ["lowmem", "switch_off", "no_method"])
def test_per_union_path_kept(tmp_path, how):
    """--lowmem, DANDD_B200_EXACT_SET_BATCH=0 and an engine without the family job count union by union, with the
    same calls as the per-union path."""
    argv = [TREE + ["-n", "2", "-k", "6"] + (["--lowmem"] if how == "lowmem" else []),
            PROG + ["-n", "2"] + (["--lowmem"] if how == "lowmem" else [])]
    engine = NoFamilyEngine if how == "no_method" else FamilyFakeEngine
    a, calls_a, _ = _run(str(tmp_path / "a"), argv, how != "switch_off", engine=engine)
    b, calls_b, _ = _run(str(tmp_path / "b"), argv, False)
    _assert_same(a, b)
    for on, off in zip(calls_a, calls_b):
        assert on["family_ks"] == [] and on == off


def test_cached_rerun_never_creates_the_store(tmp_path):
    from tests.host_harness import run_dandd
    tmp = str(tmp_path)
    argvs = [TREE + ["-n", "2", "-k", "6"], PROG + ["-n", "2"]]
    _run(tmp, argvs, True)
    before = _snapshot(tmp)

    def trap(*a, **k):
        raise AssertionError("a fully cached re-run created the sketch store")
    real = ddstore.GpuSketchStore
    ddstore.GpuSketchStore = trap
    try:
        for argv in argvs:
            random.seed(3)
            run_dandd([x.replace("<tmp>", tmp) for x in argv])
    finally:
        ddstore.GpuSketchStore = real
        ddstore.set_store(None)
    after = _snapshot(tmp)
    assert {f for f in after if "kmc_" in f} == {f for f in before if "kmc_" in f}


def test_families_end_with_their_command(tmp_path):
    """After `tree` and `progressive` no family is registered, on the host or in the store; a later count of a set
    outside any family -- find_delta_delta's subtree -- goes union by union and is right."""
    import dandd_b200
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    tmp = str(tmp_path)
    _, _, st = _run(tmp, [TREE + ["-n", "2", "-k", "6"], PROG + ["-n", "2"]], True)
    assert st.exact_family_table is None and st.stats["exact_family_jobs"] > 0
    dandd_b200.enable_compat()
    import dandd_cmd
    import sketch_classes
    assert sketch_classes._family is None
    dtree = dandd_cmd._load_tree(os.path.join(tmp, "out", "ex_5_kmc_dtree.pickle"))
    ddstore.set_store(st)
    try:
        sizes = len(st.engine.union_sizes)
        jobs = st.stats["exact_family_jobs"]
        drop = [dtree.fastas[1]]
        dtree.find_delta_delta(drop)
        rest = [f for f in dtree.fastas if f not in drop]
        assert st.stats["exact_family_jobs"] == jobs and 4 in st.engine.union_sizes[sizes:]
        k = 9
        want = orc.exact_count([orc.fasta_symbols(_read_fasta(f)) for f in rest], k, True)
        assert st.exact_count(rest, k, True) == want
    finally:
        ddstore.set_store(None)


def test_store_family_counts(tmp_path):
    """GpuSketchStore.exact_family answers singles, sets and prefixes from one job per k, leaves everything else
    (another canon, a set outside the family, k = 0 or 257) to the per-union path, and forgets the family on exit."""
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    from tests.util import make_dataset
    fastas = make_dataset(str(tmp_path / "d"), 5, 2000, seed=4)
    st = ddstore.GpuSketchStore(engine=FamilyFakeEngine())
    sets, orderings = [[0, 2], [1, 3, 4]], [[4, 1, 0, 3, 2], [2, 2, 0]]
    syms = [orc.fasta_symbols(_read_fasta(f)) for f in fastas]
    with st.exact_family(fastas, True, sets=sets, orderings=orderings):
        for k in (5, 11):
            for members in [[g] for g in range(5)] + sets + [o[:i] for o in orderings for i in range(1, len(o) + 1)]:
                got = st.exact_count([fastas[g] for g in members], k, True)
                assert got == orc.exact_count([syms[g] for g in members], k, True), (members, k)
        assert st.engine.family_ks == [5, 11] and st.engine.union_sizes == []
        assert st.exact_count([fastas[0], fastas[1]], 5, True) == orc.exact_count(syms[:2], 5, True)   # not a family set
        assert st.exact_count([fastas[0]], 5, False) == orc.exact_count(syms[:1], 5, False)            # another canon
        assert st.engine.union_sizes == [2, 1] and st.stats["exact_calls"] == 4
    assert st.exact_family_table is None
    st.exact_count([fastas[0]], 7, True)
    assert st.engine.family_ks == [5, 11]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _tree_worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from tests.host_harness import run_dandd
    st = ddstore.GpuSketchStore(engine=FamilyFakeEngine())
    ddstore.set_store(st)
    run_dandd([a.replace("<tmp>", tmp) for a in TREE + ["-n", "2", "-k", "6"]])
    with open(os.path.join(tmp, "family%d" % rank), "w") as fh:
        fh.write(repr((st.engine.family_ks, st.engine.union_sizes)))


def test_two_ranks(tmp_path):
    """`tree --exact` hill-climb under two gloo ranks: every rank runs its key range of each family job, the counts are
    summed, and rank 0 leaves what one process leaves."""
    import ast
    import torch.multiprocessing as mp
    from tests.util import make_dataset
    two = str(tmp_path / "a")
    make_dataset(os.path.join(two, "data"), 5, 3000, seed=23)
    mp.spawn(_tree_worker, args=(2, _free_port(), two), nprocs=2, join=True)
    (ks0, unions0), (ks1, unions1) = [ast.literal_eval(open(os.path.join(two, "family%d" % r)).read()) for r in (0, 1)]
    one, calls, _ = _run(str(tmp_path / "b"), [TREE + ["-n", "2", "-k", "6"]], True)
    assert ks0 == ks1 == calls[0]["family_ks"] and unions0 == unions1 == []
    got = {f: v for f, v in _snapshot(two).items() if not f.startswith("family")}
    for snap in (got, one):       # rows of a set, in the order of the process's string hashes
        snap["out/ex_5_kmc_sketchdb.txt"] = sorted(snap["out/ex_5_kmc_sketchdb.txt"].split(b"\r\n"))
    _assert_same(got, one)


def test_node_count_entry_is_declared():
    """dd_exact_pairs_node_count: in the header, the ctypes signatures and INTEGRATION.md."""
    import re
    from dandd_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    assert re.search(r"DD_API\s+int\s+dd_exact_pairs_node_count\s*\(", header)
    assert "dd_exact_pairs_node_count" in _lib.SIGNATURES and len(_lib.SIGNATURES["dd_exact_pairs_node_count"][1]) == 4
    assert "`dd_exact_pairs_node_count`" in open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert _lib.ABI_VERSION == 2


def test_node_count_entry_is_exported_and_checks_arguments():
    import subprocess
    from dandd_b200 import build, _lib
    build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "dandd_b200", "libdandd_b200.so")], text=True)
    assert "dd_exact_pairs_node_count" in {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    lib = _lib.load()
    assert lib.dd_exact_pairs_node_count(None, 4096, 1 << 20, None) == -1
    assert lib.dd_exact_pairs_node_count(1 << 20, 4096, None, None) == -1
    assert lib.dd_exact_pairs_node_count(1 << 20, 8, 1 << 20, None) == -3


def test_length_bounds_never_understate():
    from dandd_b200.engine import length_bounds, plan_pair_passes
    assert length_bounds([100, 5, 0], 2) == [16, 5, 0]
    assert length_bounds([101, 7], 40, world=2) == [51, 4]
    ws = lambda c, m: c * 16 + m * 8    # noqa: E731
    for k in (3, 12, 31, 40):
        small = plan_pair_passes([40, 7], k, ws, 1 << 40)
        big = plan_pair_passes(length_bounds([4000, 700], k), k, ws, 1 << 40)
        assert big["capacity"] >= small["capacity"] and big["max_nodes"] >= small["max_nodes"]
