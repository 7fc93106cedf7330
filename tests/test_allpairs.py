"""dandd_b200/helpers/allpairs.py on the CPU (oracle-backed store double): the same tables as the
reference's helpers/allpairs.py functions (committed golden + a live comparison where DANDD_REFERENCE
names a checkout of the reference), the sharded path under two gloo ranks, and the error behaviour."""
import importlib.util
import json
import os
import socket

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from dandd_b200.helpers import allpairs
from tests import allpairs_cases as cases
from tests.oracle_store import OracleStore
from tests.util import reference_path

REF = reference_path("helpers", "allpairs.py")


@pytest.fixture()
def oracle_store():
    st = OracleStore()
    ddstore.set_store(st)
    yield st
    ddstore.set_store(None)


def _oracle_counts(fastas, k):
    from oracle import pyoracle as orc
    return orc.exact_count([orc.fasta_symbols(open(f, "rb").read()) for f in fastas], k, True)


@pytest.mark.parametrize("name", sorted(cases.gold_cases()))
def test_tables_match_the_reference_functions(tmp_path, oracle_store, name):
    table = cases.scenario_gold(str(tmp_path), name)
    n = len(table.names)
    assert oracle_store.stats["leaf_passes"] == n            # every FASTA sketched once, whatever the k list
    assert oracle_store.stats["union_launches"] == 1         # one pair job


def test_exact_tool(tmp_path, oracle_store):
    cases.scenario_exact(str(tmp_path), _oracle_counts)


def test_errors(tmp_path, oracle_store):
    case = dict(cases.gold_cases()["six_p12"], genomes=3, length=2000)
    inputs, dataset = cases.write_dataset(str(tmp_path), case)
    names = ["a", "b", "c"]
    with pytest.raises(RuntimeError, match="cannot count k-mers of length"):
        allpairs.card_table("dashing", inputs, names, [31, 33], nest=1024)
    with pytest.raises(RuntimeError, match="power of 2"):
        allpairs.card_table("dashing", inputs, names, [12], nest=1000)
    with pytest.raises(RuntimeError, match="No card function"):
        allpairs.card_table("dashing2", inputs, names, [12])
    with pytest.raises(RuntimeError, match="Unsupported --extra"):
        allpairs.card_table("dashing", inputs, names, [12], nest=1024, extra="--min-count 2")
    with pytest.raises(RuntimeError, match="distinct"):
        allpairs.card_table("dashing", inputs, ["a", "a", "c"], [12], nest=1024)
    with pytest.raises(RuntimeError, match="No dataset file"):
        allpairs.load_dataset(str(tmp_path / "missing.json"))
    with open(tmp_path / "bad.json", "w") as fh:
        json.dump({"seqids": [str(tmp_path / "nowhere")], "treids": []}, fh)
    with pytest.raises(RuntimeError, match="Input path does not exist"):
        allpairs.load_dataset(str(tmp_path / "bad.json"))


def test_single_input_and_commands_file(tmp_path, oracle_store):
    """One FASTA: marginals only, no matrices; --write-commands lists the reference's command lines."""
    case = dict(cases.gold_cases()["six_p12"], genomes=1, length=3000, klist=[9, 10])
    inputs, dataset = cases.write_dataset(str(tmp_path), case)
    table = allpairs.go(cases.argv_for(str(tmp_path), case, dataset, write_commands="commands.txt"))
    assert table.pair.shape == (0, 2)
    with open(tmp_path / "run" / "commands.txt") as fh:
        lines = fh.read().splitlines()
    assert lines == [str(("dashing", "g0", "g0", k, "dashing hll -k %d -S 12   %s" % (k, inputs[0]))) for k in (9, 10)]
    assert not os.path.exists(tmp_path / "sim.kij.phylip")


def test_worker_processes_write_the_same_files(tmp_path, monkeypatch):
    """Large tables are written by spawned worker processes (one piece per k-block of card.tsv and per
    PHYLIP matrix): the files must equal the single-process ones byte for byte."""
    rng = np.random.default_rng(5)
    n, klist = 9, [12, 7, 31, 19]
    names = ["n%d" % i for i in rng.permutation(n)]
    table = allpairs.CardTable("dashing", names, klist, rng.uniform(1e4, 2e4, (n, 4)), rng.uniform(2e4, 3e4, (n * (n - 1) // 2, 4)))
    texts = {}
    for mode, cpu in (("serial", 1), ("workers", 3)):
        out = tmp_path / mode
        os.makedirs(out / "run")
        args = allpairs.parse_arguments(["--name", str(out / "run"), "--card-results", str(out / "card.tsv"),
                                         "--delta-results", str(out / "delta.tsv"), "--j-results-phylip", str(out / "sim.phylip"),
                                         "--ani-results-phylip", str(out / "ani.phylip"), "--cpu", str(cpu)])
        monkeypatch.setattr(allpairs, "PARALLEL_MIN_CELLS", 0)
        written = allpairs.write_outputs(table, args, {x: x for x in names})
        assert len(written) == 2 + 2 * 5 and sorted(os.listdir(out / "run")) == []       # the shared table is removed
        texts[mode] = {os.path.basename(f): open(f).read() for f in written}
        assert sorted(os.listdir(out)) == sorted(list(texts[mode]) + ["run"])            # no part files left behind
    assert texts["serial"] == texts["workers"]
    cases.assert_files_equal_tuple_path(str(tmp_path / "workers"), table)


def test_mash_distance_and_rename():
    assert allpairs.mash_distance(1.0, 21) == 0.0
    assert allpairs.mash_distance(0.0, 10) == allpairs.mash_distance(-1.0, 10) > 3.0      # clamped, not an error
    assert allpairs.rename_seqids_in_tree("(ab:1,(a:2,abc:3));", {"a": "X", "ab": "Y", "abc": "Z"}) == "(Xb:1,(X:2,Xbc:3));"


@pytest.mark.skipif(not (REF and os.path.exists(REF)),
                    reason="opt-in: runs the original DandD project, which is not part of this repository (set DANDD_REFERENCE)")
@pytest.mark.parametrize("seed", range(8))
def test_live_against_the_reference_functions(tmp_path, oracle_store, seed):
    """Random table shapes through both implementations of the summaries: identical tuples and files
    (same floats in, so exact equality)."""
    spec = importlib.util.spec_from_file_location("reference_allpairs", REF)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    rng = np.random.default_rng(seed)
    n = int(rng.integers(2, 7))
    klist = [int(k) for k in rng.permutation(np.arange(5, 30))[:int(rng.integers(1, 8))]]
    names = ["s%d" % i for i in rng.permutation(20)[:n]]
    table = allpairs.CardTable("dashing", names, klist, rng.integers(1, 9, (n, len(klist))) * 1000.0,   # ties on purpose
                               rng.integers(5, 20, (n * (n - 1) // 2, len(klist))) * 1000.0)
    results = table.results()
    assert allpairs.delta_summarize(results) == ref.delta_summarize(results) == table.delta_summary()
    dsumm = ref.delta_summarize(results)
    assert allpairs.kij_summarize(dsumm) == ref.kij_summarize(dsumm)
    ids = {name: name for name in names}
    for k in klist:
        want = ref.j_summarize(results, k)
        assert allpairs.j_summarize(results, k) == want == table.j_summary(k)
        for ani in (False, True):
            ref.summ_to_phylip(want, ids, str(tmp_path / "ref.phylip"), convert_to_ani=ani)
            allpairs.summ_to_phylip(want, ids, str(tmp_path / "ours.phylip"), convert_to_ani=ani)
            assert (tmp_path / "ours.phylip").read_text() == (tmp_path / "ref.phylip").read_text()
    for ani in (False, True):
        ref.summ_to_phylip(ref.kij_summarize(dsumm), ids, str(tmp_path / "ref.phylip"), convert_to_ani=ani)
        allpairs.summ_to_phylip(allpairs.kij_summarize(dsumm), ids, str(tmp_path / "ours.phylip"), convert_to_ani=ani)
        assert (tmp_path / "ours.phylip").read_text() == (tmp_path / "ref.phylip").read_text()
    args = allpairs.parse_arguments(["--card-results", str(tmp_path / "card.tsv"), "--delta-results", str(tmp_path / "delta.tsv"),
                                     "--j-results-phylip", str(tmp_path / "sim.phylip"),
                                     "--ani-results-phylip", str(tmp_path / "ani.phylip")])
    allpairs.write_outputs(table, args, ids)
    cases.assert_files_equal_tuple_path(str(tmp_path), table, summaries=ref)      # the files, against the reference's functions
    tree = "(s1:0.1,(s10:0.2,s2:0.3));"
    assert allpairs.rename_seqids_in_tree(tree, {"s1": "one", "s10": "ten", "s2": "two"}) == \
        ref.rename_seqids_in_tree(tree, {"s1": "one", "s10": "ten", "s2": "two"})
    for k in (1, 13, 31):
        assert ref.card_cmd("dashing", k, 4096, 8, "--no-canon", "", "a.fasta b.fasta") == \
            allpairs.reference_command("dashing", k, 4096, "--no-canon", "a.fasta b.fasta")
        assert ref.card_cmd("kmc", k, 4096, 8, "", "", "a.fasta") == allpairs.reference_command("kmc", k, 4096, "", "a.fasta")


# ---- two ranks (gloo): FASTAs sharded for sketching, registers gathered, pair list split ------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, tmp, tool):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    st = OracleStore()
    ddstore.set_store(st)
    case = dict(cases.gold_cases()["six_p12"])
    if tool == "kmc":
        case.update(genomes=3, length=2500, klist=[9, 40])
    _, dataset = cases.write_dataset(os.path.join(tmp, "in%d" % rank), case)     # same deterministic inputs on both ranks
    table = allpairs.go(cases.argv_for(tmp, case, dataset, tool=tool))
    if tool == "dashing":
        assert st.stats["leaf_passes"] == 3                    # each rank sketched only its own three FASTAs
        if rank == 0:
            cases.check_against_gold(tmp, case, table)
        with pytest.raises(RuntimeError, match="already exists"):      # rank 0 sees the directory; every rank leaves
            allpairs.go(cases.argv_for(tmp, case, dataset, tool=tool))
    else:
        inputs = [os.path.join(tmp, "in%d" % rank, "data", "g%d.fasta" % g) for g in range(3)]
        for c, k in enumerate(case["klist"]):
            assert [table.single[i, c] for i in range(3)] == [_oracle_counts([f], k) for f in inputs]
            assert [table.pair[r, c] for r in range(3)] == [_oracle_counts([inputs[a], inputs[b]], k) for a, b in table.pairs]
    dist.barrier()
    dist.destroy_process_group()
    open(os.path.join(tmp, f"ok{rank}"), "w").close()


@pytest.mark.parametrize("tool", ["dashing", "kmc"])
def test_two_ranks(tmp_path, tool):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), tool), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")


def test_config5_cli_tool_smoke(tmp_path):
    """tools/config5_cli.py (config 5 from FASTA files through the driver) on the oracle-backed store."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "rep.json"
    subprocess.run([sys.executable, os.path.join(root, "tools", "config5_cli.py"), "--genomes", "12", "--bases", "8000", "--p", "10",
                    "--kmin", "9", "--kmax", "12", "--oracle-store", "--workdir", str(tmp_path / "w"), "--out", str(out)],
                   check=True, stdout=subprocess.DEVNULL, timeout=300)
    rep = json.loads(out.read_text())
    assert rep["pairs"] == 66 and rep["oracle_max_rel_err"] == 0.0 and rep["output_files"] == 2 + 2 * 5
    assert rep["kij_within_clusters"] > 3 * rep["kij_between_clusters"]
    assert {"allpairs_sketch", "allpairs_pairs", "allpairs_outputs"} <= set(rep["stages_rank0"])
