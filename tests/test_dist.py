"""The N>1 path on CPU: world_size 2, gloo.  Sharding is deterministic and balanced, the MAX
all-reduce / all-gather of register arrays reproduces the single-process union bit for bit, and
splitting the progressive orderings across ranks loses nothing."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dandd_b200 import dist as dd_dist


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    r, w = dd_dist.init("gloo")
    assert (r, w) == (rank, world)
    rng = np.random.default_rng(0)                     # same data on every rank; each keeps its shard
    n, nk, m = 5, 3, 1 << 10
    allregs = torch.from_numpy(rng.integers(0, 40, (n, nk, m), dtype=np.uint8))
    sizes = [50, 10, 40, 30, 20]
    owners = dd_dist.shard_by_size(sizes, world)
    assert sorted(sum(owners, [])) == list(range(n))
    local = allregs[owners[rank]].clone()
    # union over ranks == union over all genomes
    mine = local.max(dim=0).values.clone() if local.shape[0] else torch.zeros((nk, m), dtype=torch.uint8)
    full = dd_dist.union_over_ranks(mine)
    assert torch.equal(full, allregs.max(dim=0).values)
    # gather restores global genome order
    got = dd_dist.gather_registers(local, owners)
    assert torch.equal(got, allregs)
    cards = dd_dist.gather_cards(local.double().mean(dim=2), owners)
    assert torch.allclose(cards, allregs.double().mean(dim=2))
    # orderings split across ranks cover everything exactly once
    mine = list(dd_dist.split_work(7))
    bucket = [None] * world
    dist.all_gather_object(bucket, mine)
    assert sorted(sum(bucket, [])) == list(range(7))
    cnt = dd_dist.sum_counts(torch.tensor([rank + 1], dtype=torch.int64))
    assert int(cnt) == world * (world + 1) // 2
    dist.barrier()
    dist.destroy_process_group()
    open(os.path.join(tmpdir, f"ok{rank}"), "w").close()


def test_two_rank_gloo(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")


def test_shard_by_size_balance():
    sizes = [3100, 3000, 2900, 50, 40, 30, 20, 10]
    owners = dd_dist.shard_by_size(sizes, 4)
    loads = [sum(sizes[i] for i in o) for o in owners]
    assert max(loads) <= 3100 and sorted(sum(owners, [])) == list(range(8))
    assert dd_dist.shard_by_size(sizes, 4) == owners        # deterministic
    assert dd_dist.shard_by_size([5, 5, 5], 1) == [[0, 1, 2]]


def test_single_process_is_identity():
    t = torch.arange(12, dtype=torch.uint8).reshape(2, 2, 3)
    assert dd_dist.world() == (0, 1)
    assert torch.equal(dd_dist.union_over_ranks(t.clone()), t)
    assert torch.equal(dd_dist.gather_registers(t, [[0, 1]]), t)
    assert list(dd_dist.split_work(5)) == [0, 1, 2, 3, 4]


def _install_store(kind):
    """'oracle': the oracle-backed double of the whole store; 'real': the shipped GpuSketchStore on the CPU
    engine double (tests/fake_engine.py) -- its sharded and split-genome paths under gloo."""
    from dandd_b200 import store as ddstore
    if kind == "real":
        from tests.fake_engine import FakeEngine
        st = ddstore.GpuSketchStore(engine=FakeEngine())
    else:
        from tests.oracle_store import OracleStore
        st = OracleStore()
    ddstore.set_store(st)
    return st


def _tree_worker(rank, world, port, tmpdir, kind="oracle"):
    """`dandd tree` under two ranks (gloo): leaves are sketched by different ranks into the shared
    sketchdb, rank 0 builds the tree; the outputs must equal the reference golden."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from tests.host_harness import run_dandd
    st = _install_store(kind)
    data = os.path.join(tmpdir, "data5")
    run_dandd(["tree", "-d", data, "-s", "runA", "-k", "14", "-o", os.path.join(tmpdir, "outA")])
    with open(os.path.join(tmpdir, f"leafpasses{rank}"), "w") as fh:
        fh.write(str(st.stats["leaf_passes"]))


@pytest.mark.parametrize("kind", ["oracle", "real"])
def test_two_rank_tree_matches_reference(tmp_path, kind):
    from tests.host_harness import assert_tree_matches, collect_tree, gold_runs
    from tests.util import make_dataset
    make_dataset(str(tmp_path / "data5"), 5, 20000, seed=21)
    mp.spawn(_tree_worker, args=(2, _free_port(), str(tmp_path), kind), nprocs=2, join=True)
    out = str(tmp_path / "outA")
    ours = collect_tree(out, "runA_5_dashing", os.path.join(out, "sketchdb"), "dashing")
    gold = gold_runs()["A_tree_hillclimb"]
    # the ranks pre-sketch a k window around kstart, so the sketchdb may hold MORE leaf sketches than
    # the reference's hill-climb visited; everything the reference has must be there and agree
    assert set(gold["files"]) <= set(ours["files"])
    assert set(gold["cardkey"]) <= set(ours["cardkey"])
    trimmed = dict(ours, files=gold["files"], cardkey={k: ours["cardkey"][k] for k in gold["cardkey"]},
                   sketchinfo=gold["sketchinfo"])
    assert set(gold["sketchinfo"]) <= set(ours["sketchinfo"])
    assert_tree_matches(trimmed, gold)
    passes = [int(open(tmp_path / f"leafpasses{r}").read()) for r in (0, 1)]
    assert passes[0] > 0 and passes[1] > 0      # both ranks sketched leaves; k outside the pre-sketched window costs rank 0 extra passes


def _cached_rerun_worker(rank, world, port, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from dandd_b200 import store as ddstore
    from tests.oracle_store import OracleStore
    from tests.host_harness import run_dandd
    argv = ["tree", "-d", os.path.join(tmpdir, "data5"), "-s", "runC", "--ksweep", "--mink", "10", "--maxk", "14",
            "-o", os.path.join(tmpdir, "outC")]
    ddstore.set_store(OracleStore())
    run_dandd(argv)
    import torch.distributed as tdist
    assert not tdist.is_initialized()          # the command leaves no process group behind

    def trap(*a, **k):
        raise AssertionError("a fully cached re-run created the sketch store (CUDA start-up)")
    ddstore.set_store(None)
    ddstore.GpuSketchStore = trap
    run_dandd(argv)
    with open(os.path.join(tmpdir, f"cached_ok{rank}"), "w") as fh:
        fh.write("ok")


def test_cached_rerun_never_creates_the_store(tmp_path):
    """`dandd tree --ksweep` twice under two ranks: the second run finds every leaf and union sketch and
    every cardinality in the database and must not create the store on any rank (that would cost
    seconds of CUDA start-up per process for zero work; reference behaviour: SURVEY.md App. C.13)."""
    from tests.util import make_dataset
    make_dataset(str(tmp_path / "data5"), 5, 20000, seed=21)
    mp.spawn(_cached_rerun_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert all((tmp_path / f"cached_ok{r}").exists() for r in (0, 1))


# ---- one genome over several ranks -------------------------------------------------------------------
def _split_cases():
    import numpy as np
    from tests.util import adversarial_fasta, random_bases, to_fasta
    rng = np.random.default_rng(3)
    big = to_fasta([(b"chr1", random_bases(rng, 120000)), (b"chr2", random_bases(rng, 30000)),
                    (b"chr3", random_bases(rng, 5000))], width=60)
    one = to_fasta([(b"x", random_bases(rng, 90000))], width=10 ** 9)
    w1 = b">r\n" + b"\n".join(bytes([c]) for c in random_bases(rng, 3000)) + b"\n"
    return {"three_records": big, "adversarial": adversarial_fasta(rng, n=40000), "one_line": one,
            "one_line_crlf": one.replace(b"\n", b"\r\n"), "width1": w1, "header_only": b">only header", "empty": b"",
            "no_records": b"ACGT\nno records\n", "no_final_newline": b">a\nACGTACGTAC"}


@pytest.mark.parametrize("nparts", [2, 3, 8])
def test_split_fasta_parts_merge_to_the_whole(nparts):
    """dist.split_fasta: the parts' HLL registers max-merge, and their k-mer sets union, to exactly
    those of the whole file, for every k up to 64 (record cuts, overlapping cuts inside a record)."""
    import numpy as np
    from oracle import pyoracle as orc
    for name, txt in _split_cases().items():
        parts = dd_dist.split_fasta(txt, nparts)
        assert len(parts) == nparts, name
        whole = orc.fasta_symbols(txt)
        syms = [orc.fasta_symbols(t) for t in parts]
        for k in (1, 5, 21, 32):
            want = orc.hll_sketch(whole, k, 10)
            got = orc.union_max([orc.hll_sketch(s, k, 10) for s in syms])
            assert np.array_equal(want, got), (name, k)
        for k in (1, 21, 32, 64):
            assert orc.exact_count([whole], k) == orc.exact_count(syms, k), (name, k)
    sizes = [len(t) for t in dd_dist.split_fasta(_split_cases()["three_records"], nparts)]
    assert max(sizes) <= 1.35 * (sum(sizes) / nparts)      # balanced by size


def _split_tree_worker(rank, world, port, tmpdir, outname, kind="oracle"):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from tests.host_harness import run_dandd
    st = _install_store(kind)
    run_dandd(["tree", "-d", os.path.join(tmpdir, "data2"), "-s", "runS", "-k", "14", "-o", os.path.join(tmpdir, outname),
               "--ksweep", "--mink", "12", "--maxk", "16"])
    with open(os.path.join(tmpdir, f"{outname}_passes{rank}"), "w") as fh:
        fh.write(str(st.stats["leaf_passes"]))


@pytest.mark.parametrize("kind", ["oracle", "real"])
def test_fewer_genomes_than_ranks_split_each_genome(tmp_path, kind):
    """`dandd tree` on 2 genomes under 3 ranks (gloo): every rank sketches a part of each genome,
    registers are max-reduced, rank 0 builds the tree -- same outputs as one process."""
    from tests.host_harness import collect_tree
    from tests.util import make_dataset
    make_dataset(str(tmp_path / "data2"), 2, 30000, seed=5)
    _split_tree_worker(0, 1, _free_port(), str(tmp_path), "out1", kind)
    mp.spawn(_split_tree_worker, args=(3, _free_port(), str(tmp_path), "out3", kind), nprocs=3, join=True)
    one = collect_tree(str(tmp_path / "out1"), "runS_2_dashing", str(tmp_path / "out1" / "sketchdb"), "dashing")
    three = collect_tree(str(tmp_path / "out3"), "runS_2_dashing", str(tmp_path / "out3" / "sketchdb"), "dashing")
    assert one["deltas"] == three["deltas"]
    assert one["files"] == three["files"]
    assert one["cardkey"] == three["cardkey"]
    passes = [int(open(tmp_path / f"out3_passes{r}").read()) for r in range(3)]
    assert all(p >= 2 for p in passes)          # every rank took part in both genomes


def _exact_tree_worker(rank, world, port, tmpdir, kind="oracle"):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from tests.host_harness import run_dandd
    st = _install_store(kind)
    run_dandd(["tree", "-d", os.path.join(tmpdir, "data5"), "-s", "runE", "-k", "14", "-o", os.path.join(tmpdir, "outE"),
               "--exact"])
    with open(os.path.join(tmpdir, f"shardcalls{rank}"), "w") as fh:
        # real: the engine's per-union counts and the hill-climb's family jobs
        fh.write(str(st.engine.calls["exact_counts"] + st.engine.calls["exact_family_counts"] if kind == "real"
                     else st.stats.get("shard_calls", 0)))


@pytest.mark.parametrize("kind", ["oracle", "real"])
def test_two_rank_exact_tree_matches_reference(tmp_path, kind):
    """`dandd tree --exact` under two ranks: rank 0 walks the tree, rank 1 serves every exact-count
    request on its key-range shard until rank 0 says stop; outputs equal the reference golden."""
    from tests.host_harness import assert_tree_matches, collect_tree, gold_runs
    from tests.util import make_dataset
    make_dataset(str(tmp_path / "data5"), 5, 20000, seed=21)
    mp.spawn(_exact_tree_worker, args=(2, _free_port(), str(tmp_path), kind), nprocs=2, join=True)
    out = str(tmp_path / "outE")
    assert_tree_matches(collect_tree(out, "runE_5_kmc", os.path.join(out, "sketchdb"), "kmc"), gold_runs()["E_tree_exact"],
                        exact=True)
    calls = [int(open(tmp_path / f"shardcalls{r}").read()) for r in (0, 1)]
    assert calls[0] > 0 and calls[0] == calls[1]       # every request of rank 0 was served by rank 1


def test_split_fasta_fuzz():
    """Property test: for ANY FASTA-ish byte string, number of parts and overlap >= k-1, the parts'
    k-mer sets union to the whole text's (and so do HLL registers) -- including '>' inside lines,
    CR/LF mixes, empty records, text before the first record and tiny inputs."""
    from hypothesis import given, settings, strategies as st
    from oracle import pyoracle as orc
    alphabet = b">ACGTACGTNacgt\n\n\r x"

    @settings(max_examples=250, deadline=None)
    @given(st.lists(st.integers(0, len(alphabet) - 1), min_size=0, max_size=600), st.integers(1, 6), st.integers(1, 10),
           st.booleans(), st.sampled_from([8, 16, 64, 4096]))
    def run(idx, nparts, k, lead_header, min_grain):
        txt = bytes(alphabet[i] for i in idx)
        if lead_header:
            txt = b">h\n" + txt
        parts = dd_dist.split_fasta(txt, nparts, overlap_symbols=k - 1 if k > 1 else 1, min_grain=min_grain)
        assert len(parts) == nparts
        whole = orc.fasta_symbols(txt)
        syms = [orc.fasta_symbols(t) for t in parts]
        assert orc.exact_count([whole], k) == orc.exact_count(syms, k)
        want = orc.hll_sketch(whole, k, 8)
        assert np.array_equal(want, orc.union_max([orc.hll_sketch(s, k, 8) for s in syms]))

    run()


def test_split_fasta_never_starts_a_piece_on_a_midline_marker():
    """'>' inside a sequence line is junk (a break symbol), but right behind a piece's synthetic
    header it would open a header line and swallow the rest of its line; pieces therefore step back
    past it.  (Without that rule ~40 % of these cases lose k-mers.)"""
    from oracle import pyoracle as orc
    rng = np.random.default_rng(4)
    for _ in range(300):
        seq = bytearray(b"ACGT"[i] for i in rng.integers(0, 4, 300))
        for pos in rng.choice(300, 25, replace=False):
            seq[pos] = 62
        txt = b">r\n" + bytes(seq) + b"\n"
        k, n = int(rng.integers(2, 8)), int(rng.integers(2, 6))
        parts = dd_dist.split_fasta(txt, n, overlap_symbols=k - 1, min_grain=8)
        assert orc.exact_count([orc.fasta_symbols(txt)], k) == orc.exact_count([orc.fasta_symbols(t) for t in parts], k)
