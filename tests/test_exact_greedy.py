"""Exact greedy ordering (`helpers/greedy.py --tool kmc`, K12) on the CPU: the numpy restatement of the cover index's
emit and step (tests/fake_engine.py), checked after every step of random orders against |A_h n U|; the store's loop on the
engine double against a brute-force greedy over oracle k-mer sets; the command line end to end with the `dandd tree
--exact` + `progressive --ksweep -r ordering.pickle` replay on the oracle store; refusals, two gloo ranks and the ABI
entries."""
import os
import pickle
import re
import socket

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from dandd_b200.helpers import greedy
from tests.fake_engine import FakeEngine, emit_rule, kmer_keys, step_rule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------- the numpy restatement of K12
def _held_cases():
    rng = np.random.default_rng(5)
    out = []
    for n in (2, 3, 40):
        held = rng.random((300, n)) < 0.3
        held[7] = True                                       # a key every genome holds
        held[:, n - 1] = held[:, 0]                          # a duplicate genome
        if n > 2:
            held[:, 1] = False
            held = np.concatenate([held, np.eye(1, n, 1, dtype=bool).repeat(20, axis=0)])   # genome 1 shares nothing
        held = held[held.any(axis=1)]                        # every key of the lists has a holder
        out.append(held)
    return out


@pytest.mark.parametrize("held", _held_cases(), ids=["n2", "n3", "n40"])
def test_lost_is_the_overlap_with_the_union(held):
    rng = np.random.default_rng(held.shape[1])
    n = held.shape[1]
    part = emit_rule(held, rng)
    assert part["offsets"][-1] == part["n_nodes"] == held.sum()
    for key in range(part["n_keys"]):                        # holders of key id i are the genomes of its nodes
        nodes = np.flatnonzero(part["key_of_node"] == key)
        got = sorted(part["holders"][part["offsets"][key]:part["offsets"][key + 1]].tolist())
        assert got == sorted(np.searchsorted(part["node_start"], nodes, side="right") - 1)
    for trial in range(3):
        part["covered"][:] = False
        lost = np.zeros(n, dtype=np.int64)
        union = np.zeros(held.shape[0], dtype=bool)
        for g in rng.permutation(n):
            step_rule(part, g, lost)
            union |= held[:, g]
            assert lost.tolist() == (held & union[:, None]).sum(axis=0).tolist()


# ---------------------------------------------------------------- the store's loop on the engine double
def _syms(fastas):
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    return [orc.fasta_symbols(_read_fasta(f)) for f in fastas]


def brute_exact_greedy(fastas, ks, steps, order="max", first=(), canon=True):
    """(order, cards [steps, nk]) from explicit k-mer sets: the lowest index wins a tie."""
    sets = [[set(kmer_keys(s, k, canon).tolist()) for k in ks] for s in _syms(fastas)]
    union = [set() for _ in ks]
    picks, cards = [], []
    for t in range(steps):
        if t < len(first):
            best = first[t]
        else:
            best, best_d = None, None
            for g in range(len(fastas)):
                if g in picks:
                    continue
                d = max(len(union[c] | sets[g][c]) / k for c, k in enumerate(ks))
                if best is None or (d > best_d if order == "max" else d < best_d):
                    best, best_d = g, d
        picks.append(best)
        union = [u | sets[best][c] for c, u in enumerate(union)]
        cards.append([len(u) for u in union])
    return picks, np.asarray(cards, dtype=np.int64)


@pytest.fixture(scope="module")
def clustered(tmp_path_factory):
    """Two clusters of near-copies plus an exact copy of genome 1 (genome 6): the lower index must win the tie."""
    import shutil
    from tests.util import make_dataset
    d = tmp_path_factory.mktemp("exact_greedy")
    a = make_dataset(str(d / "a"), 4, 2500, seed=41, prefix="a")
    b = make_dataset(str(d / "b"), 2, 2500, seed=42, prefix="b")
    dup = str(d / "dup.fasta")
    shutil.copy(a[1], dup)
    return a + b + [dup]


@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("order,first,steps", [("max", (), 7), ("min", (), 7), ("max", (3, 6), 7), ("min", (5,), 4),
                                               ("max", (), 3)])
def test_store_loop_equals_brute_force(clustered, order, first, steps, passes):
    ks = [3, 5, 8, 11]
    eng = FakeEngine()
    eng.passes = passes
    st = ddstore.GpuSketchStore(engine=eng)
    got, cards, stats = st.exact_greedy_order(clustered, ks, True, steps, order=order, first=first)
    want, want_cards = brute_exact_greedy(clustered, ks, steps, order, first)
    assert got.tolist() == want and cards.dtype == np.int64 and np.array_equal(cards, want_cards)
    assert eng.calls["exact_cover_index"] == len(ks) and eng.calls["exact_cover_step"] == steps - 1
    from oracle import pyoracle as orc
    assert stats["distinct_keys"] == [orc.exact_count(_syms(clustered), k, True) for k in ks]
    if order == "max" and not first and steps == 7:
        assert got.tolist().index(1) < got.tolist().index(6)     # the duplicate: the lower index first


def test_out_of_memory_names_the_k_and_the_bytes_held(clustered):
    import torch

    class Full(FakeEngine):
        def exact_cover_index(self, seqs, k, canon, shard=None, passes=None):
            if k == 8:
                raise torch.OutOfMemoryError("CUDA out of memory")
            return super().exact_cover_index(seqs, k, canon, shard, passes)

    st = ddstore.GpuSketchStore(engine=Full())
    held = sum(FakeEngine().exact_cover_index([st.packed(f) for f in clustered], k, True)["bytes"] for k in (3, 5))
    with pytest.raises(RuntimeError, match=r"k=8 with %d bytes.*fewer k or more ranks" % held):
        st.exact_greedy_order(clustered, [3, 5, 8], True, 3)


# ---------------------------------------------------------------- the command line
def _run(argv):
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    try:
        return greedy.go(argv), st
    finally:
        ddstore.set_store(None)


def _read_tsv(path):
    import csv
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


@pytest.mark.parametrize("order", ["max", "min"])
def test_outputs_and_exact_replay(tmp_path, order):
    """order.tsv / growth.tsv / collection.tsv against brute force over oracle k-mer sets; then `dandd tree --exact`
    and `progressive --ksweep -r ordering.pickle` on the oracle store: every summary card is growth.tsv's card."""
    from oracle import pyoracle as orc
    from tests.host_harness import read_csv, run_dandd
    from tests.oracle_store import OracleStore
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    fastas = make_dataset(data, 5, 2000, seed=19)
    names = [os.path.basename(f) for f in fastas]
    (tmp_path / "first.txt").write_text("%s\n" % names[2])
    name = str(tmp_path / "run")
    lo, hi = 3, 9
    (got, cards, _), _ = _run(["-d", data, "--tool", "kmc", "--mink", str(lo), "--maxk", str(hi), "--order", order,
                               "--first", str(tmp_path / "first.txt"), "--name", name])
    ks = list(range(lo, hi + 1))
    want, want_cards = brute_exact_greedy(fastas, ks, 5, order, (2,))
    assert got.tolist() == want and np.array_equal(cards, want_cards)
    all_cards = [orc.exact_count(_syms(fastas), k, True) for k in ks]
    all_d = max(c / k for c, k in zip(all_cards, ks))
    assert _read_tsv(os.path.join(name, "collection.tsv")) == [
        {"ngen": "5", "delta": repr(all_d), "k": str(ks[[c / k for c, k in zip(all_cards, ks)].index(all_d)])}]
    before = 0.0
    for t, r in enumerate(_read_tsv(os.path.join(name, "order.tsv"))):
        dk = [int(want_cards[t, c]) / k for c, k in enumerate(ks)]
        assert (int(r["step"]), r["genome"], int(r["forced"])) == (t + 1, names[want[t]], int(t == 0))
        assert float(r["delta"]) == max(dk) and float(r["gain"]) == max(dk) - before and float(r["fraction"]) == max(dk) / all_d
        before = max(dk)
    growth = _read_tsv(os.path.join(name, "growth.tsv"))
    assert [(int(r["ngen"]), int(r["k"]), r["card"]) for r in growth] == \
        [(t + 1, k, str(int(want_cards[t, c]))) for t in range(5) for c, k in enumerate(ks)]       # integers
    assert all(float(r["delta_pos"]) == int(r["card"]) / int(r["k"]) for r in growth)
    with open(os.path.join(name, "ordering.pickle"), "rb") as fh:
        assert pickle.load(fh) == {tuple(want)}

    out = str(tmp_path / "out")
    ddstore.set_store(OracleStore())
    try:
        run_dandd(["tree", "-d", data, "-s", "ex", "-o", out, "--exact"])
        run_dandd(["progressive", "-d", os.path.join(out, "ex_5_kmc_dtree.pickle"), "-o", out, "--ksweep",
                   "--mink", str(lo), "--maxk", str(hi), "-r", os.path.join(name, "ordering.pickle")])
    finally:
        ddstore.set_store(None)
    summary = [f for f in os.listdir(out) if f.endswith("summary.csv")]
    assert len(summary) == 1
    replay = {(int(r["ngen"]), int(r["kval"])): float(r["card"]) for r in read_csv(os.path.join(out, summary[0]))}
    assert len(replay) == len(growth)
    for r in growth:
        assert int(r["card"]) == replay[(int(r["ngen"]), int(r["k"]))], r


def test_steps_below_n_and_no_canon(tmp_path):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    fastas = make_dataset(data, 4, 1500, seed=3)
    name = str(tmp_path / "run")
    (got, cards, _), _ = _run(["-d", data, "--tool", "kmc", "--mink", "4", "--maxk", "40", "--steps", "2", "--no-canon",
                               "--name", name])
    want, want_cards = brute_exact_greedy(fastas, list(range(4, 41)), 2, canon=False)
    assert got.tolist() == want and np.array_equal(cards, want_cards)
    assert len(_read_tsv(os.path.join(name, "order.tsv"))) == 2 and len(_read_tsv(os.path.join(name, "growth.tsv"))) == 2 * 37


@pytest.mark.parametrize("argv,match", [
    (["--mink", "0"], "--mink 0 is outside 1..256 for kmc"),
    (["--maxk", "257"], "--maxk 257 is outside 1..256 for kmc"),
    (["--mink", "40", "--maxk", "33"], "above"),
    (["--steps", "4"], "--steps 4 is outside 1..3"),
])
def test_kmc_refusals(tmp_path, argv, match):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 3, 800, seed=2)
    name = str(tmp_path / "run")
    with pytest.raises(RuntimeError, match=match):
        _run(["-d", data, "--tool", "kmc", "--name", name] + argv)
    assert not os.path.exists(name)


def test_kmc_takes_k_above_32_and_ignores_registers(tmp_path):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 3, 800, seed=2)
    (got, cards, _), _ = _run(["-d", data, "--tool", "kmc", "--mink", "33", "--maxk", "34", "--registers", "4",
                               "--name", str(tmp_path / "run")])
    assert cards.shape == (3, 2)


def test_kmc_refuses_more_than_65535_inputs(tmp_path, monkeypatch):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 3, 800, seed=2)
    monkeypatch.setattr(greedy, "EXACT_MAX_N", 2)
    with pytest.raises(RuntimeError, match="--tool kmc orders at most 2 inputs, got 3"):
        _run(["-d", data, "--tool", "kmc", "--name", str(tmp_path / "run")])


# ---------------------------------------------------------------- two ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_worker(rank, world, port, argv):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    _run(argv)


def test_two_ranks_write_what_one_writes(tmp_path):
    import torch.multiprocessing as mp
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 5, 1200, seed=6)
    (tmp_path / "first.txt").write_text("g2.fasta\n")
    common = ["-d", data, "--tool", "kmc", "--mink", "3", "--maxk", "12", "--first", str(tmp_path / "first.txt")]
    two, one = str(tmp_path / "two"), str(tmp_path / "one")
    mp.spawn(_rank_worker, args=(2, _free_port(), common + ["--name", two]), nprocs=2, join=True)
    _run(common + ["--name", one])
    for fn in ("order.tsv", "growth.tsv", "collection.tsv", "ordering.pickle"):
        assert open(os.path.join(two, fn), "rb").read() == open(os.path.join(one, fn), "rb").read(), fn


# ---------------------------------------------------------------- ABI
ENTRIES = {"dd_exact_cover_count": 8, "dd_exact_cover_emit": 14, "dd_exact_cover_step": 7}


def test_entries_are_declared():
    from dandd_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    for fn, nargs in ENTRIES.items():
        assert re.search(r"DD_API\s+int\s+%s\s*\(" % fn, header), fn
        assert len(_lib.SIGNATURES[fn][1]) == nargs, fn
    assert re.search(r"#define DD_COVER_PART_BYTES %d\b" % _lib.DD_COVER_PART_BYTES, header)
    integration = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert re.search(r"\| `dd_exact_cover_count`, `dd_exact_cover_emit`, `dd_exact_cover_step` \|.*orderings_list.*kmc_tools",
                     integration)
    assert _lib.ABI_VERSION == 2


def test_entries_are_exported_and_check_arguments():
    """Arguments refused before any CUDA call (these run without a device)."""
    import subprocess
    from dandd_b200 import build, _lib
    build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "dandd_b200", "libdandd_b200.so")], text=True)
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    assert set(ENTRIES) <= exported
    lib = _lib.load()
    before = lib.dd_kernel_launches()
    WS, A, B, C_, D, E = 1 << 20, 1 << 21, 1 << 22, 1 << 23, 1 << 24, 1 << 25    # (never dereferenced: all refused)
    k, cap, nodes = 21, 1024, 4096
    wsb = lib.dd_exact_pairs_workspace_bytes(k, cap, nodes, 8)

    def count(ws=WS, wsb=wsb, k=k, cap=cap, out=A):
        return lib.dd_exact_cover_count(ws, wsb, k, cap, nodes, 8, out, None)

    assert count(ws=None) == -1 and count(out=None) == -1 and count(out=A + 4) == -1
    assert count(k=0) == -1 and count(k=257) == -1 and count(cap=1000) == -1 and count(wsb=64) == -3

    def emit(n=3, keys=10, nn=20, off=A, hol=B, kon=C_, status=D, wsb=wsb):
        return lib.dd_exact_cover_emit(WS, wsb, k, cap, nodes, 8, n, keys, nn, off, hol, kon, status, None)

    assert emit(n=0) == -1 and emit(n=65536) == -1 and b"outside [1,65535]" in lib.dd_last_error()
    assert emit(keys=1 << 32) == -1 and b"key ids are u32" in lib.dd_last_error()
    assert emit(nn=0xFFFFFFFF) == -1 and b"offsets are u32" in lib.dd_last_error()
    assert emit(off=None) == -1 and emit(status=None) == -1 and emit(hol=None) == -1 and emit(kon=None) == -1
    assert emit(off=A + 2) == -1 and emit(hol=B + 1) == -1 and emit(kon=C_ + 2) == -1 and emit(status=D + 4) == -1
    assert emit(wsb=64) == -3

    starts = np.array([0, 5, 5, 9], dtype=np.uint64)

    def part(**kw):
        row = dict(off=A, hol=B, kon=C_, cov=D, lost=E, keys=10, nn=9, start=starts.ctypes.data)
        row.update(kw)
        return [row[f] or 0 for f in ("off", "hol", "kon", "cov", "lost", "keys", "nn", "start")]

    def step(parts=None, n=3, g=0, ws=WS, wsb=128):
        table = np.array(parts or [part(), part()], dtype=np.uint64)
        return lib.dd_exact_cover_step(table.ctypes.data, table.shape[0], n, g, ws, wsb, None)

    assert lib.dd_exact_cover_step(None, 1, 3, 0, WS, 64, None) == -1
    assert step(ws=None) == -1 and step(ws=WS + 8) == -1 and step(wsb=64) == -3
    assert step(n=0) == -1 and step(n=65536) == -1
    assert step(g=3) == -1 and b"genome 3 outside [0,3)" in lib.dd_last_error() and step(g=-1) == -1
    for bad in (dict(off=None), dict(cov=None), dict(lost=None), dict(start=None), dict(hol=None), dict(kon=None),
                dict(off=A + 1), dict(hol=B + 1), dict(kon=C_ + 2), dict(lost=E + 4)):
        assert step([part(), part(**bad)]) == -1, bad
    assert step([part(keys=1 << 32)]) == -1 and b"key ids and offsets are u32" in lib.dd_last_error()
    assert step([part(nn=4)], g=2) == -1 and b"genome 2 has nodes [5,9)" in lib.dd_last_error()
    down = np.array([0, 5, 4, 9], dtype=np.uint64)
    assert step([part(start=down.ctypes.data)], g=1) == -1 and b"decreasing" in lib.dd_last_error()
    assert lib.dd_kernel_launches() == before
