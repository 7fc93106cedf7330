"""Greedy ordering (dandd_b200/helpers/greedy.py, K11) on the CPU: a numpy restatement of the dense correction rule,
the compaction and the sparse filter against explicit bincount(max(U, g)); the store's greedy loop on an engine double
against a brute-force greedy over oracle registers; the command line end to end (file formats, the `dandd
progressive -r ordering.pickle --ksweep` replay on the oracle store, refusals, two gloo ranks); the ABI entries."""
import csv
import os
import pickle
import re
import socket

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from dandd_b200.helpers import greedy
from tests.fake_engine import ListJobEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BINS = 64


# ---------------------------------------------------------------- numpy restatement of K11
def hist_of(u):
    """int64 [nk, 64] histograms of registers u [nk, m]."""
    return np.stack([np.bincount(np.minimum(row, BINS - 1), minlength=BINS) for row in np.asarray(u).astype(np.int64)])


def dense_rule(regs, union, uhist, cand):
    """(hist [C, nk, 64], live [C, nk]): hist(U) plus -1 at U[j] and +1 at g[j] for every register where g > U."""
    regs, union = np.asarray(regs).astype(np.int64), np.asarray(union).astype(np.int64)
    nk = union.shape[0]
    hist = np.zeros((len(cand), nk, BINS), dtype=np.int64)
    live = np.zeros((len(cand), nk), dtype=np.int64)
    for c, g in enumerate(cand):
        for k in range(nk):
            up = regs[g, k] > union[k]
            hist[c, k] = uhist[k]
            np.subtract.at(hist[c, k], union[k][up], 1)
            np.add.at(hist[c, k], regs[g, k][up], 1)
            live[c, k] = up.sum()
    return hist, live


def compact_rule(regs, union, cand, seg_off):
    """The sparse state: entries `j << 6 | value` of every live register in segment g * nk + k, within capacity."""
    regs, union = np.asarray(regs).astype(np.int64), np.asarray(union).astype(np.int64)
    n, nk, _ = regs.shape
    seg_off = np.asarray(seg_off, dtype=np.int64)
    entries = np.zeros(int(seg_off[-1]), dtype=np.int64)
    seg_len = np.zeros(n * nk, dtype=np.int64)
    for g in cand:
        for k in range(nk):
            s = g * nk + k
            j = np.nonzero(regs[g, k] > union[k])[0]
            cap = seg_off[s + 1] - seg_off[s]
            entries[seg_off[s]:seg_off[s] + min(cap, j.size)] = ((j << 6) | regs[g, k][j])[:cap]
            seg_len[s] = j.size
    return {"entries": entries, "seg_off": seg_off, "seg_len": seg_len, "nk": nk}


def sparse_rule(state, union, uhist, cand):
    """The sparse step: drop the entries with value <= U[k][j], keep the rest in place, count their pairs."""
    union = np.asarray(union).astype(np.int64)
    nk = state["nk"]
    hist = np.zeros((len(cand), nk, BINS), dtype=np.int64)
    live = np.zeros((len(cand), nk), dtype=np.int64)
    for c, g in enumerate(cand):
        for k in range(nk):
            s = g * nk + k
            off = state["seg_off"][s]
            n_len = min(state["seg_len"][s], state["seg_off"][s + 1] - off)
            seg = state["entries"][off:off + n_len]
            v, j = seg & 63, seg >> 6
            keep = v > union[k][j]
            state["entries"][off:off + keep.sum()] = seg[keep]
            state["seg_len"][s] = live[c, k] = keep.sum()
            hist[c, k] = uhist[k]
            np.subtract.at(hist[c, k], union[k][j[keep]], 1)
            np.add.at(hist[c, k], v[keep], 1)
    return hist, live


def explicit(regs, union, cand):
    regs, union = np.asarray(regs), np.asarray(union)
    hist = np.stack([hist_of(np.maximum(union, regs[g])) for g in cand])
    live = np.stack([(regs[g].astype(np.int64) > union).sum(axis=1) for g in cand])
    return hist, live


def offsets(live, cand, n, nk):
    counts = np.zeros((n, nk), dtype=np.int64)
    counts[list(cand)] = live
    return np.concatenate([[0], np.cumsum(counts.reshape(-1))])


@pytest.mark.parametrize("case", ["random", "zero", "equal", "maximal"])
def test_dense_rule_equals_explicit_maxima(case):
    rng = np.random.default_rng(len(case))
    n, nk, m = 6, 3, 256
    regs = rng.integers(0, 64, (n, nk, m)).astype(np.uint8)        # every value 0..63
    union = {"random": rng.integers(0, 64, (nk, m)), "zero": np.zeros((nk, m)), "equal": regs[2],
             "maximal": np.full((nk, m), 63)}[case].astype(np.uint8)
    for cand in ([0, 1, 2, 3, 4, 5], [1, 4], [5]):
        got = dense_rule(regs, union, hist_of(union), cand)
        want = explicit(regs, union, cand)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), cand
        state = compact_rule(regs, union, cand, offsets(want[1], cand, n, nk))
        got = sparse_rule(state, union, hist_of(union), cand)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), cand


def test_sparse_rule_follows_union_updates():
    """Compact once, then five union updates: the sparse step equals explicit maxima every time, with segments
    that empty (a genome equal to a chosen one) and one whose capacity bounds more than it holds."""
    rng = np.random.default_rng(5)
    n, nk, m = 8, 2, 512
    regs = np.minimum(rng.geometric(0.5, (n, nk, m)), 63).astype(np.uint8)
    regs[7] = regs[1]
    union = np.zeros((nk, m), dtype=np.uint8)
    cand = list(range(n))
    _, live = explicit(regs, union, cand)
    state = compact_rule(regs, union, cand, offsets(live, cand, n, nk))
    union = regs[0].copy()                                           # the union grew before the first sparse step
    cand.remove(0)
    for pick in (1, 3, 5, 2, 6):
        got = sparse_rule(state, union, hist_of(union), cand)
        want = explicit(regs, union, cand)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), pick
        union = np.maximum(union, regs[pick])
        cand.remove(pick)
    assert state["seg_len"][7 * nk:8 * nk].tolist() == [0] * nk      # genome 7 == genome 1: nothing left


# ---------------------------------------------------------------- the store's loop on an engine double
class GreedyFakeEngine(ListJobEngine):
    """ListJobEngine plus the K11 methods as the numpy restatement above, and Engine.cards_hist."""

    def cards_hist(self, regs, p):
        import torch
        h = torch.from_numpy(hist_of(regs.numpy().reshape(-1, 1 << p)).astype(np.int32))
        return self.mle(h, p).view(regs.shape[:-1]), h.view(tuple(regs.shape[:-1]) + (BINS,))

    def greedy_dense_hist(self, regs, union, union_hist, cand, p):
        import torch
        self.calls["greedy_dense"] = self.calls.get("greedy_dense", 0) + 1
        h, live = dense_rule(regs.numpy(), union.numpy(), union_hist.numpy(), list(cand))
        return torch.from_numpy(h.astype(np.int32)), torch.from_numpy(live.astype(np.int32))

    def greedy_compact(self, regs, union, cand, seg_off, p):
        self.calls["greedy_compact"] = self.calls.get("greedy_compact", 0) + 1
        return compact_rule(regs.numpy(), union.numpy(), list(cand), seg_off)

    def greedy_sparse_hist(self, state, union, union_hist, cand, p):
        import torch
        self.calls["greedy_sparse"] = self.calls.get("greedy_sparse", 0) + 1
        h, live = sparse_rule(state, union.numpy(), union_hist.numpy(), list(cand))
        return torch.from_numpy(h.astype(np.int32)), torch.from_numpy(live.astype(np.int32))

    def _pairs_budget(self):
        return 1 << 40


def brute_greedy(regs, ks, p, steps, order="max", first=()):
    """(order, cards [steps, nk]) by explicit unions and the oracle's estimator; the lowest index wins a tie."""
    from oracle import pyoracle as orc
    regs = np.asarray(regs)
    n, nk, m = regs.shape
    union = np.zeros((nk, m), dtype=np.uint8)
    picks, cards = [], []
    for t in range(steps):
        if t < len(first):
            best = first[t]
        else:
            best, best_d = None, None
            for g in range(n):
                if g in picks:
                    continue
                d = max(orc.card(np.maximum(union[c], regs[g, c]), p) / k for c, k in enumerate(ks))
                if best is None or (d > best_d if order == "max" else d < best_d):
                    best, best_d = g, d
        picks.append(best)
        union = np.maximum(union, regs[best])
        cards.append([orc.card(union[c], p) for c in range(nk)])
    return picks, np.asarray(cards)


def _oracle_regs(fastas, ks, p, canon=True):
    from oracle import pyoracle as orc
    return np.stack([np.stack([orc.hll_sketch(s, k, p, canon) for k in ks]) for s in _syms(fastas)])


@pytest.fixture(scope="module")
def clustered(tmp_path_factory):
    """Two clusters of near-copies plus an exact duplicate of genome 1 (genome 6): ties the lower index must win."""
    from tests.util import make_dataset
    d = tmp_path_factory.mktemp("greedy")
    a = make_dataset(str(d / "a"), 4, 3000, seed=41, prefix="a")
    b = make_dataset(str(d / "b"), 2, 3000, seed=42, prefix="b")
    fastas = a + b
    ks, p = list(range(5, 11)), 10
    regs = _oracle_regs(fastas, ks, p)
    regs = np.concatenate([regs, regs[1:2]])
    return regs, ks, p


@pytest.mark.parametrize("mode", ["dense", "sparse"])
@pytest.mark.parametrize("order,first,steps", [("max", (), 7), ("min", (), 7), ("max", (3, 6), 7), ("min", (5,), 4),
                                               ("max", (), 3)])
def test_store_loop_equals_brute_force(clustered, monkeypatch, mode, order, first, steps):
    import torch
    regs, ks, p = clustered
    st = ddstore.GpuSketchStore(engine=GreedyFakeEngine())
    if mode == "sparse":                                            # compact right after the first evaluated step
        monkeypatch.setattr(ddstore, "SPARSE_CROSS", 0)
    got, cards, stats = st.greedy_order(torch.from_numpy(regs), ks, p, steps, order=order, first=first,
                                        budget=None if mode == "sparse" else 0)
    want, want_cards = brute_greedy(regs, ks, p, steps, order, first)
    assert got.tolist() == want and np.array_equal(cards, want_cards)
    evaluated = steps - len(first)
    if mode == "dense":
        assert stats["switch_step"] is None and stats["dense_steps"] == evaluated and stats["sparse_steps"] == 0
    elif evaluated > 1:
        assert stats["switch_step"] == len(first) + 1 and stats["dense_steps"] == 1
        assert stats["sparse_steps"] == evaluated - 1 and st.engine.calls["greedy_compact"] == 1
    assert stats["live"][:len(first)] == [-1] * len(first) and len(stats["live"]) == steps
    if order == "max" and not first and steps == 7:
        assert got.tolist().index(1) < got.tolist().index(6)     # the duplicate: the lower index first


def test_store_refuses_an_engine_without_the_step():
    import torch
    st = ddstore.GpuSketchStore(engine=ListJobEngine())
    with pytest.raises(RuntimeError, match="K11"):
        st.greedy_order(torch.zeros((2, 1, 32), dtype=torch.uint8), [3], 5, 2)


# ---------------------------------------------------------------- the command line
def _run(argv, engine=GreedyFakeEngine):
    st = ddstore.GpuSketchStore(engine=engine())
    ddstore.set_store(st)
    try:
        return greedy.go(argv), st
    finally:
        ddstore.set_store(None)


def _read_tsv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


def _syms(fastas):
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    return [orc.fasta_symbols(_read_fasta(f)) for f in fastas]


@pytest.mark.parametrize("order", ["max", "min"])
def test_outputs_and_progressive_replay(tmp_path, order):
    """order.tsv / growth.tsv / collection.tsv against brute force, and growth.tsv == the summary CSV of
    `dandd progressive -r ordering.pickle --ksweep` over the same FASTAs on the oracle store."""
    from oracle import pyoracle as orc
    from tests.host_harness import read_csv, run_dandd
    from tests.oracle_store import OracleStore
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    fastas = make_dataset(data, 5, 2500, seed=17)
    names = [os.path.basename(f) for f in fastas]
    (tmp_path / "first.txt").write_text("\n%s\n" % names[3])
    name = str(tmp_path / "run")
    lo, hi, p = 4, 9, 10
    (order_, cards, _), _ = _run(["-d", data, "--mink", str(lo), "--maxk", str(hi), "--registers", str(p), "--order", order,
                                  "--first", str(tmp_path / "first.txt"), "--name", name])
    ks = list(range(lo, hi + 1))
    regs = _oracle_regs(fastas, ks, p)
    want, want_cards = brute_greedy(regs, ks, p, 5, order, (3,))
    assert order_.tolist() == want and np.array_equal(cards, want_cards)
    rows = _read_tsv(os.path.join(name, "order.tsv"))
    all_d = max(orc.card(orc.union_max(list(regs[:, c])), p) / k for c, k in enumerate(ks))
    before = 0.0
    for t, r in enumerate(rows):
        dk = [want_cards[t, c] / k for c, k in enumerate(ks)]
        assert (int(r["step"]), r["genome"], int(r["forced"])) == (t + 1, names[want[t]], int(t == 0))
        assert float(r["delta"]) == max(dk) and int(r["k"]) == ks[dk.index(max(dk))]
        assert float(r["gain"]) == max(dk) - before and float(r["fraction"]) == max(dk) / all_d
        before = max(dk)
    assert _read_tsv(os.path.join(name, "collection.tsv")) == [{"ngen": "5", "delta": repr(all_d),
                                                                "k": str(ks[[orc.card(orc.union_max(list(regs[:, c])), p) / k for c, k in enumerate(ks)].index(all_d)])}]
    growth = _read_tsv(os.path.join(name, "growth.tsv"))
    assert [(int(r["ngen"]), int(r["k"])) for r in growth] == [(t + 1, k) for t in range(5) for k in ks]
    assert all(float(r["delta_pos"]) == float(r["card"]) / int(r["k"]) for r in growth)
    with open(os.path.join(name, "ordering.pickle"), "rb") as fh:
        assert pickle.load(fh) == {tuple(want)}

    out = str(tmp_path / "out")
    ddstore.set_store(OracleStore())
    try:
        run_dandd(["tree", "-d", data, "-s", "gr", "-o", out, "-r", str(p)])
        run_dandd(["progressive", "-d", os.path.join(out, "gr_5_dashing_dtree.pickle"), "-o", out, "--ksweep",
                   "--mink", str(lo), "--maxk", str(hi), "-r", os.path.join(name, "ordering.pickle")])
    finally:
        ddstore.set_store(None)
    summary = [f for f in os.listdir(out) if f.endswith("summary.csv")]
    assert len(summary) == 1
    replay = {(int(r["ngen"]), int(r["kval"])): float(r["card"]) for r in read_csv(os.path.join(out, summary[0]))}
    assert len(replay) == len(growth)
    for r in growth:
        assert float(r["card"]) == replay[(int(r["ngen"]), int(r["k"]))], r


def test_steps_below_n(tmp_path):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 4, 1500, seed=3)
    name = str(tmp_path / "run")
    (order, cards, _), _ = _run(["-d", data, "--mink", "4", "--maxk", "6", "--registers", "8", "--steps", "2", "--name", name])
    assert len(order) == 2 and cards.shape == (2, 3)
    assert len(_read_tsv(os.path.join(name, "order.tsv"))) == 2 and len(_read_tsv(os.path.join(name, "growth.tsv"))) == 6


@pytest.mark.parametrize("argv,match", [
    (["--mink", "0"], "--mink 0 is outside"),
    (["--maxk", "33"], "--maxk 33 is outside 1..32"),
    (["--mink", "9", "--maxk", "5"], "above"),
    (["--registers", "4"], "--registers 4"),
    (["--registers", "27"], "--registers 27"),
    (["--steps", "0"], "--steps 0 is outside 1..3"),
    (["--steps", "4"], "--steps 4 is outside 1..3"),
    (["--first", "FIRST:g0.fasta,g2.fasta", "--steps", "1"], "--steps 1 is outside 2..3"),
    (["--first", "FIRST:g0.fasta,g9.fasta"], "g9.fasta is not an input"),
    (["--first", "FIRST:g1.fasta,g1.fasta"], "g1.fasta is named twice"),
    ([], None),
])
def test_refusals(tmp_path, argv, match):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 3, 800, seed=2)
    name = str(tmp_path / "run")
    for i, a in enumerate(argv):
        if a.startswith("FIRST:"):
            (tmp_path / "first.txt").write_text("\n".join(a[6:].split(",")) + "\n")
            argv[i] = str(tmp_path / "first.txt")
    if match is None:                                        # an existing --name, then no input at all
        os.makedirs(name)
        with pytest.raises(RuntimeError, match="already exists"):
            _run(["-d", data, "--name", name])
        with pytest.raises(RuntimeError, match="-d DATADIR or -f LIST"):
            _run(["--name", str(tmp_path / "other")])
        return
    with pytest.raises(RuntimeError, match=match):
        _run(["-d", data, "--name", name] + argv)
    assert not os.path.exists(name)


def test_one_input_and_duplicate_names_are_refused(tmp_path):
    from tests.util import make_dataset
    make_dataset(str(tmp_path / "one"), 1, 800, seed=2)
    with pytest.raises(RuntimeError, match="at least 2 inputs, got 1"):
        _run(["-d", str(tmp_path / "one"), "--name", str(tmp_path / "run")])
    a = make_dataset(str(tmp_path / "a"), 2, 800, seed=2)
    b = make_dataset(str(tmp_path / "b"), 1, 800, seed=3)
    listing = tmp_path / "list.txt"
    listing.write_text("\n".join(a + b) + "\n")
    with pytest.raises(RuntimeError, match="distinct.*g0.fasta"):
        _run(["-f", str(listing), "--name", str(tmp_path / "run")])


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
    common = ["-d", data, "--mink", "3", "--maxk", "8", "--registers", "10", "--first", str(tmp_path / "first.txt")]
    two, one = str(tmp_path / "two"), str(tmp_path / "one")
    mp.spawn(_rank_worker, args=(2, _free_port(), common + ["--name", two]), nprocs=2, join=True)
    _run(common + ["--name", one])
    for fn in ("order.tsv", "growth.tsv", "collection.tsv", "ordering.pickle"):
        assert open(os.path.join(two, fn), "rb").read() == open(os.path.join(one, fn), "rb").read(), fn


# ---------------------------------------------------------------- ABI
ENTRIES = {"dd_greedy_workspace_bytes": 1, "dd_greedy_dense_hist": 13, "dd_greedy_compact": 15, "dd_greedy_sparse_hist": 16}


def test_entry_is_declared():
    from dandd_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    for fn, nargs in ENTRIES.items():
        assert re.search(r"DD_API\s+(int|size_t)\s+%s\s*\(" % fn, header), fn
        assert len(_lib.SIGNATURES[fn][1]) == nargs, fn
    integration = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert re.search(r"\| `dd_greedy_workspace_bytes`, `dd_greedy_dense_hist`, `dd_greedy_compact`, `dd_greedy_sparse_hist` \|"
                     r".*orderings_list.*SubSpider", integration)
    assert _lib.ABI_VERSION == 2


def test_entry_is_exported_and_checks_arguments():
    """Arguments refused before any CUDA call (these run without a device)."""
    import subprocess
    from dandd_b200 import build, _lib
    build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "dandd_b200", "libdandd_b200.so")], text=True)
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    assert set(ENTRIES) <= exported
    lib = _lib.load()
    assert lib.dd_greedy_workspace_bytes(3) == 16 and lib.dd_greedy_workspace_bytes(0) == 0
    before = lib.dd_kernel_launches()
    R, U, UH, H, L, W = 1 << 20, 1 << 21, 1 << 22, 1 << 23, 1 << 24, 1 << 25   # (never dereferenced: all refused)
    cand = np.array([0, 2], dtype=np.int32)

    def dense(regs=R, n=3, nk=2, p=10, union=U, cand=cand, C=None, hist=H, wsb=16):
        C = len(cand) if C is None else C
        return lib.dd_greedy_dense_hist(regs, n, nk, p, union, UH, cand.ctypes.data, C, hist, L, W, wsb, None)

    assert dense(regs=None) == -1 and dense(union=None) == -1 and dense(hist=None) == -1
    assert dense(p=4) == -1 and dense(p=27) == -1 and dense(nk=0) == -1 and dense(nk=65536) == -1
    assert dense(C=0) == -1 and dense(n=0) == -1
    assert dense(cand=np.array([0, 3], dtype=np.int32)) == -1 and b"outside [0,3)" in lib.dd_last_error()
    assert dense(cand=np.array([-1], dtype=np.int32)) == -1
    assert dense(cand=np.array([1, 1], dtype=np.int32)) == -1 and b"listed twice" in lib.dd_last_error()
    big = np.arange(40000, dtype=np.int32)
    assert dense(n=40000, nk=1000, cand=big, wsb=1 << 20) == -1 and b"too many" in lib.dd_last_error()
    assert dense(regs=R + 8) == -1 and dense(union=U + 4) == -1
    assert dense(wsb=4) == -3

    off = np.zeros(3 * 2 + 1, dtype=np.int64)

    def compact(seg=off, n_entries=0, union=U, ws=W):
        return lib.dd_greedy_compact(R, 3, 2, 10, union, cand.ctypes.data, 2, seg.ctypes.data, H, L, W, n_entries, ws, 16, None)

    bad = off.copy()
    bad[0] = 1
    assert compact(seg=bad, n_entries=8) == -1 and b"start at 0" in lib.dd_last_error()
    bad = np.array([0, 4, 2, 6, 6, 6, 6], dtype=np.int64)
    assert compact(seg=bad, n_entries=8) == -1 and b"decrease" in lib.dd_last_error()
    bad = np.array([0, 4, 4, 6, 6, 6, 9], dtype=np.int64)
    assert compact(seg=bad, n_entries=8) == -1 and b"buffer holds 8" in lib.dd_last_error()
    assert compact(union=U + 8) == -1 and compact(ws=W + 4) == -1

    def sparse(n_entries=8, seg=H, C=2, union=U):
        return lib.dd_greedy_sparse_hist(L, n_entries, seg, W, 3, 2, 10, union, UH, cand.ctypes.data, C, H, L, W, 16, None)

    assert sparse(n_entries=-1) == -1 and sparse(seg=None) == -1 and sparse(seg=H + 4) == -1
    assert sparse(C=0) == -1 and sparse(union=U + 1) == -1
    assert lib.dd_kernel_launches() == before
