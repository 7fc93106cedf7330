"""Queries against a collection (dandd_b200/helpers/query.py, K13) on the CPU: the command line end to end for both tools
through the real store on an engine double, against brute force (Python k-mer sets for kmc, np.maximum unions and the
oracle MLE for dashing, per union); the gain / novel / Jaccard / containment / KIJ arithmetic and the tie rule; refusals;
two gloo ranks; and the ABI entry."""
import csv
import os
import re
import shutil
import socket

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from dandd_b200.helpers import query
from tests.fake_engine import FakeEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILES = ("union.tsv", "collection.tsv", "with.tsv", "delta.tsv", "pairs.tsv", "kij.tsv")


def _run(argv):
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    try:
        return query.go(argv), st
    finally:
        ddstore.set_store(None)


def _read_tsv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


def _syms(fastas):
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    return [orc.fasta_symbols(_read_fasta(f)) for f in fastas]


def _collection(tmp_path, n_refs=4, n_queries=3, length=1500):
    """References r0..r{R-1} and queries q0..; the last query is a copy of reference r1 under r1's name."""
    from tests.util import make_dataset
    refs = make_dataset(str(tmp_path / "refs"), n_refs, length, seed=12, prefix="r")
    queries = make_dataset(str(tmp_path / "queries"), n_queries - 1, length, seed=12, sub=0.06, prefix="q")
    shutil.copy(refs[1], str(tmp_path / "queries" / "r1.fasta"))
    return sorted(refs), sorted(queries + [str(tmp_path / "queries" / "r1.fasta")])


def _brute(refs, queries, ks, tool, canon, p=10):
    """(ref_single, query_single, union, with_q, pair) per union, from scratch."""
    from oracle import pyoracle as orc
    rs, qs = _syms(refs), _syms(queries)
    R, Q, nk = len(refs), len(queries), len(ks)
    out = [np.zeros((nk, R)), np.zeros((nk, Q)), np.zeros(nk), np.zeros((nk, Q)), np.zeros((nk, Q, R))]
    for c, k in enumerate(ks):
        if tool == "kmc":
            a = [set(orc.kmers(s, k, canon).tolist()) for s in rs]
            b = [set(orc.kmers(s, k, canon).tolist()) for s in qs]
            size, join = len, lambda xs: set().union(*xs)
        else:
            a = [orc.hll_sketch(s, k, p, canon) for s in rs]
            b = [orc.hll_sketch(s, k, p, canon) for s in qs]
            size, join = (lambda x: orc.card(x, p)), (lambda xs: np.maximum.reduce(list(xs)))
        out[0][c] = [size(x) for x in a]
        out[1][c] = [size(x) for x in b]
        out[2][c] = size(join(a))
        out[3][c] = [size(join(a + [x])) for x in b]
        out[4][c] = [[size(join([x, y])) for y in a] for x in b]
    return out


def _check_tables(name, ref_names, query_names, ks, cards, exact):
    """Every file against the arrays the run returned, restating each column's rule."""
    num = int if exact else float
    rs, qs, u, w, pr = (np.asarray(a) for a in cards)
    rows = _read_tsv(os.path.join(name, "union.tsv"))
    assert [(int(r["k"]), num(r["card"]), float(r["delta_pos"])) for r in rows] == [(k, u[c], u[c] / k) for c, k in enumerate(ks)]
    dk = [u[c] / k for c, k in enumerate(ks)]
    d_all = max(dk)
    assert _read_tsv(os.path.join(name, "collection.tsv")) == [
        {"ngen": str(len(ref_names)), "delta": repr(float(d_all)), "k": str(ks[dk.index(d_all)])}]
    rows = _read_tsv(os.path.join(name, "with.tsv"))
    assert [(int(r["k"]), r["query"]) for r in rows] == [(k, q) for k in ks for q in query_names]
    for r in rows:
        c, q = ks.index(int(r["k"])), query_names.index(r["query"])
        assert num(r["card"]) == w[c, q] and num(r["novel"]) == w[c, q] - u[c] and float(r["delta_pos"]) == w[c, q] / ks[c]
    rows = _read_tsv(os.path.join(name, "delta.tsv"))
    assert [r["query"] for r in rows] == query_names
    best = lambda col: max(((col[c] / k, k) for c, k in enumerate(ks)), key=lambda t: t[0])   # first k wins a tie
    for q, r in enumerate(rows):
        d, kk = best(w[:, q])
        assert (float(r["delta"]), int(r["k"]), float(r["gain"])) == (d, kk, d - d_all)
    rows = _read_tsv(os.path.join(name, "pairs.tsv"))
    assert [(int(r["k"]), r["query"], r["reference"]) for r in rows] == [(k, q, x) for k in ks for q in query_names for x in ref_names]
    for r in rows:
        c, q, x = ks.index(int(r["k"])), query_names.index(r["query"]), ref_names.index(r["reference"])
        a, b, ab = qs[c, q], rs[c, x], pr[c, q, x]
        assert (num(r["card_query"]), num(r["card_reference"]), num(r["card_union"])) == (a, b, ab)
        assert float(r["jaccard"]) == (a + b - ab) / ab and float(r["containment"]) == (a + b - ab) / a
    rows = _read_tsv(os.path.join(name, "kij.tsv"))
    assert [(r["query"], r["reference"]) for r in rows] == [(q, x) for q in query_names for x in ref_names]
    for r in rows:
        q, x = query_names.index(r["query"]), ref_names.index(r["reference"])
        dq, dr, dqr = best(qs[:, q])[0], best(rs[:, x])[0], best(pr[:, q, x])[0]
        assert (float(r["delta_query"]), float(r["delta_reference"]), float(r["delta_union"])) == (dq, dr, dqr)
        assert float(r["kij"]) == (dq + dr - dqr) / dqr


@pytest.mark.parametrize("tool", ["dashing", "kmc"])
@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
def test_helper_against_brute_force(tmp_path, tool, canon):
    refs, queries = _collection(tmp_path)
    ks = list(range(4, 10))
    argv = ["-d", str(tmp_path / "refs"), "-q", str(tmp_path / "queries"), "--tool", tool, "--mink", "4", "--maxk", "9",
            "--registers", "10", "--name", str(tmp_path / "run")] + ([] if canon else ["--no-canon"])
    cards, st = _run(argv)
    want = _brute(refs, queries, ks, tool, canon)
    for got, exp in zip(cards, want):
        assert np.shape(got) == exp.shape and np.array_equal(np.asarray(got, dtype=np.float64), exp)
    if tool == "kmc":
        assert all(np.asarray(a).dtype == np.int64 for a in cards)
        assert st.engine.calls["exact_query_counts"] == len(ks) and st.stats["exact_calls"] == len(ks)
    else:
        assert st.engine.calls["greedy_dense"] == 1
    R = len(refs)
    # the query that is a copy of reference r1 adds nothing and equals r1
    q = [os.path.basename(f) for f in queries].index("r1.fasta")
    assert np.array_equal(cards[3][:, q], cards[2]) and np.array_equal(cards[4][:, q, 1], cards[0][:, 1])
    _check_tables(str(tmp_path / "run"), [os.path.basename(f) for f in refs], [os.path.basename(f) for f in queries], ks, cards,
                  exact=tool == "kmc")
    assert R == 4


def test_lists_and_one_query(tmp_path):
    """-f / --query-list, one reference and one query."""
    refs, queries = _collection(tmp_path)
    (tmp_path / "r.txt").write_text(refs[2] + "\n")
    (tmp_path / "q.txt").write_text(queries[0] + "\n")
    cards, _ = _run(["-f", str(tmp_path / "r.txt"), "--query-list", str(tmp_path / "q.txt"), "--tool", "kmc", "--mink", "5",
                     "--maxk", "7", "--name", str(tmp_path / "run")])
    want = _brute([refs[2]], [queries[0]], [5, 6, 7], "kmc", True)
    assert all(np.array_equal(np.asarray(g, dtype=np.float64), w) for g, w in zip(cards, want))
    assert cards[4].shape == (3, 1, 1)


def test_arithmetic_and_ties(tmp_path):
    """Hand-made counts: a tie between two k goes to the first; gain, novel, Jaccard, containment and KIJ."""
    ks = [2, 4, 5]
    ref_single = np.array([[4, 2], [8, 6], [9, 5]])            # r0: 2.0, 2.0, 1.8 -> delta 2.0 at k = 2
    query_single = np.array([[2], [8], [10]])                  # 1.0, 2.0, 2.0 -> 2.0 at k = 4
    union = np.array([6, 12, 10])                              # 3.0, 3.0, 2.0 -> 3.0 at k = 2
    with_q = np.array([[6], [16], [20]])                       # 3.0, 4.0, 4.0 -> 4.0 at k = 4
    pair = np.array([[[5, 3]], [[12, 10]], [[15, 13]]])
    query.write_outputs(str(tmp_path), ["r0", "r1"], ["q0"], ks, ref_single, query_single, union, with_q, pair, exact=True)
    assert _read_tsv(str(tmp_path / "collection.tsv")) == [{"ngen": "2", "delta": "3.0", "k": "2"}]
    assert _read_tsv(str(tmp_path / "delta.tsv")) == [{"query": "q0", "delta": "4.0", "k": "4", "gain": "1.0"}]
    w = _read_tsv(str(tmp_path / "with.tsv"))
    assert [(r["card"], r["novel"]) for r in w] == [("6", "0"), ("16", "4"), ("20", "10")]
    p = _read_tsv(str(tmp_path / "pairs.tsv"))[0]                # k = 2, q0 x r0: |q n r| = 2 + 4 - 5 = 1
    assert (p["jaccard"], p["containment"]) == (repr(1 / 5), repr(1 / 2))
    kij = _read_tsv(str(tmp_path / "kij.tsv"))
    # q0: 2.0; r0: 2.0 (k = 2 before k = 4); q0 u r0: 12 / 4 = 3.0; KIJ = (2 + 2 - 3) / 3
    assert kij[0] == {"query": "q0", "reference": "r0", "delta_query": "2.0", "delta_reference": "2.0", "delta_union": "3.0",
                      "kij": repr((2.0 + 2.0 - 3.0) / 3.0)}
    _check_tables(str(tmp_path), ["r0", "r1"], ["q0"], ks, (ref_single, query_single, union, with_q, pair), exact=True)


# ---------------------------------------------------------------- refusals
@pytest.mark.parametrize("argv,match", [
    (["--mink", "0"], "--mink 0 is outside"),
    (["--maxk", "33"], "--maxk 33 is outside 1..32 for dashing"),
    (["--tool", "kmc", "--maxk", "257"], "--maxk 257 is outside 1..256 for kmc"),
    (["--mink", "9", "--maxk", "5"], "above"),
    (["--registers", "4"], "--registers 4"),
    (["--registers", "27"], "--registers 27"),
])
def test_refusals(tmp_path, argv, match):
    _collection(tmp_path, 2, 2, 800)
    name = str(tmp_path / "run")
    with pytest.raises(RuntimeError, match=match):
        _run(["-d", str(tmp_path / "refs"), "-q", str(tmp_path / "queries"), "--name", name] + argv)
    assert not os.path.exists(name)


def test_missing_inputs_and_existing_name(tmp_path):
    _collection(tmp_path, 2, 2, 800)
    refs, queries = str(tmp_path / "refs"), str(tmp_path / "queries")
    with pytest.raises(RuntimeError, match="give the queries"):
        _run(["-d", refs, "--name", str(tmp_path / "a")])
    with pytest.raises(RuntimeError, match="give the references"):
        _run(["-q", queries, "--name", str(tmp_path / "a")])
    os.makedirs(str(tmp_path / "empty"))
    with pytest.raises(RuntimeError, match="no queries given"):
        _run(["-d", refs, "-q", str(tmp_path / "empty"), "--name", str(tmp_path / "a")])
    assert not os.path.exists(str(tmp_path / "a"))
    os.makedirs(str(tmp_path / "b"))
    with pytest.raises(RuntimeError, match="already exists"):
        _run(["-d", refs, "-q", queries, "--name", str(tmp_path / "b")])


@pytest.mark.parametrize("side", ["references", "queries"])
def test_duplicate_names_are_refused(tmp_path, side):
    from tests.util import make_dataset
    refs, queries = _collection(tmp_path, 2, 2, 800)
    other = make_dataset(str(tmp_path / "other"), 1, 800, seed=3, prefix="r" if side == "references" else "q")
    listing = tmp_path / "list.txt"
    listing.write_text("\n".join((refs if side == "references" else queries) + other) + "\n")
    src = ["-f", str(listing), "-q", str(tmp_path / "queries")] if side == "references" else \
        ["-d", str(tmp_path / "refs"), "--query-list", str(listing)]
    with pytest.raises(RuntimeError, match="names of the %s must be distinct.*0.fasta" % side):
        _run(src + ["--name", str(tmp_path / "run")])


def test_genome_count_limits(tmp_path, monkeypatch):
    _collection(tmp_path, 2, 2, 800)
    argv = ["-d", str(tmp_path / "refs"), "-q", str(tmp_path / "queries"), "--name", str(tmp_path / "run")]
    monkeypatch.setattr(query, "MAX_CELLS", 3)
    with pytest.raises(RuntimeError, match="2 queries x 2 references is above 3 pairs"):
        _run(argv)
    monkeypatch.setattr(query, "MAX_CELLS", 1 << 32)
    monkeypatch.setattr(query, "MAX_GENOMES_LONG_K", 3)
    with pytest.raises(RuntimeError, match="above k = 64 at most 3 references"):
        _run(argv + ["--tool", "kmc", "--maxk", "65"])
    _run(argv + ["--tool", "kmc", "--mink", "60", "--maxk", "64"])       # up to k = 64 the count is not limited
    assert query.MAX_CELLS == 1 << 32 == _header_define("DD_QUERY_MAX_CELLS")


# ---------------------------------------------------------------- two ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_worker(rank, world, port, argv):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    _run(argv)


@pytest.mark.parametrize("tool", ["dashing", "kmc"])
def test_two_ranks_write_what_one_writes(tmp_path, tool):
    import torch.multiprocessing as mp
    _collection(tmp_path, 3, 3, 1200)
    common = ["-d", str(tmp_path / "refs"), "-q", str(tmp_path / "queries"), "--tool", tool, "--mink", "3", "--maxk", "8",
              "--registers", "12"]
    two, one = str(tmp_path / "two"), str(tmp_path / "one")
    mp.spawn(_rank_worker, args=(2, _free_port(), common + ["--name", two]), nprocs=2, join=True)
    _run(common + ["--name", one])
    for fn in FILES:
        assert open(os.path.join(two, fn), "rb").read() == open(os.path.join(one, fn), "rb").read(), fn


# ---------------------------------------------------------------- ABI
def _header_define(name):
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    m = re.search(r"#define\s+%s\s+\(1ll << (\d+)\)" % name, header)
    return 1 << int(m.group(1))


def test_entry_is_declared():
    from dandd_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    assert re.search(r"DD_API\s+int\s+dd_exact_query_counts\s*\(", header)
    assert len(_lib.SIGNATURES["dd_exact_query_counts"][1]) == 12
    integration = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert re.search(r"\| `dd_exact_query_counts` \|.*kmc_tools complex", integration)
    assert _lib.ABI_VERSION == 2


def test_entry_is_exported_and_checks_arguments():
    """Arguments refused before any CUDA call (these run without a device)."""
    import subprocess
    from dandd_b200 import build, _lib
    build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "dandd_b200", "libdandd_b200.so")], text=True)
    assert "dd_exact_query_counts" in {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    lib = _lib.load()
    before = lib.dd_kernel_launches()
    W, I, S, U = 1 << 20, 1 << 21, 1 << 22, 1 << 23          # (never dereferenced: every call below is refused)
    k, cap, nodes = 21, 1024, 4096
    wsb = lib.dd_exact_pairs_workspace_bytes(k, cap, nodes, 8)

    def call(ws=W, wsb=wsb, k=k, cap=cap, nodes=nodes, streams=8, R=3, Q=2, inter=I, shared=S, union=U):
        return lib.dd_exact_query_counts(ws, wsb, k, cap, nodes, streams, R, Q, inter, shared, union, None)

    assert call(ws=None) == -1 and call(inter=None) == -1 and call(shared=None) == -1 and call(union=None) == -1
    assert call(k=0) == -1 and call(k=257) == -1 and call(cap=1000) == -1 and call(nodes=0xFFFFFFFF) == -1
    assert call(wsb=wsb - 1) == -3
    assert call(R=0) == -1 and call(Q=0) == -1 and call(R=-1) == -1
    assert b"n_refs=0" in lib.dd_last_error() or b"n_refs=-1" in lib.dd_last_error()
    assert call(R=1 << 31, Q=1 << 31) == -1 and b"above 4294967295" in lib.dd_last_error()
    assert call(R=1 << 20, Q=(1 << 12) + 1) == -1 and b"cells" in lib.dd_last_error()
    big = lib.dd_exact_pairs_workspace_bytes(65, cap, nodes, 8)
    assert call(k=65, wsb=big, R=60000, Q=5537) == -1 and b"65536" in lib.dd_last_error()
    assert lib.dd_kernel_launches() == before
