"""Leave-one-out contributions (dandd_b200/helpers/leaveout.py, K10) on the CPU: a numpy restatement of K10's streaming
rule against explicit maxima over the other groups; the command line end to end for both tools through the real
store on an oracle-backed engine double, against brute force; the kmc contribution against
DeltaTree.find_delta_delta; refusals, --groups parsing, two gloo ranks and the ABI entry."""
import csv
import os
import re
import socket

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from dandd_b200.helpers import leaveout
from tests.fake_engine import BINS, FakeEngine, brute_hist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def streaming_hist(regs, group, n_groups, order=None):
    """K10's rule, restated over all registers at once, genomes visited in `order`: (max1, max2, lead) per register,
    then the union histogram plus one -1/+1 pair per register with a single leading group."""
    MULTI = -1
    regs = np.asarray(regs).astype(np.int64)
    n, nk, m = regs.shape
    m1, m2 = np.zeros((nk, m), np.int64), np.zeros((nk, m), np.int64)
    lead = np.full((nk, m), MULTI)
    for g in (range(n) if order is None else order):
        v, c = regs[g], int(group[g])
        mine = lead == c
        gt, eq, lt = v > m1, v == m1, v < m1
        m2 = np.where(gt & ~mine, m1, np.where(lt & ~mine, np.maximum(m2, v), m2))
        lead = np.where(gt, c, np.where(eq & ~mine, MULTI, lead))
        m1 = np.maximum(m1, v)
    out = np.zeros((nk, 1 + n_groups, BINS), dtype=np.int64)
    for c in range(nk):
        out[c, :] = np.bincount(m1[c], minlength=BINS)
        single = lead[c] != MULTI
        np.subtract.at(out[c], (1 + lead[c][single], m1[c][single]), 1)
        np.add.at(out[c], (1 + lead[c][single], m2[c][single]), 1)
    return out


# ---------------------------------------------------------------- the streaming rule
@pytest.mark.parametrize("case", ["ties", "duplicates", "zeros"])
@pytest.mark.parametrize("n", [1, 2, 3, 7, 12])
def test_streaming_rule_equals_explicit_maxima(case, n):
    rng = np.random.default_rng(n * 10 + len(case))
    regs = rng.integers(0, 4, (n, 3, 64)).astype(np.uint8)          # values 0..3: ties everywhere
    if case == "duplicates" and n > 1:
        regs[n - 1] = regs[0]
        regs[n // 2] = regs[0]
    if case == "zeros":
        regs[rng.integers(0, n, max(1, n // 2))] = 0
    for n_groups in range(1, n + 1):
        for trial in range(3):                                       # non-contiguous ids, every group used
            group = np.concatenate([np.arange(n_groups), rng.integers(0, n_groups, n - n_groups)])
            rng.shuffle(group)
            want = brute_hist(regs, group, n_groups)
            assert np.array_equal(streaming_hist(regs, group, n_groups), want), (n_groups, trial)
            by_group = np.argsort(group, kind="stable")              # the kernel's visiting order
            assert np.array_equal(streaming_hist(regs, group, n_groups, by_group), want)
            assert np.array_equal(streaming_hist(regs, group, n_groups, rng.permutation(n)), want)


# ---------------------------------------------------------------- the command line
def _run(argv):
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    try:
        return leaveout.go(argv), st
    finally:
        ddstore.set_store(None)


def _read_tsv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


def _syms(fastas):
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    return [orc.fasta_symbols(_read_fasta(f)) for f in fastas]


def _groups_file(tmp_path, names, labels):
    path = tmp_path / "groups.tsv"
    path.write_text("".join("%s\t%s\n" % (a, b) for a, b in zip(names, labels)))
    return str(path)


def _check_tables(name, ks, labels, union, without, ngen, exact):
    num = int if exact else float
    rows = _read_tsv(os.path.join(name, "union.tsv"))
    assert [int(r["k"]) for r in rows] == ks
    assert [num(r["card"]) for r in rows] == list(union)
    assert [float(r["delta_pos"]) for r in rows] == [u / k for u, k in zip(union, ks)]
    rows = _read_tsv(os.path.join(name, "without.tsv"))
    assert [(int(r["k"]), r["group"]) for r in rows] == [(k, lab) for k in ks for lab in labels]
    for r in rows:
        c, g = ks.index(int(r["k"])), labels.index(r["group"])
        assert num(r["card"]) == without[c][g] and num(r["novel"]) == union[c] - without[c][g]
        assert float(r["delta_pos"]) == without[c][g] / ks[c]
    dk_all = [u / k for u, k in zip(union, ks)]
    d_all = max(dk_all)
    coll = _read_tsv(os.path.join(name, "collection.tsv"))
    assert coll == [{"ngen": str(ngen), "delta": repr(d_all), "k": str(ks[dk_all.index(d_all)])}]
    rows = _read_tsv(os.path.join(name, "delta.tsv"))
    assert [r["group"] for r in rows] == labels
    for r, g in zip(rows, range(len(labels))):
        dk = [without[c][g] / k for c, k in enumerate(ks)]
        assert float(r["delta"]) == max(dk) and int(r["k"]) == ks[dk.index(max(dk))]
        assert float(r["contribution"]) == d_all - max(dk)


@pytest.mark.parametrize("grouped", [False, True], ids=["singletons", "groups"])
@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
def test_dashing_against_oracle_registers(tmp_path, canon, grouped):
    from oracle import pyoracle as orc
    from tests.util import make_dataset
    fastas = make_dataset(str(tmp_path / "data"), 5, 1500, seed=8)
    names = [os.path.basename(f) for f in fastas]
    labels_of = ["b", "a", "b", "c", "a"] if grouped else names
    argv = ["-d", str(tmp_path / "data"), "--mink", "4", "--maxk", "9", "--registers", "10", "--name", str(tmp_path / "run")]
    if grouped:
        argv += ["--groups", _groups_file(tmp_path, names, labels_of)]
    if not canon:
        argv.append("--no-canon")
    (union, without), st = _run(argv)
    labels = ["b", "a", "c"] if grouped else names
    group = [labels.index(x) for x in labels_of]
    ks = list(range(4, 10))
    syms = _syms(fastas)
    for c, k in enumerate(ks):
        regs = [orc.hll_sketch(s, k, 10, canon) for s in syms]
        assert union[c] == orc.card(orc.union_max(regs), 10)
        for g in range(len(labels)):
            assert without[c, g] == orc.card(orc.union_max([r for r, x in zip(regs, group) if x != g]), 10), (k, g)
    assert st.engine.calls["leave_out_hist"] == 1
    _check_tables(str(tmp_path / "run"), ks, labels, union.tolist(), without.tolist(), 5, exact=False)


@pytest.mark.parametrize("grouped", [False, True], ids=["singletons", "groups"])
@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
def test_kmc_against_oracle_kmer_sets(tmp_path, canon, grouped):
    from oracle import pyoracle as orc
    from tests.util import make_dataset
    fastas = make_dataset(str(tmp_path / "data"), 5, 1500, seed=9)
    names = [os.path.basename(f) for f in fastas]
    labels_of = ["x", "y", "x", "x", "z"] if grouped else names
    argv = ["-d", str(tmp_path / "data"), "--tool", "kmc", "--mink", "3", "--maxk", "12", "--name", str(tmp_path / "run")]
    if grouped:
        argv += ["--groups", _groups_file(tmp_path, names, labels_of)]
    if not canon:
        argv.append("--no-canon")
    (union, without), st = _run(argv)
    labels = ["x", "y", "z"] if grouped else names
    group = [labels.index(x) for x in labels_of]
    ks = list(range(3, 13))
    syms = _syms(fastas)
    for c, k in enumerate(ks):
        sets = [set(orc.kmers(s, k, canon).tolist()) for s in syms]
        everything = set().union(*sets)
        assert union[c] == len(everything)
        for g in range(len(labels)):
            private = set().union(*[s for s, x in zip(sets, group) if x == g]) - set().union(*[s for s, x in zip(sets, group) if x != g])
            assert without[c, g] == len(everything) - len(private), (k, g)
    job = "exact_family_counts" if grouped else "exact_spectrum"
    assert st.engine.calls[job] == len(ks) and st.stats["exact_calls"] == len(ks)
    _check_tables(str(tmp_path / "run"), ks, labels, union.tolist(), without.tolist(), 5, exact=True)


def test_kmc_contribution_equals_find_delta_delta(tmp_path):
    """`dandd tree --exact`, then find_delta_delta([g]) for every genome; where the climbs (full tree and the subtree
    without g) end at the sweep's maximum, the helper's contribution is the same float."""
    import dandd_b200
    from tests.host_harness import run_dandd
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    fastas = make_dataset(data, 4, 2500, seed=31)
    (union, without), _ = _run(["-d", data, "--tool", "kmc", "--mink", "2", "--maxk", "20", "--name", str(tmp_path / "run")])
    ks = list(range(2, 21))
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    try:
        run_dandd(["tree", "-d", data, "-s", "ex", "-o", str(tmp_path / "out"), "--exact"])
        dandd_b200.enable_compat()
        import dandd_cmd
        from huffman_dandd import SubSpider
        dtree = dandd_cmd._load_tree(os.path.join(str(tmp_path / "out"), "ex_4_kmc_dtree.pickle"))
        d_all, k_all = leaveout.best_k(ks, union)
        assert (dtree.delta, dtree.root_k()) == (float(d_all), int(k_all))      # the climb reached the sweep's maximum
        rows = {r["group"]: r for r in _read_tsv(os.path.join(str(tmp_path / "run"), "delta.tsv"))}
        for g, f in enumerate(sorted(fastas)):
            rest = [x for x in dtree.fastas if x != f]
            small = SubSpider(leafnodes=dtree.nodes_from_fastas(rest), speciesinfo=dtree.speciesinfo, experiment=dtree.experiment)
            d_out, k_out = leaveout.best_k(ks, without[:, g])
            assert (small.delta, small.root_k()) == (float(d_out), int(k_out))
            assert float(rows[os.path.basename(f)]["contribution"]) == dtree.find_delta_delta([f])
    finally:
        ddstore.set_store(None)


# ---------------------------------------------------------------- refusals and --groups
@pytest.mark.parametrize("argv,match", [
    (["--mink", "0"], "--mink 0 is outside"),
    (["--maxk", "33"], "--maxk 33 is outside 1..32 for dashing"),
    (["--tool", "kmc", "--maxk", "257"], "--maxk 257 is outside 1..256 for kmc"),
    (["--mink", "9", "--maxk", "5"], "above"),
    (["--registers", "4"], "--registers 4"),
    ([], None),
])
def test_refusals(tmp_path, argv, match):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 2, 800, seed=2)
    name = str(tmp_path / "run")
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


@pytest.mark.parametrize("lines,match", [
    (["g0.fasta\ta", "g1.fasta\ta", "g2.fasta\ta"], "at least 2 groups, got 1"),
    (["g0.fasta\ta", "g1.fasta\tb"], "does not name these inputs.*g2.fasta"),
    (["g0.fasta\ta", "g1.fasta\tb", "g2.fasta\tb", "g9.fasta\tc"], "not inputs.*g9.fasta"),
    (["g0.fasta\ta", "g1.fasta\tb", "g2.fasta\tb", "g0.fasta\tc"], "g0.fasta is named twice"),
    (["g0.fasta a", "g1.fasta\tb", "g2.fasta\tb"], "expected `basename<TAB>label`"),
])
def test_groups_refusals(tmp_path, lines, match):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 3, 800, seed=2)
    groups = tmp_path / "groups.tsv"
    groups.write_text("\n".join(lines) + "\n")
    with pytest.raises(RuntimeError, match=match):
        _run(["-d", data, "--groups", str(groups), "--name", str(tmp_path / "run")])
    assert not os.path.exists(str(tmp_path / "run"))


def test_groups_are_numbered_by_first_appearance(tmp_path):
    path = tmp_path / "g.tsv"
    path.write_text("c.fa\tone\n\na.fa\ttwo\nb.fa\tone\nd.fa\tthree\n")
    assert leaveout.parse_groups(str(path), ["a.fa", "b.fa", "c.fa", "d.fa"]) == ([0, 1, 1, 2], ["two", "one", "three"])


def test_one_genome_is_refused(tmp_path):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 1, 800, seed=2)
    with pytest.raises(RuntimeError, match="at least 2 groups, got 1"):
        _run(["-d", data, "--name", str(tmp_path / "run")])


def test_duplicate_names_are_refused(tmp_path):
    from tests.util import make_dataset
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


@pytest.mark.parametrize("tool", ["dashing", "kmc"])
def test_two_ranks_write_what_one_writes(tmp_path, tool):
    import torch.multiprocessing as mp
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 5, 1200, seed=6)
    names = ["g%d.fasta" % i for i in range(5)]
    groups = _groups_file(tmp_path, names, ["p", "q", "p", "r", "q"])
    common = ["-d", data, "--tool", tool, "--mink", "3", "--maxk", "8", "--registers", "10", "--groups", groups]
    two, one = str(tmp_path / "two"), str(tmp_path / "one")
    mp.spawn(_rank_worker, args=(2, _free_port(), common + ["--name", two]), nprocs=2, join=True)
    _run(common + ["--name", one])
    for fn in ("union.tsv", "without.tsv", "delta.tsv", "collection.tsv"):
        assert open(os.path.join(two, fn)).read() == open(os.path.join(one, fn)).read(), fn


# ---------------------------------------------------------------- ABI
def test_entry_is_declared():
    from dandd_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    assert re.search(r"DD_API\s+int\s+dd_leave_out_hist\s*\(", header)
    assert re.search(r"DD_API\s+size_t\s+dd_leave_out_workspace_bytes\s*\(", header)
    assert len(_lib.SIGNATURES["dd_leave_out_hist"][1]) == 12 and len(_lib.SIGNATURES["dd_leave_out_workspace_bytes"][1]) == 2
    integration = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert re.search(r"\| `dd_leave_out_workspace_bytes`, `dd_leave_out_hist` \|.*find_delta_delta", integration)
    assert _lib.ABI_VERSION == 2


def test_entry_is_exported_and_checks_arguments():
    """Arguments refused before any CUDA call (these run without a device)."""
    import subprocess
    from dandd_b200 import build, _lib
    build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "dandd_b200", "libdandd_b200.so")], text=True)
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    assert {"dd_leave_out_hist", "dd_leave_out_workspace_bytes"} <= exported
    lib = _lib.load()
    ws = lib.dd_leave_out_workspace_bytes(3, 2)
    assert ws == 2 * 64 * 4 + 3 * 8 and lib.dd_leave_out_workspace_bytes(0, 2) == 0
    before = lib.dd_kernel_launches()
    R, G, H, W = 1 << 20, 1 << 21, 1 << 22, 1 << 23          # (never dereferenced: every call below is refused)

    def call(regs=R, n=3, nk=2, p=10, group=G, n_groups=2, b=0, e=1024, hist=H, wsp=W, wsb=ws):
        return lib.dd_leave_out_hist(regs, n, nk, p, group, n_groups, b, e, hist, wsp, wsb, None)

    assert call(regs=None) == -1 and call(group=None) == -1 and call(hist=None) == -1 and call(wsp=None) == -1
    assert call(p=4) == -1 and call(p=27) == -1
    assert call(nk=0) == -1 and call(nk=65536) == -1
    assert call(n_groups=0) == -1 and call(n_groups=4) == -1
    assert b"n_groups" in lib.dd_last_error()
    assert call(n=70000, n_groups=65536) == -1
    assert call(nk=65535, n=40000, n_groups=40000) == -1 and b"too many" in lib.dd_last_error()
    assert call(b=8) == -1 and call(e=1000) == -1 and call(e=1040) == -1 and call(b=32, e=16) == -1
    assert b"register range" in lib.dd_last_error()
    assert call(regs=R + 8) == -1
    assert call(wsb=ws - 1) == -3
    assert lib.dd_kernel_launches() == before
