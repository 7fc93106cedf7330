"""The exact sharing spectrum and the all-orderings mean growth curve (dandd_b200/helpers/spectrum.py) on the CPU: the
closed forms against brute force and exact rationals; `growth.tsv` against `dandd progressive --exact --ksweep` over
all n! orderings through the real store; the integer identities of the spectrum; the command line's refusals and two
gloo ranks; the ABI entry.  The store runs on the oracle-backed engine double."""
import csv
import itertools
import math
import os
import pickle
import random
import re
import socket
from fractions import Fraction

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from dandd_b200.helpers import spectrum
from tests.fake_engine import FakeEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read_tsv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


# ---------------------------------------------------------------- closed forms
@pytest.mark.parametrize("n", range(1, 9))
def test_closed_forms_equal_brute_force(n):
    """Random k-mer holder sets for a random spectrum; the mean union and intersection over every m-subset in exact
    rationals."""
    rng = random.Random(n)
    hist = [rng.randint(0, 6) for _ in range(n)]
    hist[rng.randrange(n)] += 1
    holders = [frozenset(rng.sample(range(n), c)) for c in range(1, n + 1) for _ in range(hist[c - 1])]
    card, core = spectrum.mean_growth(hist)
    for m in range(1, n + 1):
        subsets = [frozenset(s) for s in itertools.combinations(range(n), m)]
        want_card = Fraction(sum(sum(1 for h in holders if h & s) for s in subsets), len(subsets))
        want_core = Fraction(sum(sum(1 for h in holders if s <= h) for s in subsets), len(subsets))
        assert card[m - 1] == pytest.approx(float(want_card), rel=1e-13, abs=1e-13)
        assert core[m - 1] == pytest.approx(float(want_core), rel=1e-13, abs=1e-13)


def test_closed_forms_at_2000_genomes():
    n = 2000
    rng = np.random.default_rng(5)
    hist = rng.integers(1, 10 ** 7, n).tolist()
    hist[0] *= 50                                             # many private k-mers: the small-m union is a small share
    card, core = spectrum.mean_growth(hist)
    for m in [1, 2, 3, 17, 250, 999, 1000, 1001, 1500, 1998, 1999, 2000]:
        total = math.comb(n, m)
        want_card = Fraction(sum(h * (total - math.comb(n - c, m)) for c, h in enumerate(hist, start=1)), total)
        want_core = Fraction(sum(h * math.comb(c, m) for c, h in enumerate(hist, start=1)), total)
        assert abs(Fraction(card[m - 1]) - want_card) <= want_card * Fraction(1, 10 ** 12), m
        assert abs(Fraction(core[m - 1]) - want_core) <= want_core * Fraction(1, 10 ** 12), m


def test_delta_of_the_mean_curve_takes_the_first_k_on_a_tie():
    delta, k = spectrum.delta_of_mean([2, 3, 4], np.array([[2.0, 8.0], [3.0, 12.0], [4.0, 10.0]]))
    assert delta.tolist() == [1.0, 4.0] and k.tolist() == [2, 2]           # 8 / 2 == 12 / 3: k = 2 wins


# ---------------------------------------------------------------- against progressive over all n! orderings
def _spectrum_run(tmp, argv):
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    try:
        return spectrum.go(argv), st
    finally:
        ddstore.set_store(None)


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("ngen", [4, 5])
def test_growth_equals_the_mean_over_all_orderings(tmp_path, ngen, canon):
    """`dandd tree --exact`, then `dandd progressive --ksweep -r <all n! orderings>` on that tree: the mean of `card` per
    (ngen, kval) in summary.csv is growth.tsv's mean_card."""
    from tests.host_harness import read_csv, run_dandd
    from tests.util import make_dataset
    tmp = str(tmp_path)
    data = os.path.join(tmp, "data")
    make_dataset(data, ngen, 2500, seed=31)
    lo, hi = 3, 9
    flags = [] if canon else ["--no-canon"]
    orderings = os.path.join(tmp, "all.pickle")
    with open(orderings, "wb") as fh:
        pickle.dump(set(itertools.permutations(range(ngen))), fh)
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    try:
        random.seed(3)
        run_dandd(["tree", "-d", data, "-s", "ex", "-o", os.path.join(tmp, "out"), "--exact"] + flags)
        run_dandd(["progressive", "-d", os.path.join(tmp, "out", "ex_%d_kmc_dtree.pickle" % ngen), "-o",
                   os.path.join(tmp, "out"), "--ksweep", "--mink", str(lo), "--maxk", str(hi),
                   "-r", orderings, "-n", str(math.factorial(ngen))])
    finally:
        ddstore.set_store(None)
    summary = [f for f in os.listdir(os.path.join(tmp, "out")) if f.endswith("summary.csv")]
    assert len(summary) == 1
    sums, counts = {}, {}
    for row in read_csv(os.path.join(tmp, "out", summary[0])):
        key = (int(row["ngen"]), int(row["kval"]))
        sums[key] = sums.get(key, 0.0) + float(row["card"])
        counts[key] = counts.get(key, 0) + 1
    assert set(counts.values()) == {math.factorial(ngen)}
    name = os.path.join(tmp, "spec")
    _spectrum_run(tmp, ["-d", data, "--mink", str(lo), "--maxk", str(hi), "--name", name] + flags)
    growth = _read_tsv(os.path.join(name, "growth.tsv"))
    assert len(growth) == (hi - lo + 1) * ngen
    for row in growth:
        key = (int(row["ngen"]), int(row["k"]))
        assert float(row["mean_card"]) == pytest.approx(sums[key] / counts[key], rel=1e-12)
        assert float(row["mean_delta_pos"]) == float(row["mean_card"]) / key[1]
    delta = _read_tsv(os.path.join(name, "delta.tsv"))
    assert [int(r["ngen"]) for r in delta] == list(range(1, ngen + 1))
    for r in delta:
        cands = [(float(g["mean_delta_pos"]), int(g["k"])) for g in growth if int(g["ngen"]) == int(r["ngen"])]
        best = max(c[0] for c in cands)
        assert float(r["delta"]) == best and int(r["k"]) == min(k for d, k in cands if d == best)


# ---------------------------------------------------------------- integer identities
@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
def test_integer_identities(tmp_path, canon):
    """At every k: sum c h_c = sum of the singles; sum h_c = |union|; h_n = |intersection|; private_g = |A_g| -
    |A_g n union of the others|.  Also an identical pair and a genome without k-mers."""
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    fastas = make_dataset(data, 4, 2000, seed=12)
    with open(fastas[0], "rb") as src, open(os.path.join(data, "h_copy.fasta"), "wb") as dst:
        dst.write(src.read())
    with open(os.path.join(data, "z_empty.fasta"), "wb") as fh:
        fh.write(b">nothing\nACGNNN\n")
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    files = sorted(os.path.join(data, f) for f in os.listdir(data))
    ks = [1, 2, 5, 9, 14]
    hist, singles, priv = st.exact_spectrum(files, ks, canon)
    assert hist.shape == singles.shape == priv.shape == (len(ks), len(files)) and hist.dtype == np.int64
    assert st.stats["exact_calls"] == len(ks) and st.engine.calls["exact_spectrum"] == len(ks)
    sets_at = {k: [set(orc.kmers(orc.fasta_symbols(_read_fasta(f)), k, canon).tolist()) for f in files] for k in ks}
    for c, k in enumerate(ks):
        sets = sets_at[k]
        n = len(sets)
        assert int((np.arange(1, n + 1) * hist[c]).sum()) == int(singles[c].sum())
        assert int(hist[c].sum()) == st.exact_count(files, k, canon) == len(set().union(*sets))
        assert hist[c, n - 1] == len(set.intersection(*sets))
        for g in range(n):
            others = set().union(*(sets[j] for j in range(n) if j != g))
            assert priv[c, g] == singles[c, g] - len(sets[g] & others) == len(sets[g] - others)
        copy = files.index(os.path.join(data, "h_copy.fasta"))
        assert priv[c, 0] == priv[c, copy] == 0
    assert singles[ks.index(5):, -1].tolist() == [0, 0, 0] and singles[0, -1] > 0     # "ACG": k-mers up to k = 3 only


# ---------------------------------------------------------------- command line
def test_outputs(tmp_path):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 3, 1500, seed=8)
    listing = tmp_path / "list.txt"
    listing.write_text("".join(os.path.join(data, "g%d.fasta" % g) + "\n" for g in (2, 0)))
    name = str(tmp_path / "run")
    (hist, singles, priv), st = _spectrum_run(str(tmp_path), ["-f", str(listing), "--mink", "4", "--maxk", "6", "--name", name])
    assert sorted(os.listdir(name)) == ["delta.tsv", "genomes.tsv", "growth.tsv", "spectrum.tsv"]
    spec = _read_tsv(os.path.join(name, "spectrum.tsv"))
    assert [(int(r["k"]), int(r["genomes"])) for r in spec] == [(k, c) for k in (4, 5, 6) for c in (1, 2)]
    assert [int(r["kmers"]) for r in spec] == hist.reshape(-1).tolist()
    gen = _read_tsv(os.path.join(name, "genomes.tsv"))
    assert [r["name"] for r in gen] == ["g0.fasta", "g2.fasta"] * 3                # list_fastas sorts the inputs
    assert [int(r["distinct"]) for r in gen] == singles.reshape(-1).tolist()
    assert [int(r["private"]) for r in gen] == priv.reshape(-1).tolist()
    growth = _read_tsv(os.path.join(name, "growth.tsv"))
    for r in growth:
        v = float(r["mean_card"])
        assert repr(v) == r["mean_card"]
    at2 = [float(r["mean_card"]) for r in growth if r["ngen"] == "2"]
    assert at2 == [float(h.sum()) for h in hist]                                     # all genomes: the whole union
    core2 = [float(r["mean_core"]) for r in growth if r["ngen"] == "2"]
    assert core2 == [float(h[-1]) for h in hist]


@pytest.mark.parametrize("argv,match", [
    (["--mink", "0"], "--mink 0 is outside"),
    (["--maxk", "257"], "--maxk 257 is outside"),
    (["--mink", "9", "--maxk", "5"], "above"),
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
            _spectrum_run(str(tmp_path), ["-d", data, "--name", name])
        with pytest.raises(RuntimeError, match="-d DATADIR or -f LIST"):
            _spectrum_run(str(tmp_path), ["--name", str(tmp_path / "other")])
        return
    with pytest.raises(RuntimeError, match=match):
        _spectrum_run(str(tmp_path), ["-d", data, "--name", name] + argv)
    assert not os.path.exists(name)


def test_duplicate_names_are_refused(tmp_path):
    from tests.util import make_dataset
    a = make_dataset(str(tmp_path / "a"), 2, 800, seed=2)
    b = make_dataset(str(tmp_path / "b"), 1, 800, seed=3)
    listing = tmp_path / "list.txt"
    listing.write_text("\n".join(a + b) + "\n")
    with pytest.raises(RuntimeError, match="distinct.*g0.fasta"):
        _spectrum_run(str(tmp_path), ["-f", str(listing), "--name", str(tmp_path / "run")])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_worker(rank, world, port, data, name):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    _spectrum_run(os.path.dirname(name), ["-d", data, "--mink", "3", "--maxk", "8", "--no-canon", "--name", name])


def test_two_ranks_write_what_one_writes(tmp_path):
    import torch.multiprocessing as mp
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 4, 1500, seed=6)
    two, one = str(tmp_path / "two"), str(tmp_path / "one")
    mp.spawn(_rank_worker, args=(2, _free_port(), data, two), nprocs=2, join=True)
    _spectrum_run(str(tmp_path), ["-d", data, "--mink", "3", "--maxk", "8", "--no-canon", "--name", one])
    for fn in ("spectrum.tsv", "genomes.tsv", "growth.tsv", "delta.tsv"):
        assert open(os.path.join(two, fn)).read() == open(os.path.join(one, fn)).read(), fn


# ---------------------------------------------------------------- ABI
def test_entry_is_declared():
    from dandd_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    assert re.search(r"DD_API\s+int\s+dd_exact_occupancy_hist\s*\(", header)
    assert len(_lib.SIGNATURES["dd_exact_occupancy_hist"][1]) == 10
    assert "`dd_exact_occupancy_hist`" in open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert _lib.ABI_VERSION == 2


def test_entry_is_exported_and_checks_arguments():
    import subprocess
    from dandd_b200 import build, _lib
    build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "dandd_b200", "libdandd_b200.so")], text=True)
    assert "dd_exact_occupancy_hist" in {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    lib = _lib.load()
    need = lib.dd_exact_pairs_workspace_bytes(21, 1024, 4096, 2)
    before = lib.dd_kernel_launches()
    assert lib.dd_exact_occupancy_hist(None, need, 21, 1024, 4096, 2, 2, 1 << 20, None, None) == -1
    assert lib.dd_exact_occupancy_hist(1 << 20, need, 21, 1024, 4096, 2, 2, None, 1 << 20, None) == -1
    assert lib.dd_exact_occupancy_hist(1 << 20, need, 21, 1024, 4096, 2, 0, 1 << 20, None, None) == -1
    assert b"n_genomes" in lib.dd_last_error()
    assert lib.dd_exact_occupancy_hist(1 << 20, need, 21, 1024, 4096, 2, 1 << 32, 1 << 20, None, None) == -1
    assert lib.dd_exact_occupancy_hist(1 << 20, need, 0, 1024, 4096, 2, 2, 1 << 20, None, None) == -1
    assert lib.dd_exact_occupancy_hist(1 << 20, need - 1, 21, 1024, 4096, 2, 2, 1 << 20, None, None) == -3
    assert lib.dd_kernel_launches() == before
