"""Live differential runs against the UNMODIFIED reference Python, on randomly drawn scenarios.

tests/golden/reference_runs.json pins twenty fixed scenarios; here the same comparison is made on
inputs and option combinations drawn from a seeded generator, so that host-logic parity (naming,
caching, the k hill-climb, tree shapes, progressive and KIJ tables) does not rest on the fixtures
alone.  The reference runs with the oracle-backed dashing/kmc/parallel stand-ins first on PATH
(oracle/shims), the drop-in layer with the oracle-backed store double -- so both sides see the same
arithmetic and any difference is host logic.

Opt-in: the original project is not part of this repository, so these run only where DANDD_REFERENCE
names a checkout of it (tests/util.py) and are skipped everywhere else.  CPU only."""
import importlib.util
import os
import random

import pytest

from dandd_b200 import store as ddstore
from tests.host_harness import assert_tree_matches, close, collect_tree, read_csv, run_dandd
from tests.oracle_store import OracleStore
from tests.util import make_dataset, reference_path

REF = reference_path("lib")
pytestmark = pytest.mark.skipif(not (REF and os.path.isdir(REF)),
                                reason="opt-in: runs the original DandD project, which is not part of this repository (set DANDD_REFERENCE)")


@pytest.fixture(scope="module")
def golden():
    """tests/golden/make_reference_golden.py as a module (run_ref, collect_tree) + the shims on a PATH dir."""
    here = os.path.dirname(os.path.abspath(__file__))
    spec = importlib.util.spec_from_file_location("make_reference_golden", os.path.join(here, "golden", "make_reference_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture()
def oracle_store():
    st = OracleStore()
    ddstore.set_store(st)
    yield st
    ddstore.set_store(None)


def _draw(seed):
    rng = random.Random(seed)
    n = rng.randint(3, 8)
    case = {"n": n, "length": rng.choice([3000, 8000, 15000]), "seed": 100 + seed, "kstart": rng.randint(9, 15),
            "sub": rng.choice([0.01, 0.05, 0.15]), "registers": rng.choice([10, 12, 14]), "canon": rng.random() < 0.75,
            "nchildren": rng.choice([None, None, 2, 3, 4]), "sweep": None}
    if rng.random() < 0.5:
        lo = rng.randint(6, 12)
        case["sweep"] = (lo, lo + rng.randint(2, 5))
    return case


def _tree_argv(case, data, out, tag):
    argv = ["tree", "-d", data, "-s", tag, "-k", str(case["kstart"]), "-o", out, "-r", str(case["registers"])]
    if not case["canon"]:
        argv.append("-C")
    if case["nchildren"]:
        argv += ["-n", str(case["nchildren"])]
    if case["sweep"]:
        argv += ["--ksweep", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])]
    return argv


def _both(golden, bindir, ref_argv, our_argv, exact=False):
    """Run one command on both sides.  True if both succeeded; False if the reference failed and the
    drop-in failed with the same exception (error behaviour is part of the interface: several option
    combinations crash the reference as shipped, e.g. n-ary shapes whose cursor runs off the node
    list, or `kij` hill-climbing out of the k range a sweep-built tree holds)."""
    import subprocess
    try:
        golden.run_ref(bindir, ref_argv, exact=exact)
    except subprocess.CalledProcessError as failed:
        last = failed.stderr.decode(errors="replace").strip().split("\n")[-1]
        with pytest.raises(Exception) as ours_err:
            run_dandd(our_argv)
        assert type(ours_err.value).__name__ in last, (last, repr(ours_err.value))
        return False
    run_dandd(our_argv)
    return True


@pytest.mark.parametrize("seed", range(int(os.environ.get("DANDD_LIVE_SEEDS", "2"))))
def test_random_tree_progressive_kij_match_the_reference(tmp_path, golden, oracle_store, seed):
    from oracle import pyoracle
    case = _draw(seed)
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    make_dataset(data, case["n"], case["length"], seed=case["seed"], sub=case["sub"])
    tag = f"r{seed}"
    prefix = f"{tag}_{case['n']}_dashing"
    ref_out, our_out = str(tmp_path / "ref"), str(tmp_path / "ours")
    # ---- tree
    if not _both(golden, bindir, _tree_argv(case, data, ref_out, tag), _tree_argv(case, data, our_out, tag)):
        print(f"LIVE seed {seed}: both fail at tree {case}")
        return
    want = golden.collect_tree(ref_out, prefix, os.path.join(ref_out, "sketchdb"), "dashing")
    ours = collect_tree(our_out, prefix, os.path.join(our_out, "sketchdb"), "dashing")
    assert_tree_matches(ours, want)
    # ---- progressive, identity ordering (the reference draws random orderings for -n > 1)
    sweep = ["--ksweep", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])] if case["sweep"] else []
    prog = lambda out: ["progressive", "-d", os.path.join(out, prefix + "_dtree.pickle"), "-n", "1", "-o", out] + sweep   # noqa: E731
    if not _both(golden, bindir, prog(ref_out), prog(our_out)):
        print(f"LIVE seed {seed}: both fail at progressive {case}")
        return
    name = f"{tag}_progu1_{case['n']}_dashing"
    def prog_rows(path):      # with --ksweep the reference leaves `delta` empty (SubSpider.delta stays None)
        from tests.host_harness import norm_fastas
        return [{"ngen": int(r["ngen"]), "kval": int(r["kval"]), "delta": float(r["delta"]) if r["delta"] else None,
                 "fastas": norm_fastas(r["fastas"], ",")} for r in read_csv(path)]
    rows_ref, rows_our = prog_rows(os.path.join(ref_out, name + ".csv")), prog_rows(os.path.join(our_out, name + ".csv"))
    assert [(r["ngen"], r["kval"], r["fastas"]) for r in rows_our] == [(r["ngen"], r["kval"], r["fastas"]) for r in rows_ref]
    assert all((a["delta"] is None and b["delta"] is None) or close(a["delta"], b["delta"]) for a, b in zip(rows_our, rows_ref))
    summ_ref = read_csv(os.path.join(ref_out, name + "summary.csv"))
    summ_our = read_csv(os.path.join(our_out, name + "summary.csv"))
    key = lambda r: (int(r["ngen"]), int(r["kval"]), r["title"])     # noqa: E731
    assert sorted(map(key, summ_our)) == sorted(map(key, summ_ref))
    cards_ref = {key(r): float(r["card"]) for r in summ_ref}
    assert all(close(float(r["card"]), cards_ref[key(r)]) for r in summ_our)
    # ---- kij (+ per-k Jaccard when a k range is known), batched pair table on our side
    jac = ["--jaccard", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])] if case["sweep"] else []
    kij = lambda out: ["kij", "-d", os.path.join(out, prefix + "_dtree.pickle"), "-o", out] + jac   # noqa: E731
    if not _both(golden, bindir, kij(ref_out), kij(our_out)):
        print(f"LIVE seed {seed}: both fail at kij {case}")
        return
    kij_ref = read_csv(os.path.join(ref_out, prefix + ".kij.csv"))
    kij_our = read_csv(os.path.join(our_out, prefix + ".kij.csv"))
    pair = lambda r: (r["Atitle"], r["Btitle"])     # noqa: E731
    assert sorted(map(pair, kij_our)) == sorted(map(pair, kij_ref)) and len(kij_ref) == case["n"] * (case["n"] - 1) // 2
    by_pair = {pair(r): r for r in kij_ref}
    for r in kij_our:
        g = by_pair[pair(r)]
        assert (int(r["Ak"]), int(r["Bk"]), int(r["ABk"])) == (int(g["Ak"]), int(g["Bk"]), int(g["ABk"])), pair(r)
        for col in ("Adelta", "Bdelta", "ABdelta"):
            assert close(float(r[col]), float(g[col])), (pair(r), col)
        assert float(r["KIJ"]) == pytest.approx(float(g["KIJ"]), rel=1e-6, abs=1e-6)
    if jac:
        j_ref = {(r["Atitle"], r["Btitle"], int(r["kval"])): r for r in read_csv(os.path.join(ref_out, prefix + ".j.csv"))}
        j_our = read_csv(os.path.join(our_out, prefix + ".j.csv"))
        assert sorted((r["Atitle"], r["Btitle"], int(r["kval"])) for r in j_our) == sorted(j_ref)
        for r in j_our:
            g = j_ref[(r["Atitle"], r["Btitle"], int(r["kval"]))]
            assert close(float(r["ABcard"]), float(g["ABcard"]))
            assert float(r["jaccard"]) == pytest.approx(float(g["jaccard"]), rel=1e-6, abs=1e-6)
    # ---- what the whole session left in the sketch database
    want_db = golden.collect_tree(ref_out, prefix, os.path.join(ref_out, "sketchdb"), "dashing")
    ours_db = collect_tree(our_out, prefix, os.path.join(our_out, "sketchdb"), "dashing")
    assert ours_db["files"] == want_db["files"]
    assert sorted(ours_db["cardkey"]) == sorted(want_db["cardkey"])
    assert all(close(ours_db["cardkey"][k], v) for k, v in want_db["cardkey"].items())
    assert ours_db["fastahex"] == want_db["fastahex"] and ours_db["sketchinfo"] == want_db["sketchinfo"]
    print(f"LIVE seed {seed}: tree + progressive + kij compared {case}")


def _draw_options(seed):
    rng = random.Random(1000 + seed)
    n = rng.randint(3, 6)
    case = {"n": n, "length": rng.choice([2000, 5000]), "seed": 300 + seed, "kstart": rng.randint(10, 14),
            "exact": rng.random() < 0.5, "sweep": None, "step": rng.choice([1, 1, 2]),
            "orderings": {tuple(range(n))} | {tuple(rng.sample(range(n), n)) for _ in range(rng.randint(1, 3))},
            "subset": sorted(rng.sample(range(n), rng.randint(2, n - 1))), "safe": rng.random() < 0.5, "fast": rng.random() < 0.3}
    if rng.random() < 0.6:
        lo = rng.randint(9, 12)
        case["sweep"] = (lo, lo + rng.randint(2, 4))
    return case


@pytest.mark.parametrize("seed", range(int(os.environ.get("DANDD_LIVE_SEEDS", "2"))))
def test_random_exact_orderings_subsets_match_the_reference(tmp_path, golden, oracle_store, seed):
    """More of the option space, same method: --exact (with the one-method run-time patch of the reference that
    tests/golden/make_reference_golden.py documents), progressive over an orderings file with --step,
    and a tree over a file-list subset with --safe / --fast."""
    import pickle
    from oracle import pyoracle
    case = _draw_options(seed)
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    files = make_dataset(data, case["n"], case["length"], seed=case["seed"], sub=0.05)
    tool = "kmc" if case["exact"] else "dashing"
    tag = f"x{seed}"
    prefix = f"{tag}_{case['n']}_{tool}"
    ref_out, our_out = str(tmp_path / "ref"), str(tmp_path / "ours")
    sweep = ["--ksweep", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])] if case["sweep"] else []
    extra = ["--exact"] if case["exact"] else ["-r", "12"]

    def both(ref_argv, our_argv):
        import subprocess
        try:
            golden.run_ref(bindir, ref_argv, exact=case["exact"])
        except subprocess.CalledProcessError as failed:
            last = failed.stderr.decode(errors="replace").strip().split("\n")[-1]
            with pytest.raises(Exception) as ours_err:
                run_dandd(our_argv)
            assert type(ours_err.value).__name__ in last, (last, repr(ours_err.value))
            return False
        run_dandd(our_argv)
        return True

    tree = lambda out: ["tree", "-d", data, "-s", tag, "-k", str(case["kstart"]), "-o", out] + extra + sweep   # noqa: E731
    if not both(tree(ref_out), tree(our_out)):
        print(f"LIVE options seed {seed}: both fail at tree {case}")
        return
    assert_tree_matches(collect_tree(our_out, prefix, os.path.join(our_out, "sketchdb"), tool),
                        golden.collect_tree(ref_out, prefix, os.path.join(ref_out, "sketchdb"), tool), exact=case["exact"])
    # ---- progressive over an orderings file (+ --step): cells keyed by member set, the ordering numbers follow
    #      list(set) order, which is process-specific
    ofile = str(tmp_path / "orderings.pickle")
    with open(ofile, "wb") as fh:
        pickle.dump(case["orderings"], fh)
    prog = lambda out: (["progressive", "-d", os.path.join(out, prefix + "_dtree.pickle"), "-r", ofile, "-s", tag + "o", "-o", out,   # noqa: E731
                         "--step", str(case["step"])] + sweep)
    if both(prog(ref_out), prog(our_out)):
        name = f"{tag}o_progu0_{case['n']}_{tool}"
        cells = {}
        for side, out in (("ref", ref_out), ("ours", our_out)):
            rows = read_csv(os.path.join(out, name + "summary.csv"))
            cells[side] = sorted({(r["title"], int(r["kval"]), float(r["card"])) for r in rows})
        assert [c[:2] for c in cells["ours"]] == [c[:2] for c in cells["ref"]]
        assert all((a[2] == b[2]) if case["exact"] else close(a[2], b[2]) for a, b in zip(cells["ours"], cells["ref"]))
        main = {}
        for side, out in (("ref", ref_out), ("ours", our_out)):
            main[side] = sorted((int(r["ngen"]), r["kval"], r["delta"][:12], r["fastas"].count(",")) for r in read_csv(os.path.join(out, name + ".csv")))
        assert [(m[0], m[1], m[3]) for m in main["ours"]] == [(m[0], m[1], m[3]) for m in main["ref"]]
    else:
        print(f"LIVE options seed {seed}: both fail at progressive {case}")
    # ---- a tree over a subset given as a file list, into the SAME sketch database (cached leaves are reused)
    flist = str(tmp_path / "flist.txt")
    with open(flist, "w") as fh:
        fh.write("\n".join(files[i] for i in case["subset"]) + "\n")
    opts = (["--safe"] if case["safe"] else []) + (["--fast"] if case["fast"] else [])
    sub = lambda out: (["tree", "-f", flist, "-s", tag + "s", "-k", str(case["kstart"]), "-o", out, "--sketchdir",   # noqa: E731
                        os.path.join(out, "sketchdb")] + extra + sweep + opts)
    if not both(sub(ref_out), sub(our_out)):
        print(f"LIVE options seed {seed}: both fail at subset tree {case}")
        return
    sub_prefix = f"{tag}s_{len(case['subset'])}_{tool}"
    rows = {}
    for side, out in (("ref", ref_out), ("ours", our_out)):
        rows[side] = [(r["title"], int(r["ngen"]), int(r["k"]), float(r["card"]), float(r["delta"]))
                      for r in read_csv(os.path.join(out, sub_prefix + "_deltas.csv"))]
        outputs = sorted(f for f in os.listdir(out) if f.startswith(tag + "s_"))
        rows[side + "_outputs"] = outputs
    assert [r[:3] for r in rows["ours"]] == [r[:3] for r in rows["ref"]]
    assert all(close(a[3], b[3]) and close(a[4], b[4]) for a, b in zip(rows["ours"], rows["ref"]))
    assert rows["ours_outputs"] == rows["ref_outputs"]                  # --fast writes the deltas table only
    want_db = golden.collect_tree(ref_out, prefix, os.path.join(ref_out, "sketchdb"), tool)
    ours_db = collect_tree(our_out, prefix, os.path.join(our_out, "sketchdb"), tool)
    assert ours_db["files"] == want_db["files"]
    if not case["fast"]:          # (--fast skips saving the caches)
        assert sorted(ours_db["cardkey"]) == sorted(want_db["cardkey"])
        assert ours_db["fastahex"] == want_db["fastahex"] and ours_db["sketchinfo"] == want_db["sketchinfo"]
    print(f"LIVE options seed {seed}: tree + orderings + subset tree compared {case}")


def _draw_lowmem(seed):
    rng = random.Random(5000 + seed)
    n = rng.randint(4, 6)
    case = {"n": n, "length": rng.choice([3000, 6000]), "seed": 700 + seed, "kstart": rng.randint(10, 14),
            "registers": rng.choice([10, 12]), "nchildren": rng.choice([None, 2, 3]), "sweep": None,
            "label": rng.choice(["", "lab"]), "subset": sorted(rng.sample(range(n), rng.randint(3, n - 1))),
            "jaccard": rng.random() < 0.5, "drop": rng.choice(["unions", "all-unions-and-a-leaf-k"])}
    if rng.random() < 0.6:
        lo = rng.randint(9, 12)
        case["sweep"] = (lo, lo + rng.randint(2, 4))
    return case


@pytest.mark.parametrize("seed", range(int(os.environ.get("DANDD_LIVE_SEEDS", "2"))))
def test_random_lowmem_labels_and_subsets_match_the_reference(tmp_path, golden, oracle_store, seed):
    """`--lowmem` re-runs over a sketch database whose multi-FASTA sketches were deleted (cardinalities on
    record are trusted, anything else is rebuilt), output labels (-l), and `kij` / `progressive` over a
    file-list subset with --afproject -- same method as above: both sides, same inputs, same outputs
    (or the same failure)."""
    import pickle
    import shutil
    from oracle import pyoracle
    case = _draw_lowmem(seed)
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    files = make_dataset(data, case["n"], case["length"], seed=case["seed"], sub=0.05)
    tag = f"m{seed}"
    label = ("_" + case["label"]) if case["label"] else ""
    prefix = f"{tag}{label}_{case['n']}_dashing"
    ref_out, our_out = str(tmp_path / "ref"), str(tmp_path / "ours")
    sweep = ["--ksweep", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])] if case["sweep"] else []

    def tree(out, more=()):
        argv = ["tree", "-d", data, "-s", tag, "-k", str(case["kstart"]), "-o", out, "-r", str(case["registers"])] + sweep
        if case["label"]:
            argv += ["-l", case["label"]]
        if case["nchildren"]:
            argv += ["-n", str(case["nchildren"])]
        return argv + list(more)

    def compare(stage):
        want = golden.collect_tree(ref_out, prefix, os.path.join(ref_out, "sketchdb"), "dashing")
        ours = collect_tree(our_out, prefix, os.path.join(our_out, "sketchdb"), "dashing")
        assert_tree_matches(ours, want)
        return want

    if not _both(golden, bindir, tree(ref_out), tree(our_out)):
        print(f"LIVE lowmem seed {seed}: both fail at tree {case}")
        return
    first = compare("tree")
    # ---- drop sketches from BOTH databases (the same relative files), then re-run with --lowmem
    doomed = [f for f in first["files"] if not f.startswith("ngen1" + os.sep)]
    if case["drop"] != "unions":
        doomed += [f for f in first["files"] if f.startswith("ngen1" + os.sep)][:1]
    for out in (ref_out, our_out):
        for rel_path in doomed:
            os.remove(os.path.join(out, "sketchdb", rel_path))
    oracle_store._regs.clear()                                   # (a new process would not hold them either)
    if not _both(golden, bindir, tree(ref_out, ["--lowmem"]), tree(our_out, ["--lowmem"])):
        print(f"LIVE lowmem seed {seed}: both fail at the --lowmem re-run {case}")
        return
    again = compare("lowmem re-run")                             # same tables; the same files (not) rebuilt on both sides
    assert len(again["files"]) <= len(first["files"])
    # ---- the ONE deliberate difference in this area.  Under --lowmem the reference answers 0 for the cardinality of
    #      any sketch that is not yet in its table -- also one it has just built (lib/sketch_classes.py:280-284) -- so a
    #      search over NEW sketches sees delta = 0 everywhere, climbs to k = 33 and raises; the flag is carried into
    #      `kij` by the tree pickle.  The drop-in records a cardinality when it creates the sketch.  Pinned here: where
    #      the reference gives up with that error, the drop-in's table equals what BOTH produce from a tree saved
    #      without the flag (next step).
    import subprocess
    kij_plain = lambda out: ["kij", "-d", os.path.join(out, prefix + "_dtree.pickle"), "-o", out, "-s", tag + "low"]   # noqa: E731
    kij_under_lowmem = None
    for out in (ref_out, our_out):                                  # (both databases are put back afterwards)
        shutil.copytree(os.path.join(out, "sketchdb"), os.path.join(out, "sketchdb.before"))
    try:
        golden.run_ref(bindir, kij_plain(ref_out))
    except subprocess.CalledProcessError as failed:
        last = failed.stderr.decode(errors="replace").strip().split("\n")[-1]
        try:
            run_dandd(kij_plain(our_out))
        except Exception as ours_err:  # noqa: BLE001 -- another of the reference's failures (e.g. a sweep-built tree): the same one
            assert type(ours_err).__name__ in last, (last, repr(ours_err))
        else:
            assert "Exploratory k value is too high" in last, last         # the only failure the drop-in does not share
            kij_under_lowmem = read_csv(os.path.join(our_out, f"{tag}low_{case['n']}_dashing.kij.csv"))
    else:
        run_dandd(kij_plain(our_out))
    for out in (ref_out, our_out):
        shutil.rmtree(os.path.join(out, "sketchdb"))
        os.rename(os.path.join(out, "sketchdb.before"), os.path.join(out, "sketchdb"))
    oracle_store._regs.clear()
    if not _both(golden, bindir, tree(ref_out), tree(our_out)):           # no flag: what lowmem skipped is rebuilt, on both sides
        print(f"LIVE lowmem seed {seed}: both fail at the plain re-run {case}")
        return
    compare("plain re-run")
    # ---- kij with --afproject and its own label; then over a subset given as a file list, which the reference
    #      cannot do as shipped (it hands file NAMES to SubSpider, lib/huffman_dandd.py:672-685): same failure
    rng = random.Random(seed)
    order = [files[i] for i in rng.sample(case["subset"], len(case["subset"]))]
    flist = str(tmp_path / "subset.txt")
    with open(flist, "w") as fh:
        fh.write("\n".join(order) + "\n")
    jac = ["--jaccard", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])] if (case["sweep"] and case["jaccard"]) else []
    kij = lambda out, more=(): (["kij", "-d", os.path.join(out, prefix + "_dtree.pickle"), "-o", out, "--afproject"] + jac   # noqa: E731
                                + (["-l", "sub"] if case["label"] else []) + list(more))
    assert not _both(golden, bindir, kij(ref_out, ["-f", flist]), kij(our_out, ["-f", flist]))
    if _both(golden, bindir, kij(ref_out), kij(our_out)):
        # (the kij output prefix is the tag with kij's OWN label, not the tree's: reference dandd_cmd.py:113-116)
        kij_prefix = f"{tag}{'_sub' if case['label'] else ''}_{case['n']}_dashing"
        pair = lambda r: (r["Atitle"], r["Btitle"])              # noqa: E731
        kij_ref = {pair(r): r for r in read_csv(os.path.join(ref_out, kij_prefix + ".kij.csv"))}
        kij_our = read_csv(os.path.join(our_out, kij_prefix + ".kij.csv"))
        k = case["n"]
        assert sorted(map(pair, kij_our)) == sorted(kij_ref) and len(kij_our) == k * (k - 1) // 2
        for r in kij_our:
            g = kij_ref[pair(r)]
            assert (int(r["Ak"]), int(r["Bk"]), int(r["ABk"])) == (int(g["Ak"]), int(g["Bk"]), int(g["ABk"]))
            assert float(r["KIJ"]) == pytest.approx(float(g["KIJ"]), rel=1e-6, abs=1e-6)
        tuples = {}
        for side, out in (("ref", ref_out), ("ours", our_out)):
            with open(os.path.join(out, kij_prefix + "_AFtuples.pickle"), "rb") as fh:
                tuples[side] = sorted((t[0], t[1], t[2], t[3], t[5], t[6], t[7]) for t in pickle.load(fh))
        assert tuples["ours"] == tuples["ref"]
        if kij_under_lowmem is not None:
            cols = ("Atitle", "Btitle", "Ak", "Bk", "ABk", "Adelta", "Bdelta", "ABdelta", "KIJ")
            assert [[r[c] for c in cols] for r in kij_under_lowmem] == [[r[c] for c in cols] for r in kij_our]
    else:
        print(f"LIVE lowmem seed {seed}: both fail at kij {case}")
    # ---- progressive over the file list: without -n / -r there is nothing to order by (same ValueError), with
    #      -n 1 the order of the FILE is the ordering (reference lib/huffman_dandd.py:581-589)
    prog = lambda out, more=(): (["progressive", "-d", os.path.join(out, prefix + "_dtree.pickle"), "-f", flist, "-s", tag + "p",   # noqa: E731
                                  "-o", out] + sweep + list(more))
    assert not _both(golden, bindir, prog(ref_out), prog(our_out))
    if _both(golden, bindir, prog(ref_out, ["-n", "1"]), prog(our_out, ["-n", "1"])):
        name = f"{tag}p_progu1_{case['n']}_dashing"
        from tests.host_harness import norm_fastas
        rows = {side: [(int(r["ngen"]), r["kval"], norm_fastas(r["fastas"], ",")) for r in read_csv(os.path.join(out, name + ".csv"))]
                for side, out in (("ref", ref_out), ("ours", our_out))}
        assert rows["ours"] == rows["ref"] and len(rows["ours"]) >= len(order)
        assert rows["ours"][-1][2] == ",".join(os.path.basename(f) for f in order)        # the file's order, not the sorted one
        cells = {side: sorted((r["title"], int(r["kval"]), float(r["card"])) for r in read_csv(os.path.join(out, name + "summary.csv")))
                 for side, out in (("ref", ref_out), ("ours", our_out))}
        assert [c[:2] for c in cells["ours"]] == [c[:2] for c in cells["ref"]]
        assert all(close(a[2], b[2]) for a, b in zip(cells["ours"], cells["ref"]))
    else:
        print(f"LIVE lowmem seed {seed}: both fail at progressive -n 1 {case}")
    shutil.rmtree(str(tmp_path / "bin"), ignore_errors=True)
    print(f"LIVE lowmem seed {seed}: tree, --lowmem re-run, kij -f --afproject, progressive -f compared {case}")


def _draw_inputs(seed):
    rng = random.Random(9000 + seed)
    n = rng.randint(3, 5)
    case = {"n": n, "length": rng.choice([2500, 5000]), "seed": 900 + seed, "kstart": rng.randint(10, 13),
            "exact": rng.random() < 0.4, "canon": rng.random() < 0.6, "threads": rng.choice([0, 2]),
            "ext": [rng.choice([".fasta", ".fa", ".fa.gz", ".fna.gz", ".fasta.gz"]) for _ in range(n)],
            "crlf": rng.random() < 0.3, "headless": rng.random() < 0.25, "sweep": None, "custom_db": rng.random() < 0.5,
            "nchildren": rng.choice([None, None, 2])}
    if rng.random() < 0.5:
        lo = rng.randint(9, 11)
        case["sweep"] = (lo, lo + rng.randint(2, 3))
    return case


@pytest.mark.parametrize("seed", range(int(os.environ.get("DANDD_LIVE_SEEDS", "2"))))
def test_random_input_formats_exact_kij_and_shared_databases_match_the_reference(tmp_path, golden, oracle_store, seed):
    """Input side of the path: gzip-compressed and plain FASTAs under every extension the reference names, CRLF line
    ends, a file whose records hold no sequence at all; --exact with -C / --nthreads; `kij` in exact mode; a second
    tree (other tag, fewer genomes) into the same --sketchdir.  Same outputs, or the same failure."""
    import gzip
    from oracle import pyoracle
    case = _draw_inputs(seed)
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    files = make_dataset(data, case["n"], case["length"], seed=case["seed"], sub=0.08)
    final = []
    for i, (path, ext) in enumerate(zip(files, case["ext"])):
        with open(path, "rb") as fh:
            text = fh.read()
        if case["crlf"] and i % 2 == 0:
            text = text.replace(b"\n", b"\r\n")
        if case["headless"] and i == case["n"] - 1:        # records without sequence between real ones
            text = b">nothing here\n>nor here\n\n" + text + b">empty at the end\n"
        os.remove(path)
        new = path[:-len(".fasta")] + ext
        with open(new, "wb") as fh:
            fh.write(gzip.compress(text, mtime=0) if ext.endswith(".gz") else text)
        final.append(new)
    tool = "kmc" if case["exact"] else "dashing"
    tag = f"i{seed}"
    prefix = f"{tag}_{case['n']}_{tool}"
    ref_out, our_out = str(tmp_path / "ref"), str(tmp_path / "ours")
    sweep = ["--ksweep", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])] if case["sweep"] else []
    mode = (["--exact"] + (["-e", str(case["threads"])] if case["threads"] else [])) if case["exact"] else ["-r", "10"]
    mode += [] if case["canon"] else ["-C"]
    if case["nchildren"]:
        mode += ["-n", str(case["nchildren"])]
    db = lambda out: os.path.join(out, "shared_db" if case["custom_db"] else "sketchdb")       # noqa: E731
    extra_db = lambda out: ["-c", db(out)] if case["custom_db"] else []                         # noqa: E731

    def both(ref_argv, our_argv):
        import subprocess
        try:
            golden.run_ref(bindir, ref_argv, exact=case["exact"])
        except subprocess.CalledProcessError as failed:
            last = failed.stderr.decode(errors="replace").strip().split("\n")[-1]
            with pytest.raises(Exception) as ours_err:
                run_dandd(our_argv)
            assert type(ours_err.value).__name__ in last, (last, repr(ours_err.value))
            return False
        run_dandd(our_argv)
        return True

    tree = lambda out: ["tree", "-d", data, "-s", tag, "-k", str(case["kstart"]), "-o", out] + mode + sweep + extra_db(out)   # noqa: E731
    if not both(tree(ref_out), tree(our_out)):
        print(f"LIVE inputs seed {seed}: both fail at tree {case}")
        return
    assert_tree_matches(collect_tree(our_out, prefix, db(our_out), tool), golden.collect_tree(ref_out, prefix, db(ref_out), tool),
                        exact=case["exact"])
    # ---- kij (exact mode goes pair by pair on both sides; HLL mode through the batched table on ours)
    kij = lambda out: ["kij", "-d", os.path.join(out, prefix + "_dtree.pickle"), "-o", out] + (   # noqa: E731
        ["--jaccard", "--mink", str(case["sweep"][0]), "--maxk", str(case["sweep"][1])] if case["sweep"] else [])
    if both(kij(ref_out), kij(our_out)):
        pair = lambda r: (r["Atitle"], r["Btitle"])     # noqa: E731
        kij_ref = {pair(r): r for r in read_csv(os.path.join(ref_out, prefix + ".kij.csv"))}
        kij_our = read_csv(os.path.join(our_out, prefix + ".kij.csv"))
        assert sorted(map(pair, kij_our)) == sorted(kij_ref)
        for r in kij_our:
            g = kij_ref[pair(r)]
            assert (int(r["Ak"]), int(r["Bk"]), int(r["ABk"])) == (int(g["Ak"]), int(g["Bk"]), int(g["ABk"])), pair(r)
            assert float(r["KIJ"]) == pytest.approx(float(g["KIJ"]), rel=1e-6, abs=1e-6)
        if case["sweep"]:
            j_ref = {(r["Atitle"], r["Btitle"], int(r["kval"])): r for r in read_csv(os.path.join(ref_out, prefix + ".j.csv"))}
            j_our = read_csv(os.path.join(our_out, prefix + ".j.csv"))
            assert sorted((r["Atitle"], r["Btitle"], int(r["kval"])) for r in j_our) == sorted(j_ref)
            for r in j_our:
                g = j_ref[(r["Atitle"], r["Btitle"], int(r["kval"]))]
                assert float(r["jaccard"]) == pytest.approx(float(g["jaccard"]), rel=1e-6, abs=1e-6)
    else:
        print(f"LIVE inputs seed {seed}: both fail at kij {case}")
    # ---- a second tree, other tag, over the first n-1 files, into the SAME database: leaves are found, not redone
    flist = str(tmp_path / "fewer.txt")
    with open(flist, "w") as fh:
        fh.write("\n".join(final[:-1]) + "\n")
    tag2 = tag + "b"
    second = lambda out: (["tree", "-f", flist, "-s", tag2, "-k", str(case["kstart"]), "-o", out, "-c", db(out)] + mode + sweep)   # noqa: E731
    passes = oracle_store.stats["leaf_passes"]
    if both(second(ref_out), second(our_out)):
        prefix2 = f"{tag2}_{case['n'] - 1}_{tool}"
        rows = {side: [(r["title"], int(r["ngen"]), int(r["k"]), float(r["card"]), float(r["delta"]))
                       for r in read_csv(os.path.join(out, prefix2 + "_deltas.csv"))] for side, out in (("ref", ref_out), ("ours", our_out))}
        assert [r[:3] for r in rows["ours"]] == [r[:3] for r in rows["ref"]]
        assert all((a[3] == b[3]) if case["exact"] else (close(a[3], b[3]) and close(a[4], b[4])) for a, b in zip(rows["ours"], rows["ref"]))
        want_db = golden.collect_tree(ref_out, prefix, db(ref_out), tool)
        ours_db = collect_tree(our_out, prefix, db(our_out), tool)
        assert ours_db["files"] == want_db["files"] and ours_db["fastahex"] == want_db["fastahex"]
        assert ours_db["sketchinfo"] == want_db["sketchinfo"]
    else:
        print(f"LIVE inputs seed {seed}: both fail at the second tree {case}")
    print(f"LIVE inputs seed {seed}: tree, kij, second tree into the same database compared {case}")


def test_a_genome_without_any_kmer(tmp_path, golden, oracle_store):
    """The second deliberate difference in error behaviour.  A FASTA whose records hold no sequence has
    cardinality 0 at every k; the reference reads a stored 0 as "not computed yet", recomputes, stores 0 again and
    ends in its retry path with an UnboundLocalError (lib/sketch_classes.py:254-291).  The drop-in keeps the 0:
    a sweep completes, and a hill-climb ends with the reference's own message for data that is amiss."""
    import subprocess
    from oracle import pyoracle
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    files = make_dataset(data, 3, 2500, seed=9, sub=0.05)
    with open(files[-1], "wb") as fh:
        fh.write(b">nothing here\n>nor here\n\n")
    sweep = ["--ksweep", "--mink", "11", "--maxk", "13"]
    for mode in (sweep, []):
        argv = lambda out: ["tree", "-d", data, "-s", "e", "-k", "10", "-o", out, "-r", "10"] + mode     # noqa: E731
        with pytest.raises(subprocess.CalledProcessError) as ref_err:
            golden.run_ref(bindir, argv(str(tmp_path / ("ref%d" % len(mode)))))
        assert "UnboundLocalError" in ref_err.value.stderr.decode(errors="replace")
        if mode:
            run_dandd(argv(str(tmp_path / "ours")))
            db = collect_tree(str(tmp_path / "ours"), "e_3_dashing", str(tmp_path / "ours" / "sketchdb"), "dashing")
            empty = [v for k, v in db["cardkey"].items() if os.sep + "ngen1" + os.sep in os.sep + k and "g2" in k]
            assert len(empty) == 3 and all(v == 0 for v in empty)
            assert all(v > 0 for k, v in db["cardkey"].items() if "g2." not in os.path.basename(k))
        else:
            with pytest.raises(ValueError, match="Exploratory k value is too high"):
                run_dandd(argv(str(tmp_path / "ours_climb")))


def test_changed_inputs_and_damaged_databases(tmp_path, golden, oracle_store):
    """What both sides do when the world changes between runs: a FASTA is replaced (the stale name is reused
    without --safe, --safe refuses with the same message), a database pickle is damaged (both recover from the
    .bkp copy).  With the .bkp gone as well the reference stops (it catches FileExistsError where it means
    FileNotFoundError, lib/species_specifics.py:23-38) and the drop-in starts from an empty table, as the
    reference's own comment there intends -- the third and last deliberate difference."""
    import shutil
    import subprocess
    from oracle import pyoracle
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    files = make_dataset(data, 4, 3000, seed=19, sub=0.05)
    ref_out, our_out = str(tmp_path / "ref"), str(tmp_path / "ours")
    argv = lambda out, more=(): ["tree", "-d", data, "-s", "t", "-k", "11", "-o", out, "-r", "10"] + list(more)   # noqa: E731

    def same():
        assert_tree_matches(collect_tree(our_out, "t_4_dashing", os.path.join(our_out, "sketchdb"), "dashing"),
                            golden.collect_tree(ref_out, "t_4_dashing", os.path.join(ref_out, "sketchdb"), "dashing"))
    assert _both(golden, bindir, argv(ref_out), argv(our_out))
    same()
    for side in (ref_out, our_out):
        shutil.copytree(side, side + ".pristine")
    # ---- a FASTA is replaced by another genome
    other = make_dataset(str(tmp_path / "other"), 4, 3000, seed=99, sub=0.05)
    shutil.copy(other[2], files[2])
    oracle_store._syms.clear()
    oracle_store._regs.clear()
    assert _both(golden, bindir, argv(ref_out), argv(our_out))                        # stale name, stale sketches: on both sides
    same()
    with pytest.raises(subprocess.CalledProcessError) as ref_err:
        golden.run_ref(bindir, argv(ref_out, ["--safe"]))
    with pytest.raises(RuntimeError) as our_err:
        run_dandd(argv(our_out, ["--safe"]))
    assert str(our_err.value) in ref_err.value.stderr.decode(errors="replace")        # "Checksum does not match stored value for g2.fasta: ..."
    make_dataset(data, 4, 3000, seed=19, sub=0.05)                                    # the original genome is back
    oracle_store._syms.clear()
    # ---- damaged pickles
    for name in ("dandd_fastahex.pickle", "dandd_sketchinfo.pickle", "t_dashing_cardinalities.pickle"):
        for keep_backup in (True, False):
            for side in (ref_out, our_out):
                shutil.rmtree(side)
                shutil.copytree(side + ".pristine", side)
                with open(os.path.join(side, "sketchdb", name), "wb") as fh:
                    fh.write(b"\\x80\\x04garbage")
                if not keep_backup:
                    os.remove(os.path.join(side, "sketchdb", name + ".bkp"))
            oracle_store._regs.clear()
            if keep_backup:
                assert _both(golden, bindir, argv(ref_out), argv(our_out))
            else:
                with pytest.raises(subprocess.CalledProcessError) as ref_err:
                    golden.run_ref(bindir, argv(ref_out))
                assert "FileNotFoundError" in ref_err.value.stderr.decode(errors="replace")
                run_dandd(argv(our_out))                                              # starts from an empty table, rebuilds, saves
                assert os.path.getsize(os.path.join(our_out, "sketchdb", name)) > 20


EXTREMES = [
    # (name, extra argv, exact, what to expect: "same" = same outputs or the same failure; otherwise the exception the
    #  REFERENCE dies with where the drop-in completes -- deliberate difference (4) of DESIGN.md section 2)
    ("k2", ["-k", "2"], False, "same"), ("k3", ["-k", "3"], False, "same"), ("k30", ["-k", "30"], False, "same"),
    ("k31", ["-k", "31"], False, "same"), ("k32", ["-k", "32"], False, "same"), ("k33", ["-k", "33"], False, "same"),
    ("k1", ["-k", "1"], False, "KeyError"),                       # exploring k - 1 = 0 collides with the k = 0 template slot
    ("sweep_1_3", ["-k", "10", "--ksweep", "--mink", "1", "--maxk", "3"], False, "same"),
    ("sweep_0_2", ["-k", "10", "--ksweep", "--mink", "0", "--maxk", "2"], False, "KeyError"),
    ("sweep_30_34", ["-k", "10", "--ksweep", "--mink", "30", "--maxk", "34"], False, "same"),   # names of k = 33, 34 are registered, no more
    ("sweep_32_32", ["-k", "10", "--ksweep", "--mink", "32", "--maxk", "32"], False, "same"),
    ("sweep_5_4", ["-k", "10", "--ksweep", "--mink", "5", "--maxk", "4"], False, "same"),
    ("registers_4", ["-k", "10", "-r", "4"], False, "same"), ("registers_24", ["-k", "10", "-r", "24"], False, "same"),
    ("exact_k2", ["-k", "2", "--exact"], True, "same"),
    ("exact_k1", ["-k", "1", "--exact"], True, "KeyError"),
    ("exact_k33", ["-k", "33", "--exact"], True, "same"), ("exact_k64", ["-k", "64", "--exact"], True, "same"),
    ("exact_k65", ["-k", "65", "--exact"], True, "same"),
    ("exact_sweep_30_36", ["-k", "31", "--exact", "--ksweep", "--mink", "30", "--maxk", "36"], True, "same"),    # across the 64-bit k-mer
    ("exact_sweep_62_67", ["-k", "31", "--exact", "--ksweep", "--mink", "62", "--maxk", "67"], True, "same"),    # across the 128-bit k-mer
    ("exact_sweep_99_100_nocanon", ["-k", "31", "--exact", "-C", "--ksweep", "--mink", "99", "--maxk", "100"], True, "same"),
]


CORNERS_EXACT = [   # on an --exact tree: k-mer sets instead of sketches, ranges that cross k = 32 (real for KMC, the stand-in follows)
    ("exact_progressive_identity", ["progressive", "-n", "1"], ["x_progu1_4_kmc.csv", "x_progu1_4_kmcsummary.csv"]),
    ("exact_progressive_sweep_31_35", ["progressive", "-n", "1", "-s", "xh", "--ksweep", "--mink", "31", "--maxk", "35"],
     ["xh_progu1_4_kmc.csv", "xh_progu1_4_kmcsummary.csv"]),
    ("exact_kij", ["kij"], ["x_4_kmc.kij.csv"]),
    ("exact_kij_jaccard_31_35", ["kij", "-s", "xk", "--jaccard", "--mink", "31", "--maxk", "35"], ["xk_4_kmc.kij.csv", "xk_4_kmc.j.csv"]),
]


@pytest.mark.parametrize("name,extra,exact,expect", EXTREMES, ids=[e[0] for e in EXTREMES])
def test_extreme_k_sweeps_and_register_counts(tmp_path, golden, oracle_store, name, extra, exact, expect):
    import subprocess
    from oracle import pyoracle
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    make_dataset(data, 3, 3000, seed=5, sub=0.05)
    tool = "kmc" if exact else "dashing"
    ref_out, our_out = str(tmp_path / "ref"), str(tmp_path / "ours")
    argv = lambda out: ["tree", "-d", data, "-s", "t", "-o", out] + ([] if exact or "-r" in extra else ["-r", "10"]) + extra   # noqa: E731
    if expect == "same":
        try:
            golden.run_ref(bindir, argv(ref_out), exact=exact)
        except subprocess.CalledProcessError as failed:
            last = failed.stderr.decode(errors="replace").strip().split("\n")[-1]
            with pytest.raises(Exception) as ours_err:
                run_dandd(argv(our_out))
            assert type(ours_err.value).__name__ in last, (last, repr(ours_err.value))
            return
        run_dandd(argv(our_out))
        assert_tree_matches(collect_tree(our_out, f"t_3_{tool}", os.path.join(our_out, "sketchdb"), tool),
                            golden.collect_tree(ref_out, f"t_3_{tool}", os.path.join(ref_out, "sketchdb"), tool), exact=exact)
    else:
        with pytest.raises(subprocess.CalledProcessError) as ref_err:
            golden.run_ref(bindir, argv(ref_out), exact=exact)
        assert expect in ref_err.value.stderr.decode(errors="replace").strip().split("\n")[-1]
        run_dandd(argv(our_out))
        rows = read_csv(os.path.join(our_out, f"t_3_{tool}_deltas.csv"))
        assert len(rows) == 4 and ("--ksweep" in extra or all(float(r["delta"]) > 0 and int(r["k"]) >= 1 for r in rows))


def _rows_for_comparison(path):
    """CSV rows with directories stripped from path-like fields and numbers parsed; the `command` column (the
    shell line the reference ran / the drop-in stands in for) is left out."""
    import re
    out = []
    for r in read_csv(path):
        row = {}
        for key, value in r.items():
            if key == "command":
                continue
            value = re.sub(r"/[^ ,|'\\]]*/", "", value or "")
            try:
                row[key] = float(value)
            except ValueError:
                row[key] = value
        out.append(row)
    return out


def assert_csv_close(ref_path, our_path):
    ref, ours = _rows_for_comparison(ref_path), _rows_for_comparison(our_path)
    label = lambda r: tuple(sorted((k, v) for k, v in r.items() if not isinstance(v, float)))     # noqa: E731
    assert sorted(map(label, ours)) == sorted(map(label, ref)), os.path.basename(ref_path)
    by_label = {}
    for r in ref:
        by_label.setdefault(label(r), []).append(r)
    for r in ours:
        candidates = by_label[label(r)]
        assert any(all(close(r[k], g[k]) for k in r if isinstance(r[k], float)) for g in candidates), (os.path.basename(ref_path), r)


CORNERS = [
    # (name, command argv after the pickle, files to compare -- same outputs, or the same failure)
    ("progressive_identity", ["progressive", "-n", "1"], ["t_progu1_4_dashing.csv", "t_progu1_4_dashingsummary.csv"]),
    ("progressive_sweep_on_a_climbed_tree", ["progressive", "-n", "1", "-s", "ps", "--ksweep", "--mink", "9", "--maxk", "12"],
     ["ps_progu1_4_dashing.csv", "ps_progu1_4_dashingsummary.csv"]),
    ("progressive_step_3", ["progressive", "-n", "1", "-s", "s3", "--step", "3"], ["s3_progu1_4_dashing.csv"]),
    ("progressive_step_beyond_n", ["progressive", "-n", "1", "-s", "s9", "--step", "9"], ["s9_progu1_4_dashing.csv"]),
    ("progressive_step_0", ["progressive", "-n", "1", "-s", "s0", "--step", "0"], []),
    ("progressive_every_permutation", ["progressive", "-n", "24", "-s", "all"], ["all_progu24_4_dashing.csv"]),
    ("progressive_more_than_every_permutation", ["progressive", "-n", "100", "-s", "many"], ["many_progu100_4_dashing.csv"]),
    ("kij_plain", ["kij"], ["t_4_dashing.kij.csv"]),
    ("kij_jaccard_without_a_range", ["kij", "-s", "j0", "--jaccard"], ["j0_4_dashing.kij.csv"]),
    ("kij_jaccard_empty_range", ["kij", "-s", "j1", "--jaccard", "--mink", "12", "--maxk", "10"], ["j1_4_dashing.kij.csv"]),
    ("kij_jaccard_9_12", ["kij", "-s", "j2", "--jaccard", "--mink", "9", "--maxk", "12"], ["j2_4_dashing.kij.csv", "j2_4_dashing.j.csv"]),
    ("kij_jaccard_past_k32", ["kij", "-s", "j3", "--jaccard", "--mink", "30", "--maxk", "34"], []),
    ("kij_sweep_without_jaccard", ["kij", "-s", "j4", "--ksweep", "--mink", "9", "--maxk", "12"], ["j4_4_dashing.kij.csv"]),
]


def test_progressive_and_kij_corner_options(tmp_path, golden, oracle_store):
    """One climbed tree on each side, then every corner command in turn on the same pair of databases (their
    tags differ, what they add to the databases they add on both sides)."""
    from oracle import pyoracle
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    make_dataset(data, 4, 3000, seed=5, sub=0.05)
    ref_out, our_out = str(tmp_path / "ref"), str(tmp_path / "ours")
    tree = lambda out: ["tree", "-d", data, "-s", "t", "-k", "11", "-o", out, "-r", "10"]     # noqa: E731
    assert _both(golden, bindir, tree(ref_out), tree(our_out))
    xtree = lambda out: ["tree", "-d", data, "-s", "x", "-k", "11", "-o", out, "--exact"]     # noqa: E731
    golden.run_ref(bindir, xtree(ref_out), exact=True)
    run_dandd(xtree(our_out))
    for name, command, outputs in CORNERS + CORNERS_EXACT:
        pickle_name = "x_4_kmc_dtree.pickle" if name.startswith("exact_") else "t_4_dashing_dtree.pickle"
        argv = lambda out: [command[0], "-d", os.path.join(out, pickle_name), "-o", out] + command[1:]   # noqa: E731
        if _both(golden, bindir, argv(ref_out), argv(our_out), exact=name.startswith("exact_")):
            assert outputs, name + ": both succeeded where a shared failure was expected"
            for filename in outputs:
                if "progu24" in filename or "progu100" in filename:       # random orderings: every permutation, whatever the order
                    ref_rows, our_rows = (_rows_for_comparison(os.path.join(out, filename)) for out in (ref_out, our_out))
                    key = lambda r: (r["ngen"], r["kval"], round(r["delta"], 3), r["fastas"])     # noqa: E731
                    assert len(our_rows) == len(ref_rows) == 24 * 4 and sorted(map(key, our_rows)) == sorted(map(key, ref_rows)), name
                else:
                    assert_csv_close(os.path.join(ref_out, filename), os.path.join(our_out, filename))
        else:
            assert not outputs, name + ": both failed (the same way) where outputs were expected"
        print("LIVE corner", name, "compared")


def test_input_listing_corners(tmp_path, golden, oracle_store):
    """How the inputs of `tree` are found: --nchildren beyond what can be built, file lists with blank lines,
    duplicates, missing files, one file, no file; directories with one FASTA, none, a trailing slash, a relative
    path; tags with underscores -- same outputs or the same failure.  Deliberate difference (5):
    for a --datadir that does not exist the reference CONSTRUCTS a ValueError but never raises it
    (lib/huffman_dandd.py:866-867) and fails later on an empty file name; the drop-in raises that ValueError."""
    import shutil
    import subprocess
    from oracle import pyoracle
    bindir = pyoracle.install_shims(str(tmp_path / "bin"))
    data = str(tmp_path / "data")
    files = make_dataset(data, 4, 3000, seed=5, sub=0.05)
    base = lambda out, more: ["tree", "-s", "t", "-k", "11", "-o", out, "-r", "10"] + more     # noqa: E731
    flist = str(tmp_path / "list.txt")
    one, none = str(tmp_path / "one"), str(tmp_path / "none")
    os.makedirs(one)
    os.makedirs(none)
    shutil.copy(files[0], one)
    cases = [("nchildren_2", ["-d", data, "-n", "2"], None, 4), ("nchildren_4", ["-d", data, "-n", "4"], None, 4),
             ("nchildren_5", ["-d", data, "-n", "5"], None, 4), ("nchildren_9", ["-d", data, "-n", "9"], None, 4),
             ("list_blank_line", ["-f", flist], "\n".join(files[:3]) + "\n\n", 3),
             ("list_duplicate", ["-f", flist], "\n".join([files[0], files[1], files[0]]) + "\n", 3),
             ("list_missing_file", ["-f", flist], "\n".join([files[0], files[1], str(tmp_path / "nope.fasta")]) + "\n", 3),
             ("list_single", ["-f", flist], files[0] + "\n", 1), ("list_empty", ["-f", flist], "", 0),
             ("dir_single", ["-d", one], None, 1), ("dir_empty", ["-d", none], None, 0),
             ("dir_trailing_slash", ["-d", data + "/"], None, 4), ("tag_with_underscores", ["-d", data, "-s", "my_tag_1"], None, 4)]
    for name, more, list_text, n in cases:
        if list_text is not None:
            with open(flist, "w") as fh:
                fh.write(list_text)
        ref_out, our_out = str(tmp_path / ("ref_" + name)), str(tmp_path / ("ours_" + name))
        oracle_store._regs.clear()
        if _both(golden, bindir, base(ref_out, more), base(our_out, more)):
            tag = "my_tag_1" if "my_tag_1" in more else "t"
            assert_tree_matches(collect_tree(our_out, f"{tag}_{n}_dashing", os.path.join(our_out, "sketchdb"), "dashing"),
                                golden.collect_tree(ref_out, f"{tag}_{n}_dashing", os.path.join(ref_out, "sketchdb"), "dashing"))
        print("LIVE inputs", name, "compared")
    missing = ["-d", str(tmp_path / "no_such_directory")]
    with pytest.raises(subprocess.CalledProcessError) as ref_err:
        golden.run_ref(bindir, base(str(tmp_path / "ref_missing"), missing))
    assert "FileNotFoundError" in ref_err.value.stderr.decode(errors="replace")
    with pytest.raises(ValueError, match="You must provide either an existing directory of fastas"):
        run_dandd(base(str(tmp_path / "ours_missing"), missing))
    for side in ("ref", "ours"):                                   # neither input option: both print the same line and exit 1
        try:
            (golden.run_ref(bindir, base(str(tmp_path / "ref_nothing"), [])) if side == "ref"
             else run_dandd(base(str(tmp_path / "ours_nothing"), [])))
            raise AssertionError(side + " accepted a run without inputs")
        except subprocess.CalledProcessError as failed:
            assert failed.returncode == 1
        except SystemExit as stop:
            assert stop.code == 1


def test_command_line_surface_equals_the_reference():
    """Every sub-command, option string, destination, default, type, nargs and choice of the reference's argparse
    tree exists unchanged in the drop-in's; the drop-in adds --device and --gpus, and a handler for `info`."""
    import argparse
    import subprocess
    import sys
    import textwrap
    probe = textwrap.dedent("""
        import argparse, json, sys
        sys.path.insert(0, sys.argv[1])
        if len(sys.argv) > 2:
            sys.path.insert(1, sys.argv[2])
        import dandd_cmd
        parser = dandd_cmd.parse_arguments()[0]
        subs = [a for a in parser._actions if isinstance(a, argparse._SubParsersAction)][0]
        out = {}
        for name, sp in subs.choices.items():
            out[name] = {"|".join(a.option_strings): [a.dest, repr(a.default), repr(a.nargs), getattr(a.type, "__name__", repr(a.type)),
                                                       a.required, repr(a.choices), type(a).__name__]
                         for a in sp._actions if not isinstance(a, argparse._HelpAction)}
            out[name]["<handler>"] = sp.get_default("func") is not None
        print(json.dumps(out))
    """)
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    surfaces = {}
    for side, args in (("ref", [REF]), ("ours", [os.path.join(root, "dandd_b200", "lib"), root])):
        done = subprocess.run([sys.executable, "-W", "ignore", "-c", probe] + args, capture_output=True, text=True, check=True)
        surfaces[side] = json.loads(done.stdout)
    assert sorted(surfaces["ours"]) == sorted(surfaces["ref"]) == ["info", "kij", "progressive", "tree"]
    for command, options in surfaces["ref"].items():
        for option, spec in options.items():
            if option == "<handler>":
                continue
            ours = surfaces["ours"][command][option]
            if option == "-o|--out" or option == "-o|--outdir":
                spec, ours = spec[:1] + spec[2:], ours[:1] + ours[2:]          # default = the current directory of each probe
            assert ours == spec, (command, option, spec, ours)
        extra = set(surfaces["ours"][command]) - set(options)
        assert extra == {"--device", "--gpus"}, (command, extra)
    assert surfaces["ref"]["info"]["<handler>"] is False and surfaces["ours"]["info"]["<handler>"] is True
    assert all(surfaces[s][c]["<handler>"] for s in surfaces for c in ("tree", "progressive", "kij"))
