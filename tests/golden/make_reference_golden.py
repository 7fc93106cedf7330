"""Runs the UNMODIFIED reference Python (lib/dandd of the checkout DANDD_REFERENCE names) on small synthetic datasets
with oracle-backed stand-ins for dashing / kmc / kmc_tools / parallel first on PATH
(oracle/shims, SURVEY.md Appendix C technique) and records what it produced -- deltas, argmax k,
cardinalities, sketchdb layout, progressive and KIJ tables -- as tests/golden/reference_runs.json.

These fixtures pin the HOST LOGIC of the drop-in layer (dandd_b200/lib/*) to the reference's own
behaviour: the tests re-create the same inputs and require the same outputs.  They cannot pin the
arithmetic to real Dashing/KMC (absent here; parity unpinned, see oracle/dandd_oracle.c).

The reference is not part of this repository, hence committed fixtures.  Run from the repository root:
    DANDD_REFERENCE=<checkout of the reference> python tests/golden/make_reference_golden.py
"""
import csv
import json
import os
import pickle
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle  # noqa: E402
from tests.util import make_dataset, reference_path  # noqa: E402

REF = reference_path("lib")

# --exact is broken as shipped (KMCSketchObj.sketch_check <-> check_cardinality recurse forever,
# SURVEY.md App. B).  The golden for exact mode is produced with that ONE method replaced at run
# time by the existence test it was meant to be; the reference files are not modified.
EXACT_WRAPPER = r'''
import os, sys
sys.path.insert(0, %(ref)r)
import sketch_classes
def sketch_check(self, path=None):
    path = path or self.sfp.full
    return all(os.path.exists(path + e) and os.stat(path + e).st_size != 0 for e in (".kmc_pre", ".kmc_suf"))
sketch_classes.KMCSketchObj.sketch_check = sketch_check
from dandd_cmd import parse_arguments
parser, _ = parse_arguments()
args = parser.parse_args(sys.argv[1:])
args.func(args)
'''


def run_ref(bindir, argv, exact=False, cwd=None):
    # (TMPDIR: the reference's ksweep_update_node makes a temporary directory per call and never removes it,
    # lib/huffman_dandd.py:161,187 -- keep those next to the stand-ins, where the caller's clean-up finds them)
    scratch = os.path.join(bindir, "tmp")
    os.makedirs(scratch, exist_ok=True)
    env = dict(os.environ, PATH=bindir + os.pathsep + os.environ["PATH"], PYTHONPATH=REF, PYTHONHASHSEED="0",
               ORC_PARALLEL_JOBS="4", TMPDIR=scratch)
    if exact:
        wrapper = os.path.join(bindir, "exact_wrapper.py")
        with open(wrapper, "w") as fh:
            fh.write(EXACT_WRAPPER % {"ref": REF})
        cmd = [sys.executable, wrapper] + argv
    else:
        cmd = [sys.executable, os.path.join(REF, "dandd")] + argv
    subprocess.run(cmd, check=True, env=env, cwd=cwd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)


def read_csv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh))


def rel(path, base):
    return os.path.relpath(path, base) if path and os.path.isabs(path) else path


def norm_fastas(text, sep):
    return sep.join(os.path.basename(f.strip(" '[]")) for f in text.split(sep))


def collect_tree(outdir, prefix, sketchdir, tool):
    rows = []
    for r in read_csv(os.path.join(outdir, prefix + "_deltas.csv")):
        rows.append({"title": r["title"], "ngen": int(r["ngen"]), "k": int(r["k"]), "delta": float(r["delta"]),
                     "card": float(r["card"]), "sketchloc": rel(r["sketchloc"], sketchdir),
                     "fastas": norm_fastas(r["fastas"], "|")})
    files = sorted(os.path.relpath(os.path.join(d, f), sketchdir) for d, _, fs in os.walk(sketchdir) for f in fs
                   if not f.endswith((".pickle", ".bkp")))
    cardkey = {}
    for name in os.listdir(sketchdir):
        if name.endswith(f"_{tool}_cardinalities.pickle"):
            with open(os.path.join(sketchdir, name), "rb") as fh:
                cardkey.update({rel(k, sketchdir): float(v) for k, v in pickle.load(fh).items()})
    with open(os.path.join(sketchdir, "dandd_fastahex.pickle"), "rb") as fh:
        fastahex = pickle.load(fh)
    with open(os.path.join(sketchdir, "dandd_sketchinfo.pickle"), "rb") as fh:
        sketchinfo = sorted(pickle.load(fh).keys())
    with open(os.path.join(outdir, prefix + "_dtree.pickle"), "rb") as fh:
        pass  # unpickling needs the reference modules; existence is enough here
    return {"deltas": rows, "files": files, "cardkey": cardkey, "fastahex": fastahex, "sketchinfo": sketchinfo}


def prog_rows(path):
    return [{"ngen": int(r["ngen"]), "kval": int(r["kval"]), "delta": float(r["delta"]), "fastas": norm_fastas(r["fastas"], ",")}
            for r in read_csv(path)]


def more_runs(work, bindir, data5, dtreeA, outA, gold):
    """Option coverage: --no-canon / --registers, -f file lists, --safe, --fast, progressive -f and
    --step, kij --afproject.  (`--lowmem` and `kij -f` fail in the reference as shipped -- a runaway
    hill-climb after the union sketches are deleted, and strings where nodes are expected,
    lib/huffman_dandd.py:685 -- so there is nothing to pin for them.)"""
    # H: non-canonical k-mers, 2^12 registers
    outH = os.path.join(work, "outH")
    run_ref(bindir, ["tree", "-d", data5, "-s", "runH", "-k", "12", "-o", outH, "-C", "-r", "12"])
    gold["runs"]["H_tree_noncanon_p12"] = collect_tree(outH, "runH_5_dashing", os.path.join(outH, "sketchdb"), "dashing")
    # I: a file list instead of a directory (3 of the 5 FASTAs), with --safe
    flist = os.path.join(work, "flist.txt")
    with open(flist, "w") as fh:
        fh.write("\n".join(os.path.join(data5, f) for f in sorted(os.listdir(data5))[1:4]) + "\n")
    outI = os.path.join(work, "outI")
    run_ref(bindir, ["tree", "-f", flist, "-s", "runI", "-k", "14", "-o", outI, "--safe"])
    gold["runs"]["I_tree_flist_safe"] = collect_tree(outI, "runI_3_dashing", os.path.join(outI, "sketchdb"), "dashing")
    # K: --fast writes the deltas table only
    outK = os.path.join(work, "outK")
    run_ref(bindir, ["tree", "-d", data5, "-s", "runK", "-k", "14", "-o", outK, "--fast"])
    gold["runs"]["K_tree_fast"] = {"outputs": sorted(f for f in os.listdir(outK) if f != "sketchdb"),
                                   "deltas": [{"title": r["title"], "ngen": int(r["ngen"]), "k": int(r["k"]),
                                               "delta": float(r["delta"]), "card": float(r["card"])}
                                              for r in read_csv(os.path.join(outK, "runK_5_dashing_deltas.csv"))]}
    # L: progressive over a subset of the tree's FASTAs; N: --step 2
    run_ref(bindir, ["progressive", "-d", dtreeA, "-f", flist, "-n", "1", "-o", outA, "-s", "sub"])
    gold["runs"]["L_progressive_subset"] = {"rows": prog_rows(os.path.join(outA, "sub_progu1_5_dashing.csv"))}
    run_ref(bindir, ["progressive", "-d", dtreeA, "-n", "1", "--step", "2", "-o", outA, "-s", "st2"])
    gold["runs"]["N_progressive_step2"] = {"rows": prog_rows(os.path.join(outA, "st2_progu1_5_dashing.csv"))}
    # O: kij --afproject (the tuples handed to the AFproject helper)
    run_ref(bindir, ["kij", "-d", dtreeA, "-o", outA, "--afproject", "-s", "af"])
    with open(os.path.join(outA, "af_5_dashing_AFtuples.pickle"), "rb") as fh:
        tuples = pickle.load(fh)
    gold["runs"]["O_kij_afproject"] = {"type": type(tuples).__name__, "tuples": json.loads(json.dumps(tuples, default=list))}


def exact_runs(work, bindir, data5, gold):
    """--exact beyond the hill-climb: a k sweep, progressive unions with and without the sweep
    (all with the one-method run-time patch described at EXACT_WRAPPER), and a binary tree."""
    outP = os.path.join(work, "outP")
    sweep = ["--ksweep", "--mink", "12", "--maxk", "15"]
    run_ref(bindir, ["tree", "-d", data5, "-s", "runP", "-k", "14", "-o", outP, "--exact"] + sweep, exact=True)
    gold["runs"]["P_tree_exact_ksweep"] = collect_tree(outP, "runP_5_kmc", os.path.join(outP, "sketchdb"), "kmc")
    dtreeP = os.path.join(outP, "runP_5_kmc_dtree.pickle")
    run_ref(bindir, ["progressive", "-d", dtreeP, "-n", "1", "-o", outP] + sweep, exact=True)
    summ = read_csv(os.path.join(outP, "runP_progu1_5_kmcsummary.csv"))
    gold["runs"]["Q_progressive_exact_ksweep"] = {
        "summary": [{"ngen": int(r["ngen"]), "kval": int(r["kval"]), "card": float(r["card"]), "delta_pos": float(r["delta_pos"]),
                     "title": r["title"]} for r in summ]}
    run_ref(bindir, ["progressive", "-d", dtreeP, "-n", "1", "-o", outP, "-s", "hc"], exact=True)
    gold["runs"]["Q_progressive_exact_hillclimb"] = {"rows": prog_rows(os.path.join(outP, "hc_progu1_5_kmc.csv"))}
    outS = os.path.join(work, "outS")
    run_ref(bindir, ["tree", "-d", data5, "-s", "runS", "-k", "13", "-o", outS, "-n", "2"])
    gold["runs"]["S_tree_nchildren2"] = collect_tree(outS, "runS_5_dashing", os.path.join(outS, "sketchdb"), "dashing")
    # T: the default sweep (k = 2..32) -- small k included -- on three short genomes
    data3 = os.path.join(work, "data3")
    make_dataset(data3, 3, 6000, seed=23, prefix="s")
    outT = os.path.join(work, "outT")
    run_ref(bindir, ["tree", "-d", data3, "-s", "runT", "-k", "10", "-o", outT, "--ksweep"])
    gold["runs"]["T_tree_default_sweep"] = collect_tree(outT, "runT_3_dashing", os.path.join(outT, "sketchdb"), "dashing")


def main():
    if not REF:
        sys.exit("set DANDD_REFERENCE to a checkout of the reference")
    work = tempfile.mkdtemp(prefix="dandd_golden_")
    bindir = pyoracle.install_shims(os.path.join(work, "bin"))
    gold = {"generator": "tests/golden/make_reference_golden.py", "runs": {}}
    try:
        data5 = os.path.join(work, "data5")
        make_dataset(data5, 5, 20000, seed=21)
        data7 = os.path.join(work, "data7")
        make_dataset(data7, 7, 12000, seed=22, prefix="h")

        # A: hill-climb spider, -k 14
        outA = os.path.join(work, "outA")
        run_ref(bindir, ["tree", "-d", data5, "-s", "runA", "-k", "14", "-o", outA])
        gold["runs"]["A_tree_hillclimb"] = collect_tree(outA, "runA_5_dashing", os.path.join(outA, "sketchdb"), "dashing")

        # B: k sweep 10..16, then progressive (identity ordering and 3 fixed orderings)
        outB = os.path.join(work, "outB")
        run_ref(bindir, ["tree", "-d", data5, "-s", "runB", "-k", "14", "-o", outB, "--ksweep", "--mink", "10", "--maxk", "16"])
        gold["runs"]["B_tree_ksweep"] = collect_tree(outB, "runB_5_dashing", os.path.join(outB, "sketchdb"), "dashing")
        dtreeB = os.path.join(outB, "runB_5_dashing_dtree.pickle")
        run_ref(bindir, ["progressive", "-d", dtreeB, "-n", "1", "-o", outB, "--ksweep", "--mink", "10", "--maxk", "16"])
        prog = read_csv(os.path.join(outB, "runB_progu1_5_dashing.csv"))
        summ = read_csv(os.path.join(outB, "runB_progu1_5_dashing" + "summary.csv"))
        gold["runs"]["B_progressive_identity"] = {
            "rows": [{"ngen": int(r["ngen"]), "kval": int(r["kval"]), "delta": r["delta"], "ordering": int(r["ordering"]),
                      "fastas": norm_fastas(r["fastas"], ",")} for r in prog],
            "summary": [{"ngen": int(r["ngen"]), "kval": int(r["kval"]), "card": float(r["card"]),
                         "delta_pos": float(r["delta_pos"]), "title": r["title"], "ordering": int(r["ordering"])} for r in summ]}
        orderings = {(0, 1, 2, 3, 4), (4, 2, 0, 1, 3), (3, 4, 1, 0, 2)}
        ofile = os.path.join(work, "orderings.pickle")
        with open(ofile, "wb") as fh:
            pickle.dump(orderings, fh)
        run_ref(bindir, ["progressive", "-d", dtreeB, "-r", ofile, "-s", "runBo", "-o", outB, "--ksweep", "--mink", "10",
                         "--maxk", "16"])
        summ = read_csv(os.path.join(outB, "runBo_progu0_5_dashing" + "summary.csv"))
        # ordering numbers follow list(set) order, which is process-specific: key rows by member set instead
        gold["runs"]["B_progressive_orderings"] = {
            "orderings": sorted(orderings),
            "cells": sorted({(r["title"], int(r["kval"]), float(r["card"])) for r in summ})}

        # F: progressive with the hill-climb (no k sweep), identity ordering, on A's tree
        dtreeA = os.path.join(outA, "runA_5_dashing_dtree.pickle")
        run_ref(bindir, ["progressive", "-d", dtreeA, "-n", "1", "-o", outA])
        prog = read_csv(os.path.join(outA, "runA_progu1_5_dashing.csv"))
        gold["runs"]["F_progressive_hillclimb"] = {
            "rows": [{"ngen": int(r["ngen"]), "kval": int(r["kval"]), "delta": float(r["delta"]),
                      "fastas": norm_fastas(r["fastas"], ",")} for r in prog]}

        # C: KIJ + per-k Jaccard on A's tree
        run_ref(bindir, ["kij", "-d", dtreeA, "-o", outA, "--jaccard", "--mink", "12", "--maxk", "14"])
        kij = read_csv(os.path.join(outA, "runA_5_dashing.kij.csv"))
        jac = read_csv(os.path.join(outA, "runA_5_dashing.j.csv"))
        gold["runs"]["C_kij"] = {
            "kij": [{"Atitle": r["Atitle"], "Btitle": r["Btitle"], "Ak": int(r["Ak"]), "Bk": int(r["Bk"]), "ABk": int(r["ABk"]),
                     "Adelta": float(r["Adelta"]), "Bdelta": float(r["Bdelta"]), "ABdelta": float(r["ABdelta"]),
                     "KIJ": float(r["KIJ"])} for r in kij],
            "jaccard": [{"Atitle": r["Atitle"], "Btitle": r["Btitle"], "kval": int(r["kval"]), "Acard": float(r["Acard"]),
                         "Bcard": float(r["Bcard"]), "ABcard": float(r["ABcard"]), "jaccard": float(r["jaccard"])} for r in jac]}

        # D: --nchildren 3 over 7 FASTAs (the lopsided tree of SURVEY.md App. C.14)
        outD = os.path.join(work, "outD")
        run_ref(bindir, ["tree", "-d", data7, "-s", "runD", "-k", "13", "-o", outD, "-n", "3"])
        gold["runs"]["D_tree_nchildren3"] = collect_tree(outD, "runD_7_dashing", os.path.join(outD, "sketchdb"), "dashing")

        # G: config 1 of BASELINE.json -- the example/ tutorial shape (25 mito-like genomes of 16-17 kbp,
        # `dandd tree -k 14`); the tutorial data itself is not in the reference repository
        data25 = os.path.join(work, "mito25")
        make_dataset(data25, 25, 16500, seed=1, sub=0.10, indel=0.003, prefix="mito")
        outG = os.path.join(work, "outG")
        run_ref(bindir, ["tree", "-d", data25, "-s", "fish-mito", "-k", "14", "-o", outG])
        gold["runs"]["G_config1_tree"] = collect_tree(outG, "fish-mito_25_dashing", os.path.join(outG, "sketchdb"), "dashing")

        # E: --exact (one reference method patched at run time, see EXACT_WRAPPER)
        outE = os.path.join(work, "outE")
        run_ref(bindir, ["tree", "-d", data5, "-s", "runE", "-k", "14", "-o", outE, "--exact"], exact=True)
        gold["runs"]["E_tree_exact"] = collect_tree(outE, "runE_5_kmc", os.path.join(outE, "sketchdb"), "kmc")
        more_runs(work, bindir, data5, dtreeA, outA, gold)
        exact_runs(work, bindir, data5, gold)
    finally:
        shutil.rmtree(work, ignore_errors=True)
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_runs.json")
    with open(out, "w") as fh:
        json.dump(gold, fh, indent=1, sort_keys=True)
    print("wrote", out, {k: len(v.get("deltas", v.get("rows", v.get("kij", v.get("cells", []))))) for k, v in gold["runs"].items()})


if __name__ == "__main__":
    main()
