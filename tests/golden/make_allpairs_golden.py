"""Runs the UNMODIFIED functions of the reference's helpers/allpairs.py on a small synthetic dataset and
records what they produce as tests/golden/allpairs_golden.json.

The reference's `go()` cannot run as shipped (undefined `args.name`, helpers/allpairs.py:333; undefined
`run_fneighbor`, :418), so this script replays the part of it that can -- the command list (:356-370),
`mp_runner` on every command with the oracle-backed `dashing` stand-in first on PATH (oracle/shims),
`delta_summarize`, `kij_summarize`, `j_summarize` and `summ_to_phylip` (:381-432) -- calling the
reference's own functions, imported from the checkout DANDD_REFERENCE names.  The fixtures pin the HOST LOGIC of
dandd_b200/helpers/allpairs.py to the reference's behaviour; the cardinalities are the oracle's, printed
by the stand-in with six decimals as `dashing hll` text output is parsed (parity unpinned, see
oracle/dandd_oracle.c).  Run from the repository root:
    DANDD_REFERENCE=<checkout of the reference> python tests/golden/make_allpairs_golden.py
"""
import importlib.util
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle  # noqa: E402
from tests.util import make_dataset, reference_path  # noqa: E402

REF = reference_path("helpers", "allpairs.py")
CASES = {
    # name: (genomes, length, seed, substitution rate, klist, nest, extra)
    "six_p12": (6, 20000, 71, 0.05, list(range(8, 21)), 4096, ""),
    "five_nocanon_unsorted_klist": (5, 8000, 72, 0.10, [15, 9, 12, 21, 10], 1024, "--no-canon"),
}


def load_reference():
    spec = importlib.util.spec_from_file_location("reference_allpairs", REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_case(ref, work, case):
    n, length, seed, sub, klist, nest, extra = case
    inputs = make_dataset(os.path.join(work, "data"), n, length, seed=seed, sub=sub)
    names = [os.path.basename(f).split(".")[0] for f in inputs]
    commands = []                                   # helpers/allpairs.py:356-370, verbatim shape
    for k in klist:
        for i in range(n):
            commands.append(("dashing", names[i], names[i], k, ref.card_cmd("dashing", k, nest, 8, extra, "", inputs[i])))
            for j in range(i + 1, n):
                commands.append(("dashing", names[i], names[j], k,
                                 ref.card_cmd("dashing", k, nest, 8, extra, "", inputs[i] + " " + inputs[j])))
    results = [ref.mp_runner(c) for c in commands]
    dsumm = ref.delta_summarize(results)
    summ = ref.kij_summarize(dsumm)
    for k in klist:
        summ += ref.j_summarize(results, k)
    ids = {name: name for name in names}
    phylip = {}
    for k in [0] + klist:
        part = [x for x in summ if x[3] == k]
        for ani in (False, True):
            fn = os.path.join(work, "out.phylip")
            ref.summ_to_phylip(part, ids, fn, convert_to_ani=ani)
            with open(fn) as fh:
                phylip[("ani" if ani else "sim") + ("kij" if k == 0 else "k%d" % k)] = fh.read()
    return {"genomes": n, "length": length, "seed": seed, "sub": sub, "klist": klist, "nest": nest, "extra": extra,
            "names": names, "results": [list(r) for r in results], "delta_summary": [list(r) for r in dsumm],
            "summary": [list(r) for r in summ], "phylip": phylip}


def main():
    if not REF:
        sys.exit("set DANDD_REFERENCE to a checkout of the reference")
    ref = load_reference()
    work = tempfile.mkdtemp(prefix="allpairs_golden_")
    bindir = pyoracle.install_shims(os.path.join(work, "bin"))
    ref.bin_dict["dashing"] = os.path.join(bindir, "dashing")
    out = {"made_by": "tests/golden/make_allpairs_golden.py", "reference": REF, "cases": {}}
    for name, case in CASES.items():
        out["cases"][name] = run_case(ref, os.path.join(work, name), case)
        print(name, len(out["cases"][name]["results"]), "cardinalities")
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "allpairs_golden.json"), "w") as fh:
        json.dump(out, fh)


if __name__ == "__main__":
    main()
