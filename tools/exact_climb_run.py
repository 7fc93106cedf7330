#!/usr/bin/env python3
"""Exact hill-climb unions from one family job per visited k, on one GPU: 12 clustered synthetic genomes of 5 Mbp
(tools/synth.py; 3 clusters of 4 copies of a random root, 1 % substitutions each) -- the config-2 shape -- through
`dandd tree --exact -n 2` and then `dandd progressive --exact -n 30`, both hill-climb (no --ksweep).

Each command runs on the family path and on the per-union path (DANDD_B200_EXACT_SET_BATCH=0), alternated, each run
in a fresh output directory, in this one process (the commands are called the way the `dandd` launcher calls them,
so the engine -- CUDA context, library -- is started once, before the first timed run, and is not in any time).  Per
run: wall time (host clock around the command; every count ends in a device->host copy), kernel launches
(dd_kernel_launches), family jobs and per-union counts (store stats).  The outputs of the two paths are compared
file for file (CSVs, sketch database listing, descriptors, cardinality / name pickles byte for byte; the tree pickles
by content).  The card name and power limit are read in the same run.

    python tools/exact_climb_run.py --out profiles/r05_exact_climb.json"""
import argparse
import json
import os
import pickle
import random
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.exact_pairs_run import card_info  # noqa: E402


def _content(obj, path=()):
    """A tree object's content as plain data (which objects share identity is not part of it)."""
    if isinstance(obj, dict):
        return {k: _content(v, path) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return [_content(v, path) for v in obj]
    if isinstance(obj, set):
        return sorted(_content(v, path) for v in obj)
    if hasattr(obj, "__dict__"):
        if id(obj) in path:
            return "<cycle>"
        return (type(obj).__name__, _content(vars(obj), path + (id(obj),)))
    return obj


def snapshot(root):
    out = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            raw = open(p, "rb").read()
            if f.endswith("_dtree.pickle"):
                raw = repr(_content(pickle.loads(raw))).encode()
            out[os.path.relpath(p, root)] = raw.replace(root.encode(), b"<out>")
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--genomes", type=int, default=12)
    ap.add_argument("--clusters", type=int, default=3)
    ap.add_argument("--bases", type=int, default=5_000_000)
    ap.add_argument("--orderings", type=int, default=30)
    ap.add_argument("--kstart", type=int, default=14)
    ap.add_argument("--reps", type=int, default=2, help="rounds of (family, per-union), the order swapped every round")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_exact_climb.json"))
    args = ap.parse_args()

    from dandd_b200 import build
    build.build()
    import dandd_b200
    from dandd_b200 import store as ddstore
    from dandd_b200.engine import get_engine
    from tools.synth import mutate_text, synth_fasta
    eng = get_engine()
    lib = eng.lib
    dandd_b200.enable_compat()
    import dandd_cmd
    parser, _ = dandd_cmd.parse_arguments()

    work = tempfile.mkdtemp(prefix="dd_exclimb_")
    try:
        data = os.path.join(work, "fastas")
        os.makedirs(data)
        per = max(1, args.genomes // args.clusters)
        g = 0
        for c in range(args.clusters):
            root = synth_fasta(args.bases, 1, seed=2000 + c, device=eng.device)
            for i in range(per):
                if g < args.genomes:
                    with open(os.path.join(data, "genome%02d.fasta" % g), "wb") as fh:
                        fh.write(mutate_text(root, 0.01, seed=200 * c + i).cpu().numpy().tobytes())
                    g += 1
        n = g

        def run(mode, rep):
            out = os.path.join(work, "%s%d" % (mode, rep))
            os.environ["DANDD_B200_EXACT_SET_BATCH"] = "1" if mode == "family" else "0"
            st = ddstore.GpuSketchStore(engine=eng)
            ddstore.set_store(st)
            rows = {}
            try:
                for name, argv in (("tree", ["tree", "-d", data, "-s", "cfg2", "-k", str(args.kstart), "-n", "2", "-o", out, "--exact"]),
                                   ("progressive", ["progressive", "-d", os.path.join(out, "cfg2_%d_kmc_dtree.pickle" % n),
                                                    "-n", str(args.orderings), "-o", out])):
                    random.seed(11)            # the same orderings on both paths
                    before = dict(st.stats)
                    l0 = lib.dd_kernel_launches()
                    t0 = time.perf_counter()
                    a = parser.parse_args(argv)
                    a.func(a)
                    wall = time.perf_counter() - t0
                    jobs = st.stats["exact_family_jobs"] - before["exact_family_jobs"]
                    rows[name] = {"wall_s": wall, "kernel_launches": int(lib.dd_kernel_launches() - l0), "family_jobs": jobs,
                                  "per_union_counts": st.stats["exact_calls"] - before["exact_calls"] - jobs}
            finally:
                os.environ.pop("DANDD_B200_EXACT_SET_BATCH", None)
                ddstore.set_store(None)
            return out, rows

        runs = []
        outputs = {}
        for rep in range(args.reps):
            for mode in (("family", "per_union") if rep % 2 == 0 else ("per_union", "family")):
                out, rows = run(mode, rep)
                runs.append({"rep": rep, "mode": mode, **rows})
                print(json.dumps(runs[-1]), flush=True)
                snap = snapshot(out)
                if mode in outputs:
                    assert snap == outputs[mode], "%s: a repeated run left different files" % mode
                outputs[mode] = snap
                shutil.rmtree(out, ignore_errors=True)
        a, b = outputs["family"], outputs["per_union"]
        differ = sorted(f for f in set(a) | set(b) if a.get(f) != b.get(f))
        summary = {}
        for name in ("tree", "progressive"):
            for mode in ("family", "per_union"):
                walls = [r[name]["wall_s"] for r in runs if r["mode"] == mode]
                summary["%s_%s_wall_s" % (name, mode)] = {"min": min(walls), "max": max(walls)}
        rep = dict(card_info(), genomes=n, bases=args.bases, clusters=args.clusters, orderings=args.orderings,
                   kstart=args.kstart, runs=runs, summary=summary, files_compared=len(a), outputs_equal=not differ,
                   differing_files=differ[:20],
                   timing="host clock around each command in one process, engine started before the first run; "
                          "the two paths alternate, the order swapped every round")
        print(json.dumps(summary), "outputs_equal=%s (%d files)" % (not differ, len(a)), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(rep, fh, indent=1)
        print("wrote", args.out)
        if differ:
            raise SystemExit("the family path left different files: %s" % differ[:5])
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
