#!/usr/bin/env python3
"""Exact progressive unions (K7 lists + K8 first-rank histograms) on one GPU: 12 clustered synthetic genomes of
5 Mbp (tools/synth.py; 3 clusters of 4 copies of a random root, 1 % substitutions each), 30 orderings, k = 10..32
-- the shape of `dandd progressive --exact --ksweep` at config-2 scale.

Per k it reports the wall time of the single counts (one K5 set per genome, listed separately: the leaves of a
progressive run are on record), of the batched job that gives all 30 x 12 prefix counts (host clock around work
that ends in a device->host copy), and the kernel launches of that job.  The per-prefix path (one fresh K5 set
per prefix union, as before K8) runs on a subset of the orderings; its time is scaled to all 30 orderings and
labelled as an extrapolation.  Every subset count must equal the batched count, and a few cells are checked
against the CPU oracle.  Then the command line itself: `dandd tree --exact --ksweep` once, and `dandd progressive
--exact --ksweep` over the 30 orderings from copies of that sketch database, with and without
DANDD_B200_EXACT_SET_BATCH=0.  The card name and power limit are read in the same run.

    python tools/exact_progressive_run.py --out profiles/r04_exact_progressive.json"""
import argparse
import json
import os
import pickle
import random
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.exact_pairs_run import card_info  # noqa: E402

CLI = os.path.join(ROOT, "dandd_b200", "lib", "dandd")


def run_cli(argv, env=None):
    t0 = time.perf_counter()
    subprocess.run([sys.executable, CLI] + argv, check=True, stdout=subprocess.DEVNULL, env=dict(os.environ, **(env or {})))
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--genomes", type=int, default=12)
    ap.add_argument("--clusters", type=int, default=3)
    ap.add_argument("--bases", type=int, default=5_000_000)
    ap.add_argument("--orderings", type=int, default=30)
    ap.add_argument("--subset", type=int, default=3, help="orderings timed on the per-prefix path")
    ap.add_argument("--mink", type=int, default=10)
    ap.add_argument("--maxk", type=int, default=32)
    ap.add_argument("--no-cli", action="store_true", help="skip the command-line A/B")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_exact_progressive.json"))
    args = ap.parse_args()

    import torch
    from dandd_b200 import build
    build.build()
    from dandd_b200 import _lib, engine as E
    from tools.synth import mutate_text, synth_fasta
    eng = E.Engine(0)
    lib = eng.lib
    ks = list(range(args.mink, args.maxk + 1))
    per = max(1, args.genomes // args.clusters)
    texts = []
    for c in range(args.clusters):
        root = synth_fasta(args.bases, 1, seed=2000 + c, device=eng.device)
        texts += [mutate_text(root, 0.01, seed=200 * c + i) for i in range(per)]
    texts = texts[:args.genomes]
    seqs = [eng.pack(t).check() for t in texts]
    n = len(seqs)
    random.seed(4)
    orderings = set()
    while len(orderings) < args.orderings:
        orderings.add(tuple(random.sample(range(n), n)))
    orderings = sorted(orderings)
    ranks = np.full((len(orderings), n), 0xFFFF, dtype=np.uint16)
    for o, order in enumerate(orderings):
        ranks[o, list(order)] = np.arange(n)
    sub = orderings[:args.subset]
    torch.cuda.synchronize()

    rows = []
    for k in ks:
        t0 = time.perf_counter()
        singles = [eng.exact_counts([s], k)[0] for s in seqs]
        t_single = time.perf_counter() - t0
        l0 = lib.dd_kernel_launches()
        t0 = time.perf_counter()
        hist = eng.exact_first_rank_hist(seqs, k, True, ranks, singles)
        t_job = time.perf_counter() - t0
        launches = lib.dd_kernel_launches() - l0
        prefix = np.cumsum(hist.astype(np.int64), axis=1)       # [ordering, i - 1]
        t0 = time.perf_counter()
        per_prefix = [[eng.exact_counts([seqs[g] for g in order[:i]], k)[-1] for i in range(2, n + 1)] for order in sub]
        t_sub = time.perf_counter() - t0
        equal = per_prefix == prefix[:len(sub), 1:].tolist()
        rows.append({
            "k": k, "passes": eng.last_pair_plan["passes"], "singles_s": t_single, "batched_s": t_job, "launches": int(launches),
            "subset_orderings": len(sub), "subset_per_prefix_s": t_sub,
            "per_prefix_extrapolated_to_all_orderings_s": t_sub / len(sub) * len(orderings),
            "subset_counts_equal_per_prefix": bool(equal),
        })
        print(json.dumps(rows[-1]), flush=True)
        if not equal:
            raise SystemExit("k=%d: batched prefix counts differ from the per-prefix path" % k)

    from oracle import pyoracle as orc
    checks = []
    for o, i, k in [(0, 3, 21), (1, 12, 12), (2, 6, 31)]:
        if k not in ks or i > n:
            continue
        order = orderings[o]
        syms = [orc.fasta_symbols(texts[g].cpu().numpy().tobytes()) for g in order[:i]]
        want = orc.exact_count(syms, k)
        got = int(np.cumsum(eng.exact_first_rank_hist(seqs, k, True, ranks[o:o + 1]).astype(np.int64))[i - 1])
        checks.append({"ordering": o, "prefix": i, "k": k, "oracle": want, "batched": got})
        if want != got:
            raise SystemExit("oracle mismatch: %s" % checks[-1])

    cli = None
    if not args.no_cli:
        work = tempfile.mkdtemp(prefix="dd_exprog_")
        try:
            data = os.path.join(work, "fastas")
            os.makedirs(data)
            for g, t in enumerate(texts):
                with open(os.path.join(data, "genome%02d.fasta" % g), "wb") as fh:
                    fh.write(t.cpu().numpy().tobytes())
            ofile = os.path.join(work, "orderings.pickle")
            with open(ofile, "wb") as fh:
                pickle.dump(set(orderings), fh)
            sweep = ["--ksweep", "--mink", str(args.mink), "--maxk", str(args.maxk)]
            base = os.path.join(work, "tree")
            cli = {"tree_s": run_cli(["tree", "-d", data, "-s", "exp", "-k", "14", "-o", base, "--exact"] + sweep)}
            outs = {}
            for mode, switch in (("batched", "1"), ("per_union", "0")):
                out = outs[mode] = os.path.join(work, mode)
                shutil.copytree(base, out)
                dtree = os.path.join(out, "exp_%d_kmc_dtree.pickle" % n)
                cli["progressive_%s_s" % mode] = run_cli(["progressive", "-d", dtree, "-r", ofile, "-o", out] + sweep,
                                                         {"DANDD_B200_EXACT_SET_BATCH": switch})
            csvs = [[open(os.path.join(outs[m], "exp_progu0_%d_kmc%s.csv" % (n, s)), "rb").read().replace(outs[m].encode(), b"")
                     for s in ("", "summary")] for m in ("batched", "per_union")]
            cli["csvs_equal"] = csvs[0] == csvs[1]
            print(json.dumps(cli), flush=True)
        finally:
            shutil.rmtree(work, ignore_errors=True)

    rep = dict(card_info(), genomes=n, bases=args.bases, clusters=args.clusters, orderings=len(orderings), ks=ks, rows=rows,
               oracle_cells=checks, cli=cli,
               timing="host clock around each call; every call ends in a device->host copy of its result",
               extrapolation="per_prefix_extrapolated_to_all_orderings_s = subset per-prefix time / subset orderings x "
                             "all orderings (not measured)")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
