#!/usr/bin/env python3
"""The exact sharing spectrum (K7 lists + K9) on one GPU, per k, against today's sampled route to the growth curve.

Shapes (clustered synthetic genomes of 5 Mbp, tools/synth.py: clusters of copies of a random root, 1 % substitutions
each): config 2 -- 12 genomes in 3 clusters, k = 10..32; the r3 shape -- 100 genomes in 10 clusters, k = 14..32.
Per k, alternated in this one process (the order swapped every k): the spectrum job (Engine.exact_spectrum, which
gives the mean over ALL n! orderings in closed form) and the store's exact_prefix_cards over 30 random orderings (one
K8 job per k, sized from the sequence lengths as the spectrum job is, so no single count runs first).  Times are a
host clock around a call that ends in a device->host copy; launches are dd_kernel_launches() over the call.  One
spectrum job at the first k runs untimed first (module load).  A few cells are checked against oracle k-mer sets; the card name and power limit
are read in the same run.

    python tools/exact_spectrum_run.py --out profiles/r06_exact_spectrum.json"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.exact_pairs_run import card_info  # noqa: E402

SHAPES = {"config2": (12, 3, 10, 32), "r3": (100, 10, 14, 32)}


def oracle_check(texts, k, hist, priv):
    """hist and priv at k <= 32 from the oracle's k-mer arrays of the whole genomes."""
    from oracle import pyoracle as orc
    sets = [np.unique(orc.kmers(orc.fasta_symbols(t.cpu().numpy().tobytes()), k, True)) for t in texts]
    keys, counts = np.unique(np.concatenate(sets), return_counts=True)
    want_hist = np.bincount(counts, minlength=len(texts) + 1)[1:].tolist()
    alone = keys[counts == 1]
    want_priv0 = int(np.isin(sets[0], alone, assume_unique=True).sum())
    got = {"k": k, "hist_equal": want_hist == hist.astype(np.int64).tolist(), "priv0": int(priv[0]), "oracle_priv0": want_priv0}
    if not got["hist_equal"] or got["priv0"] != want_priv0:
        raise SystemExit("oracle mismatch: %s" % got)
    return got


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--shapes", default="config2,r3")
    ap.add_argument("--bases", type=int, default=5_000_000)
    ap.add_argument("--orderings", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_exact_spectrum.json"))
    args = ap.parse_args()

    import torch
    from dandd_b200 import build
    build.build()
    from dandd_b200 import store as ddstore
    from dandd_b200.engine import get_engine, length_bounds
    from dandd_b200.helpers.spectrum import mean_growth
    from tools.synth import mutate_text, synth_fasta
    eng = get_engine()
    lib = eng.lib
    work = tempfile.mkdtemp(prefix="dd_spectrum_")
    report = dict(card_info(), bases=args.bases, orderings=args.orderings, shapes={},
                  timing="host clock around each call; every call ends in a device->host copy of its result")
    for shape in args.shapes.split(","):
        n_gen, clusters, mink, maxk = SHAPES[shape]
        per = n_gen // clusters
        texts = []
        for c in range(clusters):
            root = synth_fasta(args.bases, 1, seed=2000 + c, device=eng.device)
            texts += [mutate_text(root, 0.01, seed=200 * c + i) for i in range(per)]
        files = []
        for g, t in enumerate(texts):
            files.append(os.path.join(work, "%s_g%03d.fa" % (shape, g)))
            t.cpu().numpy().tofile(files[-1])
        st = ddstore.GpuSketchStore(engine=eng)
        seqs = [st.packed(f) for f in files]
        rng = np.random.default_rng(4)
        orderings = [rng.permutation(n_gen).tolist() for _ in range(args.orderings)]
        rows, checks = [], []
        ks = list(range(mink, maxk + 1))
        eng.exact_spectrum(seqs, ks[0], True)                 # warm-up: module load, workspace
        torch.cuda.synchronize()
        for i, k in enumerate(ks):
            row = {"k": k}
            bounds = length_bounds([s.nsym for s in seqs], k)   # the spectrum job's own sizing, so both plans are equal
            for which in (("spectrum", "sampled") if i % 2 == 0 else ("sampled", "spectrum")):
                l0, t0 = lib.dd_kernel_launches(), time.perf_counter()
                if which == "spectrum":
                    hist, singles, priv = eng.exact_spectrum(seqs, k, True)
                else:
                    prefix = st.exact_prefix_cards(files, orderings, [k], True, singles=np.array(bounds)[:, None])
                row[which + "_s"] = time.perf_counter() - t0
                row[which + "_launches"] = lib.dd_kernel_launches() - l0
                row[which + "_passes"] = eng.last_pair_plan["passes"]
            card, core = mean_growth(hist)
            row["union_all"] = int(hist.sum())
            row["core_all"] = int(hist[-1])
            row["singles_equal_sampled"] = prefix[:, 0, 0].tolist() == [int(singles[o[0]]) for o in orderings]
            row["union_equal_sampled"] = bool((prefix[:, -1, 0] == hist.sum()).all())
            row["sampled_mean_vs_exact_max_rel"] = float(np.max(np.abs(prefix[:, :, 0].mean(axis=0) - card) / card))
            rows.append(row)
            print(json.dumps(dict(row, shape=shape)), flush=True)
            if not (row["singles_equal_sampled"] and row["union_equal_sampled"]):
                raise SystemExit("spectrum and prefix job disagree at k=%d" % k)
            if shape == "config2" and k in (12, 21, 32):
                checks.append(oracle_check(texts, k, hist, priv))
        report["shapes"][shape] = dict(genomes=n_gen, clusters=clusters, ks=ks, rows=rows, oracle_cells=checks,
                                       spectrum_total_s=sum(r["spectrum_s"] for r in rows),
                                       sampled_total_s=sum(r["sampled_s"] for r in rows))
        del st, seqs, texts
        for f in files:
            os.remove(f)
    os.rmdir(work)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(report, fh, indent=1)
    print(json.dumps({s: {k: v for k, v in r.items() if k.endswith("_s")} for s, r in report["shapes"].items()}))


if __name__ == "__main__":
    main()
