#!/usr/bin/env python3
"""Exact all pairs (K7) on one GPU: 100 clustered synthetic genomes of 5 Mbp (tools/synth.py; 10 clusters of
10 copies of a random root, 1 % substitutions each) at k = 10..32, 40, 64, 99 -- the klist of an exact
`helpers/allpairs.py --tool kmc` run.  Per k it reports the path the engine took, its passes, sum(occ^2)
over the k-mers (= 2 sum|A n B| + sum|A|: the work of the list path), the wall time of the batched job
(host clock around work that ends in a device synchronise) and the kernel launches it made.

A 20-genome subset also runs through the per-pair path (one exact_counts call per pair, as before K7): every
count must be equal, and its time per pair is scaled to 100 genomes -- labelled as an extrapolation.  A few
cells are checked against the CPU oracle, and both paths are timed at k = 12..15, around the switch of the rule
that picks one (engine.dense_pairs).  The card name and power limit are read in the same run.

    python tools/exact_pairs_run.py --out profiles/r03_exact_pairs.json"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info():
    try:
        line = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in line.splitlines()[0].split(",")]
        return {"card": name, "power_limit": power}
    except (OSError, subprocess.CalledProcessError, ValueError):
        import torch
        return {"card": torch.cuda.get_device_name(0), "power_limit": "unknown"}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--genomes", type=int, default=100)
    ap.add_argument("--clusters", type=int, default=10)
    ap.add_argument("--bases", type=int, default=5_000_000)
    ap.add_argument("--subset", type=int, default=20)
    ap.add_argument("--klist", default=",".join(str(k) for k in list(range(10, 33)) + [40, 64, 99]))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_exact_pairs.json"))
    args = ap.parse_args()

    import torch
    from dandd_b200 import build
    build.build()
    from dandd_b200 import _lib, engine as E
    from tools.synth import mutate_text, synth_fasta
    eng = E.Engine(0)
    lib = eng.lib
    ks = [int(k) for k in args.klist.split(",")]
    per = max(1, args.genomes // args.clusters)
    texts = []
    for c in range(args.clusters):
        root = synth_fasta(args.bases, 1, seed=1000 + c, device=eng.device)
        texts += [mutate_text(root, 0.01, seed=100 * c + i) for i in range(per)]
    texts = texts[:args.genomes]
    seqs = [eng.pack(t).check() for t in texts]
    n = len(seqs)
    sub = list(range(0, n, max(1, n // args.subset)))[:args.subset]   # two per cluster: pairs inside and across clusters
    torch.cuda.synchronize()

    rows = []
    for k in ks:
        t0 = time.perf_counter()
        singles = [eng.exact_counts([s], k)[0] for s in seqs]
        t_single = time.perf_counter() - t0
        l0 = _lib.load().dd_kernel_launches()
        t0 = time.perf_counter()
        inter = eng.exact_pair_intersections(seqs, k, True, singles)
        t_pairs = time.perf_counter() - t0
        launches = lib.dd_kernel_launches() - l0
        plan = dict(eng.last_pair_plan)
        sub_seqs = [seqs[g] for g in sub]
        sub_singles = [singles[g] for g in sub]
        t0 = time.perf_counter()
        sub_inter = eng.exact_pair_intersections(sub_seqs, k, True, sub_singles)
        t_sub_batched = time.perf_counter() - t0
        t0 = time.perf_counter()
        per_pair = [eng.exact_counts([sub_seqs[a], sub_seqs[b]], k)[-1]
                    for a in range(len(sub)) for b in range(a + 1, len(sub))]
        t_sub_pairs = time.perf_counter() - t0
        iu = np.triu_indices(len(sub), 1)
        batched_unions = (np.asarray(sub_singles, dtype=np.int64)[iu[0]] + np.asarray(sub_singles, dtype=np.int64)[iu[1]]
                          - sub_inter.astype(np.int64))
        # the subset's rows of the 100-genome job must be the subset job's
        full_rows = [a * n - a * (a + 1) // 2 + (b - a - 1) for a, b in zip(np.asarray(sub)[iu[0]], np.asarray(sub)[iu[1]])]
        equal = batched_unions.tolist() == per_pair and inter[full_rows].tolist() == sub_inter.tolist()
        sub_pairs = len(per_pair)
        rows.append({
            "k": k, "path": plan["path"], "passes": plan["passes"],
            "sum_occ_sq": int(2 * int(inter.astype(np.uint64).sum()) + sum(singles)),
            "mean_single": float(np.mean(singles)),
            "batched_s": t_pairs, "singles_s": t_single, "launches": int(launches),
            "subset_batched_s": t_sub_batched, "subset_per_pair_s": t_sub_pairs,
            "per_pair_extrapolated_to_all_pairs_s": t_sub_pairs / sub_pairs * (n * (n - 1) // 2),
            "subset_counts_equal_per_pair": bool(equal),
        })
        print(json.dumps(rows[-1]), flush=True)
        if not equal:
            raise SystemExit("k=%d: batched counts differ from the per-pair path" % k)

    # the dense/sparse crossover: both engine-level paths on all genomes at the k values around the rule's switch
    crossover = []
    for k in (12, 13, 14, 15):
        singles = [eng.exact_counts([s], k)[0] for s in seqs]
        t0 = time.perf_counter()
        dense = eng.exact_pairs_dense(seqs, k, True)
        t_dense = time.perf_counter() - t0
        t0 = time.perf_counter()
        sparse = eng.exact_pairs_sparse(seqs, k, True, singles)
        t_sparse = time.perf_counter() - t0
        crossover.append({"k": k, "rule_picks": "dense" if E.dense_pairs(k, singles) else "sparse",
                          "kmer_space_over_mean_single": 4 ** k / float(np.mean(singles)),
                          "dense_s": t_dense, "sparse_s": t_sparse, "equal": dense.tolist() == sparse.tolist()})
        print(json.dumps(crossover[-1]), flush=True)
        if not crossover[-1]["equal"]:
            raise SystemExit("k=%d: dense and sparse paths differ" % k)

    # a few cells against the CPU oracle (whole 5 Mbp genomes)
    from oracle import pyoracle as orc
    checks = []
    for (a, b, k) in [(0, 1, 21), (0, per, 40), (1, 2, 12)]:
        if k not in ks or b >= n:
            continue
        sa, sb = orc.fasta_symbols(texts[a].cpu().numpy().tobytes()), orc.fasta_symbols(texts[b].cpu().numpy().tobytes())
        want = orc.exact_count([sa, sb], k)
        singles = [eng.exact_counts([seqs[g]], k)[0] for g in (a, b)]
        inter = int(eng.exact_pair_intersections([seqs[a], seqs[b]], k, True, singles)[0])
        checks.append({"a": a, "b": b, "k": k, "oracle_union": want, "batched_union": singles[0] + singles[1] - inter})
        if checks[-1]["oracle_union"] != checks[-1]["batched_union"]:
            raise SystemExit("oracle mismatch: %s" % checks[-1])

    rep = dict(card_info(), genomes=n, bases=args.bases, clusters=args.clusters, subset=len(sub), ks=ks,
               dense_bits_per_kmer=E.DENSE_BITS_PER_KMER, rows=rows, crossover=crossover, oracle_cells=checks,
               timing="host clock around each call; every call ends in a device->host copy of its result",
               extrapolation="per_pair_extrapolated_to_all_pairs_s = subset per-pair time / subset pairs x all pairs (not measured)")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
