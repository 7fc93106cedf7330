#!/usr/bin/env python3
"""Queries against a collection (helpers/query.py) on one GPU: K13 against K7 on the same lists, and the whole helper at
the config-5 shape.

Genomes are synthetic (tools/synth.py) in clusters of 10 mutated copies (2 % substitutions) of one ancestor, written to a
temporary directory; queries are further mutated copies (2 %) of the first genome of some clusters.

  (a) 10 queries against 100 x 5 Mbp references, k = 10..32, exact.  Per k, one K7 list job over references + queries;
      on its lists, --reps alternating launches of K13 (dd_exact_query_counts) and K7 accumulate over all R + Q genomes
      (dd_exact_pairs_accumulate), each timed by CUDA events.  The increments each one counts, from its own output:
      sum q_on r_on (the sum of K13's Q x R block) against sum occ (occ - 1) / 2 (the sum of K7's triangle).  Checks on
      the same lists: K13's Q x R block equals the (reference, query) cells of K7's triangle, |U_R| and |U_R u A_q| equal
      K8's set rows; a few cells equal the oracle's k-mer sets.
  (b) 1 and 10 queries against the config-5 shape (1000 x 5 Mbp references, k = 10..32, p = 18), dashing: the whole
      helper in this process, host clock, a fresh store per run (sketching of every genome included; the FASTA files
      are in the page cache).  Checks: a few with.tsv cells equal the oracle's MLE over np.maximum of the device
      registers of the references and the query (to 1e-9 relative).
The card name and power limit are read in the same run.

    python tools/query_run.py --out profiles/r11_query.json"""
import argparse
import csv
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.exact_pairs_run import card_info  # noqa: E402
from tools.synth import mutate_text, synth_fasta  # noqa: E402


def write_genomes(directory, n_refs, n_queries, bases, seed, dev):
    """(references, queries): n_refs genomes in clusters of 10, then n_queries mutated copies of cluster heads."""
    os.makedirs(os.path.join(directory, "refs"))
    os.makedirs(os.path.join(directory, "queries"))
    refs, queries, heads = [], [], []
    for g in range(n_refs):
        if g % 10 == 0:
            anc = synth_fasta(int(bases), 1, seed=seed + g // 10, device=dev)
            heads.append(anc)
        text = anc if g % 10 == 0 else mutate_text(anc, 0.02, seed * 10 + g)
        refs.append(os.path.join(directory, "refs", "r%04d.fasta" % g))
        with open(refs[-1], "wb") as fh:
            fh.write(text.cpu().numpy().tobytes())
    for q in range(n_queries):
        text = mutate_text(heads[(3 * q) % len(heads)], 0.02, seed * 10 + 100000 + q)
        queries.append(os.path.join(directory, "queries", "q%02d.fasta" % q))
        with open(queries[-1], "wb") as fh:
            fh.write(text.cpu().numpy().tobytes())
    return refs, queries


def shape_a(eng, refs, queries, ks, reps):
    from dandd_b200 import store as ddstore
    from dandd_b200._lib import check
    from dandd_b200.engine import length_bounds
    from oracle import pyoracle as orc
    st = ddstore.GpuSketchStore(engine=eng)
    seqs = [st.packed(f) for f in refs + queries]
    R, Q, n = len(refs), len(queries), len(refs) + len(queries)
    lib, stream, dev = eng.lib, eng.stream, eng.device
    tri_cells = n * (n - 1) // 2
    per_k, ok = [], True
    for k in ks:
        rec = {"k": k, "k13_ms": [], "k7_ms": []}
        ranks = np.full((1 + Q, n), 0xFFFF, dtype=np.uint16)
        ranks[:, :R] = 0
        ranks[1 + np.arange(Q), R + np.arange(Q)] = 0
        d_ranks = torch.from_numpy(ranks.view(np.int16)).to(dev)

        def launch(ws, cap, nodes, part):
            check(lib.dd_exact_query_counts(ws.data_ptr(), ws.numel(), k, cap, nodes, n, R, Q, part, part + 8 * Q * R,
                                            part + 8 * (Q * R + Q), stream))

        def after(ws, cap, nodes, got):
            inter = torch.zeros(Q * R + Q + 1, dtype=torch.int64, device=dev)
            tri = torch.zeros(tri_cells, dtype=torch.int64, device=dev)
            for _ in range(reps):          # alternated on the same lists
                for which, out in (("k13", inter), ("k7", tri)):
                    out.zero_()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    if which == "k13":
                        launch(ws, cap, nodes, out.data_ptr())
                    else:
                        check(lib.dd_exact_pairs_accumulate(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, out.data_ptr(), stream))
                    b.record()
                    b.synchronize()
                    rec[which + "_ms"].append(a.elapsed_time(b))
            hist = torch.zeros(ranks.size, dtype=torch.int64, device=dev)
            check(lib.dd_exact_first_rank_hist(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, d_ranks.data_ptr(), 1 + Q,
                                               hist.data_ptr(), stream))
            rec["after"] = (inter.cpu().numpy(), tri.cpu().numpy(), hist.cpu().numpy().reshape(1 + Q, n))

        got, singles = eng._list_job(seqs, k, True, length_bounds([s.nsym for s in seqs], k), None, None, Q * R + Q + 1, True,
                                     launch, "overflow", after=after)
        inter, tri, hist = rec.pop("after")
        block = inter[:Q * R].reshape(Q, R)
        rows = np.array([[r * (2 * n - r - 1) // 2 + (R + q - r - 1) for r in range(R)] for q in range(Q)])
        union = int(inter[-1])
        with_q = union + singles[R:].astype(np.int64) - inter[Q * R:Q * R + Q]
        rec.update(passes=eng.last_pair_plan["passes"],
                   k13_ms_median=float(np.median(rec["k13_ms"])), k7_ms_median=float(np.median(rec["k7_ms"])),
                   increments_k13=int(block.sum()), increments_k7=int(tri.sum()),
                   block_equals_k7=bool(np.array_equal(block, tri[rows])),
                   sets_equal_k8=bool(union == hist[0, 0] and np.array_equal(with_q, hist[1:, 0])),
                   job_equals_timed=bool(np.array_equal(got.astype(np.int64), inter)))
        if k in (ks[0], 21, ks[-1]):   # oracle k-mer sets: the singles and (query 0, reference 0..2)
            sets = [np.unique(orc.kmers(orc.fasta_symbols(open(f, "rb").read()), k, True)) for f in [queries[0]] + refs[:3]]
            rec["oracle_cells_equal"] = bool(
                [int(singles[R])] + [int(singles[r]) for r in range(3)] == [a.size for a in sets]
                and [int(block[0, r]) for r in range(3)] == [np.intersect1d(sets[0], sets[1 + r]).size for r in range(3)])
            ok &= rec["oracle_cells_equal"]
        ok &= rec["block_equals_k7"] and rec["sets_equal_k8"] and rec["job_equals_timed"]
        per_k.append(rec)
        print(json.dumps({x: y for x, y in rec.items() if not x.endswith("_ms")}), flush=True)
    return {"shape": "(a) %d queries against %d references, exact, k = %d..%d" % (Q, R, ks[0], ks[-1]), "per_k": per_k,
            "k13_ms_total": sum(r["k13_ms_median"] for r in per_k), "k7_ms_total": sum(r["k7_ms_median"] for r in per_k),
            "increments_k13_total": sum(r["increments_k13"] for r in per_k),
            "increments_k7_total": sum(r["increments_k7"] for r in per_k), "checks_pass": bool(ok)}


def shape_b(eng, refs, queries, ks, p, tmp):
    from dandd_b200 import store as ddstore
    from dandd_b200.helpers import query
    from oracle import pyoracle as orc
    runs, ok = [], True
    for nq in (1, len(queries)):
        qlist = os.path.join(tmp, "q%d.txt" % nq)
        with open(qlist, "w") as fh:
            fh.write("\n".join(queries[:nq]) + "\n")
        st = ddstore.GpuSketchStore(engine=eng)
        ddstore.set_store(st)
        name = os.path.join(tmp, "run%d" % nq)
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            cards = query.go(["-d", os.path.dirname(refs[0]), "--query-list", qlist, "--mink", str(ks[0]), "--maxk", str(ks[-1]),
                              "--registers", str(p), "--name", name])
            torch.cuda.synchronize()
            secs = time.perf_counter() - t0
            with open(os.path.join(name, "with.tsv"), newline="") as fh:
                with_rows = list(csv.DictReader(fh, delimiter="\t"))
            checks, cols = [], (0, len(ks) // 2)
            leaf = lambda f: eng.sketch(eng.pack(open(f, "rb").read()), [ks[c] for c in cols], p)[0]
            union = leaf(refs[0])
            for f in refs[1:]:                     # oracle MLE over explicit maxima of the device registers
                union = torch.maximum(union, leaf(f))
            qr = torch.maximum(union, leaf(queries[0])).cpu().numpy()
            for i, c in enumerate(cols):
                want = orc.card(qr[i], p)
                got = float(with_rows[c * nq]["card"])
                checks.append({"k": ks[c], "helper": got, "oracle": want, "rel": abs(got - want) / want})
                ok &= abs(got - want) <= 1e-9 * want
        finally:
            ddstore.set_store(None)
        runs.append({"queries": nq, "helper_host_s": secs, "oracle_checks": checks,
                     "union_card_k_first": float(cards[2][0]), "pairs": int(cards[4][0].size)})
        print(json.dumps(runs[-1]), flush=True)
    return {"shape": "(b) 1 and %d queries against %d references, dashing, k = %d..%d, p = %d" % (
        len(queries), len(refs), ks[0], ks[-1], p), "runs": runs, "checks_pass": bool(ok)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--bases", type=float, default=5e6)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="a,b")
    ap.add_argument("--refs-b", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_query.json"))
    args = ap.parse_args()
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    eng = Engine(0)
    ks = list(range(10, 33))
    rep = dict(card_info(), shapes=[])
    for shape in args.shapes.split(","):
        with tempfile.TemporaryDirectory() as tmp:
            if shape == "a":
                refs, queries = write_genomes(tmp, 100, 10, args.bases, 5000, eng.device)
                rep["shapes"].append(shape_a(eng, refs, queries, ks, args.reps))
            else:
                refs, queries = write_genomes(tmp, args.refs_b, 10, args.bases, 5000, eng.device)
                rep["shapes"].append(shape_b(eng, refs, queries, ks, 18, tmp))
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    if not all(s["checks_pass"] for s in rep["shapes"]):
        raise SystemExit("a check failed: see %s" % args.out)


if __name__ == "__main__":
    main()
