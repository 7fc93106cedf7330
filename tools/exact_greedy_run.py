#!/usr/bin/env python3
"""K12 exact greedy ordering (store.exact_greedy_order) on one GPU, against the per-step K8 route and the HLL order.

Shapes (k = 10..32, canonical):
  (a) 12 x 5 Mbp: 12 mutated copies (2 % substitutions) of one synthetic ancestor;
  (b) 100 x 5 Mbp in clusters of 10 mutated copies (2 % substitutions), as tools/leaveout_run.py builds config 5.
The FASTAs are generated on the device (tools/synth.py) and written to a temporary directory; packing is not timed.

  index     Engine.exact_cover_index per k, timed by CUDA events (the K7 list job, the count read-back, the index
            allocation and the emit); its device bytes against the formula 6 B x sum |A_g| + 5 B x distinct keys.
  order     the whole order by store.exact_greedy_order, host clock with a device synchronise at the end (index
            build included), then its steps replayed on a fresh index: each K12 step launch timed by CUDA events.
  k8        the per-step baseline: store.exact_union_cards over every (chosen + candidate) set, timed by the host
            clock for the first --k8-steps steps (one K7 list job + K8 per k each); its picks and cards must equal
            K12's.  Scaled to the whole order it is an extrapolation, labelled as one.
  hll       the HLL order (store.greedy_order, p = 20) of the same FASTAs: the first step where it differs from the
            exact order (informative only).
The card name and power limit are read in the same run.

    python tools/exact_greedy_run.py --out profiles/r10_exact_greedy.json"""
import argparse
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


def write_genomes(directory, n, per_cluster, bases, seed, dev):
    paths, anc = [], None
    for g in range(n):
        if g % per_cluster == 0:
            anc = synth_fasta(int(bases), 1, seed=seed + g // per_cluster, device=dev)
        text = mutate_text(anc, 0.02, seed * 100 + g)
        path = os.path.join(directory, "g%04d.fasta" % g)
        with open(path, "wb") as fh:
            fh.write(text.cpu().numpy().tobytes())
        paths.append(path)
    return paths


def shape_run(eng, fastas, ks, k8_steps, label):
    from dandd_b200 import store as ddstore
    st = ddstore.GpuSketchStore(engine=eng)
    seqs = [st.packed(f) for f in fastas]
    n = len(fastas)
    torch.cuda.synchronize()

    index = []
    for k in ks:                                   # index build per k, device events; freed before the next k
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ix = eng.exact_cover_index(seqs, k, True)
        b.record()
        b.synchronize()
        nodes = sum(p["n_nodes"] for p in ix["parts"])
        index.append({"k": k, "build_ms": a.elapsed_time(b), "bytes": ix["bytes"], "formula_bytes": 6 * nodes + 5 * ix["keys"],
                      "distinct_keys": ix["keys"], "nodes": nodes, "passes": len(ix["parts"])})
        del ix

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    order, cards, stats = st.exact_greedy_order(fastas, ks, True, n)
    torch.cuda.synchronize()
    whole_s = time.perf_counter() - t0

    indices = [eng.exact_cover_index(seqs, k, True) for k in ks]      # the same steps, each K12 launch timed
    lost = torch.zeros((len(ks), n), dtype=torch.int64, device=eng.device)
    step_ms = []
    for g in order.tolist():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.exact_cover_step(indices, g, lost)
        b.record()
        b.synchronize()
        step_ms.append(a.elapsed_time(b))
    del indices, lost

    k8_s, k8_picks, k8_cards = [], [], []
    for t in range(min(k8_steps, n)):
        cand = [g for g in range(n) if g not in k8_picks]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = st.exact_union_cards(fastas, [k8_picks + [g] for g in cand], ks, True)
        torch.cuda.synchronize()
        k8_s.append(time.perf_counter() - t0)
        d = [max(got[i, c] / k for c, k in enumerate(ks)) for i in range(len(cand))]
        best = d.index(max(d))
        k8_picks.append(cand[best])
        k8_cards.append(got[best].tolist())
    k8_equal = k8_picks == order.tolist()[:len(k8_picks)] and k8_cards == cards[:len(k8_picks)].tolist()

    p = 20
    regs = torch.empty((n, len(ks), 1 << p), dtype=torch.uint8, device=eng.device)
    hist = torch.empty((len(ks), 64), dtype=torch.int32, device=eng.device)
    for g, s in enumerate(seqs):
        eng.sketch(s, ks, p=p, out=regs[g], hist_out=hist)
    hll_order, _, _ = st.greedy_order(regs, ks, p, n)
    del regs
    differ = [t for t in range(n) if hll_order[t] != order[t]]

    med_step = float(np.median(step_ms))
    return {"shape": label, "n": n, "ks": [ks[0], ks[-1]], "index_per_k": index,
            "index_build_ms_total": sum(x["build_ms"] for x in index),
            "index_bytes_total": sum(x["bytes"] for x in index),
            "formula_bytes_total": sum(x["formula_bytes"] for x in index),
            "whole_order_host_s_including_index_build": whole_s, "stats_distinct_keys_equal_index":
                stats["distinct_keys"] == [x["distinct_keys"] for x in index],
            "step_ms": step_ms, "step_ms_median": med_step, "step_ms_total": float(np.sum(step_ms)),
            "k8_steps_timed": len(k8_s), "k8_step_s": k8_s, "k8_step_s_mean": float(np.mean(k8_s)),
            "k8_whole_order_s_extrapolated": float(np.mean(k8_s)) * n,
            "k8_picks_and_cards_equal_k12": bool(k8_equal),
            "hll_p20_first_differing_step": (differ[0] + 1) if differ else None,
            "hll_p20_steps_differing": len(differ)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--bases", type=float, default=5e6)
    ap.add_argument("--k8-steps", type=int, default=3)
    ap.add_argument("--shapes", default="a,b")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_exact_greedy.json"))
    args = ap.parse_args()
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    eng = Engine(0)
    ks = list(range(10, 33))
    rep = dict(card_info(), shapes=[])
    for shape in args.shapes.split(","):
        n, per = (12, 12) if shape == "a" else (100, 10)
        with tempfile.TemporaryDirectory() as tmp:
            fastas = write_genomes(tmp, n, per, args.bases, 7000 if shape == "a" else 5000, eng.device)
            label = "(%s) %d x %.0f bp, %d mutated copies (2 %%) per ancestor, k = 10..32" % (shape, n, args.bases, per)
            rep["shapes"].append(shape_run(eng, fastas, ks, args.k8_steps, label))
        print(json.dumps({k: v for k, v in rep["shapes"][-1].items() if k not in ("index_per_k", "step_ms")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    if not all(s["k8_picks_and_cards_equal_k12"] and s["stats_distinct_keys_equal_index"] for s in rep["shapes"]):
        raise SystemExit("the K12 order disagrees with the K8 steps: see %s" % args.out)


if __name__ == "__main__":
    main()
