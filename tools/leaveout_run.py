#!/usr/bin/env python3
"""K10 leave-one-out histograms at the config-5 shape, against the per-union path, on one GPU.

Shape (BASELINE.json config 5): 1000 synthetic 5 Mbp genomes in clusters of 10 mutated copies (2 % substitutions,
as tools/config5_run.py builds them), k = 10..32, p = 18: 1000 x 23 x 2^18 registers = 6.0 GB, sketched on the
device and kept there (sketching is not timed).

  k10       Engine.leave_out_hist with every genome its own group (1000 leave-outs), timed by CUDA events around
            each of --reps calls after one untimed call.  The event window covers the whole entry point: the group
            table's round trip, the member upload, K10 and its finishing kernel.  Algorithmic bytes = n nk 2^p (each
            register read once); bytes / time is set against the HBM bandwidth measured in the same run (a 4 GiB
            device-to-device copy: read + write bytes over time) and the data sheet's 7.7 TB/s.
  per-union the union of the other 999 genomes for --subset leave-outs, all k in one K3 launch each
            (Engine.union_sets over the 999 member sketches, as a SubSpider's union goes), alternated with K10 in
            this process; scaled to 1000 leave-outs that is an extrapolation, labelled as one.
  check     the K10 cards of those leave-outs equal the per-union cards (same histograms, same MLE: ==); a few
            (genome, k) cells equal the oracle's estimator over explicit maxima of the device registers (to 1e-9: the
            oracle's MLE is the sequential form); genome 0's
            registers at two k equal the oracle's sketch.
The card name and power limit are read in the same run.

    python tools/leaveout_run.py --out profiles/r08_leaveout.json"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.exact_pairs_run import card_info  # noqa: E402
from tools.synth import mutate_text, synth_fasta  # noqa: E402


def events(fn, reps):
    """Per-call milliseconds by CUDA events, one pair per call."""
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--bases", type=float, default=5e6)
    ap.add_argument("--p", type=int, default=18)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--subset", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_leaveout.json"))
    args = ap.parse_args()
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    from oracle import pyoracle as orc
    eng = Engine(0)
    dev = eng.device
    ks = list(range(10, 33))
    n, nk, p = args.genomes, len(ks), args.p
    m = 1 << p
    regs = torch.empty((n, nk, m), dtype=torch.uint8, device=dev)
    hist = torch.empty((nk, 64), dtype=torch.int32, device=dev)
    anc, text0 = None, None
    t0 = time.perf_counter()
    for g in range(n):
        if g % 10 == 0:
            anc = synth_fasta(int(args.bases), 1, seed=5000 + g // 10, device=dev)
        text = anc if g % 10 == 0 else mutate_text(anc, 0.02, 50000 + g)
        if g == 0:
            text0 = text.cpu().numpy().tobytes()
        eng.sketch(eng.pack(text, start=0), ks, p=p, out=regs[g], hist_out=hist)
    torch.cuda.synchronize()
    t_sketch = time.perf_counter() - t0

    # HBM bandwidth of this card, measured here: a device-to-device copy
    src = torch.empty(1 << 32, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    copy_ms = events(lambda: dst.copy_(src), 10)
    hbm = 2 * src.numel() / (np.median(copy_ms) / 1e3)
    del src, dst

    group = np.arange(n, dtype=np.int32)
    algo_bytes = n * nk * m
    k10 = lambda: eng.leave_out_hist(regs, group, n, p)                  # noqa: E731
    subset = np.linspace(0, n - 1, args.subset).astype(int)
    base = regs.data_ptr()
    tables = [base + (np.delete(np.arange(n), g)[None, :] * nk + np.arange(nk)[:, None]) * m for g in subset]   # [nk, n - 1]
    per_union = lambda: [eng.union_sets(t, p, final_only=True) for t in tables]   # noqa: E731
    k10()
    per_union()
    torch.cuda.synchronize()
    t_k10, t_pu = [], []
    for r in range(args.rounds):                                          # alternated, order swapped every round
        for which in ((0, 1) if r % 2 == 0 else (1, 0)):
            if which == 0:
                t_k10 += events(k10, args.reps)
            else:
                t_pu += events(per_union, 1)

    out = k10()
    cards = eng.mle(out, p).cpu().numpy()                                 # [nk, 1 + n]
    pu = np.stack([c.cpu().numpy().reshape(nk) for c in per_union()])     # [subset, nk]
    equal_per_union = bool(np.array_equal(pu, cards[:, 1 + subset].T))
    oracle_cells = []
    for c in (0, nk // 2, nk - 1):
        host = regs[:, c].cpu().numpy()
        for g in subset[:3]:
            want = orc.card(np.delete(host, g, axis=0).max(axis=0), p)
            oracle_cells.append({"k": ks[c], "genome": int(g), "k10": float(cards[c, 1 + g]), "oracle": want,
                                 "equal": abs(float(cards[c, 1 + g]) - want) <= 1e-9 * want})
        want = orc.card(host.max(axis=0), p)
        oracle_cells.append({"k": ks[c], "genome": "union", "k10": float(cards[c, 0]), "oracle": want,
                             "equal": abs(float(cards[c, 0]) - want) <= 1e-9 * want})
    sym0 = orc.fasta_symbols(text0)
    regs_ok = all(np.array_equal(regs[0, c].cpu().numpy(), orc.hll_sketch(sym0, ks[c], p)) for c in (0, nk - 1))

    med_k10 = float(np.median(t_k10))
    med_pu = float(np.median(t_pu))
    rep = dict(card_info(), shape="config 5: %d x %.0f bp clustered (10 per cluster), k = 10..32, p = %d" % (n, args.bases, p),
               register_bytes=algo_bytes, sketch_s_untimed_setup=t_sketch,
               hbm_copy_GB_per_s_measured=hbm / 1e9, k10_call_ms=t_k10, k10_call_ms_median=med_k10,
               k10_algorithmic_GB_per_s=algo_bytes / (med_k10 / 1e3) / 1e9,
               k10_share_of_measured_hbm=algo_bytes / (med_k10 / 1e3) / hbm,
               k10_share_of_datasheet_7p7TBs=algo_bytes / (med_k10 / 1e3) / 7.7e12,
               per_union_subset=int(args.subset), per_union_subset_ms=t_pu, per_union_subset_ms_median=med_pu,
               per_union_1000_ms_extrapolated=med_pu * n / args.subset,
               speedup_extrapolated=med_pu * n / args.subset / med_k10,
               k10_equals_per_union=equal_per_union, oracle_cells=oracle_cells,
               oracle_cells_equal=all(x["equal"] for x in oracle_cells), genome0_registers_equal_oracle=bool(regs_ok),
               launches_per_k10_call="K10 + finishing kernel (2), plus a memset and two small copies")
    print(json.dumps(rep))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    if not (equal_per_union and rep["oracle_cells_equal"] and regs_ok):
        raise SystemExit("leave-out cards disagree: see %s" % args.out)


if __name__ == "__main__":
    main()
