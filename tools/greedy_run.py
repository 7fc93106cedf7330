#!/usr/bin/env python3
"""K11 greedy ordering at the config-5 shape on one GPU: the whole order, its phases, and the K6 per-step baseline.

Shape (BASELINE.json config 5): 1000 synthetic 5 Mbp genomes in clusters of 10 mutated copies (2 % substitutions, as
tools/leaveout_run.py builds them), k = 10..32, p = 18: 6.0 GB of registers, sketched on the device (not timed).

  order      GpuSketchStore.greedy_order over all 1000 steps, host clock around the call (it ends in a device read),
             with the store's dense/sparse selection and with the sparse phase off (budget 0): same order, same cards?
  phases     replaying that order: per step t in a sample, CUDA events around the dense step over the remaining
             candidates (bytes = C nk 2^p + nk 2^p over its time, against a device-to-device copy of this run), the
             MLE of the C nk rows, and the pick + union update + K4 of U; the compaction at the store's switch step;
             then dense and sparse steps alternated on the same steps after the switch, histograms compared.
  k6         the per-step baseline: U written as one more sketch into bit planes of all genomes, then
             Engine.pairwise_cards of every (candidate, U) pair (K6), on three windows of 20 steps; picks and cards
             equal to K11's; scaled by the candidate count to the whole order, an extrapolation.
The card name and power limit are read in the same run.

    python tools/greedy_run.py --out profiles/r09_greedy.json"""
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
from tools.leaveout_run import events  # noqa: E402
from tools.synth import mutate_text, synth_fasta  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--bases", type=float, default=5e6)
    ap.add_argument("--p", type=int, default=18)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_greedy.json"))
    args = ap.parse_args()
    from dandd_b200 import build
    build.build()
    from dandd_b200 import store as ddstore
    from dandd_b200.engine import Engine
    eng = Engine(0)
    st = ddstore.GpuSketchStore(engine=eng)
    dev = eng.device
    ks = list(range(10, 33))
    n, nk, p = args.genomes, len(ks), args.p
    m = 1 << p
    regs = torch.empty((n, nk, m), dtype=torch.uint8, device=dev)
    hist = torch.empty((nk, 64), dtype=torch.int32, device=dev)
    anc = None
    for g in range(n):
        if g % 10 == 0:
            anc = synth_fasta(int(args.bases), 1, seed=5000 + g // 10, device=dev)
        text = anc if g % 10 == 0 else mutate_text(anc, 0.02, 50000 + g)
        eng.sketch(eng.pack(text, start=0), ks, p=p, out=regs[g], hist_out=hist)
    torch.cuda.synchronize()

    src = torch.empty(1 << 32, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    copy_ms = events(lambda: dst.copy_(src), 10)
    hbm = 2 * src.numel() / (np.median(copy_ms) / 1e3)
    del src, dst

    # ---- the whole order, both selections (the first call also warms every shape)
    st.greedy_order(regs, ks, p, 30)
    runs = {}
    for label, budget in (("selected", None), ("dense_only", 0), ("selected_again", None)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        order, cards, stats = st.greedy_order(regs, ks, p, n, budget=budget)
        runs[label] = dict(seconds=time.perf_counter() - t0, order=order, cards=cards, stats=stats)
    order, stats = runs["selected"]["order"], runs["selected"]["stats"]
    same = all(np.array_equal(runs[x]["order"], order) and np.array_equal(runs[x]["cards"], runs["selected"]["cards"])
               for x in runs)

    # ---- phases, replaying the order
    kdiv = torch.tensor(ks, dtype=torch.float64, device=dev)

    def union_at(t):
        u = torch.zeros((nk, m), dtype=torch.uint8, device=dev)
        for g in order[:t]:
            u = torch.maximum(u, regs[int(g)])
        return u

    sample = [1, 2, 5, 10, 20, 50, 100, 200, 400, 700, 999]
    per_step = []
    for t in sample:
        u = union_at(t)
        _, uh = eng.cards_hist(u, p)
        rest = sorted(set(range(n)) - set(int(g) for g in order[:t]))
        h, live = eng.greedy_dense_hist(regs, u, uh, rest, p)
        d_ms = float(np.median(events(lambda: eng.greedy_dense_hist(regs, u, uh, rest, p), 5)))
        mle_ms = float(np.median(events(lambda: eng.mle(h, p), 5)))
        chosen = torch.zeros(n, dtype=torch.bool, device=dev)

        def pick_update():
            full = torch.zeros((n, nk), dtype=torch.float64, device=dev)
            full[torch.as_tensor(rest, device=dev)] = eng.mle(h, p)
            pk = (full / kdiv).amax(dim=1).masked_fill(chosen, float("-inf")).argmax()
            eng.cards_hist(torch.maximum(u, regs.index_select(0, pk.view(1))[0]), p)
        pu_ms = float(np.median(events(pick_update, 5)))
        nbytes = (len(rest) + 1) * nk * m
        live_n = int(live.to(torch.int64).sum())
        per_step.append(dict(step=t, candidates=len(rest), live=live_n, live_fraction=live_n / (len(rest) * nk * m),
                             dense_ms=d_ms, dense_GB_per_s=nbytes / d_ms / 1e6, dense_share_of_copy=nbytes / (d_ms / 1e3) / hbm,
                             mle_ms=mle_ms, mle_pick_update_k4_ms=pu_ms))

    alternated, compact_ms = [], None
    s0 = stats["switch_step"]
    if s0 is not None:
        u_prev, u = union_at(s0 - 1), union_at(s0)
        _, uh = eng.cards_hist(u_prev, p)
        cand = sorted(set(range(n)) - set(int(g) for g in order[:s0 - 1]))
        _, live = eng.greedy_dense_hist(regs, u_prev, uh, cand, p)
        counts = np.zeros((n, nk), dtype=np.int64)
        counts[cand] = live.cpu().numpy()
        counts[int(order[s0 - 1])] = 0
        off = np.concatenate([[0], np.cumsum(counts.reshape(-1))])
        rest = [g for g in cand if g != int(order[s0 - 1])]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        state = eng.greedy_compact(regs, u, rest, off, p)
        b.record()
        b.synchronize()
        compact_ms = a.elapsed_time(b)
        for t in range(s0, min(n, s0 + 40)):
            _, uh = eng.cards_hist(u, p)
            rest = sorted(set(range(n)) - set(int(g) for g in order[:t]))
            hd, ld = eng.greedy_dense_hist(regs, u, uh, rest, p)
            d_ms = events(lambda: eng.greedy_dense_hist(regs, u, uh, rest, p), 1)[0]
            a.record()
            hs, ls = eng.greedy_sparse_hist(state, u, uh, rest, p)
            b.record()
            b.synchronize()
            alternated.append(dict(step=t, dense_ms=d_ms, sparse_ms=a.elapsed_time(b), live=int(ls.to(torch.int64).sum()),
                                   equal=bool(torch.equal(hd, hs) and torch.equal(ld, ls))))
            u = torch.maximum(u, regs[int(order[t])])

    # ---- K6 per-step baseline on three windows
    planes = torch.empty(((n + 1) * nk, 6, m // 32), dtype=torch.int32, device=dev)
    eng.to_planes(regs, p, out=planes[:n * nk])
    k6, k6_equal = [], True
    for w0 in (0, n // 2, n - 20):
        u = union_at(w0)
        for t in range(w0, w0 + 20):
            rest = sorted(set(range(n)) - set(int(g) for g in order[:t]))
            pairs = np.array([[g, n] for g in rest], dtype=np.int32)

            def k6_step():
                eng.to_planes(u, p, out=planes[n * nk:])
                return eng.pairwise_cards(None, pairs, p, planes=planes, n_genomes=n + 1, nk=nk)
            ms = events(k6_step, 1)[0]
            c6 = k6_step()
            _, uh = eng.cards_hist(u, p)
            c11 = eng.mle(eng.greedy_dense_hist(regs, u, uh, rest, p)[0], p)
            pick6 = rest[int((c6 / kdiv).amax(dim=1).argmax())]
            k6_equal &= bool(torch.equal(c6, c11)) and pick6 == int(order[t])
            k6.append(dict(step=t, candidates=len(rest), ms=ms))
            u = torch.maximum(u, regs[int(order[t])])
    k6_cands = sum(x["candidates"] for x in k6)
    k6_ms = sum(x["ms"] for x in k6)
    total_cands = n * (n + 1) // 2

    rep = dict(card_info(), shape="config 5: %d x %.0f bp clustered (10 per cluster), k = 10..32, p = %d" % (n, args.bases, p),
               sparse_cross=ddstore.SPARSE_CROSS, hbm_copy_GB_per_s_measured=hbm / 1e9,
               order_seconds={x: runs[x]["seconds"] for x in runs}, orders_and_cards_equal=bool(same),
               switch_step=stats["switch_step"], dense_steps=stats["dense_steps"], sparse_steps=stats["sparse_steps"],
               live_per_step=stats["live"], dense_only_stats={x: runs["dense_only"]["stats"][x] for x in ("dense_steps", "sparse_steps")},
               per_step=per_step, compact_ms=compact_ms, alternated=alternated,
               alternated_equal=all(x["equal"] for x in alternated),
               k6_windows=k6, k6_equal_to_k11=bool(k6_equal),
               k6_whole_order_s_extrapolated=k6_ms / k6_cands * total_cands / 1e3,
               order=[int(g) for g in order])
    print(json.dumps({x: rep[x] for x in rep if x not in ("live_per_step", "order", "k6_windows")}))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    if not (same and rep["alternated_equal"] and k6_equal):
        raise SystemExit("greedy results disagree: see %s" % args.out)


if __name__ == "__main__":
    main()
