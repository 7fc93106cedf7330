#!/usr/bin/env python
"""A/B of the prefix-union paths at the bench shape (12 x 5 Mbp genomes, k = 10..32, p = 20, 30 orderings of
12 steps) in one process: dd_prefix_union_card with dd_set_option("prefix_lattice", 1) (subset table,
lattice.cu) and 0 (bit planes, planes.cu), rounds alternated, each call timed with CUDA events.  Checks
that both give the same histograms and cardinalities, records the card and its power limit, and writes
--out (JSON).  A separate torch.profiler pass over --profile-calls calls of Engine.prefix_union_cards (lattice
path) adds the device time of every launch of the call, grouped by kernel, under "launches"."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (the benchmark's own genome and ordering generators)


def card_info():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().split("\n")[0]
    except Exception as e:   # noqa: BLE001
        return "unavailable: %s" % e


def launch_split(eng, regs, orders, p, calls):
    """Device time of each launch of Engine.prefix_union_cards (lattice path) under torch.profiler, per kernel
    name over `calls` calls: {name: {"per_call": launches per call, "median_us", "min_us", "max_us"}}."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        eng.prefix_union_cards(regs, orders, p)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            eng.prefix_union_cards(regs, orders, p)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = ev.name
        for short in ("lattice_levels", "lattice_prefix", "lattice_sets", "lattice_zeta", "lattice_finish", "mle_kernel"):
            if short in name:
                name = short
        if "emset" in name or "Memset" in name:
            name = "memset"
        if "emcpy" in name or "Memcpy" in name:
            name = "memcpy " + ("HtoD" if "HtoD" in name else "DtoH" if "DtoH" in name else "DtoD")
        per.setdefault(name, []).append(ev.time_range.elapsed_us())
    out = {}
    for name, t in sorted(per.items(), key=lambda kv: -sum(kv[1])):
        out[name] = {"per_call": len(t) / calls, "median_us": round(statistics.median(t), 2), "min_us": round(min(t), 2),
                     "max_us": round(max(t), 2)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--calls", type=int, default=10, help="calls per path per round")
    ap.add_argument("--profile-calls", type=int, default=10, help="calls traced by torch.profiler (0 = no trace)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_prefix_lattice.json"))
    args = ap.parse_args()

    import torch
    from dandd_b200 import build
    build.build()
    from dandd_b200._lib import check
    from dandd_b200.engine import Engine
    eng = Engine(0)
    P, KS = bench.P, bench.KS
    regs = torch.empty((bench.N_GENOMES, len(KS), 1 << P), dtype=torch.uint8, device="cuda")
    for g, (text, _) in enumerate(bench.make_genomes(seed=2)):
        eng.sketch(eng.pack(text), KS, p=P, out=regs[g])
    orders = bench.make_orderings(bench.N_GENOMES, bench.N_ORDERINGS, seed=2)
    order = torch.as_tensor(orders).cuda().contiguous()
    n_g, nk, _ = regs.shape
    n_ord, n_steps = order.shape
    ws = torch.empty(eng.lib.dd_prefix_union_workspace_bytes(n_ord, n_steps, n_g, nk, P), dtype=torch.uint8, device="cuda")
    out = {}
    for name in ("lattice", "planes"):
        out[name] = (torch.empty((n_ord, n_steps, nk, 64), dtype=torch.int32, device="cuda"),
                     torch.empty((n_ord, n_steps, nk), dtype=torch.float64, device="cuda"))

    def call(name):
        check(eng.lib.dd_set_option(b"prefix_lattice", int(name == "lattice")), "dd_set_option")
        hist, cards = out[name]
        check(eng.lib.dd_prefix_union_card(regs.data_ptr(), order.data_ptr(), n_ord, n_steps, n_g, nk, P, 0, cards.data_ptr(),
                                           hist.data_ptr(), None, ws.data_ptr(), ws.numel(), None), "dd_prefix_union_card")

    times = {"lattice": [], "planes": []}
    for name in times:   # warm-up
        for _ in range(3):
            call(name)
    torch.cuda.synchronize()
    for _ in range(args.rounds):
        for name in times:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.calls):
                call(name)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.calls)
    check(eng.lib.dd_set_option(b"prefix_lattice", 1), "dd_set_option")
    same_hist = bool(torch.equal(out["lattice"][0], out["planes"][0]))
    same_cards = bool(torch.equal(out["lattice"][1], out["planes"][1]))

    def summary(t):
        return {"median_ms": round(statistics.median(t), 4), "min_ms": round(min(t), 4), "max_ms": round(max(t), 4)}
    launches = launch_split(eng, regs, orders, P, args.profile_calls) if args.profile_calls > 0 else None
    rep = {"card": card_info(),
           "what": "dd_prefix_union_card (hist + MLE) at the bench shape: 12 genomes x 23 k x 2^20 registers, 30 orderings "
                   "x 12 steps; CUDA events around %d back-to-back calls, %d rounds, paths alternated" % (args.calls, args.rounds),
           "lattice": summary(times["lattice"]), "planes": summary(times["planes"]),
           "hist_equal": same_hist, "cards_equal": same_cards}
    if launches is not None:
        rep["launches"] = launches
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps(rep))
    if not (same_hist and same_cards):
        sys.exit("prefix_lattice_run: the two paths disagree")


if __name__ == "__main__":
    main()
