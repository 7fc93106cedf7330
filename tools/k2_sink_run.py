#!/usr/bin/env python
"""A/B of K2's rank-1 sink (dd_set_option("sketch_sink", 1/0)) in one process, rounds alternated:
  * serialised K2 time per config-2 genome (CUDA events around dd_sketch_update_sched, 12 genomes); at
    config 2 that call is one sketch_sink_kernel launch, so with the sink on this is the sink kernel's time;
  * the bench-shaped step: 12 genomes on 2 streams (pack + K2 + finalize), leaf MLE, prefix unions;
  * one 100 Mbp and one 1 Gbp stream at k = 2..32, p = 20, which cross the first floor cut early and
    must not regress.
Also records the card, its power limit and SM clock, the static SASS of one k block of the sink
kernel (cuobjdump on dandd_b200/build/sketch.o, when available), the device time of every launch of
one bench-shaped step under torch.profiler (a run of its own), and the rank >= 2 updates of one bench
genome counted on the CPU with the oracle (the L2 reductions the sink cannot absorb).
--lib loads another build of the library (e.g. a one-off variant of the sink kernel); --sink-only then
records just the serialised per-genome K2 time with the sink on.  Writes --out (JSON)."""
import argparse
import json
import os
import re
import shutil
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


def sink_sass():
    """Median length of the per-k blocks of sketch_sink_kernel<canon=true> (from one hash start to the next):
    the static instructions of one k's tile loop, window extraction through REDG."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(ROOT, "dandd_b200", "build", "sketch.o")
    if not (os.path.exists(tool) and os.path.exists(obj)):
        return None
    sass = subprocess.check_output([tool, "-sass", obj], text=True).split("\n")
    heads = [i for i, ln in enumerate(sass) if "Function :" in ln]
    for n, h in enumerate(heads):
        if "sketch_sink_kernelILb1E" not in sass[h]:
            continue
        body = sass[h:heads[n + 1] if n + 1 < len(heads) else len(sass)]
        ins = [m.group(1).strip() for ln in body if (m := re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", ln))]
        starts = [i for i, t in enumerate(ins) if "IMAD.WIDE.U32" in t and "0x1fffff" in t]
        spans = [b - a for a, b in zip(starts, starts[1:])]
        return {"kernel_instructions": len(ins), "hash_sites": len(starts),
                "median_instr_between_k_blocks": statistics.median(spans) if spans else None,
                "atoms_or": sum("ATOMS.OR" in t for t in ins), "redg": sum(t.startswith("REDG") or " REDG" in t for t in ins)}
    return None


def rank2_updates(text, ks, p):
    """(updates, updates of rank >= 2) of one genome over ks: every valid canonical k-mer is one update, and its
    rank is >= 2 exactly when the hash bit just below the p register bits is 0."""
    from oracle import pyoracle as orc
    from oracle.ref_numpy import wang_np
    sym = orc.fasta_symbols(text)
    total = high = 0
    for k in ks:
        h = wang_np(orc.kmers(sym, k, True))
        total += int(h.size)
        high += int(np.count_nonzero(((h >> np.uint64(63 - p)) & np.uint64(1)) == 0))
    return total, high


def step_launches(step, torch):
    """Device time of every kernel and memset of one step, under torch.profiler: {name: {calls, total_ms}}."""
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0 or ev.key.startswith("cuda"):
            continue
        out[ev.key] = {"calls": ev.count, "total_ms": t / 1e3}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["total_ms"]))


def long_fasta(n, seed):
    rng = np.random.default_rng(seed)
    s = bench.ACGT[rng.integers(0, 4, n, dtype=np.uint8)]
    nfull = n // bench.LINE
    body = np.empty((nfull, bench.LINE + 1), dtype=np.uint8)
    body[:, :bench.LINE] = s[:nfull * bench.LINE].reshape(nfull, bench.LINE)
    body[:, bench.LINE] = 10
    return b">long\n" + body.tobytes() + s[nfull * bench.LINE:].tobytes() + b"\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r15_k2_sink.json"))
    ap.add_argument("--lib", default=None, help="load this build of libdandd_b200.so instead of the in-tree one")
    ap.add_argument("--sink-only", action="store_true", help="only the serialised per-genome K2 time, sink on")
    args = ap.parse_args()
    import torch
    from dandd_b200 import _lib
    if args.lib:
        _lib.LIB_PATH = os.path.abspath(args.lib)
    else:
        from dandd_b200 import build
        build.build()
    from dandd_b200._lib import check
    from dandd_b200.engine import Engine
    eng = Engine(0)
    dev = eng.device
    report = {"card": card_info(), "lib": _lib.LIB_PATH if args.lib else "in-tree", "rounds": args.rounds}
    if not args.lib:
        report["sass_sink_kernel_canon"] = sink_sass()

    def set_sink(on):
        check(eng.lib.dd_set_option(b"sketch_sink", int(on)), "dd_set_option")

    texts = bench.make_genomes(seed=2)
    d_texts = [torch.from_numpy(np.frombuffer(t, dtype=np.uint8).copy()).to(dev) for t, _ in texts]
    orders = bench.make_orderings(bench.N_GENOMES, bench.N_ORDERINGS, seed=2)
    nk, m = len(bench.KS), 1 << bench.P
    regs = torch.empty((bench.N_GENOMES, nk, m), dtype=torch.uint8, device=dev)
    hist = torch.empty((bench.N_GENOMES, nk, 64), dtype=torch.int32, device=dev)
    side = [torch.cuda.Stream(device=dev) for _ in range(2)]
    orig_update = eng._update_from_state
    events = []

    def hooked(seq, kmask, p, canon, ws, st):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_update(seq, kmask, p, canon, ws, st)
        e1.record()
        events.append((e0, e1))

    def step():
        main_st = torch.cuda.current_stream()
        for s_ in side:
            s_.wait_stream(main_st)
        for g, dt in enumerate(d_texts):
            with torch.cuda.stream(side[g % 2]):
                seq = eng.pack(dt, start=0, ws_tag=f"pack{g % 2}")
                eng.sketch(seq, bench.KS, p=bench.P, out=regs[g], hist_out=hist[g], ws_tag=f"sketch{g % 2}")
        for s_ in side:
            main_st.wait_stream(s_)
        return eng.mle(hist, bench.P), eng.prefix_union_cards(regs, orders, bench.P)

    def timed_step():
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            out = step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps, out

    packed = [eng.pack(dt, start=0) for dt in d_texts]

    def k2_serial():
        eng._update_from_state = hooked
        events.clear()
        for g, seq in enumerate(packed):
            eng.sketch(seq, bench.KS, p=bench.P, out=regs[g], hist_out=hist[g])
        torch.cuda.synchronize()
        eng._update_from_state = orig_update
        return [a.elapsed_time(b) for a, b in events]

    def write(rep):
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(rep, fh, indent=1)

    set_sink(1)
    k2_serial()
    if args.sink_only:
        per = [statistics.median(k2_serial()) for _ in range(args.rounds)]
        report["sink_ms_per_genome"] = {"median": statistics.median(per), "min": min(per), "max": max(per), "all": per,
                                        "how": "median over the 12 genomes of CUDA events around each serialised call, per round"}
        write(report)
        print(json.dumps(report, indent=1))
        return
    report["step_launches"] = step_launches(step, torch)
    per = [statistics.median(k2_serial()) for _ in range(args.rounds)]
    report["sink_ms_per_genome"] = {"median": statistics.median(per), "min": min(per), "max": max(per), "all": per,
                                    "how": "median over the 12 genomes of CUDA events around each serialised call, per round"}
    total, high = rank2_updates(texts[0][0], bench.KS, bench.P)
    report["bench_genome0_updates"] = {"all": total, "rank_ge2": high,
                                       "rank_ge2_ms_at_187_g_per_s": high / 187e9 * 1e3}

    longs = {}
    for name, n in (("100mbp", 100_000_000), ("1gbp", 1_000_000_000)):
        txt = long_fasta(n, seed=7 if n < 10**9 else 8)
        longs[name] = eng.pack(txt)
        del txt
    ks_long = list(range(2, 33))

    def long_ms(seq):
        eng._update_from_state = hooked
        events.clear()
        r, _ = eng.sketch(seq, ks_long, p=20, ws_tag="long")
        torch.cuda.synchronize()
        eng._update_from_state = orig_update
        return events[0][0].elapsed_time(events[0][1]), r

    res = {on: {"k2_ms_per_genome": [], "step_ms": [], "long_100mbp_ms": [], "long_1gbp_ms": []} for on in (1, 0)}
    outputs = {}
    for on in (1, 0):          # warm-up of both arms
        set_sink(on)
        step()
        k2_serial()
        for seq in longs.values():
            long_ms(seq)
    for rnd in range(args.rounds):
        for on in ((1, 0) if rnd % 2 == 0 else (0, 1)):
            set_sink(on)
            res[on]["k2_ms_per_genome"].append(statistics.mean(k2_serial()))
            ms, (leaf, prog) = timed_step()
            res[on]["step_ms"].append(ms)
            t100, _ = long_ms(longs["100mbp"])
            t1g, r1g = long_ms(longs["1gbp"])
            res[on]["long_100mbp_ms"].append(t100)
            res[on]["long_1gbp_ms"].append(t1g)
            if rnd == 0:
                outputs[on] = (leaf.cpu().numpy(), prog.cpu().numpy(), regs.cpu().numpy(), r1g.cpu().numpy())
    set_sink(1)
    report["identical_outputs_on_off"] = all(np.array_equal(a, b) for a, b in zip(outputs[1], outputs[0]))
    for on in (1, 0):
        arm = "sink_on" if on else "sink_off"
        report[arm] = {key: {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v} for key, v in res[on].items()}
    report["ratio_on_over_off"] = {key: report["sink_on"][key]["median"] / report["sink_off"][key]["median"] for key in res[1]}
    updates = sum(n for _, n in texts) / len(texts) * nk
    report["updates_per_genome"] = updates
    report["update_rate_g_per_s"] = {arm: updates / (report[arm]["k2_ms_per_genome"]["median"] / 1e3) / 1e9
                                     for arm in ("sink_on", "sink_off")}
    write(report)
    print(json.dumps({key: report[key] for key in ("card", "sink_ms_per_genome", "bench_genome0_updates", "ratio_on_over_off",
                                                   "identical_outputs_on_off", "update_rate_g_per_s")}, indent=1))


if __name__ == "__main__":
    main()
