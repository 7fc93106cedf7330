#!/usr/bin/env python3
"""K14 register sharing spectrum and the all-orderings mean growth curve (helpers/spectrum.py --tool dashing) at the
config-5 shape, on one GPU.

Shape (BASELINE.json config 5): 1000 synthetic 5 Mbp genomes in clusters of 10 mutated copies (2 % substitutions, as
tools/config5_run.py builds them), k = 10..32, p = 18: 1000 x 23 x 2^18 registers = 6.0 GB.  The genomes are written
as FASTA files to a temporary directory and sketched on the device as they are written.

  k14       Engine.register_spectrum over all registers, timed by CUDA events around each of --reps calls after one
            untimed call (the window covers the workspace memset, K14 and its finishing kernel).  Algorithmic bytes =
            n nk 2^p (each register read once); bytes / time is set against a 4 GiB device-to-device copy in the same
            run (read + write bytes over time) and the data sheet's 7.7 TB/s.
  reductions  the L2 reductions K14 makes per register, counted from the registers with torch: a level whose
            count c is neither 1 nor n adds up to two cells of the global table (n > 128: the table is not kept whole
            in shared memory); also the levels per register.
  helper    helpers/spectrum.py --tool dashing on the FASTA files by the host clock, a fresh store (reading and
            sketching every genome included).
  gap       the estimator gap: the mean over --orderings random orderings of the prefix-union cards of the existing
            path (Engine.prefix_union_cards), against the helper's mean_card, as the largest relative difference
            over m per k, beside the 95 % sampling spread of those orderings' mean (1.96 standard errors, relative).
  check     the helper's table equals K14 on the sketched registers; its m = n cards equal K4 on the union; T on the
            first 4096 registers of every k equals torch counts.
The card name and power limit are read in the same run.

    python tools/register_spectrum_run.py --out profiles/r13_register_spectrum.json"""
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
from tools.leaveout_run import events  # noqa: E402
from tools.synth import mutate_text, synth_fasta  # noqa: E402


def reductions(regs, p):
    """(levels per register, L2 reductions per register) over all k of regs [n, nk, 2^p] (table not kept whole)."""
    n, nk, m = regs.shape
    levels = red = 0
    for k in range(nk):
        x = torch.clamp(regs[:, k], max=63)
        cv = torch.stack([(x >= v).sum(dim=0, dtype=torch.int32) for v in range(1, 64)])    # [63, m], v = 1..63
        prev = torch.cat([torch.full((1, m), -1, dtype=torch.int32, device=x.device), cv[:-1]])
        nxt = torch.cat([cv[1:], torch.full((1, m), -1, dtype=torch.int32, device=x.device)])
        live = cv > 0
        far = (cv != 1) & (cv != n)
        start = live & (cv != prev)                       # +1 at (v, c_v)
        end = live & (cv != nxt)                          # -1 at (v + 1, c_v), none at v = 63
        end[-1] = False
        levels += int(start.sum())
        red += int((start & far).sum()) + int((end & far).sum())
    return levels / (nk * m), red / (nk * m)


def brute(regs):
    x = torch.clamp(regs, max=63)
    n, nk, _ = x.shape
    out = torch.zeros((nk, 64, n), dtype=torch.int64, device=regs.device)
    rowid = torch.arange(nk, device=regs.device)[:, None] * (n + 1)
    for v in range(1, 64):
        c = (x >= v).sum(dim=0)
        out[:, v] = torch.bincount((rowid + c).flatten(), minlength=nk * (n + 1)).view(nk, n + 1)[:, 1:]
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--genomes", type=int, default=1000)
    ap.add_argument("--bases", type=float, default=5e6)
    ap.add_argument("--p", type=int, default=18)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--orderings", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r13_register_spectrum.json"))
    args = ap.parse_args()
    from dandd_b200 import build
    build.build()
    from dandd_b200 import store as ddstore
    from dandd_b200.engine import Engine
    from dandd_b200.helpers import spectrum
    eng = Engine(0)
    dev = eng.device
    ks = list(range(10, 33))
    n, nk, p = args.genomes, len(ks), args.p
    m = 1 << p
    rep = dict(card_info(), shape="config 5: %d x %.0f bp clustered (10 per cluster), k = 10..32, p = %d" % (n, args.bases, p),
               register_bytes=n * nk * m)
    with tempfile.TemporaryDirectory() as tmp:
        data = os.path.join(tmp, "data")
        os.makedirs(data)
        regs = torch.empty((n, nk, m), dtype=torch.uint8, device=dev)
        hist = torch.empty((nk, 64), dtype=torch.int32, device=dev)
        t0 = time.perf_counter()
        for g in range(n):
            if g % 10 == 0:
                anc = synth_fasta(int(args.bases), 1, seed=5000 + g // 10, device=dev)
            text = anc if g % 10 == 0 else mutate_text(anc, 0.02, 50000 + g)
            with open(os.path.join(data, "g%04d.fasta" % g), "wb") as fh:
                fh.write(text.cpu().numpy().tobytes())
            eng.sketch(eng.pack(text, start=0), ks, p=p, out=regs[g], hist_out=hist)
        torch.cuda.synchronize()
        rep["write_and_sketch_s_untimed_setup"] = time.perf_counter() - t0

        # HBM bandwidth of this card, measured here: a device-to-device copy
        src = torch.empty(1 << 32, dtype=torch.uint8, device=dev)
        dst = torch.empty_like(src)
        dst.copy_(src)
        copy_ms = events(lambda: dst.copy_(src), 10)
        hbm = 2 * src.numel() / (np.median(copy_ms) / 1e3)
        del src, dst
        torch.cuda.empty_cache()

        acc = torch.zeros((nk, 64, n), dtype=torch.int32, device=dev)
        eng.register_spectrum(regs, p, out=acc)
        t_k14 = events(lambda: eng.register_spectrum(regs, p, out=acc), args.reps)
        one = eng.register_spectrum(regs, p)
        adds_up = bool(torch.equal(acc, one * (1 + args.reps)))
        med = float(np.median(t_k14))
        rep.update(hbm_copy_GB_per_s_measured=hbm / 1e9, k14_call_ms=t_k14, k14_call_ms_median=med,
                   k14_call_ms_range=[float(min(t_k14)), float(max(t_k14))],
                   k14_algorithmic_GB_per_s=n * nk * m / (med / 1e3) / 1e9,
                   k14_share_of_measured_hbm=n * nk * m / (med / 1e3) / hbm,
                   k14_share_of_datasheet_7p7TBs=n * nk * m / (med / 1e3) / 7.7e12, repeated_calls_add_up=adds_up)
        print(json.dumps({k: v for k, v in rep.items() if k != "k14_call_ms"}), flush=True)
        head = brute(regs[:, :, :4096].contiguous())
        slice_ok = bool(torch.equal(eng.register_spectrum(regs, p, reg_range=(0, 4096)).long(), head))
        lv, red = reductions(regs, p)
        rep.update(levels_per_register=lv, l2_reductions_per_register=red, first_4096_registers_equal_torch=slice_ok)
        print(json.dumps(dict(levels_per_register=lv, l2_reductions_per_register=red)), flush=True)

        st = ddstore.GpuSketchStore(engine=eng)
        ddstore.set_store(st)
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            spec, single, cards = spectrum.go(["-d", data, "--tool", "dashing", "--mink", "10", "--maxk", "32",
                                               "--registers", str(p), "--name", os.path.join(tmp, "run")])
            torch.cuda.synchronize()
            rep["helper_host_s"] = time.perf_counter() - t0
        finally:
            ddstore.set_store(None)
        del st
        torch.cuda.empty_cache()
    table_ok = bool(np.array_equal(spec, one.long().cpu().numpy()))
    union_cards = eng.cards_hist(regs.amax(dim=0).contiguous(), p)[0].cpu().numpy()
    union_ok = bool(np.array_equal(cards[:, n - 1], union_cards))
    rep.update(helper_table_equals_k14=table_ok, helper_last_row_equals_union_card=union_ok)
    print(json.dumps(dict(helper_host_s=rep["helper_host_s"], table_ok=table_ok, union_ok=union_ok)), flush=True)

    rng = np.random.default_rng(13)
    orders = np.stack([rng.permutation(n) for _ in range(args.orderings)]).astype(np.int32)
    total = np.zeros((n, nk))
    total2 = np.zeros((n, nk))
    for o in range(0, args.orderings, 10):
        c = eng.prefix_union_cards(regs, orders[o:o + 10], p).cpu().numpy()         # [10, n, nk]
        total += c.sum(axis=0)
        total2 += (c ** 2).sum(axis=0)
    mean = total / args.orderings
    sd = np.sqrt(np.maximum(total2 / args.orderings - mean ** 2, 0.0) * args.orderings / (args.orderings - 1))
    gap = np.abs(mean.T - cards) / mean.T                                             # [nk, n]
    spread = 1.96 * sd.T / np.sqrt(args.orderings) / mean.T
    rep["gap"] = [{"k": k, "largest_relative_gap": float(gap[c].max()), "at_m": int(gap[c].argmax()) + 1,
                   "sampling_spread_95_at_that_m": float(spread[c, gap[c].argmax()]),
                   "largest_sampling_spread_95": float(spread[c].max())} for c, k in enumerate(ks)]
    rep["gap_largest_over_k"] = float(gap.max())
    print(json.dumps(rep["gap"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    if not (adds_up and slice_ok and table_ok and union_ok):
        raise SystemExit("a check failed: see %s" % args.out)


if __name__ == "__main__":
    main()
