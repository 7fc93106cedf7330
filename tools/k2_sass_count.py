#!/usr/bin/env python
"""Instruction counts of K2's per-(symbol, k) update, read off the SASS of the built object
(dandd_b200/build/sketch.o) -- the number bench.py's INT32-issue view uses, so that it is derived
from a committed listing and not a remembered constant.

For each static-k-set instantiation of sketch_allk_kernel<canon=true> the unrolled k blocks are
delimited by the hash's first multiply (`IMAD.WIDE.U32 ..., 0x1fffff`); inside a block the update
tail (rank, register index, address, REDG) sits behind the branch that follows the threshold
compare, so   always-executed = block length - tail length.
Writes profiles/r02_k2_sass.json and profiles/r02_k2_sass.md (one k block, annotated).

--sink instead counts sketch_sink_kernel<canon=true>: on the all-valid warp path a k's 16 symbols are unrolled,
one hash per symbol, and every warp runs both the rank-1 and the rank >= 2 side of the tail, so the distance
between consecutive hashes of one unrolled run is the instructions a warp executes per (symbol, k).  That count
goes into profiles/r15_k2_sink.json ("sass_sink_all_valid"), next to the kernel's measured times."""
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "dandd_b200", "build", "sketch.o")
VARIANTS = {"4294966784": "k10_32", "4294967294": "k2_32", "4294967295": "k1_32"}


def blocks_of(ins):
    """One block per k: from the instruction after a REDG up to and including the next REDG."""
    reds = [i for i, t in enumerate(ins) if "REDG" in t]
    return [(a + 1, b + 1) for a, b in zip(reds, reds[1:])]


def instructions(body):
    return [mm.group(1).strip() for ln in body if (mm := re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", ln))]


def sink_counts(sass, heads):
    for n, h in enumerate(heads):
        if "sketch_sink_kernelILb1E" not in sass[h]:
            continue
        ins = instructions(sass[h:heads[n + 1] if n + 1 < len(heads) else len(sass)])
        hashes = [i for i, t in enumerate(ins) if "IMAD.WIDE.U32" in t and "0x1fffff" in t]
        gaps = [b - a for a, b in zip(hashes, hashes[1:])]
        # an unrolled run: a k's 16 hashes, 15 gaps, of which scheduling makes the first and last differ; the
        # per-symbol path has one hash per k, so 10 equal gaps in a row only occur inside a run
        runs = [gaps[i:i + 10] for i in range(len(gaps) - 9)
                if len(set(gaps[i:i + 10])) == 1 and (i == 0 or gaps[i - 1] != gaps[i])]
        per = statistics.median(r[0] for r in runs)
        return {"kernel_instructions": len(ins), "hash_sites": len(hashes), "unrolled_runs": len(runs),
                "instr_per_update_all_valid": per, "bssy": sum("BSSY" in t for t in ins),
                "atoms_or": sum("ATOMS.OR" in t for t in ins), "redg": sum("REDG" in t for t in ins),
                "how": "tools/k2_sass_count.py --sink on dandd_b200/build/sketch.o (cuobjdump -sass): median distance between "
                       "consecutive hashes of the unrolled all-valid runs of sketch_sink_kernel<true>"}
    raise SystemExit("sketch_sink_kernel<true> not found in " + OBJ)


def main():
    sass = subprocess.check_output(["cuobjdump", "-sass", OBJ], text=True).split("\n")
    heads = [i for i, ln in enumerate(sass) if "Function :" in ln]
    if "--sink" in sys.argv:
        counts = sink_counts(sass, heads)
        path = os.path.join(ROOT, "profiles", "r15_k2_sink.json")
        report = json.load(open(path)) if os.path.exists(path) else {}
        report["sass_sink_all_valid"] = counts
        with open(path, "w") as fh:
            json.dump(report, fh, indent=1)
        print(json.dumps(counts, indent=1))
        return 0
    out, listing = {}, []
    for n, h in enumerate(heads):
        name = sass[h]
        m = re.search(r"sketch_allk_kernelILb1ELj(\d+)ELi(\d+)", name)
        if not m or m.group(1) not in VARIANTS:
            continue
        body = sass[h:heads[n + 1] if n + 1 < len(heads) else len(sass)]
        ins = instructions(body)
        lengths, always, chosen = [], [], None
        for a, b in blocks_of(ins):
            blk = ins[a:b]
            if not any("ISETP.LT.U32.AND.EX" in t for t in blk):      # 64-bit k-mers only (k > 16): the common, costlier case
                continue
            cmp_at = next((i for i, t in enumerate(blk) if "ISETP.GT.U32" in t), None)
            thr = next((i for i, t in enumerate(blk) if cmp_at is not None and i > cmp_at and t.startswith("@") and "BRA" in t), None)
            if thr is None:
                continue
            lengths.append(len(blk))
            always.append(thr + 1)
            chosen = blk
        tag = VARIANTS[m.group(1)]
        L, A = statistics.median(lengths), statistics.median(always)
        out[f"static_instr_per_k_block_{tag}"] = L
        out[f"always_executed_{tag}"] = A
        out[f"tail_instr_{tag}"] = L - A
        if tag == "k10_32":
            listing = chosen
    # what bench.py uses: at config-2 size (floor 0) every update runs its tail; on a long genome almost none does
    out["instr_per_update_k10_32"] = out["static_instr_per_k_block_k10_32"]
    out["instr_per_update_k2_32_floor"] = out["always_executed_k2_32"]
    out["how"] = "tools/k2_sass_count.py on dandd_b200/build/sketch.o (cuobjdump -sass), median over the k > 16 blocks"
    os.makedirs(os.path.join(ROOT, "profiles"), exist_ok=True)
    with open(os.path.join(ROOT, "profiles", "r02_k2_sass.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    with open(os.path.join(ROOT, "profiles", "r02_k2_sass.md"), "w") as fh:
        fh.write("# K2 `sketch_allk_kernel<true, k=10..32, 256>`: one k block (k > 16) of the unrolled update\n\n")
        fh.write("From `cuobjdump -sass dandd_b200/build/sketch.o`; counts in `r02_k2_sass.json`.\n\n```\n")
        fh.write("\n".join(listing) + "\n```\n")
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    sys.exit(main())
