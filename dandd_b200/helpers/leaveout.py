#!/usr/bin/env python3
"""Leave-one-out contribution of every genome, or every group of genomes, to a collection's delta.

For each group g this gives delta(all) - delta(all without g): how much the group adds to the collection's
diversity.  Near-duplicates contribute about nothing, outliers and contaminated assemblies a lot.  It is what
`DeltaTree.find_delta_delta([g])` answers for one subset at a time, with a fresh climb over the remaining FASTAs;
here every group is answered at once:

  --tool dashing  one read of the HLL registers of all genomes per rank (store.leave_out_cards, K10) gives the
                  register histograms of the union and of every leave-out union; the histograms are the ones the
                  union of the remaining sketches would have, so the estimates are the same floats.
  --tool kmc      one exact device job per k (store.exact_leave_out): the sharing-spectrum job when every group is
                  one genome, else one first-rank job with a row per group.

delta is the maximum over the swept k of card / k, the first k winning a tie (delta_summarize's rule).  It equals
find_delta_delta where the reference's hill-climb over the remaining FASTAs reaches that maximum; a climb that stops
at a local maximum gives a smaller delta.  Under HLL, `novel` is the difference of two estimates: its error is that
of the union's estimate, not a fraction of itself.

Inputs are listed as `dandd tree` lists them (-d DATADIR or -f LIST, sorted); names are the FASTA base names and must
be distinct.  --groups TSV names every input exactly once as `basename<TAB>label`; groups are numbered in order of
first appearance in the sorted input list.  Without it every genome is its own group, labelled by its name.  Written
into --name (a directory that must not exist yet), tab-separated, floats by repr, integers for kmc:
  union.tsv       k  card  delta_pos                   the union of all genomes; delta_pos = card / k
  without.tsv     k  group  card  novel  delta_pos     the union without the group; novel = union card - card
  delta.tsv       group  delta  k  contribution        delta without the group; contribution = delta(all) - delta
  collection.tsv  ngen  delta  k                       delta of the whole collection
Under torchrun every rank sketches its share of the genomes (dashing) or counts its key range (kmc), and rank 0
writes."""
import argparse
import os
import sys
from typing import List, Sequence

import numpy as np

HLL_MAX_K = 32       # Dashing's
EXACT_MAX_K = 256    # KMC's


def get_store():
    from dandd_b200.store import get_store as _get   # torch + CUDA start only when a job is actually run
    return _get()


def best_k(ks: Sequence[int], cards: np.ndarray):
    """(delta, k) per column of cards [nk, ...]: the largest card / k, the first k of the list winning a tie."""
    dk = np.asarray(cards, dtype=np.float64) / np.asarray(ks, dtype=np.float64).reshape((-1,) + (1,) * (np.ndim(cards) - 1))
    best = np.argmax(dk, axis=0)
    return np.take_along_axis(dk, best[None], axis=0)[0], np.asarray(ks, dtype=np.int64)[best]


def parse_groups(path: str, names: Sequence[str]):
    """(group ids [n], labels [G]) from a `basename<TAB>label` file naming every input exactly once; ids in order of
    first appearance along names.  Raises ValueError with the reason."""
    label_of = {}
    with open(path) as fh:
        for num, line in enumerate(fh, start=1):
            line = line.rstrip("\n").rstrip("\r")
            if not line.strip():
                continue
            parts = line.split("\t")
            if len(parts) != 2 or not parts[0] or not parts[1]:
                raise ValueError("%s:%d: expected `basename<TAB>label`" % (path, num))
            if parts[0] in label_of:
                raise ValueError("%s:%d: %s is named twice" % (path, num, parts[0]))
            label_of[parts[0]] = parts[1]
    unknown = sorted(set(label_of) - set(names))
    if unknown:
        raise ValueError("--groups names files that are not inputs: %s" % unknown)
    missing = [x for x in names if x not in label_of]
    if missing:
        raise ValueError("--groups does not name these inputs: %s" % missing)
    labels: List[str] = []
    for x in names:
        if label_of[x] not in labels:
            labels.append(label_of[x])
    return [labels.index(label_of[x]) for x in names], labels


# ---------------------------------------------------------------- outputs
def write_outputs(directory: str, n: int, labels: Sequence[str], ks: Sequence[int], union, without, exact: bool) -> List[str]:
    """The four tables from union [nk] and without [nk, G] (float64 for HLL, int64 for exact counts)."""
    num = (lambda v: "%d" % v) if exact else repr
    rows = {"union.tsv": ["k\tcard\tdelta_pos"], "without.tsv": ["k\tgroup\tcard\tnovel\tdelta_pos"],
            "delta.tsv": ["group\tdelta\tk\tcontribution"], "collection.tsv": ["ngen\tdelta\tk"]}
    union = np.asarray(union)
    without = np.asarray(without)
    for c, k in enumerate(ks):
        u = union[c].item()
        rows["union.tsv"].append("%d\t%s\t%s" % (k, num(u), repr(u / k)))
        for g, label in enumerate(labels):
            w = without[c, g].item()
            rows["without.tsv"].append("%d\t%s\t%s\t%s\t%s" % (k, label, num(w), num(u - w), repr(w / k)))
    if len(ks):
        d_all, k_all = best_k(ks, union)
        rows["collection.tsv"].append("%d\t%s\t%d" % (n, repr(float(d_all)), int(k_all)))
        d_out, k_out = best_k(ks, without)
        for label, d, kk in zip(labels, d_out.tolist(), k_out.tolist()):
            rows["delta.tsv"].append("%s\t%s\t%d\t%s" % (label, repr(d), kk, repr(float(d_all) - d)))
    written = []
    for fn, lines in rows.items():
        path = os.path.join(directory, fn)
        with open(path, "w") as fh:
            fh.write("\n".join(lines) + "\n")
        written.append(path)
    return written


# ---------------------------------------------------------------- command line
def parse_arguments(argv=None):
    parser = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    src = parser.add_mutually_exclusive_group()
    src.add_argument("-d", "--datadir", dest="genomedir", default=None, help="directory of FASTA files (every file is an input)")
    src.add_argument("-f", "--fastas", dest="flist_loc", default=None, help="file listing one FASTA path per line")
    parser.add_argument("--tool", choices=["dashing", "kmc"], default="dashing",
                        help="dashing: HLL estimates (default); kmc: exact distinct k-mer counts")
    parser.add_argument("--mink", type=int, default=2, help="smallest k (1..%d for dashing, 1..%d for kmc)" % (HLL_MAX_K, EXACT_MAX_K))
    parser.add_argument("--maxk", type=int, default=32, help="largest k")
    parser.add_argument("--registers", type=int, default=20, help="log2 of the number of HLL registers (dashing)")
    parser.add_argument("--no-canon", dest="canon", action="store_false", help="count k-mers as read, not canonical")
    parser.add_argument("--groups", default=None, help="TSV of `fasta_basename<TAB>label` naming every input once")
    parser.add_argument("--name", default="leaveout", help="output directory; it must not exist yet")
    return parser.parse_args(argv)


def _inputs(args):
    """(fastas, names, ks, group, labels) or a refusal message."""
    import dandd_b200
    dandd_b200.enable_compat()         # the mirrors import each other by the reference's top-level module names
    from dandd_b200.lib.huffman_dandd import list_fastas
    if not (args.genomedir or args.flist_loc):
        return None, "give the inputs: -d DATADIR or -f LIST"
    limit = HLL_MAX_K if args.tool == "dashing" else EXACT_MAX_K
    for flag, k in (("--mink", args.mink), ("--maxk", args.maxk)):
        if not 1 <= k <= limit:
            return None, "%s %d is outside 1..%d for %s" % (flag, k, limit, args.tool)
    if args.mink > args.maxk:
        return None, "--mink %d is above --maxk %d" % (args.mink, args.maxk)
    if args.tool == "dashing" and not 5 <= args.registers <= 26:
        return None, "--registers %d is outside 5..26" % args.registers
    try:
        fastas = list_fastas(args.genomedir, args.flist_loc)
    except (OSError, ValueError) as err:
        return None, "cannot list the inputs: %s" % err
    names = [os.path.basename(f) for f in fastas]
    dup = sorted({x for x in names if names.count(x) > 1})
    if dup:
        return None, "input names must be distinct: %s" % dup
    if args.groups:
        try:
            group, labels = parse_groups(args.groups, names)
        except (OSError, ValueError) as err:
            return None, "cannot read --groups: %s" % err
    else:
        group, labels = list(range(len(names))), list(names)
    if len(labels) < 2:
        return None, "leaving a group out needs at least 2 groups, got %d" % len(labels)
    if len(labels) > 65535:
        return None, "at most 65535 groups, got %d" % len(labels)
    return (fastas, names, list(range(args.mink, args.maxk + 1)), group, labels), None


def go(argv=None):
    args = parse_arguments(argv)
    from dandd_b200 import dist as dd_dist
    from dandd_b200 import timing
    rank, world = dd_dist.init()
    got, refusal = _inputs(args)
    if rank == 0 and refusal is None:
        if os.path.exists(args.name):
            refusal = 'Output directory with name "%s" already exists' % args.name
        else:
            os.makedirs(args.name)
    if world > 1:                      # every rank leaves together, none is left waiting in a collective
        refusal = dd_dist.broadcast_object(refusal)
    if refusal:
        raise RuntimeError(refusal)
    fastas, names, ks, group, labels = got
    n, shard = len(fastas), ((rank, world) if world > 1 else None)
    try:
        store = get_store()
        if args.tool == "dashing":
            from dandd_b200 import ingest
            from dandd_b200.helpers.allpairs import gather_leaf_registers
            owners = [[g for g in range(n) if g % world == r] for r in range(world)]
            ingest.prefetch([fastas[g] for g in owners[rank]], want_digest=False)
            regs, _ = gather_leaf_registers(store, fastas, ks, args.registers, args.canon, owners, tag="leaveout")
            with timing.span("leaveout_hist"):
                union, without = store.leave_out_cards(regs, group, len(labels), args.registers, shard=shard)
        else:
            with timing.span("leaveout_exact"):
                union, without, _ = store.exact_leave_out(fastas, ks, args.canon, group, len(labels), shard=shard)
                if world > 1:          # each k-mer belongs to exactly one rank's key range: the counts add up
                    import torch
                    dev = getattr(getattr(store, "engine", None), "device", "cpu")
                    both = torch.as_tensor(np.concatenate([union[:, None], without], axis=1), device=dev)
                    both = dd_dist.sum_counts(both).cpu().numpy()
                    union, without = both[:, 0], both[:, 1:]
        if rank == 0:
            with timing.span("leaveout_outputs"):
                write_outputs(args.name, n, labels, ks, union, without, exact=args.tool == "kmc")
    finally:
        timing.dump()          # DANDD_B200_TIMING=<file>: one JSON line of stage times per process
    return union, without


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    go()
