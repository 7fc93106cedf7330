#!/usr/bin/env python3
"""Greedy most-diverse-first (or least-diverse-first) ordering of a collection of genomes.

Step t adds the genome not chosen yet whose union with the genomes chosen so far has the largest delta (--order max)
or the smallest (--order min), the lowest input index winning a tie; genomes listed in --first take the first steps
in the order given.  delta is the maximum over the swept k of card / k, the first k winning a tie.  The greedy
growth curve is the upper edge of the band `dandd progressive` samples (--order min gives a lower curve), and its
first m genomes answer "which m assemblies capture most of the diversity".
  --tool dashing  every step evaluates every remaining candidate on the HLL registers resident on the device
                  (store.greedy_order, K11): the time grows with steps x n.
  --tool kmc      exact distinct k-mer counts (store.exact_greedy_order, K12): a cover index per k is built once and
                  held on the device (about 6 bytes per (genome, distinct k-mer) plus 5 per distinct k-mer, per k);
                  then every step is one device launch over all k, and the whole order costs one visit per holder of
                  every k-mer.  Late in an order the candidates differ by few novel k-mers, which HLL estimates blur;
                  these counts do not.  At most 65535 inputs; k up to 256; --registers is not used.

Inputs are listed as `dandd tree` lists them (-d DATADIR or -f LIST, sorted); genome i is index i of that list and
names are the FASTA base names, which must be distinct.  --first names input base names, one per line.  Written
into --name (a directory that must not exist yet), tab-separated, floats by repr, integer cards for kmc:
  order.tsv       step  genome  forced  delta  k  gain  fraction   gain = delta - delta before the step (0 before
                                                                     the first), fraction = delta / delta(all inputs)
  growth.tsv      ngen  k  card  delta_pos                          the union of the first ngen genomes, every k
  collection.tsv  ngen  delta  k                                    the union of all inputs
  ordering.pickle {tuple(order)}: `dandd progressive -d <tree of the same inputs> -r DIR/ordering.pickle --ksweep`
                  replays it (-n 0; with --steps n, -n 30 adds random orderings beside it).
Under torchrun every rank sketches its share of the genomes and evaluates its share of the candidates (dashing) or
indexes its key range of every genome (kmc), and rank 0 writes."""
import argparse
import os
import pickle
import sys
from typing import List, Sequence

import numpy as np

HLL_MAX_K = 32       # Dashing's
EXACT_MAX_K = 256    # KMC's
EXACT_MAX_N = 65535  # the cover index keeps genome ids in 16 bits


def get_store():
    from dandd_b200.store import get_store as _get   # torch + CUDA start only when a job is actually run
    return _get()


def read_first(path: str, names: Sequence[str]) -> List[int]:
    """Input indices of the base names listed in `path`, one per line (blank lines skipped).  Raises ValueError."""
    out: List[int] = []
    with open(path) as fh:
        for num, line in enumerate(fh, start=1):
            name = line.strip()
            if not name:
                continue
            if name not in names:
                raise ValueError("%s:%d: %s is not an input" % (path, num, name))
            if names.index(name) in out:
                raise ValueError("%s:%d: %s is named twice" % (path, num, name))
            out.append(names.index(name))
    return out


# ---------------------------------------------------------------- outputs
def write_outputs(directory: str, names: Sequence[str], ks: Sequence[int], order, n_forced: int, cards, all_cards) -> None:
    """order.tsv, growth.tsv, collection.tsv and ordering.pickle from order [steps], cards [steps, nk] (the union
    after each step) and all_cards [nk] (the union of every input)."""
    from dandd_b200.helpers.leaveout import best_k
    cards = np.asarray(cards)
    if cards.dtype.kind not in "iu":      # integer (exact) cards stay integers
        cards = cards.astype(np.float64)
    d_all, k_all = best_k(ks, np.asarray(all_cards, dtype=np.float64))
    d_all = float(d_all)
    rows = {"order.tsv": ["step\tgenome\tforced\tdelta\tk\tgain\tfraction"], "growth.tsv": ["ngen\tk\tcard\tdelta_pos"],
            "collection.tsv": ["ngen\tdelta\tk", "%d\t%s\t%d" % (len(names), repr(d_all), int(k_all))]}
    before = 0.0
    for t, g in enumerate(order):
        d, kk = best_k(ks, cards[t])
        d = float(d)
        rows["order.tsv"].append("%d\t%s\t%d\t%s\t%d\t%s\t%s" % (t + 1, names[int(g)], int(t < n_forced), repr(d), int(kk),
                                                                repr(d - before), repr(d / d_all)))
        before = d
        for c, k in enumerate(ks):
            rows["growth.tsv"].append("%d\t%d\t%s\t%s" % (t + 1, k, repr(cards[t, c].item()), repr(cards[t, c].item() / k)))
    for fn, lines in rows.items():
        with open(os.path.join(directory, fn), "w") as fh:
            fh.write("\n".join(lines) + "\n")
    with open(os.path.join(directory, "ordering.pickle"), "wb") as fh:
        pickle.dump({tuple(int(g) for g in order)}, fh)


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
    parser.add_argument("--registers", type=int, default=20, help="log2 of the number of HLL registers")
    parser.add_argument("--no-canon", dest="canon", action="store_false", help="count k-mers as read, not canonical")
    parser.add_argument("--order", choices=["max", "min"], default="max",
                        help="max: the most diverse union first (default); min: the least diverse")
    parser.add_argument("--first", default=None, help="file of input base names, one per line, that take the first steps")
    parser.add_argument("--steps", type=int, default=None, help="number of steps (default: every input)")
    parser.add_argument("--name", default="greedy", help="output directory; it must not exist yet")
    return parser.parse_args(argv)


def _inputs(args):
    """(fastas, names, ks, first, steps) or a refusal message."""
    import dandd_b200
    dandd_b200.enable_compat()         # the mirrors import each other by the reference's top-level module names
    from dandd_b200.lib.huffman_dandd import list_fastas
    if not (args.genomedir or args.flist_loc):
        return None, "give the inputs: -d DATADIR or -f LIST"
    for flag, k in (("--mink", args.mink), ("--maxk", args.maxk)):
        if args.tool == "dashing" and not 1 <= k <= HLL_MAX_K:
            return None, "%s %d is outside 1..%d" % (flag, k, HLL_MAX_K)
        if args.tool == "kmc" and not 1 <= k <= EXACT_MAX_K:
            return None, "%s %d is outside 1..%d for kmc" % (flag, k, EXACT_MAX_K)
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
    if len(names) < 2:
        return None, "an ordering needs at least 2 inputs, got %d" % len(names)
    if args.tool == "kmc" and len(names) > EXACT_MAX_N:
        return None, "--tool kmc orders at most %d inputs, got %d" % (EXACT_MAX_N, len(names))
    first: List[int] = []
    if args.first:
        try:
            first = read_first(args.first, names)
        except (OSError, ValueError) as err:
            return None, "cannot read --first: %s" % err
    steps = len(names) if args.steps is None else args.steps
    if not max(1, len(first)) <= steps <= len(names):
        return None, "--steps %d is outside %d..%d" % (steps, max(1, len(first)), len(names))
    return (fastas, names, list(range(args.mink, args.maxk + 1)), first, steps), None


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
    fastas, names, ks, first, steps = got
    n, shard = len(fastas), ((rank, world) if world > 1 else None)
    try:
        store = get_store()
        from dandd_b200 import ingest
        if args.tool == "kmc":
            ingest.prefetch(fastas, want_digest=False)          # every rank indexes its key range of every genome
            with timing.span("greedy_order"):
                order, cards, stats = store.exact_greedy_order(fastas, ks, args.canon, steps, order=args.order, first=first,
                                                               shard=shard)
            all_cards = np.asarray(stats["distinct_keys"], dtype=np.int64)   # the index's keys: |union of all|
        else:
            from dandd_b200.helpers.allpairs import gather_leaf_registers
            owners = [[g for g in range(n) if g % world == r] for r in range(world)]
            ingest.prefetch([fastas[g] for g in owners[rank]], want_digest=False)
            regs, _ = gather_leaf_registers(store, fastas, ks, args.registers, args.canon, owners, tag="greedy")
            with timing.span("greedy_order"):
                order, cards, stats = store.greedy_order(regs, ks, args.registers, steps, order=args.order, first=first,
                                                         shard=shard)
            with timing.span("greedy_collection"):
                engine = store.engine
                all_cards = engine.cards(engine.union([regs[g] for g in range(n)]), args.registers).cpu().numpy()
        if rank == 0:
            with timing.span("greedy_outputs"):
                write_outputs(args.name, names, ks, order, len(first), cards, all_cards)
    finally:
        timing.dump()          # DANDD_B200_TIMING=<file>: one JSON line of stage times per process
    return order, cards, stats


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    go()
