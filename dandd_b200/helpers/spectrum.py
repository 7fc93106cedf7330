#!/usr/bin/env python3
"""Sharing spectrum of a collection of FASTA files, and the growth curve averaged over ALL n! orderings.

`dandd progressive` samples orderings (-n 30) and leaves the averaging to its user; the average it approximates -- the
mean over every ordering of the union of the first m genomes -- follows in closed form from a sharing spectrum, because
prefix m of a uniformly random ordering is a uniformly random m-subset.

  --tool kmc (default)  exact counts.  h_c, the number of distinct k-mers held by exactly c of the n genomes, gives
                        mean |union of the first m|        = sum_c h_c (1 - C(n - c, m) / C(n, m))
                        mean |intersection of the first m| = sum_c h_c C(c, m) / C(n, m)
                        The spectrum of one k is one device job (store.exact_spectrum: K7 co-occurrence lists + K9),
                        whatever n is.
  --tool dashing        HLL sketches.  Registers do not record which genomes hold a k-mer, but they carry the register
                        counterpart: T[v][c], the number of registers where exactly c genomes hold a value >= v.  The
                        union of a subset has a value >= v at such a register exactly when the subset meets those c
                        genomes, so the MEAN register histogram of the m-prefix union over all orderings is
                        cnt>=(v) = sum_c T[v][c] (1 - C(n - c, m) / C(n, m)), with the weights of the exact mode
                        (hit_weights).  One read of all registers per rank gives T for every k (store.
                        register_spectrum_cards, K14).  mean_card is the Ertl MLE of that mean histogram: an estimate
                        of the mean union, NOT the mean of the per-ordering estimates (max, MLE and mean do not
                        commute).  The two differ most when the m-subset unions differ widely in size, i.e. for strongly
                        clustered collections: on synthetic sets of 8 genomes the largest relative gap over m was
                        1.6e-4 for near-copies of one ancestor (p = 12, where the HLL error is about 1.6e-2), 2.7e-3 for
                        two ancestors, 1.4e-2 for three unrelated ancestors (p = 14).  m = n is the union's own
                        histogram, so its card is the union's estimate.  There is no HLL counterpart of mean_core.

Inputs are listed as `dandd tree` lists them (-d DATADIR or -f LIST, sorted); names are the FASTA base names and must
be distinct.  Written into --name (a directory that must not exist yet), tab-separated, floats by repr:
  kmc
  spectrum.tsv   k  genomes  kmers                                 one row per k and c = 1..n, zeros included
  genomes.tsv    k  name  distinct  private                        input order
  growth.tsv     k  ngen  mean_card  mean_core  mean_delta_pos     m = 1..n; mean_delta_pos = mean_card / k
  dashing
  registers.tsv  k  value  genomes  registers                      T[v][c] per k, nonzero entries only
  genomes.tsv    k  name  card                                     each genome's own estimate, input order
  growth.tsv     k  ngen  mean_card  mean_delta_pos                m = 1..n; mean_delta_pos = mean_card / k
  both
  delta.tsv      ngen  delta  k                                    the delta of the MEAN curve: max over k of
                                                                   mean_card / k, the first k winning a tie
The delta of the mean curve is not the mean of the per-ordering deltas (max and mean do not commute), and the
spectrum cannot give the latter.  Under torchrun every rank counts its key range (kmc) or sketches its share of the
genomes and reads its slice of the registers (dashing), and rank 0 writes."""
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


# ---------------------------------------------------------------- closed forms
def _hits(n: int):
    """(m, hit) for m = 1..n: hit[c - 1] = 1 - C(n - c, m) / C(n, m), float64 [n], the chance that a uniformly random
    m-subset of the n genomes meets a given set of c of them.  The ratios C(n - c, m) / C(n, m) are running products
    over c, no big binomial."""
    c = np.arange(n, dtype=np.float64)                       # c = 0 .. n-1
    for m in range(1, n + 1):
        # miss(c) = C(n - c, m) / C(n, m), the chance that none of a c-genome k-mer's genomes is among the first m:
        # miss(c + 1) = miss(c) (n - c - m) / (n - c), so hit(c) = 1 - miss(c) = sum_{j < c} miss(j) m / (n - j)
        miss = np.concatenate([[1.0], np.maximum(np.cumprod((n - c[:-1] - m) / (n - c[:-1])), 0.0)])   # miss(0 .. n-1)
        yield m, np.cumsum(miss * (m / (n - c)))                                                         # hit(1 .. n)


def hit_weights(n: int) -> np.ndarray:
    """float64 [n, n]: W[c - 1][m - 1] = 1 - C(n - c, m) / C(n, m), the weight of a k-mer (kmc) or a register level
    (dashing) held by c genomes in the mean union of the first m.  A sum of positive terms (no 1 - x cancellation);
    W[c - 1][n - 1] = 1 exactly.  O(n^2) memory."""
    w = np.zeros((n, n))
    for m, hit in _hits(n):
        w[:, m - 1] = hit
    return w


def mean_growth(hist: Sequence[int]):
    """(mean_card, mean_core), float64 [n] each, entry m - 1 for the first m genomes of a uniformly random ordering of
    the n genomes, from the spectrum hist[c - 1] = k-mers held by exactly c genomes.  O(n) memory, O(n^2) time: for each
    m the ratios C(n - c, m) / C(n, m) and C(c, m) / C(n, m) are running products over c, no big binomial.  Both means
    are sums of positive terms (no 1 - x cancellation), so the relative error stays within a few n ulps."""
    h = np.asarray(hist, dtype=np.float64)
    n = len(h)
    card, core = np.zeros(n), np.zeros(n)
    for m, hit in _hits(n):
        card[m - 1] = float(np.dot(h, hit))
        # hold(c) = C(c, m) / C(n, m), the chance that all of the first m are among its c genomes: hold(n) = 1,
        # hold(c - 1) = hold(c) (c - m) / c, and 0 below c = m
        top = np.arange(n, m, -1, dtype=np.float64)          # c = n .. m+1
        hold = np.cumprod(np.concatenate([[1.0], (top - m) / top]))[::-1]                                # hold(m .. n)
        core[m - 1] = float(np.dot(h[m - 1:], hold))
    return card, core


def delta_of_mean(ks: Sequence[int], mean_card: np.ndarray):
    """(delta, k) per ngen from mean_card [nk, n]: the largest mean_card / k, the first k of the list winning a tie
    (delta_summarize's rule)."""
    dk = np.asarray(mean_card, dtype=np.float64) / np.asarray(ks, dtype=np.float64)[:, None]
    best = np.argmax(dk, axis=0)
    return dk[best, np.arange(dk.shape[1])], np.asarray(ks, dtype=np.int64)[best]


# ---------------------------------------------------------------- outputs
def write_outputs(directory: str, names: Sequence[str], ks: Sequence[int], hist, singles, priv) -> List[str]:
    """The four tables from the int64 [nk, n] spectrum, singles and private counts; returns the files written."""
    n = len(names)
    rows = {"spectrum.tsv": ["k\tgenomes\tkmers"], "genomes.tsv": ["k\tname\tdistinct\tprivate"],
            "growth.tsv": ["k\tngen\tmean_card\tmean_core\tmean_delta_pos"], "delta.tsv": ["ngen\tdelta\tk"]}
    cards = np.zeros((len(ks), n))
    for c, k in enumerate(ks):
        rows["spectrum.tsv"] += ["%d\t%d\t%d" % (k, i + 1, v) for i, v in enumerate(hist[c].tolist())]
        rows["genomes.tsv"] += ["%d\t%s\t%d\t%d" % (k, name, d, p) for name, d, p in zip(names, singles[c].tolist(), priv[c].tolist())]
        cards[c], core = mean_growth(hist[c])
        rows["growth.tsv"] += ["\t".join([str(k), str(m + 1), repr(a), repr(b), repr(a / k)])
                               for m, (a, b) in enumerate(zip(cards[c].tolist(), core.tolist()))]
    if len(ks):
        delta, best = delta_of_mean(ks, cards)
        rows["delta.tsv"] += ["%d\t%s\t%d" % (m + 1, repr(d), kk) for m, (d, kk) in enumerate(zip(delta.tolist(), best.tolist()))]
    written = []
    for fn, lines in rows.items():
        path = os.path.join(directory, fn)
        with open(path, "w") as fh:
            fh.write("\n".join(lines) + "\n")
        written.append(path)
    return written


def write_register_outputs(directory: str, names: Sequence[str], ks: Sequence[int], spec, single, cards) -> List[str]:
    """The four dashing tables from the int64 [nk, 64, n] register spectrum, the genomes' own cards [n, nk] and the
    mean cards [nk, n]; returns the files written."""
    rows = {"registers.tsv": ["k\tvalue\tgenomes\tregisters"], "genomes.tsv": ["k\tname\tcard"],
            "growth.tsv": ["k\tngen\tmean_card\tmean_delta_pos"], "delta.tsv": ["ngen\tdelta\tk"]}
    spec, single, cards = np.asarray(spec), np.asarray(single, dtype=np.float64), np.asarray(cards, dtype=np.float64)
    for c, k in enumerate(ks):
        v, g = np.nonzero(spec[c])
        rows["registers.tsv"] += ["%d\t%d\t%d\t%d" % (k, a, b + 1, t) for a, b, t in zip(v.tolist(), g.tolist(), spec[c][v, g].tolist())]
        rows["genomes.tsv"] += ["%d\t%s\t%s" % (k, name, repr(x)) for name, x in zip(names, single[:, c].tolist())]
        rows["growth.tsv"] += ["\t".join([str(k), str(m + 1), repr(a), repr(a / k)]) for m, a in enumerate(cards[c].tolist())]
    if len(ks):
        delta, best = delta_of_mean(ks, cards)
        rows["delta.tsv"] += ["%d\t%s\t%d" % (m + 1, repr(d), kk) for m, (d, kk) in enumerate(zip(delta.tolist(), best.tolist()))]
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
    parser.add_argument("--tool", choices=["kmc", "dashing"], default="kmc",
                        help="kmc: exact distinct k-mer counts (default); dashing: HLL register spectrum")
    parser.add_argument("--mink", type=int, default=2, help="smallest k (1..%d for kmc, 1..%d for dashing)" % (EXACT_MAX_K, HLL_MAX_K))
    parser.add_argument("--maxk", type=int, default=32, help="largest k")
    parser.add_argument("--registers", type=int, default=20, help="log2 of the number of HLL registers (dashing)")
    parser.add_argument("--no-canon", dest="canon", action="store_false", help="count k-mers as read, not canonical")
    parser.add_argument("--name", default="spectrum", help="output directory; it must not exist yet")
    return parser.parse_args(argv)


def _inputs(args):
    """(fastas, names, ks) or a refusal message."""
    import dandd_b200
    dandd_b200.enable_compat()         # the mirrors import each other by the reference's top-level module names
    from dandd_b200.lib.huffman_dandd import list_fastas
    if not (args.genomedir or args.flist_loc):
        return None, "give the inputs: -d DATADIR or -f LIST"
    limit, tool = (HLL_MAX_K, " for dashing") if args.tool == "dashing" else (EXACT_MAX_K, "")
    for flag, k in (("--mink", args.mink), ("--maxk", args.maxk)):
        if not 1 <= k <= limit:
            return None, "%s %d is outside 1..%d%s" % (flag, k, limit, tool)
    if args.mink > args.maxk:
        return None, "--mink %d is above --maxk %d" % (args.mink, args.maxk)
    if args.tool == "dashing" and not 5 <= args.registers <= 26:
        return None, "--registers %d is outside 5..26" % args.registers
    try:
        fastas = list_fastas(args.genomedir, args.flist_loc)
    except (OSError, ValueError) as err:
        return None, "cannot list the inputs: %s" % err
    if not fastas:
        return None, "no FASTA files given"
    names = [os.path.basename(f) for f in fastas]
    dup = sorted({x for x in names if names.count(x) > 1})
    if dup:
        return None, "input names must be distinct: %s" % dup
    if args.tool == "dashing" and len(names) > 65535:
        return None, "at most 65535 inputs for dashing, got %d" % len(names)
    return (fastas, names, list(range(args.mink, args.maxk + 1))), None


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
    fastas, names, ks = got
    n = len(fastas)
    try:
        store = get_store()
        if args.tool == "dashing":
            from dandd_b200 import ingest
            from dandd_b200.helpers.allpairs import gather_leaf_registers
            owners = [[g for g in range(n) if g % world == r] for r in range(world)]
            ingest.prefetch([fastas[g] for g in owners[rank]], want_digest=False)
            regs, single = gather_leaf_registers(store, fastas, ks, args.registers, args.canon, owners, tag="spectrum")
            with timing.span("spectrum_registers"):
                spec, cards = store.register_spectrum_cards(regs, args.registers, shard=(rank, world) if world > 1 else None)
            if rank == 0:
                with timing.span("spectrum_outputs"):
                    write_register_outputs(args.name, names, ks, spec, single, cards)
            return spec, single, cards
        with timing.span("spectrum_exact"):
            hist, singles, priv = store.exact_spectrum(fastas, ks, args.canon, shard=(rank, world) if world > 1 else None)
            if world > 1:              # each k-mer belongs to exactly one rank's key range: the counts add up
                import torch
                dev = getattr(getattr(store, "engine", None), "device", "cpu")
                both = torch.as_tensor(np.concatenate([hist, singles, priv], axis=1), device=dev)
                both = dd_dist.sum_counts(both).cpu().numpy()
                hist, singles, priv = both[:, :n], both[:, n:2 * n], both[:, 2 * n:]
        if rank == 0:
            with timing.span("spectrum_outputs"):
                write_outputs(args.name, names, ks, hist, singles, priv)
    finally:
        timing.dump()          # DANDD_B200_TIMING=<file>: one JSON line of stage times per process
    return hist, singles, priv


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    go()
