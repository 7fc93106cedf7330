#!/usr/bin/env python3
"""Query genomes against a collection: how much each query would raise the collection's delta, and how close it is to
every member.

For a new assembly, a batch of new strains or a suspect sample, this answers what `find_delta_delta` answers for removal,
for addition instead: the delta of the collection plus the query, and, for every (query, reference) pair, the cards of
the two genomes and of their union, Jaccard, containment and KIJ.  Queries are not added to one another.

  --tool dashing  the HLL registers of references and queries (one read per rank), then store.query_cards: the union of
                  the references (K3, K4), card(U u q) for every query from one K11 dense step, and the Q x R pair cards
                  (K6).  The histograms are the ones the per-union path builds for the same members, so the estimates are
                  the same floats.
  --tool kmc      one exact device job per k (store.exact_query_cards, K7 lists + K13): |U u q| = |U| + |q| - |q n U| and
                  |q u r| = |q| + |r| - |q n r|, in integers.

delta is the maximum over the swept k of card / k, the first k winning a tie (delta_summarize's rule); KIJ is
kij_summarize's (delta_q + delta_r - delta_qr) / delta_qr.  Under HLL, `novel` and `gain` are differences of two
estimates: their error is that of the estimates, not a fraction of themselves.

References are listed as `dandd tree` lists its inputs (-d DATADIR or -f LIST, sorted), queries likewise (-q DIR or
--query-list FILE, sorted); names are the FASTA base names and must be distinct among the references and among the
queries (a file may be both).  Written into --name (a directory that must not exist yet), tab-separated, floats by repr,
integers for kmc:
  union.tsv       k  card  delta_pos                     the union of the references; delta_pos = card / k
  collection.tsv  ngen  delta  k                         delta of the references
  with.tsv        k  query  card  novel  delta_pos       the references plus the query; novel = card - union card
  delta.tsv       query  delta  k  gain                  delta of the references plus the query; gain = delta - delta(collection)
  pairs.tsv       k  query  reference  card_query  card_reference  card_union  jaccard  containment
                                                         containment = |q n r| / |q|
  kij.tsv         query  reference  delta_query  delta_reference  delta_union  kij
Under torchrun every rank sketches its share of the genomes and takes the queries q = rank (mod world) (dashing), or
counts its key range (kmc); rank 0 writes."""
import argparse
import os
import sys
from typing import List, Sequence

import numpy as np

HLL_MAX_K = 32               # Dashing's
EXACT_MAX_K = 256            # KMC's
MAX_CELLS = 1 << 32          # query x reference pairs of one job (DD_QUERY_MAX_CELLS)
MAX_GENOMES_LONG_K = 65536   # references + queries of one exact job above k = 64


def get_store():
    from dandd_b200.store import get_store as _get   # torch + CUDA start only when a job is actually run
    return _get()


# ---------------------------------------------------------------- outputs
def write_outputs(directory: str, refs: Sequence[str], queries: Sequence[str], ks: Sequence[int], ref_single, query_single,
                  union, with_q, pair, exact: bool) -> List[str]:
    """The six tables from ref_single [nk, R], query_single [nk, Q], union [nk], with_q [nk, Q] and pair [nk, Q, R]
    (float64 for HLL, int64 for exact counts)."""
    from dandd_b200.helpers.allpairs import jaccard_of
    from dandd_b200.helpers.leaveout import best_k
    num = (lambda v: "%d" % v) if exact else repr
    ref_single, query_single, union = np.asarray(ref_single), np.asarray(query_single), np.asarray(union)
    with_q, pair = np.asarray(with_q), np.asarray(pair)
    rows = {"union.tsv": ["k\tcard\tdelta_pos"], "collection.tsv": ["ngen\tdelta\tk"],
            "with.tsv": ["k\tquery\tcard\tnovel\tdelta_pos"], "delta.tsv": ["query\tdelta\tk\tgain"],
            "pairs.tsv": ["k\tquery\treference\tcard_query\tcard_reference\tcard_union\tjaccard\tcontainment"],
            "kij.tsv": ["query\treference\tdelta_query\tdelta_reference\tdelta_union\tkij"]}
    cq, cr = query_single[:, :, None], ref_single[:, None, :]
    with np.errstate(divide="ignore", invalid="ignore"):     # an empty union or query (k above its length): nan
        jac = jaccard_of(cq, cr, pair)
        cont = (cq + cr - pair) / cq
    for c, k in enumerate(ks):
        u = union[c].item()
        rows["union.tsv"].append("%d\t%s\t%s" % (k, num(u), repr(u / k)))
        for q, qn in enumerate(queries):
            w = with_q[c, q].item()
            rows["with.tsv"].append("%d\t%s\t%s\t%s\t%s" % (k, qn, num(w), num(w - u), repr(w / k)))
        for q, qn in enumerate(queries):
            a = query_single[c, q].item()
            for r, rn in enumerate(refs):
                rows["pairs.tsv"].append("%d\t%s\t%s\t%s\t%s\t%s\t%s\t%s" % (
                    k, qn, rn, num(a), num(ref_single[c, r].item()), num(pair[c, q, r].item()), repr(jac[c, q, r].item()),
                    repr(cont[c, q, r].item())))
    if len(ks):
        d_all, k_all = best_k(ks, union)
        rows["collection.tsv"].append("%d\t%s\t%d" % (len(refs), repr(float(d_all)), int(k_all)))
        d_with, k_with = best_k(ks, with_q)
        for qn, d, kk in zip(queries, d_with.tolist(), k_with.tolist()):
            rows["delta.tsv"].append("%s\t%s\t%d\t%s" % (qn, repr(d), kk, repr(d - float(d_all))))
        d_q, _ = best_k(ks, query_single)
        d_r, _ = best_k(ks, ref_single)
        d_qr, _ = best_k(ks, pair)
        with np.errstate(divide="ignore", invalid="ignore"):
            kij = jaccard_of(d_q[:, None], d_r[None, :], d_qr)
        for q, qn in enumerate(queries):
            for r, rn in enumerate(refs):
                rows["kij.tsv"].append("%s\t%s\t%s\t%s\t%s\t%s" % (qn, rn, repr(d_q[q].item()), repr(d_r[r].item()),
                                                                   repr(d_qr[q, r].item()), repr(kij[q, r].item())))
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
    src.add_argument("-d", "--datadir", dest="genomedir", default=None, help="directory of reference FASTA files")
    src.add_argument("-f", "--fastas", dest="flist_loc", default=None, help="file listing one reference FASTA path per line")
    qsrc = parser.add_mutually_exclusive_group()
    qsrc.add_argument("-q", "--queries", dest="querydir", default=None, help="directory of query FASTA files")
    qsrc.add_argument("--query-list", dest="qlist_loc", default=None, help="file listing one query FASTA path per line")
    parser.add_argument("--tool", choices=["dashing", "kmc"], default="dashing",
                        help="dashing: HLL estimates (default); kmc: exact distinct k-mer counts")
    parser.add_argument("--mink", type=int, default=2, help="smallest k (1..%d for dashing, 1..%d for kmc)" % (HLL_MAX_K, EXACT_MAX_K))
    parser.add_argument("--maxk", type=int, default=32, help="largest k")
    parser.add_argument("--registers", type=int, default=20, help="log2 of the number of HLL registers (dashing)")
    parser.add_argument("--no-canon", dest="canon", action="store_false", help="count k-mers as read, not canonical")
    parser.add_argument("--name", default="query", help="output directory; it must not exist yet")
    return parser.parse_args(argv)


def _inputs(args):
    """(refs, ref_names, queries, query_names, ks) or a refusal message."""
    import dandd_b200
    dandd_b200.enable_compat()         # the mirrors import each other by the reference's top-level module names
    from dandd_b200.lib.huffman_dandd import list_fastas
    if not (args.genomedir or args.flist_loc):
        return None, "give the references: -d DATADIR or -f LIST"
    if not (args.querydir or args.qlist_loc):
        return None, "give the queries: -q DIR or --query-list FILE"
    limit = HLL_MAX_K if args.tool == "dashing" else EXACT_MAX_K
    for flag, k in (("--mink", args.mink), ("--maxk", args.maxk)):
        if not 1 <= k <= limit:
            return None, "%s %d is outside 1..%d for %s" % (flag, k, limit, args.tool)
    if args.mink > args.maxk:
        return None, "--mink %d is above --maxk %d" % (args.mink, args.maxk)
    if args.tool == "dashing" and not 5 <= args.registers <= 26:
        return None, "--registers %d is outside 5..26" % args.registers
    got = []
    for what, d, listing in (("references", args.genomedir, args.flist_loc), ("queries", args.querydir, args.qlist_loc)):
        try:
            fastas = list_fastas(d, listing)
        except (OSError, ValueError) as err:
            return None, "cannot list the %s: %s" % (what, err)
        if not fastas:
            return None, "no %s given" % what
        names = [os.path.basename(f) for f in fastas]
        dup = sorted({x for x in names if names.count(x) > 1})
        if dup:
            return None, "the names of the %s must be distinct: %s" % (what, dup)
        got += [fastas, names]
    refs, queries = got[0], got[2]
    if len(refs) * len(queries) > MAX_CELLS:
        return None, "%d queries x %d references is above %d pairs" % (len(queries), len(refs), MAX_CELLS)
    if args.tool == "kmc" and args.maxk > 64 and len(refs) + len(queries) > MAX_GENOMES_LONG_K:
        return None, "above k = 64 at most %d references + queries, got %d" % (MAX_GENOMES_LONG_K, len(refs) + len(queries))
    return (got[0], got[1], got[2], got[3], list(range(args.mink, args.maxk + 1))), None


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
    refs, ref_names, queries, query_names, ks = got
    R, shard = len(refs), ((rank, world) if world > 1 else None)
    try:
        store = get_store()
        if args.tool == "dashing":
            from dandd_b200 import ingest
            from dandd_b200.helpers.allpairs import gather_leaf_registers
            inputs = refs + queries
            owners = [[g for g in range(len(inputs)) if g % world == r] for r in range(world)]
            ingest.prefetch([inputs[g] for g in owners[rank]], want_digest=False)
            regs, _ = gather_leaf_registers(store, inputs, ks, args.registers, args.canon, owners, tag="query")
            with timing.span("query_cards"):
                cards = store.query_cards(regs, R, args.registers, shard=shard)
        else:
            with timing.span("query_exact"):
                cards = store.exact_query_cards(refs, queries, ks, args.canon, shard=shard)
                if world > 1:          # each k-mer belongs to exactly one rank's key range: the counts add up
                    import torch
                    dev = getattr(getattr(store, "engine", None), "device", "cpu")
                    flat = torch.as_tensor(np.concatenate([np.asarray(a).reshape(len(ks), -1) for a in cards], axis=1), device=dev)
                    flat = dd_dist.sum_counts(flat).cpu().numpy()
                    split = np.cumsum([np.asarray(a).reshape(len(ks), -1).shape[1] for a in cards])[:-1]
                    cards = tuple(part.reshape(np.shape(a)) for part, a in zip(np.split(flat, split, axis=1), cards))
        if rank == 0:
            with timing.span("query_outputs"):
                write_outputs(args.name, ref_names, query_names, ks, *cards, exact=args.tool == "kmc")
    finally:
        timing.dump()          # DANDD_B200_TIMING=<file>: one JSON line of stage times per process
    return cards


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    go()
