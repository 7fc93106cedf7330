#!/usr/bin/env python3
"""All-pairs k-independent Jaccard (KIJ) / per-k Jaccard / ANI tables over a set of FASTA files: the
GPU-backed counterpart of the reference's helpers/allpairs.py (BASELINE config 5 shape).

The reference composes |klist| x N(N+1)/2 shell commands -- `dashing hll -k K -S log2(nest) A [B]`
(helpers/allpairs.py:32-35, 356-370), i.e. BOTH FASTAs are parsed and sketched again for every pair
and every k -- and maps them over a process pool (:376-380).  Here every FASTA is sketched ONCE for
all k (K1 + K2, `store.leaf_block`), the N(N-1)/2 x |klist| union cardinalities come from one
batched pair job on the resident registers (K6, `store.pair_cards`), and the rest is the reference's
arithmetic on that table:

    delta(A)   = max_k card_k(A) / k, first k of --klist wins ties        (delta_summarize, :103-118)
    KIJ(A,B)   = (delta(A) + delta(B) - delta(A u B)) / delta(A u B)       (kij_summarize,   :121-148)
    J_k(A,B)   = (|A| + |B| - |A u B|) / |A u B|                           (j_summarize,     :151-179)
    PHYLIP     lower-triangular 1 - J or Mash distance -ln(2J/(1+J))/k     (summ_to_phylip,  :182-218)

Same function names, tuple layouts, file formats and option names as the reference, with these
deliberate differences (the reference's `go()` cannot run as shipped: it reads an undefined
`args.name` (:333) and calls `run_fneighbor`, which is commented out (:418)):
  * `--name` exists (default "allpairs"); as in the reference the directory must not exist yet;
  * neighbour-joining trees (EMBOSS fneighbor + ete3, both external) are not built: the PHYLIP
    matrices they would be built from are the last product;
  * `--write-commands` defaults to "" -- no commands are run, so the list is only written on request;
  * `--tool kmc` counts the union of a pair exactly (the reference's kmc command line for a pair is
    malformed: it passes "A B" where kmc expects one input, :38-44), all pairs of one k in one device
    job (K7, `store.exact_pair_cards`) that reads every FASTA once;
  * `--extra` understands `--no-canon` (the only sketching flag DandD itself ever passes).
Under torchrun / several ranks the FASTAs are sharded over the GPUs for sketching, the registers
are all-gathered and the pair list is split over the ranks; rank 0 writes the files."""
import argparse
import itertools
import json
import math
import os
import sys
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

HLL_MAX_K = 32       # Dashing's k limit (reference README.md:82)
EXACT_MAX_K = 256    # KMC's
_default_klist = ",".join(str(k) for k in range(2, 100))   # helpers/allpairs.py:295


def get_store():
    from dandd_b200.store import get_store as _get   # torch + CUDA start only when a job is actually run
    return _get()


# ---------------------------------------------------------------- the card table (one batched job)
class CardTable:
    """Cardinalities of every FASTA and of every pair union at every k of the list.
    single[i, c] = card(input i at ks[c]); pair[r, c] = card(input a u input b at ks[c]) with
    (a, b) = pairs[r], the r-th of (0,1), (0,2) .. (n-2,n-1).  The summaries below are the reference's
    (delta_summarize / kij_summarize / j_summarize / summ_to_phylip) evaluated on whole columns: the same
    IEEE operations in the same order, so the same floats, without 10^7 Python tuples."""

    def __init__(self, tool: str, names: Sequence[str], ks: Sequence[int], single: np.ndarray, pair: np.ndarray):
        self.tool, self.names, self.ks = tool, list(names), [int(k) for k in ks]
        n = len(self.names)
        self.single = np.asarray(single, dtype=np.float64).reshape(n, len(self.ks))
        self.pair = np.asarray(pair, dtype=np.float64).reshape(n * (n - 1) // 2, len(self.ks))
        self.pairs = np.stack(np.triu_indices(n, 1), axis=1) if n > 1 else np.zeros((0, 2), dtype=np.int64)
        # the reference's command order within one k: input i alone, then i with every later input
        # (helpers/allpairs.py:358-370), as indices into [single rows; pair rows]
        first = np.concatenate([[0], np.cumsum(n - 1 - np.arange(n))[:-1]]).astype(np.int64) if n else np.zeros(0, np.int64)
        self._order = np.concatenate([np.concatenate([[i], n + first[i] + np.arange(n - 1 - i)]) for i in range(n)]
                                     or [np.zeros(0)]).astype(np.int64)
        both = np.concatenate([np.stack([np.arange(n), np.arange(n)], axis=1), self.pairs]).astype(np.int64)
        self._who = both[self._order]                                             # [(i, j)] per row, i <= j
        self._heads = None
        self._in_order = None

    def pair_row(self, a: int, b: int) -> int:
        a, b = (a, b) if a < b else (b, a)
        n = len(self.names)
        return a * n - a * (a + 1) // 2 + (b - a - 1)

    def cards_in_command_order(self) -> np.ndarray:
        """[n(n+1)/2, nk]: row r = the r-th command of one k."""
        if self._in_order is None:
            self._in_order = np.concatenate([self.single, self.pair])[self._order]
        return self._in_order

    def row_names(self) -> List[Tuple[str, str]]:
        return [(self.names[i], self.names[j]) for i, j in self._who.tolist()]

    def row_heads(self) -> List[str]:
        """"tool<TAB>name1<TAB>name2<TAB>" per row of one k (card.tsv)."""
        if self._heads is None:
            self._heads = ["\t".join((self.tool, a, b)) + "\t" for a, b in self.row_names()]
        return self._heads

    def save(self, directory: str) -> None:
        os.makedirs(directory, exist_ok=True)
        np.save(os.path.join(directory, "single.npy"), self.single)
        np.save(os.path.join(directory, "pair.npy"), self.pair)
        with open(os.path.join(directory, "meta.json"), "w") as fh:
            json.dump({"tool": self.tool, "names": self.names, "ks": self.ks}, fh)

    @classmethod
    def load(cls, directory: str) -> "CardTable":
        with open(os.path.join(directory, "meta.json")) as fh:
            meta = json.load(fh)
        return cls(meta["tool"], meta["names"], meta["ks"], np.load(os.path.join(directory, "single.npy")),
                   np.load(os.path.join(directory, "pair.npy"), mmap_mode="r"))

    def results(self) -> List[Tuple[str, str, str, int, float]]:
        """[(tool, name1, name2, k, card)] exactly as the reference's pool.map returns them (k-major)."""
        who, cards = self.row_names(), self.cards_in_command_order()
        return [(self.tool, a, b, k, card) for c, k in enumerate(self.ks) for (a, b), card in zip(who, cards[:, c].tolist())]

    def _best(self, cards: np.ndarray):
        """(delta, card, k) per row: the largest card/k, the first k of the list winning a tie (numpy's
        first maximum = the reference's strict `>` in --klist order)."""
        dkk = cards / np.asarray(self.ks, dtype=np.float64)
        c = np.argmax(dkk, axis=1) if len(self.ks) else np.zeros(len(cards), dtype=np.int64)
        rows = np.arange(len(cards))
        return dkk[rows, c], cards[rows, c], np.asarray(self.ks, dtype=np.int64)[c]

    def delta_summary(self) -> List[Tuple[str, str, str, float, float, int]]:
        """delta_summarize(self.results()): rows sorted by (name1, name2)."""
        delta, card, k = self._best(self.cards_in_command_order())
        rank = np.empty(len(self.names), dtype=np.int64)
        rank[sorted(range(len(self.names)), key=self.names.__getitem__)] = np.arange(len(self.names))
        by_name = np.argsort(rank[self._who[:, 0]] * len(self.names) + rank[self._who[:, 1]], kind="stable")
        who = self.row_names()
        return [(self.tool,) + who[r] + (d, c, kk) for r, d, c, kk in
                zip(by_name.tolist(), delta[by_name].tolist(), card[by_name].tolist(), k[by_name].tolist())]

    def kij_values(self):
        """(KIJ, k1, k2, k12) per pair of self.pairs (kij_summarize without the dictionaries)."""
        d1, _, k1 = self._best(self.single)
        d12, _, k12 = self._best(self.pair)
        a, b = self.pairs[:, 0], self.pairs[:, 1]
        return jaccard_of(d1[a], d1[b], d12), k1[a], k1[b], k12

    def j_values(self, target_k: int) -> np.ndarray:
        """J at one k per pair of self.pairs."""
        c = self.ks.index(target_k)
        return jaccard_of(self.single[self.pairs[:, 0], c], self.single[self.pairs[:, 1], c], self.pair[:, c])

    def j_summary(self, target_k: int) -> List[tuple]:
        """j_summarize(self.results(), target_k)."""
        if target_k not in self.ks:
            return []
        return [(self.tool, self.names[a], self.names[b], target_k, j, None, None, None)
                for (a, b), j in zip(self.pairs.tolist(), self.j_values(target_k).tolist())]

    def write_phylip(self, values: np.ndarray, filename: str) -> None:
        """One value per pair of self.pairs -> lower-triangular PHYLIP matrix over the sorted names, the
        text summ_to_phylip writes for the same numbers."""
        n = len(self.names)
        full = np.zeros((n, n))
        full[self.pairs[:, 0], self.pairs[:, 1]] = values
        full[self.pairs[:, 1], self.pairs[:, 0]] = values
        by_name = sorted(range(n), key=self.names.__getitem__)
        full = full[by_name][:, by_name]
        with open(filename, "wt") as fh:
            fh.write("%d\n" % n)
            fh.write("".join(" ".join([self.names[g]] + list(map(repr, full[i, :i].tolist()))) + "\n"
                             for i, g in enumerate(by_name)))


def mash_distances(j: np.ndarray, k) -> np.ndarray:
    """mash_distance over a column: the products and quotients are IEEE-exact in numpy as in Python, the
    logarithm is taken with math.log value by value (numpy's vector log may differ in the last bit)."""
    j = np.maximum(j, sys.float_info.epsilon)
    return -np.asarray(list(map(math.log, (2.0 * j / (1.0 + j)).tolist()))).reshape(j.shape) / k


def gather_leaf_registers(store, inputs: Sequence[str], ks: Sequence[int], p: int, canon: bool, owners, tag: str = "allpairs"):
    """(regs, single): the registers uint8 [n, nk, 2^p] of every input on this rank's device, on every rank, and their
    cardinalities float64 [n, nk] on the host.  Rank r sketches the inputs owners[r] lists (each once, all k) into its
    slice of the job's array; one all-gather then gives every rank the whole array."""
    import torch
    from dandd_b200 import dist as dd_dist
    from dandd_b200 import timing
    rank, _ = dd_dist.world()
    dev = getattr(getattr(store, "engine", None), "device", "cpu")
    local = torch.empty((len(owners[rank]), len(ks), 1 << p), dtype=torch.uint8, device=dev)
    local_cards = np.zeros((len(owners[rank]), len(ks)))
    with timing.span(tag + "_sketch"):
        for j, g in enumerate(owners[rank]):      # the registers land in their slice of the job's array
            local_cards[j] = store.leaf_block(inputs[g], ks, p, canon, out=local[j])[1]
    local_cards = torch.as_tensor(local_cards, dtype=torch.float64, device=dev)
    with timing.span(tag + "_gather"):
        regs = dd_dist.gather_registers(local, owners)                     # [n, nk, 2^p] on every rank
        single = dd_dist.gather_cards(local_cards, owners).cpu().numpy()
    return regs, single


def card_table(tool: str, inputs: Sequence[str], names: Sequence[str], klist: Sequence[int], nest: int = 262144,
               extra: str = "", store=None, tile_pairs: int = 1 << 16) -> CardTable:
    """Every cardinality the reference's command list asks for, as one device job per rank.
    tool 'dashing': HLL with log2(nest) register bits (`dashing hll -k K -S p [extra] A [B]`);
    tool 'kmc': exact distinct canonical k-mer counts (`kmc -k K -fm -ci1 -cs2` + `kmc_tools info`)."""
    import torch
    from dandd_b200 import dist as dd_dist
    if len(set(names)) != len(names):
        raise RuntimeError("input names must be distinct: %s" % sorted(n for n in set(names) if list(names).count(n) > 1))
    ks = [int(k) for k in klist]
    canon = True
    for token in extra.split():
        if token == "--no-canon":
            canon = False
        else:
            raise RuntimeError('Unsupported --extra argument "%s" (only --no-canon is understood)' % token)
    limit = {"dashing": HLL_MAX_K, "kmc": EXACT_MAX_K}.get(tool)
    if limit is None:
        raise RuntimeError("No card function for tool %s" % tool)      # reference: dashing2 raises the same way (:74-80)
    bad = [k for k in ks if not 1 <= k <= limit]
    if bad:
        raise RuntimeError('%s cannot count k-mers of length %s (1 <= k <= %d)' % (tool, bad, limit))
    store = store or get_store()
    rank, world = dd_dist.world()
    n = len(inputs)
    owners = [[g for g in range(n) if g % world == r] for r in range(world)]
    pairs = np.stack(np.triu_indices(n, 1), axis=1).astype(np.int32) if n > 1 else np.zeros((0, 2), dtype=np.int32)
    span = dd_dist.split_work(len(pairs))
    mine = pairs[span.start:span.stop]
    if tool == "dashing" and (nest < 1 or nest & (nest - 1)):
        raise RuntimeError("--nest must be a power of 2 for dashing (got %d)" % nest)
    from dandd_b200 import ingest, timing
    batched_exact = tool == "kmc" and hasattr(store, "exact_pair_cards")        # every rank reads every FASTA
    ingest.prefetch(list(inputs) if batched_exact else [inputs[g] for g in owners[rank]], want_digest=False)   # file i+1.. are read while the GPU works on file i
    if tool == "dashing":
        p = int(math.log2(nest))
        uniq = sorted(set(ks))
        regs, single = gather_leaf_registers(store, inputs, uniq, p, canon, owners)
        with timing.span("allpairs_pairs"):
            part = store.pair_cards(regs, mine, p, tile_pairs)
        col = [uniq.index(k) for k in ks]
        single, part = single[:, col], part[:, col]
    elif batched_exact:
        # one batched job per k; under several ranks every rank counts its key range of the same job and
        # the integer counts are summed (each k-mer belongs to exactly one rank's range)
        with timing.span("allpairs_exact"):
            single, pair = store.exact_pair_cards(inputs, ks, canon, shard=(rank, world) if world > 1 else None)
            if world > 1:
                dev = getattr(getattr(store, "engine", None), "device", "cpu")
                both = torch.as_tensor(np.concatenate([single, pair]).astype(np.int64), device=dev)
                both = dd_dist.sum_counts(both).cpu().numpy().astype(np.float64)
                single, pair = both[:n], both[n:]
        return CardTable(tool, names, ks, single, pair)
    else:
        with timing.span("allpairs_exact"):
            single_mine = np.array([[store.exact_count([inputs[g]], k, canon) for k in ks] for g in owners[rank]],
                                   dtype=np.float64).reshape(len(owners[rank]), len(ks))
            part = np.array([[store.exact_count([inputs[a], inputs[b]], k, canon) for k in ks] for a, b in mine],
                            dtype=np.float64).reshape(len(mine), len(ks))
        single = np.zeros((n, len(ks)))
        for r, rows in enumerate(_gather_objects(single_mine, world)):
            single[owners[r]] = rows
    pair = np.concatenate(_gather_objects(part, world), axis=0) if world > 1 else part
    return CardTable(tool, names, ks, single, pair)


def _gather_objects(obj, world):
    if world == 1:
        return [obj]
    import torch.distributed as dist
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


# ---------------------------------------------------------------- the reference's summaries, on tuple lists
def jaccard_of(a, b, ab):
    """(a + b - ab) / ab: the Jaccard index from the sizes of two sets and of their union; over deltas instead of
    sizes, KIJ (helpers/allpairs.py:121-179).  Scalars or numpy arrays."""
    return (a + b - ab) / ab


def delta_summarize(results):
    """[(tool, name1, name2, k, card)] -> [(tool, name1, name2, delta, card, k)] sorted by the names:
    the largest card/k per (tool, name1, name2); the first k seen wins a tie (helpers/allpairs.py:103-118)."""
    best: Dict[tuple, tuple] = {}
    for tool, name1, name2, k, card in results:
        key, score = (tool, name1, name2), card / k
        if key not in best or score > best[key][0]:
            best[key] = (score, card, k)
    return [key + best[key] for key in sorted(best)]


def kij_summarize(delta_summary):
    """-> [(tool, name1, name2, 0, KIJ, k1, k2, k12)] over every two inputs, in the order of the
    sorted names; k = 0 marks "no single k" (helpers/allpairs.py:121-148)."""
    alone, together, tool = {}, {}, None
    for tool, name1, name2, delta, _card, k in delta_summary:
        if name1 == name2:
            alone[name1] = (delta, k)
        else:
            together[frozenset((name1, name2))] = (delta, k)
    out = []
    for a, b in itertools.combinations(alone, 2):
        (da, ka), (db, kb), (dab, kab) = alone[a], alone[b], together[frozenset((a, b))]
        out.append((tool, a, b, 0, jaccard_of(da, db, dab), ka, kb, kab))
    return out


def j_summarize(results, target_k):
    """-> [(tool, name1, name2, target_k, J, None, None, None)] from the cardinalities at one fixed k
    (helpers/allpairs.py:151-179)."""
    alone, together, tool = {}, {}, None
    for tool_, name1, name2, k, card in results:
        tool = tool_
        if k != target_k:
            continue
        if name1 == name2:
            alone[name1] = card
        else:
            together[frozenset((name1, name2))] = card
    out = []
    for a, b in itertools.combinations(alone, 2):
        out.append((tool, a, b, target_k, jaccard_of(alone[a], alone[b], together[frozenset((a, b))]), None, None, None))
    return out


def mash_distance(j, k):
    """-ln(2J / (1 + J)) / k, J clamped to the smallest positive float; already a distance
    (helpers/allpairs.py:210-218)."""
    try:
        j = max(j, sys.float_info.epsilon)
        return -(math.log(2.0 * j / (1.0 + j))) / k
    except ValueError:
        raise RuntimeError("Could not compute mash distance for k=%d, j=%f" % (k, j))


def summ_to_phylip(summ, seqid_to_treid, phylip_fn, convert_to_ani=False):
    """Lower-triangular PHYLIP distance matrix over the sorted names: 1 - J, or the Mash distance at
    k (k = 0: at max(k1, k2, k12)) (helpers/allpairs.py:182-207)."""
    assert len(summ) > 0
    dist_of = {}
    for _tool, name1, name2, k, j, k1, k2, k12 in summ:
        if convert_to_ani:
            if k == 0:
                assert k1 is not None and k2 is not None and k12 is not None
            value = mash_distance(j, k if k else max(k1, k2, k12))
        else:
            value = 1 - j
        dist_of[frozenset((name1, name2))] = value
    names = sorted(set().union(*dist_of))
    assert len(names) == len(seqid_to_treid), (len(names), len(seqid_to_treid))
    with open(phylip_fn, "wt") as fh:
        fh.write("%d\n" % len(names))
        for i, name1 in enumerate(names):
            fh.write(" ".join([name1] + [str(dist_of[frozenset((name1, name2))]) for name2 in names[:i]]) + "\n")


def rename_seqids_in_tree(orig_tree, seqid_to_treid):
    """Replace every sequence id in a Newick string by its tree id (helpers/allpairs.py:273-289): at each
    position the first id (in dict order) that matches there wins."""
    out, i = [], 0
    while i < len(orig_tree):
        hit = next((sid for sid in seqid_to_treid if orig_tree.startswith(sid, i)), None)
        out.append(seqid_to_treid[hit] if hit is not None else orig_tree[i])
        i += len(hit) if hit is not None else 1
    return "".join(out)


# ---------------------------------------------------------------- command line
def reference_command(tool, k, nest, extra, inputs):
    """The shell command the reference would have run for this cell (for --write-commands only)."""
    if tool == "dashing":
        return "dashing hll -k %d -S %d %s %s %s" % (k, int(math.log2(nest)), extra, "", inputs)
    count = "test -f %s.kmc_pre || kmc -v -k%d -fm -ci1 -cs2 %s %s /tmp/" % (inputs, k, inputs, inputs)
    # (the database name is never substituted into the reference's `kmc_tools info %s`, :38-44)
    return "(" + count + ") && kmc_tools info %s | head -n 2 | tail -n 1 | awk '{print $NF}'"


OPTIONS = [
    ("--tool", str, "kmc", "which tool's numbers to produce: dashing (HLL) or kmc (exact)"),
    ("--name", str, "allpairs", "run name; a directory of this name is created and must not exist yet"),
    ("--dataset", str, "dataset.json", "AFproject dataset json file (seqids, treids)"),
    ("--write-commands", str, "", "write the reference's command list to <name>/<this file> (nothing is run from it)"),
    ("--card-results", str, "card.tsv", "write raw cardinalities results here"),
    ("--delta-results", str, "delta.tsv", "write delta results here"),
    ("--j-results-phylip", str, "sim.phylip", "write all-pairs 1-minus-Js and 1-minus-KIJs here, PHYLIP format"),
    ("--ani-results-phylip", str, "ani.phylip", "write all-pairs Mash distances here, PHYLIP format"),
    ("--extra", str, "", "extra arguments for the sketching tool (--no-canon)"),
    ("--nest", int, 262144, "# estimators (power of 2 required for dashing)"),
    ("--bitsper", int, 8, "bits per estimator (default 8; 8 required for dashing)"),
    ("--klist", str, _default_klist, "ks to try"),
    ("--cpu", int, -1, "accepted for compatibility; the device job is not a process pool"),
]


def parse_arguments(argv=None):
    parser = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    for flag, kind, default, text in OPTIONS:
        parser.add_argument(flag, type=kind, default=default, help=text)
    return parser.parse_args(argv)


def _with_tag(filename: str, tag: str) -> str:
    """sim.phylip -> sim.kij.phylip / sim.k21.phylip (helpers/allpairs.py:404-406)."""
    parts = filename.split(".")
    return ".".join(parts[:-1] + [tag, parts[-1]])


def load_dataset(path: str):
    """-> (inputs, names, seqid_to_treid) from an AFproject dataset file (helpers/allpairs.py:338-357):
    `<seqid>.fasta` must exist; its base name holds exactly one dot."""
    if not os.path.exists(path):
        raise RuntimeError('No dataset file "%s"' % path)
    with open(path, "rt") as fh:
        data = json.load(fh)
    assert len(data["treids"]) == 0 or len(data["treids"]) == len(data["seqids"])
    seqid_to_treid = dict(zip(data["seqids"], data["treids"] or data["seqids"]))
    assert len(seqid_to_treid) > 0
    inputs, names = [], []
    for seqid in data["seqids"]:
        fasta = seqid + ".fasta"
        if not os.path.exists(fasta):
            raise RuntimeError('Input path does not exist: "%s"' % fasta)
        base = os.path.basename(fasta)
        assert base.count(".") == 1
        inputs.append(fasta)
        names.append(base.split(".")[0])
    return inputs, names, seqid_to_treid


def write_outputs(table: CardTable, args, seqid_to_treid, inputs: Optional[List[str]] = None) -> List[str]:
    """card.tsv, delta.tsv and the PHYLIP matrices, in the reference's formats (helpers/allpairs.py:381-432).
    Returns the files written."""
    written = []
    klist = table.ks
    if args.write_commands and inputs is not None:
        fn = os.path.join(args.name, args.write_commands)
        n = len(inputs)
        with open(fn, "wt") as fh:
            lines = []
            for k in klist:
                for i in range(n):
                    lines.append(str((table.tool, table.names[i], table.names[i], k,
                                      reference_command(table.tool, k, args.nest, args.extra, inputs[i]))))
                    for j in range(i + 1, n):
                        lines.append(str((table.tool, table.names[i], table.names[j], k,
                                          reference_command(table.tool, k, args.nest, args.extra, inputs[i] + " " + inputs[j]))))
            fh.write("\n".join(lines) + "\n")
        written.append(fn)
    with open(args.delta_results, "wt") as fh:
        # (the reference's header says delta, card, k but its rows hold k, card, delta: kept, :386-389)
        fh.write("\t".join(["tool", "name1", "name2", "delta", "card", "k"]) + "\n")
        fh.write("".join(["\t".join([tool, name1, name2, str(k), repr(card), repr(delta)]) + "\n"
                         for tool, name1, name2, delta, card, k in table.delta_summary()]))
    written.append(args.delta_results)
    # the big files -- one block of card.tsv per k, two PHYLIP matrices per k -- are independent pieces:
    # 3.5 x 10^7 float -> text conversions for 1000 inputs x 23 k, spread over worker processes when large
    pieces = [("card", k, args.card_results + ".part%d" % c) for c, k in enumerate(klist)]
    if len(table.names) >= 2:
        assert len(table.names) == len(seqid_to_treid), (len(table.names), len(seqid_to_treid))
        for k in [0] + klist:
            tag = "kij" if k == 0 else "k%d" % k
            if args.j_results_phylip:
                pieces.append(("sim", k, _with_tag(args.j_results_phylip, tag)))
            if args.ani_results_phylip:
                pieces.append(("ani", k, _with_tag(args.ani_results_phylip, tag)))
    cells = len(table._order) * len(klist)
    workers = min(len(pieces), 32, args.cpu if args.cpu > 0 else (os.cpu_count() or 1))
    if workers > 1 and cells >= PARALLEL_MIN_CELLS and os.path.isdir(args.name):
        import concurrent.futures
        import multiprocessing
        import shutil
        shared = os.path.join(args.name, ".table")
        table.save(shared)
        try:    # spawn, not fork: this process holds a CUDA context
            with concurrent.futures.ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("spawn")) as pool:
                list(pool.map(_write_piece, [(shared,) + piece for piece in pieces]))
        finally:
            shutil.rmtree(shared, ignore_errors=True)
    else:
        for piece in pieces:
            write_piece(table, *piece)
    with open(args.card_results, "wb") as fh:
        fh.write(("\t".join(["tool", "name1", "name2", "k", "card"]) + "\n").encode())
        for kind, _k, part in pieces:
            if kind == "card":
                with open(part, "rb") as src:
                    while chunk := src.read(1 << 24):
                        fh.write(chunk)
                os.remove(part)
    written.append(args.card_results)
    return written + [fn for kind, _k, fn in pieces if kind != "card"]


PARALLEL_MIN_CELLS = int(os.environ.get("DANDD_B200_ALLPAIRS_PARALLEL_MIN", str(2_000_000)))


def write_piece(table: CardTable, kind: str, k: int, filename: str) -> None:
    """One independent piece of the output: the card.tsv block of one k, or one PHYLIP matrix
    (k = 0: the KIJ matrix; its Mash distances are taken at the largest of the pair's three k)."""
    if kind == "card":
        c = table.ks.index(k)
        tail = "%d\t" % k
        with open(filename, "wt") as fh:
            fh.write("".join([head + tail + repr(card) + "\n"
                             for head, card in zip(table.row_heads(), table.cards_in_command_order()[:, c].tolist())]))
        return
    if k == 0:
        sim, k1, k2, k12 = table.kij_values()
        at_k = np.maximum(np.maximum(k1, k2), k12)
    else:
        sim, at_k = table.j_values(k), k
    table.write_phylip(1 - sim if kind == "sim" else mash_distances(sim, at_k), filename)


_worker_tables: Dict[str, CardTable] = {}


def _write_piece(spec) -> None:
    """Worker-process entry: the table is loaded once per process from the directory the parent saved it in."""
    directory, kind, k, filename = spec
    if directory not in _worker_tables:
        _worker_tables[directory] = CardTable.load(directory)
    write_piece(_worker_tables[directory], kind, k, filename)


def go(argv=None):
    args = parse_arguments(argv)
    from dandd_b200 import dist as dd_dist
    rank, world = dd_dist.init()
    refusal = None
    if rank == 0:
        print('Performing run with name "%s"' % args.name)
        if os.path.exists(args.name):
            refusal = 'Output directory with name "%s" already exists' % args.name
        else:
            os.makedirs(args.name)
    if world > 1:                      # every rank leaves together, none is left waiting in a collective
        refusal = dd_dist.broadcast_object(refusal)
    if refusal:
        raise RuntimeError(refusal)
    inputs, names, seqid_to_treid = load_dataset(args.dataset)
    klist = [int(k) for k in args.klist.split(",")]
    from dandd_b200 import timing
    try:
        table = card_table(args.tool, inputs, names, klist, nest=args.nest, extra=args.extra)
        if rank == 0:
            with timing.span("allpairs_outputs"):
                write_outputs(table, args, seqid_to_treid, inputs)
    finally:
        timing.dump()          # DANDD_B200_TIMING=<file>: one JSON line of stage times per process
    return table


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    go()
