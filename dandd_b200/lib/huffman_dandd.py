"""Delta trees: which sketches DandD asks for, in which order, and what it reports.

Drop-in for the reference module of the same name (reference lib/huffman_dandd.py): same classes
(DeltaTreeNode, DeltaTree, SubSpider, DeltaSpider), same public methods, same pickled attributes,
same CSV/pickle outputs.  The experiment logic -- the stateful k hill-climb, the odd n-ary tree
shape, orderings, KIJ/Jaccard formulas -- is reproduced decision for decision, because it defines
which (node, k) cells exist and therefore what the output files contain.

What differs is the one place where the reference hands work to the outside world:
DeltaTreeNode.ksweep_update_node builds `parallel -j 95% '<dashing|kmc command with {}>' ::: k...`
(reference :148-239).  Here that line becomes ONE batched SketchStore call per node: a fused all-k
GPU pass for a leaf, one union+histogram+MLE launch over all missing k for an inner node; the
sketch files and the cardinality cache are then filled for the whole k range at once, so the
per-k SketchObj constructors that follow find everything cached.  Progressive unions
(DeltaTree.progressive_union, reference :624-663) additionally pre-compute every prefix union of
every ordering in a single launch (a running max: n sketch reads per ordering instead of the
reference's n(n+1)/2).
"""
import contextlib
import csv
import os
import pickle
import sys
from itertools import permutations
from math import factorial
from random import sample, shuffle
from typing import Dict, List, Set, Tuple

from sketch_classes import DashSketchObj, KMCSketchObj, SketchFilePath, SketchObj, ensure_dir, exact_family, nonempty_file  # noqa: F401
from species_specifics import SpeciesSpecifics

from dandd_b200 import ingest, timing


def get_store():
    """The process-wide sketch store (dandd_b200.store), imported on first use: a run that is served
    entirely from the sketch database -- or ends in an argument error -- never pays for importing
    torch and starting CUDA."""
    from dandd_b200.store import get_store as _get
    return _get()


HLL_MAX_K = 32      # "maxk<=32 for estimation" (reference README.md:82, lib/huffman_dandd.py:109-110)
EXACT_MAX_K = 256   # KMC's own k limit
MIN_KSLOTS = 100    # default length of DeltaTreeNode.ksketches (index = k, slot 0 = sweep template)


def write_listdict_to_csv(outfile: str, listdict: List[Dict], suffix: str = "", last_col: str = None):
    """Rows (dicts) -> CSV with the union of their keys as header.  The column order of the reference
    comes from a set (reference :18-21) and so varies from run to run; here it is first-seen order,
    with `fastas` / `files` forced last as in the reference because they may contain commas."""
    columns: List[str] = []
    for row in listdict:
        for key in row:
            if key not in columns:
                columns.append(key)
    for special in ("fastas", "files"):
        if special in columns:
            last_col = special
    if last_col in columns:
        columns.remove(last_col)
        columns.append(last_col)
    to_stdout = outfile is None or outfile == "-"
    handle = sys.stdout if to_stdout else open(outfile + suffix, "w", newline="")
    try:
        writer = csv.DictWriter(handle, fieldnames=columns)
        writer.writeheader()
        writer.writerows(listdict)
    finally:
        if not to_stdout:
            handle.close()


def permute(length, norder, preexist=set(), exhaust=False, verbose=False) -> Set[Tuple[int]]:
    """A set of `norder` distinct orderings of range(length), extending `preexist` (reference :36-60):
    all permutations shuffled when there are few (< 7!+1) or all are wanted, random draws otherwise."""
    total = factorial(length)
    norder = min(norder, total)
    chosen = set(preexist)
    if verbose:
        print(f"{norder} permutations will be produced.")
    if total < 5041 or norder == total or exhaust:
        pool = list(permutations(range(length)))
        shuffle(pool)
    else:
        pool = []
        while len(pool) < norder:
            pool.extend(tuple(sample(range(length), length)) for _ in range(norder))
            pool = list(set(pool))
    for candidate in pool:
        if len(chosen) >= norder:
            break
        chosen.add(candidate)
    return chosen


def _sketch_class(tool: str):
    return {"dashing": DashSketchObj, "kmc": KMCSketchObj}[tool]


class DeltaTreeNode:
    """A FASTA (leaf) or the union of its children's FASTAs (inner node).

    ksketches[k] is the SketchObj of this node at k (None until requested); ksketches[0] holds the
    k-sweep template whose names contain a literal '{}' (reference :150,183)."""

    def __init__(self, node_title: str, children: list, speciesinfo: SpeciesSpecifics, experiment: dict, progeny: list = []):
        self.node_title = node_title
        self.progeny = progeny
        self.experiment = experiment
        self.speciesinfo = speciesinfo
        self.children = children
        self.mink, self.maxk = experiment["ksweep"] if experiment["ksweep"] is not None else (0, 0)
        self.bestk = 0
        self.delta = 0
        self.ksketches = [None] * max(MIN_KSLOTS, self.maxk + 2)
        self.assign_progeny()
        self.fastas = [leaf.fastas[0] for leaf in self.progeny]
        self.ngen = len(self.progeny)

    def __repr__(self):
        return (f"{self.__class__.__name__}['{self.node_title}', k: {self.bestk}, delta: {self.delta}, "
                f"ngen: {self.ngen}, children: {repr(self.children)} ]")

    def __lt__(self, other):
        return self.ngen < other.ngen

    def assign_progeny(self):
        """A node created without progeny is a leaf: its title is the FASTA path, shortened to the
        file stem for display (reference :97-102)."""
        if not self.progeny:
            self.progeny = [self]
            self.fastas = [self.node_title]
            self.node_title = os.path.splitext(os.path.basename(self.node_title))[0]

    def _grow_slots(self, upto: int) -> None:
        if upto >= len(self.ksketches):
            self.ksketches.extend([None] * (upto - len(self.ksketches) + 2))

    # ---------------------------------------------------------------- argmax-k search (reference :106-146)
    def find_delta_helper(self, kval: int, direction=1):
        """One step of the local hill-climb: make k-1..k+1 available, take k if it does not lower
        delta (ties move on), remember it as the species' next starting k, continue in `direction`."""
        if self.experiment["tool"] == "dashing" and kval > HLL_MAX_K:
            raise ValueError("Exploratory k value is too high for dashing. Either something is amiss with your data "
                             "or you need to be using --exact mode")
        self._grow_slots(kval + 1)
        self.node_ksweep(mink=kval - abs(direction), maxk=kval + abs(direction))
        self.update_node(kval)
        if direction < 0:
            self.mink = kval
        else:
            self.maxk = kval
        if self.delta == 0 and self.experiment["verbose"]:
            print("delta is 0 post update_node")
        candidate = self.ksketches[kval].delta_pos
        if self.delta <= candidate:
            self.speciesinfo.kstart = kval
            self.bestk = kval
            self.delta = candidate
            self.find_delta_helper(kval=kval + direction, direction=direction)

    def find_delta(self, kval: int):
        """Climb upwards from kval, then downwards from the same kval."""
        self.find_delta_helper(kval=kval, direction=1)
        self.find_delta_helper(kval=kval, direction=-1)
        self.card = self.ksketches[self.bestk].card

    # ---------------------------------------------------------------- batched sketching (reference :148-239)
    def ksweep_update_node(self, mink, maxk):
        """Make this node's sketches exist for every k in [mink, maxk] that it does not hold yet,
        children first.  Returns the list of sketch paths of the range (the reference feeds it to a
        batched `card` call that never runs, reference :256-257,274-275; kept for API parity)."""
        lo, hi = max(1, int(mink)), int(maxk)
        if self.experiment["tool"] == "dashing":
            hi = min(hi, HLL_MAX_K)
        template = SketchFilePath(filenames=self.fastas, kval=0, speciesinfo=self.speciesinfo, experiment=self.experiment)
        self._grow_slots(hi)
        wanted = [k for k in range(lo, hi + 1) if self.ksketches[k] is None]
        if not wanted:
            return []
        paths = {k: template.full.replace("{}", str(k)) for k in range(lo, hi + 1)}
        sketchlist = []
        for k in range(lo, hi + 1):
            ensure_dir(template.dir.replace("{}", str(k)))
            sketchlist.append(paths[k])
            self.experiment["baseset"].add(template.base.replace("{}", str(k)))

        child_templates = []
        if self.ngen > 1:
            for child in self.children:
                sketchlist += child.ksweep_update_node(mink=mink, maxk=maxk)
                if child.ksketches[0] is None:   # child had nothing to do this time and never swept before
                    child.ksketches[0] = _sketch_class(self.experiment["tool"])(
                        kval=0, sfp=SketchFilePath(filenames=child.fastas, kval=0, speciesinfo=self.speciesinfo,
                                                   experiment=self.experiment),
                        speciesinfo=self.speciesinfo, experiment=self.experiment)
                child_templates.append(child.ksketches[0].sfp.full)
        self.ksketches[0] = _sketch_class(self.experiment["tool"])(
            kval=0, sfp=template, speciesinfo=self.speciesinfo, experiment=self.experiment, presketches=child_templates)

        # ks whose sketch is already on disk are left alone, like the reference's existence test (:191-212)
        cardkey = self.speciesinfo.cardkey
        missing = []
        for k in wanted:
            on_disk = self.ksketches[0].sketch_check(path=paths[k])
            trusted = (not on_disk and self.experiment["lowmem"] and self.ngen > 1
                       and float(cardkey.get(paths[k]) or 0) > 0)
            if not on_disk and not trusted:
                missing.append(k)
        if not missing:
            return []

        command = (self.ksketches[0]._leaf_command(tmpdir="") if self.ngen < 2 else self.ksketches[0]._union_command())
        self._announce("parallel -j 95% ' " + command + " ' ::: " + " ".join(map(str, missing)))
        self._sketch_batch(missing, paths, child_templates)
        return sketchlist

    def _announce(self, text: str) -> None:
        if self.experiment["debug"]:
            print(text)
        elif self.experiment["verbose"]:
            print(text if len(text) < 400 else text[:200] + " .. " + text[-200:])

    def _sketch_batch(self, ks: List[int], paths: Dict[int, str], child_templates: List[str]) -> None:
        """The GPU stand-in for the `parallel` line: all `ks` of this node in one store call, files
        written, cardinalities cached."""
        store = get_store()
        registers = int(self.experiment["registers"])
        canon = bool(self.experiment["canonicalize"])
        out_paths = {k: paths[k] for k in ks}
        if self.experiment["tool"] == "dashing":
            if self.ngen < 2:
                cards = store.leaf_sketches(self.fastas[0], ks, registers, canon, out_paths)
            else:
                if self.experiment["lowmem"]:
                    members = {k: self._union_members(k) for k in ks}
                else:
                    members = {k: [tpl.replace("{}", str(k)) for tpl in child_templates] for k in ks}
                cards = store.union_sketches(members, registers, out_paths)
            for k, card in cards.items():
                self.speciesinfo.cardkey[out_paths[k]] = card
        else:
            for k in ks:   # exact mode: one GPU k-mer set per k (sets of different k share nothing)
                KMCSketchObj.build_db(out_paths[k], k, canon, self.fastas, self.speciesinfo.cardkey)

    def _union_members(self, k: int) -> List[str]:
        """The sketches whose register-wise max is this node's sketch at k: its children's -- except that under
        --lowmem a child union may be a cardinality on record without a file (it is trusted and not rebuilt,
        reference lib/sketch_classes.py:223-225), in which case the child's own members stand in for it.  (The
        reference hands `dashing union` the missing path; the union comes out empty, its cardinality 0.)"""
        out = []
        for child in self.children:
            template = child.ksketches[0].sfp if child.ksketches[0] is not None else SketchFilePath(
                filenames=child.fastas, kval=0, speciesinfo=self.speciesinfo, experiment=self.experiment)
            path = template.full.replace("{}", str(k))
            if child.ngen > 1 and not nonempty_file(path):
                out.extend(child._union_members(k))
            else:
                out.append(path)
        return out

    # ---------------------------------------------------------------- per-k objects (reference :243-287)
    def update_node(self, kval):
        """Own a SketchObj at kval, after making sure every child owns one too."""
        sweep = self.experiment["ksweep"]
        if sweep is not None and not (sweep[0] <= kval <= sweep[1]):
            print(f"k={kval} is outside of ksweep range ", sweep)
            return
        self._grow_slots(kval)
        if self.ksketches[kval]:
            return
        sfp = SketchFilePath(filenames=self.fastas, kval=kval, speciesinfo=self.speciesinfo, experiment=self.experiment)
        presketches = []
        if self.ngen > 1:
            for child in self.children:
                child.update_node(kval)
                presketches.append(child.ksketches[kval].sketch)
        self.ksketches[kval] = _sketch_class(self.experiment["tool"])(
            kval=kval, sfp=sfp, speciesinfo=self.speciesinfo, experiment=self.experiment, presketches=presketches)

    def node_ksweep(self, mink, maxk):
        """Sketch objects for every k in [mink, maxk] at this node and below."""
        self.ksweep_update_node(mink=mink, maxk=maxk)
        lo, hi = max(1, int(mink)), int(maxk)
        if self.experiment["tool"] == "dashing":
            for kval in range(max(lo, HLL_MAX_K + 1), hi + 1):
                self._name_only(kval)
            hi = min(hi, HLL_MAX_K)
        for kval in range(lo, hi + 1):
            if self.ksketches[kval] is None:
                self.update_node(kval)
        self.mink = mink
        self.maxk = maxk

    def _name_only(self, kval: int) -> None:
        """A k beyond Dashing's limit: the reference still NAMES the sketch (and its children's) in the sketch
        database's registry before `dashing` refuses to build it (reference :243-269); nothing else happens."""
        SketchFilePath(filenames=self.fastas, kval=kval, speciesinfo=self.speciesinfo, experiment=self.experiment)
        if self.ngen > 1:
            for child in self.children:
                child._name_only(kval)

    def summarize(self, mink: int = 0, maxk: int = 0, ordering_number=0):
        """One row per k with the candidate delta card/k (reference :289-301)."""
        rows = []
        for kval in range(mink, maxk + 1):
            obj = self.ksketches[kval]
            rows.append({"ngen": self.ngen, "kval": kval, "card": obj.card, "delta_pos": obj.delta_pos,
                         "title": self.node_title, "command": obj.cmd, "ordering": ordering_number})
        return rows


DEFAULT_EXPERIMENT = {"tool": "dashing", "registers": 20, "canonicalize": True, "debug": False, "nthreads": 0,
                      "baseset": set(), "safety": False, "fast": False, "verbose": False, "ksweep": None, "lowmem": False}


class DeltaTree:
    """Leaves = FASTAs, inner nodes = unions; every node carries its argmax k and delta = card/k there."""

    def __init__(self, fasta_files, speciesinfo, nchildren=2, leafnodes=[], experiment=DEFAULT_EXPERIMENT, padding=True):
        self.experiment = experiment
        self.mink, self.maxk = experiment["ksweep"] if experiment["ksweep"] is not None else (0, 0)
        self.kstart = speciesinfo.kstart
        self.speciesinfo = speciesinfo
        if self.experiment["verbose"]:
            print("Now making tree for fastas: " + ", ".join(fasta_files))
        with self._exact_tree_family(fasta_files, nchildren):
            self._build_tree(fasta_files, nchildren)
            self.fill_tree(padding=padding)
        self.ngen = len(fasta_files)
        self.root = self._dt[-1]
        self.delta = self.root_delta()
        self.fastas = fasta_files
        if self.experiment["ksweep"] is None:
            speciesinfo.kstart = self.root_k()
        self.speciesinfo.save_references(fast=experiment["fast"])
        self.speciesinfo.save_cardkey(tool=self.experiment["tool"])

    def __sub__(self, other):
        print("Larger Tree Delta: ", self.delta)
        print("Subtree Delta: ", other.delta)
        print("Subtraction Result: ", self.delta - other.delta)
        return self.delta - other.delta

    def __repr__(self):
        return "{}(FASTAS: {}, NODES: {})".format(self.__class__.__name__, self.fastas, repr(self._dt[-1]))

    def print_tree(self):
        """Depth-first dump of the nodes."""
        def walk(node, depth):
            print("  " * depth + repr(node.node_title), node.bestk, node.delta)
            for child in node.children:
                walk(child, depth + 1)
        walk(self._dt[-1], 0)

    def print_list(self) -> None:
        print(" -> ".join(f"'{n.node_title}'({n.ngen}'({' '.join(p.node_title for p in n.progeny)})" for n in self._dt))

    def root_delta(self):
        return self._dt[-1].delta

    def root_k(self):
        return self._dt[-1].bestk

    def delete_sketches(self):
        """Remove the union sketches of every node but the root (never called by the reference, :329)."""
        for node in self._dt[:-1]:
            if node.ngen > 1:
                for obj in node.ksketches:
                    if obj is not None:
                        obj.remove_sketch()

    # ---------------------------------------------------------------- construction (reference :377-438)
    def _evaluate(self, node: DeltaTreeNode) -> None:
        if self.experiment["ksweep"] is None:
            node.find_delta(self.speciesinfo.kstart)
        else:
            node.node_ksweep(mink=self.mink, maxk=self.maxk)

    def _build_tree(self, symbol: list, nchildren: int, leafnodes: List[DeltaTreeNode] = []) -> None:
        """Leaves in order of size, each evaluated in turn (the hill-climb's starting k is carried
        from node to node through speciesinfo.kstart); then groups of `nchildren` consecutive
        nodes get a parent, which is inserted behind the last node that is not larger than it.
        When the insertion cursor reaches the end of the list the next parent takes everything that
        is left (reference :436-438) -- so the shape is NOT a balanced n-ary tree (SURVEY.md App. C.14)."""
        nodes = list(leafnodes) if leafnodes else [
            DeltaTreeNode(node_title=path, children=[], speciesinfo=self.speciesinfo, experiment=self.experiment, progeny=[])
            for path in symbol]
        nodes.sort()
        for leaf in nodes:
            self._evaluate(leaf)
        self._prefetch_tree_unions(nodes, nchildren)
        self._dt = nodes
        cursor = 0       # first node not yet given a parent
        insert_at = 0    # where the previous parent went
        while cursor != len(self._dt) - 1:
            stride = nchildren - 1
            group = self._dt[cursor:cursor + nchildren]
            parent = DeltaTreeNode(node_title="_".join(c.node_title for c in group), speciesinfo=self.speciesinfo,
                                   children=group, progeny=[leaf for c in group for leaf in c.progeny],
                                   experiment=self.experiment)
            self._evaluate(parent)
            while insert_at < len(self._dt) - stride and self._dt[insert_at + stride].ngen <= parent.ngen:
                insert_at += stride
            self._dt.insert(insert_at + stride, parent)
            cursor += nchildren
            if insert_at + stride > len(self._dt) - 1:
                nchildren = len(self._dt) - cursor

    @staticmethod
    def plan_tree(ngens: List[int], nchildren: int) -> List[List[int]]:
        """The shape _build_tree is going to produce, from the node sizes alone: for every parent, in
        creation order, the indices (into the sorted leaf list) of its progeny leaves.  Same cursor /
        insertion arithmetic as the loop below (reference :412-438) on (size, leaves) pairs."""
        dt = [(n, [i]) for i, n in enumerate(ngens)]
        parents, cursor, insert_at = [], 0, 0
        while cursor != len(dt) - 1:
            stride = nchildren - 1
            group = dt[cursor:cursor + nchildren]
            parent = (sum(g[0] for g in group), [leaf for g in group for leaf in g[1]])
            parents.append(parent[1])
            while insert_at < len(dt) - stride and dt[insert_at + stride][0] <= parent[0]:
                insert_at += stride
            dt.insert(insert_at + stride, parent)
            cursor += nchildren
            if insert_at + stride > len(dt) - 1:
                nchildren = len(dt) - cursor
        return parents

    def _prefetch_tree_unions(self, leaves: List[DeltaTreeNode], nchildren: int) -> None:
        """--ksweep: every (inner node, k) cell of the tree is known before any parent is evaluated -- the
        shape depends on node sizes only, and a node's union is the max over its progeny LEAVES -- so all
        of them go to the device as one batched job (GpuSketchStore.union_many) instead of one launch per
        node; the parents built below then find their sketch files and cardinalities in place.  Exact mode
        takes the same cells to one first-rank histogram job per k (_prefetch_exact_sets).  The hill-climb
        visits k adaptively and keeps the per-node batches."""
        sweep = self.experiment["ksweep"]
        tool = self.experiment["tool"]
        if sweep is None or self.experiment["lowmem"] or len(leaves) < 3 or not all(leaf.ngen == 1 for leaf in leaves):
            return
        ks = list(range(max(1, int(sweep[0])), min(EXACT_MAX_K if tool == "kmc" else HLL_MAX_K, int(sweep[1])) + 1))
        plan = self.plan_tree([1] * len(leaves), nchildren)
        if len(plan) < 2 or not ks:
            return                      # a spider has one inner node: the per-node batch is already one launch
        if any(not progeny for progeny in plan):
            return                      # the reference's cursor arithmetic runs off the list for some (n, nchildren),
                                        # e.g. (4, 3) or (6, 4), and then fails naming a parent without members
                                        # (lib/huffman_dandd.py:412-438): leave that to _build_tree, same error
        if tool == "kmc":
            self._prefetch_exact_sets(leaves, [([leaves[i].fastas[0] for i in progeny], None, None) for progeny in plan], ks)
            return
        if tool != "dashing" or os.environ.get("DANDD_B200_TREE_BATCH", "1") == "0":
            return
        probe = DashSketchObj(kval=0, sfp=SketchFilePath(filenames=[leaves[0].fastas[0]], kval=0, speciesinfo=self.speciesinfo,
                                                         experiment=self.experiment),
                              speciesinfo=self.speciesinfo, experiment=self.experiment)
        jobs, targets = [], []
        for progeny in plan:
            fastas = [leaves[i].fastas[0] for i in progeny]
            template = SketchFilePath(filenames=fastas, kval=0, speciesinfo=self.speciesinfo, experiment=self.experiment)
            paths = {k: template.full.replace("{}", str(k)) for k in ks}
            missing = [k for k in ks if not probe.sketch_check(path=paths[k])]
            if not missing:
                continue
            for k in missing:
                ensure_dir(os.path.dirname(paths[k]))
            jobs.append(({k: [leaves[i].ksketches[k].sketch for i in progeny] for k in missing}, {k: paths[k] for k in missing}))
            targets.append(paths)
        if not jobs:
            return                      # a cached re-run: nothing to compute, and the store (CUDA start-up) is never created
        store = get_store()
        if not hasattr(store, "union_many"):
            return
        results = store.union_many(jobs, int(self.experiment["registers"]))
        for (members, out_paths), cards in zip(jobs, results):
            for k, card in cards.items():
                self.speciesinfo.cardkey[out_paths[k]] = card

    def _exact_climb(self) -> bool:
        """Exact hill-climb whose genome sets may be registered as a family (sketch_classes.exact_family): not under
        --ksweep (_prefetch_exact_sets batches those cells), --lowmem, or DANDD_B200_EXACT_SET_BATCH=0 (union by union)."""
        return (self.experiment["tool"] == "kmc" and self.experiment["ksweep"] is None and not self.experiment["lowmem"]
                and os.environ.get("DANDD_B200_EXACT_SET_BATCH", "1") != "0")

    def _exact_tree_family(self, fastas, nchildren: int):
        """Exact hill-climb: the climb picks k as it goes, but which sets it counts is fixed by the node sizes alone --
        the leaves (sorted by size: every leaf holds one FASTA, so in the given order) and the inner nodes of
        plan_tree.  They are registered for the whole build, fill_tree's argmax k included, and every k the climb
        visits then costs one family job (GpuSketchStore.exact_family) instead of a fresh k-mer set per (node, k).
        Shapes the reference cannot build register nothing, so that _build_tree reaches the same failure."""
        if not self._exact_climb() or not fastas or (len(fastas) > 1 and int(nchildren) < 2):
            return contextlib.nullcontext()
        try:
            plan = self.plan_tree([1] * len(fastas), int(nchildren))
        except IndexError:
            return contextlib.nullcontext()
        if any(not progeny for progeny in plan):
            return contextlib.nullcontext()
        return exact_family(fastas, bool(self.experiment["canonicalize"]), sets=plan)

    def _exact_set_path(self, fastas, k: int) -> str:
        """Where SketchFilePath puts the exact database of the set `fastas` at k -- without registering the set's
        names: the node that asks for the set later does that itself, in the order the per-union path does."""
        spec = self.speciesinfo
        files = sorted(os.path.basename(f) for f in fastas)
        stored = spec.fastahex.get("".join(files)) or hex(sum(int(spec.fastahex[name], 16) for name in files))
        nc = "" if self.experiment["canonicalize"] else "nc"
        base = f"{stored[:15]}_{self.experiment['registers']}n{len(fastas)}k{k}{nc}"
        return os.path.join(spec.sketchdir, "ngen" + str(len(fastas)), "k" + str(k), base)

    def _prefetch_exact_sets(self, leaves: List[DeltaTreeNode], cells, ks: List[int], orderings=None) -> None:
        """Exact mode: the union databases of many nodes x every k of `ks` from one batched device job per k
        (K7 lists + K8 first-rank histograms, GpuSketchStore.exact_union_cards / exact_prefix_cards) instead of
        one fresh k-mer set per (node, k).  leaves: the genomes, in index order.  cells: (fastas of the asking
        node, o, i) -- with `orderings`, the node is the union of the first i genomes of orderings[o]; without,
        it is the set of its fastas.  Only the descriptor files are written; the node objects built later find
        them, read the counts back and issue no device work, so every file, name and cardinality comes out as on
        the per-union path (DANDD_B200_EXACT_SET_BATCH=0), in the same order.  A descriptor lists its inputs in
        the order of the asking node's fastas."""
        if not ks or not cells or self.experiment["lowmem"] or os.environ.get("DANDD_B200_EXACT_SET_BATCH", "1") == "0":
            return
        todo, seen = {}, set()
        for c, (fastas, _, _) in enumerate(cells):
            for k in ks:
                path = self._exact_set_path(fastas, k)
                if path not in seen and not all(nonempty_file(path + ext) for ext in (".kmc_pre", ".kmc_suf")):
                    seen.add(path)
                    todo.setdefault(k, []).append((path, c))
        if not todo:
            return                      # a cached re-run: nothing to compute, and the store (CUDA start-up) is never created
        store = get_store()
        if not hasattr(store, "exact_union_cards") or not hasattr(getattr(store, "engine", None), "exact_first_rank_hist"):
            return
        ks = sorted(todo)
        canon = bool(self.experiment["canonicalize"])
        genomes = [leaf.fastas[0] for leaf in leaves]
        singles = None                  # exact leaf counts on record size the job; else the store counts them
        if all(k < len(leaf.ksketches) and leaf.ksketches[k] is not None for leaf in leaves for k in ks):
            singles = [[int(leaf.ksketches[k].card) for k in ks] for leaf in leaves]
        if orderings is None:
            index = {f: g for g, f in enumerate(genomes)}
            cards = store.exact_union_cards(genomes, [[index[f] for f in fastas] for fastas, _, _ in cells], ks, canon,
                                            singles=singles)
            count = lambda c, col: cards[c, col]                                                  # noqa: E731
        else:
            cards = store.exact_prefix_cards(genomes, orderings, ks, canon, singles=singles)
            count = lambda c, col: cards[cells[c][1], cells[c][2] - 1, col]                       # noqa: E731
        for col, k in enumerate(ks):
            for path, c in todo[k]:
                KMCSketchObj.write_db(path, k, canon, cells[c][0], int(count(c, col)), None)

    def fill_tree(self, padding=False) -> None:
        """Give every node a sketch at every k that is some node's argmax (hill-climb mode), or sweep
        the whole range at every node (--ksweep) (reference :447-460)."""
        if self.experiment["ksweep"] is None:
            root = self._dt[-1]
            for k in sorted({n.bestk for n in self._dt} - {0}):
                root.update_node(k)
        else:
            self.ksweep(mink=self.experiment["ksweep"][0], maxk=self.experiment["ksweep"][1])

    def leaf_nodes(self) -> List[DeltaTreeNode]:
        return [node for node in self._dt if node.ngen == 1]

    def nodes_from_fastas(self, fasta_list):
        return [node for node in self.leaf_nodes() if node.fastas[0] in fasta_list]

    def ksweep(self, mink, maxk) -> None:
        for node in self._dt:
            node.node_ksweep(mink=mink, maxk=maxk)

    # ---------------------------------------------------------------- outputs (reference :484-524)
    def make_prefix(self, tag: str, label="", outdir: str = None):
        outdir = outdir or os.getcwd()
        label = "_" + label if label != "" else ""
        return os.path.join(outdir, tag + label + "_" + str(self.ngen) + "_" + self.experiment["tool"])

    def save(self, fileprefix: str, fast=False):
        """<prefix>_dtree.pickle, <prefix>_sketchdb.txt (what every sketch base name means) and
        <prefix>_deltas.csv; with fast only the deltas."""
        filepath = fileprefix + "_dtree.pickle"
        if not fast:
            with open(filepath, "wb") as fh:
                pickle.dump(obj=self, file=fh)
            print("Tree Pickle saved to: " + filepath)
            expmaploc = fileprefix + "_sketchdb.txt"
            write_listdict_to_csv(outfile=expmaploc,
                                  listdict=[self.speciesinfo.sketchinfo[base] for base in list(self.experiment["baseset"])])
            print(f"Output Sketch/DB mapping saved to {expmaploc}.")
        deltapath = fileprefix + "_deltas.csv"
        write_listdict_to_csv(deltapath, self.report_deltas())
        print("Deltas saved to: " + deltapath)
        return filepath

    def report_deltas(self) -> List[dict]:
        """Root first, then children depth-first: delta, argmax k, sketch and cardinality at that k."""
        rows = []

        def visit(node):
            best = node.ksketches[node.bestk]
            rows.append({"delta": node.delta, "k": node.bestk, "title": node.node_title, "ngen": node.ngen,
                         "sketchloc": best.sketch, "card": best.card, "fastas": "|".join(node.fastas)})
            for child in node.children:
                visit(child)
        visit(self._dt[-1])
        return rows

    def find_delta_delta(self, fasta_subset: List[str]) -> float:
        """delta(all) - delta(all minus fasta_subset) (reference :559-566)."""
        rest = [f for f in self.fastas if f not in fasta_subset]
        small = SubSpider(leafnodes=self.nodes_from_fastas(rest), speciesinfo=self.speciesinfo, experiment=self.experiment)
        print("Full Tree Delta: ", self.delta)
        print("Subtree Delta: ", small.delta)
        return self - small

    # ---------------------------------------------------------------- progressive unions (reference :574-663)
    def orderings_list(self, ordering_file=None, flist_loc=None, count=0) -> Tuple[List[str], List[Tuple[int]]]:
        """(sorted fasta list, orderings).  count == 1 -> the identity ordering; otherwise orderings
        are read from / added to a pickled set at <sketchdir>/<tag>_<n>_orderings.pickle."""
        fastas = self.fastas
        fastas.sort()
        if flist_loc:
            with open(flist_loc) as fh:
                listed = [line.strip() for line in fh]
            fastas = [f for f in listed if f in fastas]
        if count == 1:
            return fastas, [tuple(range(len(fastas)))]
        ordering_file = ordering_file or os.path.join(
            self.speciesinfo.sketchdir, self.speciesinfo.tag + "_" + str(len(fastas)) + "_orderings.pickle")
        orderings = set()
        if os.path.exists(ordering_file):
            with open(ordering_file, "rb") as fh:
                orderings = pickle.load(fh)
            if count == 0:
                return fastas, list(orderings)
            if count <= len(orderings):
                return fastas, list(orderings)[:count]
        elif count < 1:
            raise ValueError("You must provide a value for count when there is no default ordering file")
        orderings = permute(length=len(fastas), norder=count, preexist=orderings, verbose=self.experiment["verbose"])
        with open(ordering_file, "wb") as fh:
            pickle.dump(orderings, fh)
        return fastas, list(orderings)

    def progressive_wrapper(self, flist_loc=None, count=30, ordering_file=None, step=1, debug=False) -> List[dict]:
        fastas, orderings = self.orderings_list(ordering_file=ordering_file, flist_loc=flist_loc, count=count)
        return self.progressive_union(flist=fastas, orderings=orderings, step=step)

    def progressive_union(self, flist, orderings, step) -> Tuple[List[dict], List[dict]]:
        """For every ordering, delta (or the whole k sweep) of the union of its first i FASTAs,
        i = step, 2*step, ...  The pickles are saved after every ordering, as in the reference."""
        family = contextlib.nullcontext()
        if self._exact_climb() and all(0 <= int(j) < len(flist) for ordering in orderings for j in ordering):
            # every prefix the climbs count, the spider's union included (prefix n of any ordering)
            family = exact_family(flist, bool(self.experiment["canonicalize"]), orderings=orderings)
        with family:
            smain = DeltaSpider(fasta_files=flist, speciesinfo=self.speciesinfo, experiment=self.experiment)
            smain._prefetch_prefix_unions(orderings, step)
            results, summary = [], []
            for number, ordering in enumerate(orderings, start=1):
                if self.experiment["verbose"]:
                    print(f"Now sweeping for ordering {number}")
                rows, sweep_rows = smain.sketch_ordering(ordering, ordering_number=number, step=step)
                results.extend(rows)
                summary.extend(sweep_rows)
                self.speciesinfo.save_references(fast=self.experiment["fast"])
                self.speciesinfo.save_cardkey(tool=self.experiment["tool"], fast=self.experiment["fast"])
        return results, summary

    def _prefetch_prefix_unions(self, orderings, step) -> None:
        """K3: with a k sweep requested every (ordering, prefix, k) cell is known in advance, so all
        prefix unions -- cardinalities and sketch files -- come from one running-max pass per
        ordering, stored under the names the per-prefix SubSpiders will ask for; those then find
        every file present and every cardinality cached and issue no further work.  Exact mode: the same cells
        over the k range every prefix is swept at (the sweep, else the spider's own [mink, maxk]) come from one
        first-rank histogram job per k (_prefetch_exact_sets).  HLL without a sweep goes through the per-node
        batches."""
        sweep = self.experiment["ksweep"]
        if self.experiment["tool"] == "kmc" and orderings:
            lo, hi = sweep if sweep is not None else (self.mink, self.maxk)
            by_fasta = {node.fastas[0]: node for node in self.leaf_nodes()}
            cells = [([n.fastas[0] for n in self.nodes_from_fastas([self.fastas[j] for j in ordering[:i]])], o, i)
                     for o, ordering in enumerate(orderings) for i in range(2, len(ordering) + 1) if i % step == 0]
            self._prefetch_exact_sets([by_fasta[f] for f in self.fastas], cells,
                                      list(range(max(1, int(lo)), min(EXACT_MAX_K, int(hi)) + 1)),
                                      orderings=[list(o) for o in orderings])
            return
        if sweep is None or self.experiment["tool"] != "dashing" or not orderings:
            return
        ks = list(range(max(1, int(sweep[0])), min(HLL_MAX_K, int(sweep[1])) + 1))
        if not ks:
            return
        leaves = {node.fastas[0]: node for node in self.leaf_nodes()}
        ordered_leaves = [leaves[f] for f in self.fastas]
        for leaf in ordered_leaves:
            leaf.node_ksweep(mink=ks[0], maxk=ks[-1])
        leaf_paths = {k: [leaf.ksketches[k].sketch for leaf in ordered_leaves] for k in ks}
        cardkey = self.speciesinfo.cardkey
        probe = DashSketchObj(kval=0, sfp=SketchFilePath(filenames=[self.fastas[0]], kval=0, speciesinfo=self.speciesinfo,
                                                         experiment=self.experiment),
                              speciesinfo=self.speciesinfo, experiment=self.experiment)
        cells, out_paths = {}, {}
        for o, ordering in enumerate(orderings):
            for i in range(2, len(ordering) + 1):
                if i % step:
                    continue
                members = [self.fastas[j] for j in ordering[:i]]
                template = SketchFilePath(filenames=members, kval=0, speciesinfo=self.speciesinfo, experiment=self.experiment)
                for k in ks:
                    path = template.full.replace("{}", str(k))
                    cells[(o, i - 1, k)] = path
                    if not probe.sketch_check(path=path):
                        ensure_dir(os.path.dirname(path))
                        out_paths[(o, i - 1, k)] = path
        if not out_paths and all(float(cardkey.get(path) or 0) > 0 for path in cells.values()):
            return   # everything cached already: a repeated run issues no GPU work (SURVEY.md App. C.13)
        cards = get_store().prefix_unions(leaf_paths, [list(o) for o in orderings], int(self.experiment["registers"]),
                                          out_paths=out_paths)
        for (o, st, k), path in cells.items():
            cardkey[path] = float(cards[o, st, ks.index(k)])

    def sketch_ordering(self, ordering, ordering_number, step=1) -> Tuple[List[dict], List[dict]]:
        output, summary = [], []
        lo, hi = self.experiment["ksweep"] if self.experiment["ksweep"] is not None else (self.mink, self.maxk)
        for i in range(1, len(ordering) + 1):
            if i % step:
                continue
            sublist = [self.fastas[j] for j in ordering[:i]]
            spider = SubSpider(leafnodes=self.nodes_from_fastas(sublist), speciesinfo=self.speciesinfo, experiment=self.experiment)
            spider.ksweep(mink=int(lo), maxk=int(hi))
            output.append({"ngen": i, "kval": spider.root_k(), "delta": spider.delta, "ordering": ordering_number,
                           "fastas": sublist})
            summary.extend(spider.root.summarize(mink=int(lo), maxk=int(hi), ordering_number=ordering_number))
        return output, summary

    # ---------------------------------------------------------------- pairwise (reference :666-723)
    def pairwise_spiders(self, sublist=[], mink=0, maxk=0, jaccard=True) -> Tuple[List[dict], List[dict]]:
        """K-independent Jaccard of every unordered pair of leaves, optionally per-k Jaccard too."""
        leaves = sublist if len(sublist) else self.leaf_nodes()
        pair_experiment = self.experiment.copy()
        pair_experiment.update({"fast": True, "safe": False, "ksweep": None})
        if jaccard and (mink == 0 or maxk == 0):
            if self.experiment["ksweep"]:
                mink, maxk = self.experiment["ksweep"]
                print("WARNING: If EITHER minimum OR maximum k are not provided with --mink and --maxk flags, DandD will "
                      "default to the --ksweep values embedded in the delta-tree input.")
            else:
                print("WARNING: If BOTH minimum AND maximum k are not provided either by the input delta-tree or using "
                      "--mink and --maxk, the --jaccard flag will be ignored.")
                jaccard = False
        table = self._prefetch_pair_unions(leaves)
        kij_rows, j_rows = [], []
        pair_index = 0
        for i, first in enumerate(leaves):
            for second in leaves[i + 1:]:
                rows = None
                if table is not None:
                    rows = self._pair_from_table(first, second, table, pair_index, pair_experiment, jaccard, mink, maxk)
                pair_index += 1
                if rows is None:         # --safe, no batched job in this store, or a k outside the table: one SubSpider per pair
                    pair = SubSpider(leafnodes=[first, second], speciesinfo=self.speciesinfo, experiment=pair_experiment)
                    pair.root.find_delta(self.root_k())
                    krow, jrows = pair.kij_summarize(), []
                    if jaccard:
                        pair.ksweep(mink=mink, maxk=maxk)
                        jrows = pair.jaccard_summarize(mink=mink, maxk=maxk)
                    rows = (krow, jrows)
                kij_rows.append(rows[0])
                j_rows.extend(rows[1])
        return kij_rows, j_rows

    # ---------------------------------------------------------------- pairs from the batched K6 table
    def _pair_from_table(self, first, second, table, row, pair_experiment, jaccard, mink, maxk):
        """What `SubSpider([first, second])` + `root.find_delta(root_k)` + `kij_summarize()` (+ the Jaccard
        sweep) would do (reference :666-695, :727-815), replayed on the cardinalities the batched pair job
        already holds: the same hill-climb decisions (including the species-wide start k it mutates), the
        same rows, and the same side effects on the sketch database -- a union sketch file, a cardinality
        entry and a name registration for every k the reference would have touched -- without building
        ~20 Python objects and issuing 3-8 store calls per pair.  Returns None when the replay needs a
        k the table does not cover (the caller then takes the object path for this pair)."""
        spec, exp = self.speciesinfo, pair_experiment
        col = table.col
        registers, canon = exp["registers"], exp["canonicalize"]
        exact = exp["tool"] == "kmc"
        limit = EXACT_MAX_K if exact else HLL_MAX_K
        files = sorted(os.path.basename(f) for f in (first.fastas[0], second.fastas[0]))
        set_key = "".join(files)
        stored = spec.fastahex.get(set_key)
        if stored is None:
            stored = hex(sum(int(spec.fastahex[name], 16) for name in files))
        stem = f"{stored[:15]}_{registers}n2k"
        nc = "" if canon else "nc"
        state = {"delta": 0, "bestk": 0}
        visited = []
        cells = {}

        def cell(k):
            """(path, file is there, union cardinality) of this pair at k.  Like SketchObj (reference
            lib/sketch_classes.py:244-262) a cardinality the database remembers is used when the sketch file
            is also there; only a cell the database cannot answer asks for the batched device job (which
            then evaluates every pair x every k at once)."""
            hit = cells.get(k)
            if hit is None:
                path = os.path.join(spec.sketchdir, "ngen2", "k" + str(k), stem + str(k) + nc) + ("" if exact else ".hll")
                there = all(nonempty_file(path + ext) for ext in ((".kmc_pre", ".kmc_suf") if exact else ("",)))
                card = float(spec.cardkey.get(path) or 0) if there else 0.0
                if not card > 0:
                    card = float(table.cards()[row, col[k]])
                hit = cells[k] = (path, there, card)
            return hit

        def touch(lo, hi):
            for k in range(max(1, lo), min(hi, limit) + 1):
                if k not in col:
                    raise KeyError(k)
                if k not in visited:
                    visited.append(k)

        def helper(k, direction):
            if not exact and k > HLL_MAX_K:
                raise ValueError("Exploratory k value is too high for dashing. Either something is amiss with your data "
                                 "or you need to be using --exact mode")
            touch(k - 1, k + 1)
            candidate = cell(k)[2] / k if k >= 1 else 0
            if state["delta"] <= candidate:
                spec.kstart = k
                state["bestk"], state["delta"] = k, candidate
                helper(k + direction, direction)

        def find_delta(k):
            helper(k, 1)
            helper(k, -1)

        kstart_before = spec.kstart
        try:
            find_delta(spec.kstart)                                   # SubSpider._build_tree
            for k in sorted({first.bestk, second.bestk, state["bestk"]} - {0}):
                touch(k, k)                                           # fill_tree
            find_delta(self.root_k())                                 # pairwise_spiders
            if jaccard:
                touch(int(mink), int(maxk))                           # pair.ksweep + jaccard_summarize
            for k in visited:
                cell(k)                                               # may start the batched job: before any side effect
        except KeyError:
            spec.kstart = kstart_before                               # the object path starts where this pair started
            return None
        # side effects on the database: names, files, cardinalities (SketchFilePath / DashSketchObj / store)
        spec.fastahex.setdefault(set_key, stored)
        leaf_sketch = {n: n.ksketches for n in (first, second)}
        for k in [0] + visited:
            ktok = "{}" if k == 0 else str(k)
            base = stem + ktok + nc
            if base not in spec.sketchinfo:
                spec.sketchinfo[base] = {"sketchbase": base, "files": files, "ngen": 2, "kval": k, "registers": registers}
            exp["baseset"].add(base)
            if k == 0:
                continue
            path, there, card = cell(k)
            if not there and exact:        # the descriptor pair the union's KMCSketchObj would write
                KMCSketchObj.write_db(path, k, bool(canon), [first.fastas[0], second.fastas[0]], int(card), spec.cardkey)
            elif not there:
                ensure_dir(os.path.dirname(path))
                get_store().materialize_union(path, int(registers), card, [leaf_sketch[first][k].sketch, leaf_sketch[second][k].sketch])
            if not float(spec.cardkey.get(path) or 0):
                spec.cardkey[path] = card
        a, b = (first, second) if first.node_title <= second.node_title else (second, first)
        kij = {"A": a.fastas[0], "B": b.fastas[0], "Adelta": a.delta, "Bdelta": b.delta, "Ak": a.bestk, "Bk": b.bestk,
               "ABdelta": state["delta"], "ABk": state["bestk"], "Atitle": a.node_title, "Btitle": b.node_title}
        kij["KIJ"] = (kij["Adelta"] + kij["Bdelta"] - kij["ABdelta"]) / kij["ABdelta"]
        jrows = []
        if jaccard:
            for k in range(mink, maxk + 1):
                jr = {"A": first.fastas[0], "B": second.fastas[0], "Atitle": first.node_title, "Btitle": second.node_title,
                      "kval": k, "Acard": _card_at(first, k), "Bcard": _card_at(second, k),
                      "ABcard": cell(k)[2] if k <= limit else 0.0}
                jr["jaccard"] = (jr["Acard"] + jr["Bcard"] - jr["ABcard"]) / jr["ABcard"]
                jrows.append(jr)
        return kij, jrows

    def _prefetch_pair_unions(self, leaves):
        """The union cardinality of every pair of leaves at every k the leaves hold, computed by ONE
        batched device job and kept by the store: K6 on the HLL sketches (transposed once, pair matrix
        tiled), or in exact mode K7 (one pair-intersection job per k, every FASTA read once per k).  The
        pairs below are then replayed on that table and issue no device work of their own."""
        tool = self.experiment["tool"]
        if (tool not in ("dashing", "kmc") or len(leaves) < 3 or self.experiment["safety"] or self.experiment["lowmem"]
                or os.environ.get("DANDD_B200_PAIR_TABLE", "1") == "0"
                or not all(hasattr(leaf, "ksketches") for leaf in leaves)):
            return None
        ks = [k for k in range(1, (EXACT_MAX_K if tool == "kmc" else HLL_MAX_K) + 1)
              if all(k < len(leaf.ksketches) and leaf.ksketches[k] is not None for leaf in leaves)]
        if not ks:
            return None
        registers = int(self.experiment["registers"])

        def compute():
            store = get_store()
            if tool == "kmc":
                if not hasattr(store, "exact_pair_cards"):
                    raise KeyError("this store has no batched exact pair job")     # -> the object path
                return store.exact_pair_cards([leaf.fastas[0] for leaf in leaves], ks, bool(self.experiment["canonicalize"]),
                                              remember=True)[1]
            if not hasattr(store, "pair_unions"):
                raise KeyError("this store has no batched pair job")       # -> the object path, pair by pair
            return store.pair_unions({k: [leaf.ksketches[k].sketch for leaf in leaves] for k in ks}, registers)
        return _PairTable(ks, compute)

    def prepare_AFproject(self, kijsummary, jsummary) -> List[Tuple]:
        """(tool, name1, name2, k, value, k1, k2, k12) tuples for helpers/AFproject.py: k = 0 rows carry
        KIJ and the three argmax ks, k > 0 rows carry the per-k Jaccard (reference :697-718)."""
        tool = self.experiment["tool"]
        out = {(tool, r["Atitle"], r["Btitle"], 0, r["KIJ"], r["Ak"], r["Bk"], r["ABk"]) for r in kijsummary}
        out |= {(tool, r["Atitle"], r["Btitle"], r["kval"], r["jaccard"], None, None, None) for r in jsummary}
        return list(out)


class _PairTable:
    """Union cardinalities of every pair of leaves at every k: `cards()[pair, col[k]]`.  The batched device
    job runs the first time a cell is asked for that the sketch database cannot answer -- a `kij` re-run
    whose unions are all on record never creates the store (no torch import, no CUDA start-up)."""

    def __init__(self, ks, compute):
        self.col = {k: i for i, k in enumerate(ks)}
        self._compute = compute
        self._cards = None

    def cards(self):
        if self._cards is None:
            self._cards = self._compute()
        return self._cards


class SubSpider(DeltaTree):
    """Existing leaf nodes under one new union node (reference :727-815)."""

    def __init__(self, leafnodes, speciesinfo, experiment):
        self.speciesinfo = speciesinfo
        self.fastahex = self.speciesinfo.fastahex
        self.experiment = experiment
        self.kstart = self.speciesinfo.kstart
        if self.experiment["ksweep"] is not None:
            self.mink, self.maxk = self.experiment["ksweep"]
        self._build_tree(leafnodes)
        self.root = self._dt[-1]
        self.fastas = self.root.fastas
        self.ngen = len(self.fastas)
        self.delta = None
        self.fill_tree()
        if self.experiment["ksweep"] is None:
            self.delta = self.root_delta()
        else:
            self.mink, self.maxk = self.experiment["ksweep"]

    def _build_tree(self, leafnodes):
        body = DeltaTreeNode(node_title="_".join(os.path.basename(c.node_title) for c in leafnodes),
                             speciesinfo=self.speciesinfo, children=leafnodes,
                             progeny=[leaf for c in leafnodes for leaf in c.progeny], experiment=self.experiment)
        if self.experiment["ksweep"] is None:
            body.find_delta(kval=self.speciesinfo.kstart)
        else:
            body.node_ksweep(mink=self.mink, maxk=self.maxk)
        self.mink = body.mink
        self.maxk = body.maxk
        self._dt = leafnodes + [body]

    def _ordered_pair(self):
        if len(self.fastas) != 2:
            raise ValueError("KIJ can only be calculated on spider/trees with 2 children")
        a, b = self._dt[0], self._dt[1]
        return (a, b) if a.node_title <= b.node_title else (b, a)

    def kij_summarize(self) -> Dict:
        """KIJ = (delta_A + delta_B - delta_AB) / delta_AB, each delta at its own argmax k (reference :791)."""
        a, b = self._ordered_pair()
        self.root.update_node(self.root.bestk)
        a.update_node(a.bestk)
        b.update_node(b.bestk)
        row = {"A": a.fastas[0], "B": b.fastas[0], "Adelta": a.delta, "Bdelta": b.delta, "Ak": a.bestk, "Bk": b.bestk,
               "ABdelta": self.root.delta, "ABk": self.root.bestk, "Atitle": a.node_title, "Btitle": b.node_title}
        row["KIJ"] = (row["Adelta"] + row["Bdelta"] - row["ABdelta"]) / row["ABdelta"]
        return row

    def jaccard_summarize(self, mink=2, maxk=32) -> List[Dict]:
        """J_k = (|A| + |B| - |A u B|) / |A u B| for every k of the range (reference :813); A and B
        keep their positional order here, as in the reference (its swap test can never fire, :804)."""
        if len(self.fastas) != 2:
            raise ValueError("KIJ can only be calculated on spider/trees with 2 or more children")
        a, b = self._dt[0], self._dt[1]
        self.ksweep(mink=mink, maxk=maxk)
        rows = []
        for k in range(mink, maxk + 1):
            row = {"A": a.fastas[0], "B": b.fastas[0], "Atitle": a.node_title, "Btitle": b.node_title, "kval": k,
                   "Acard": _card_at(a, k), "Bcard": _card_at(b, k), "ABcard": _card_at(self.root, k)}
            row["jaccard"] = (row["Acard"] + row["Bcard"] - row["ABcard"]) / row["ABcard"]
            rows.append(row)
        return rows


def _card_at(node, k: int) -> float:
    """Cardinality of a node's sketch at k for the Jaccard tables.  Beyond Dashing's k limit no sketch exists and
    the reference works with the 0 it gets for a sketch that could not be made -- so that a Jaccard range reaching
    past k = 32 ends in the same ZeroDivisionError there and here."""
    if k > HLL_MAX_K and node.experiment["tool"] == "dashing" and (k >= len(node.ksketches) or node.ksketches[k] is None):
        return 0.0
    return node.ksketches[k].card


class DeltaSpider(DeltaTree):
    """All FASTAs as leaves directly under one union node (reference :818-823)."""

    def __init__(self, fasta_files, speciesinfo, experiment, padding=False):
        super().__init__(fasta_files=fasta_files, speciesinfo=speciesinfo, experiment=experiment,
                         nchildren=len(fasta_files), padding=padding)

    def __init2__(self, tree: DeltaTree):
        raise NotImplementedError("initialization of spider by tree not yet implemented")


def presketch_leaves_sharded(fastas, speciesinfo, experiment, kstart, halfwidth=6) -> int:
    """One process per GPU (torchrun): every rank sketches its share of the FASTAs (largest first,
    balanced by size) into the SHARED sketch database, ranks exchange the cardinalities they
    computed, and rank 0 then builds the tree from files that already exist -- so the only work
    left after this call is the unions.  Returns this process's rank.  HLL merge is exact, so the results are
    identical to a single-GPU run (SURVEY.md 8e).  k range: the sweep if one was asked for, else a
    window around kstart (anything the hill-climb visits outside it is sketched on demand)."""
    if int(os.environ.get("WORLD_SIZE", "1")) < 2:
        return 0              # (and torch.distributed is never imported in the single-process case)
    from dandd_b200 import dist as dd_dist
    rank, world = dd_dist.world()
    if world < 2:
        return 0
    if experiment["tool"] != "dashing":
        # exact mode: k-mer sets are not mergeable files; rank 0 walks the tree, every count it needs is
        # computed by all ranks on key-range shards of the set (dandd_b200.dist.ExactWorkers)
        workers = get_store().start_exact_workers()
        if rank > 0:
            workers.serve()
        return rank
    import torch.distributed as tdist
    lo, hi = experiment["ksweep"] if experiment["ksweep"] is not None else (kstart - halfwidth, kstart + halfwidth)
    lo, hi = max(1, int(lo)), min(HLL_MAX_K, int(hi))
    if len(fastas) < world:
        _presketch_split(fastas, speciesinfo, experiment, lo, hi, rank, world)
        return rank
    owners = dd_dist.shard_by_size([os.path.getsize(f) for f in fastas], world)
    mine = [fastas[i] for i in owners[rank]]
    ingest.prefetch([f for f in mine if os.path.basename(f) not in speciesinfo.fastahex])   # (usually started already: dandd_cmd._early_prefetch)
    found = {}
    scratch = dict(experiment, baseset=set())   # pre-sketching must not leak names into the tree's own bookkeeping
    for path in mine:
        if os.path.basename(path) not in speciesinfo.fastahex and hasattr(get_store(), "warm_leaf"):
            with timing.span("warm_leaves"):      # GPU work first: the name (blake2b) is still being computed
                get_store().warm_leaf(path, int(experiment["registers"]), bool(experiment["canonicalize"]))
        leaf = DeltaTreeNode(node_title=path, children=[], speciesinfo=speciesinfo, experiment=scratch, progeny=[])
        with timing.span("presketch_leaves"):
            leaf.ksweep_update_node(mink=lo, maxk=hi)
        template = leaf.ksketches[0].sfp.full if leaf.ksketches[0] is not None else None
        for k in range(lo, hi + 1):
            if template:
                key = template.replace("{}", str(k))
                if key in speciesinfo.cardkey:
                    found[key] = speciesinfo.cardkey[key]
    bucket = [None] * world
    with timing.span("exchange_cards"):      # also where a fast rank waits for the slowest one
        tdist.all_gather_object(bucket, (found, {k: v for k, v in speciesinfo.fastahex.items()}))
    for cards, hexes in bucket:
        speciesinfo.cardkey.update(cards)
        for key, value in hexes.items():
            speciesinfo.fastahex.setdefault(key, value)
    return rank


def _presketch_split(fastas, speciesinfo, experiment, lo, hi, rank, world) -> None:
    """Fewer genomes than GPUs: every rank sketches its PART of every genome (records, or overlapping
    pieces of a large record -- dandd_b200.dist.split_fasta), the registers are max-reduced over the
    ranks and rank 0 writes the leaf sketches and remembers their cardinalities.  Which k are still
    missing on disk is decided by rank 0 alone and broadcast, so that all ranks enter the same
    collectives."""
    import torch.distributed as tdist
    store = get_store()
    scratch = dict(experiment, baseset=set())
    registers, canon = int(experiment["registers"]), bool(experiment["canonicalize"])
    for path in fastas:
        template = SketchFilePath(filenames=[path], kval=0, speciesinfo=speciesinfo, experiment=scratch)
        paths = {k: template.full.replace("{}", str(k)) for k in range(lo, hi + 1)}
        missing = None
        if rank == 0:
            probe = _sketch_class("dashing")(kval=0, sfp=template, speciesinfo=speciesinfo, experiment=scratch)
            missing = []
            for k in range(lo, hi + 1):
                ensure_dir(template.dir.replace("{}", str(k)))
                if not probe.sketch_check(path=paths[k]):
                    missing.append(k)
        box = [missing]
        tdist.broadcast_object_list(box, src=0)
        missing = box[0]
        if missing:
            cards = store.leaf_sketches(path, missing, registers, canon, {k: paths[k] for k in missing}, split=(rank, world))
            if rank == 0:
                for k, card in cards.items():
                    speciesinfo.cardkey[paths[k]] = card


def list_fastas(genomedir, flist_loc) -> List[str]:
    """The sorted FASTA list of a `tree` run: the lines of --fastas, else every file of --datadir
    (reference :858-868)."""
    if flist_loc:
        with open(flist_loc) as fh:
            fastas = [line.strip() for line in fh]
    elif genomedir and os.path.exists(genomedir):
        fastas = [os.path.join(genomedir, n) for n in os.listdir(genomedir)]
    else:
        raise ValueError("no FASTA directory or list")
    fastas.sort()
    return fastas


def _warm_fresh_leaves(fastas, speciesinfo, experiment) -> None:
    """Single process: sketch the large FASTAs the database has never named BEFORE the tree is built.
    Building a leaf node needs the file's blake2b name, seconds of hashing for a multi-GB genome (it
    runs on background threads since prefetch); the GPU pass needs only the bytes.  Doing the passes
    first puts the device work under the hashing instead of behind it; the leaf constructors then find
    their all-k blocks in HBM and only name and write them.  (presketch_leaves_sharded does the same per
    rank.)  Small files are not worth it, and a run without large fresh files never creates the store here."""
    if experiment["tool"] != "dashing":
        return
    fresh = [f for f in fastas if os.path.basename(f) not in speciesinfo.fastahex and os.path.isfile(f)
             and os.path.getsize(f) >= ingest.HASH_ONLY_MIN_BYTES]
    if not fresh:
        return
    store = get_store()
    if not hasattr(store, "warm_leaf"):
        return
    registers = int(experiment["registers"])
    fit = int(getattr(store, "cache_bytes", 0) // 2 // (HLL_MAX_K << registers))    # all-k blocks that stay resident
    for path in fresh[:fit]:
        with timing.span("warm_leaves"):
            store.warm_leaf(path, registers, bool(experiment["canonicalize"]))


def create_delta_tree(tag: str, genomedir: str, sketchdir: str, kstart: int, nchildren=None, registers=0, flist_loc=None,
                      canonicalize=True, tool="dashing", debug=False, nthreads=0, safety=False, fast=False, verbose=False,
                      ksweep=None, lowmem=False):
    """Entry point of `dandd tree` (reference :839-877): FASTA list -> DeltaSpider (default) or
    DeltaTree (--nchildren), with the per-experiment option dict threaded through every object."""
    experiment = {"registers": registers, "canonicalize": canonicalize, "tool": tool, "nthreads": int(nthreads),
                  "debug": debug, "baseset": set(), "safety": safety, "fast": fast, "verbose": verbose, "ksweep": ksweep,
                  "lowmem": lowmem}
    speciesinfo = SpeciesSpecifics(tag=tag, genomedir=genomedir, sketchdir=sketchdir, kstart=kstart, tool=tool,
                                   flist_loc=flist_loc)
    if flist_loc:
        with open(flist_loc) as fh:
            fastas = [line.strip() for line in fh]
    elif speciesinfo.inputdir and os.path.exists(speciesinfo.inputdir):
        fastas = speciesinfo.retrieve_fasta_files(full=True)
    else:
        raise ValueError("You must provide either an existing directory of fastas or a file listing the paths of the "
                         f"desired fastas. The directory you provided was {speciesinfo.inputdir}.")
    fastas.sort()
    if nchildren and int(nchildren) == 1 and len(fastas) > 1:
        # (the reference never returns from such a run: every new node takes ONE node off its list and puts one
        # back, lib/huffman_dandd.py:377-438.  Refused before any rank reads or sketches anything.)
        raise ValueError("--nchildren 1 cannot build a tree over more than one fasta: every node would have a single child")
    if presketch_leaves_sharded(fastas, speciesinfo, experiment, kstart) > 0:
        return None           # ranks > 0 only contribute leaf sketches; rank 0 builds and saves the tree
    # read / gunzip / blake2b in the background while the GPU works -- only files the database has never
    # named (a cached re-run reads nothing; usually started already by dandd_cmd._early_prefetch)
    ingest.prefetch([f for f in fastas if os.path.basename(f) not in speciesinfo.fastahex])
    _warm_fresh_leaves(fastas, speciesinfo, experiment)
    if nchildren:
        dtree = DeltaTree(fasta_files=fastas, speciesinfo=speciesinfo, nchildren=nchildren, experiment=experiment)
    else:
        dtree = DeltaSpider(fasta_files=fastas, speciesinfo=speciesinfo, experiment=experiment)
    speciesinfo.save_cardkey(tool=tool, fast=fast)
    speciesinfo.save_references(fast=fast)
    ingest.drop_all()         # prefetched bytes nobody asked for (their sketches were cached)
    return dtree
