"""SketchStore: what the drop-in sketch objects (dandd_b200/lib/sketch_classes.py) call instead of
shelling out to dashing / kmc / kmc_tools / GNU parallel.

The reference's only state between commands is the sketchdb directory (files + cardinality
pickle).  The store keeps that contract -- every sketch it produces is written to the path DandD
expects -- and adds an HBM-resident cache of registers and packed sequences so that unions,
progressive prefix unions and pairwise unions never re-read a file or re-sketch a FASTA:

    dashing sketch (x nk via parallel)  -> leaf_sketches()      one fused all-k pass on the GPU
    dashing union  (x nk via parallel)  -> union_sketches()     one batched max+histogram+MLE launch
    dashing card                        -> card_of_file()
    kmc + kmc_tools info / complex      -> exact_count()        GPU k-mer set (bitmap / hash set)
    kmc_tools complex over all pairs    -> exact_pair_cards()   one pair-intersection job per k
    kmc_tools complex over prefixes,    -> exact_prefix_cards() / exact_union_cards()
      over tree nodes                                            one first-rank histogram job per k

One store per process; it talks to one Engine (one GPU).  There is no CPU path here.
"""
import os
from collections import OrderedDict
from contextlib import contextmanager
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import hllfile, ingest, timing
from .engine import Engine, get_engine

ALL_HLL_KS = tuple(range(1, 33))
EXACT_MAX_K = 256   # KMC's own k limit, and the exact kernels'
# The greedy ordering compacts its live registers once 4 bytes per live register, times this, is at most what a
# dense step reads (1 byte per register of every remaining candidate): sparse entries cost more than their 4 bytes
# (a random L2 read of U, a write back, a CTA per segment).
SPARSE_CROSS = 2
STREAM_MIN_BYTES = int(os.environ.get("DANDD_B200_STREAM_MIN", str(32 << 20)))   # larger FASTAs take the chunked pipeline


def greedy_pick(cards: torch.Tensor, kdiv: torch.Tensor, chosen: torch.Tensor, order: str) -> torch.Tensor:
    """One greedy step's pick, on the device: the genome not `chosen` whose delta = max_k cards[g, k] / k is the largest
    (order="max") or the smallest ("min"), the lowest index winning a tie.  cards float64 [n, nk], kdiv the ks [nk]."""
    fill = float("-inf") if order == "max" else float("inf")
    delta = (cards / kdiv).amax(dim=1).masked_fill(chosen, fill)
    return delta.argmax() if order == "max" else delta.argmin()   # the first extremum: the lowest index


def read_fasta_bytes(path: str) -> bytes:
    """Whole FASTA as bytes; .gz is inflated on the host (dashing/kmc read .gz transparently).
    Served from the background ingest pool when the file was prefetched."""
    return ingest.fasta_bytes(path)


class GpuSketchStore:
    def __init__(self, engine: Engine = None, prefetch_all_k: bool = True, cache_bytes: int = 64 << 30,
                 hll_compresslevel: int = None, union_files: str = None):
        self.engine = engine or get_engine()
        self.prefetch_all_k = prefetch_all_k
        self.cache_bytes = cache_bytes
        self.hll_compresslevel = int(os.environ.get("DANDD_B200_HLL_GZIP", "0")) if hll_compresslevel is None else hll_compresslevel
        # 'full': union sketches are written out like `dashing union -o` does; 'stub': a header-only
        # marker file (registers stay in HBM / are recomputed from the leaves on demand)
        self.union_files = union_files or os.environ.get("DANDD_B200_UNION_FILES", "full")
        # all-pairs jobs leave N(N-1)/2 x (a few k) union sketches behind: markers unless full files were asked for
        self.pair_union_files = union_files or os.environ.get("DANDD_B200_UNION_FILES", "stub")
        # One LRU over everything resident in HBM, keyed by kind: ("sketch", path) -> [2^p] u8,
        # ("leaf", fasta, p, canon) -> {"regs","cards","ks"}, ("packed", fasta) -> PackedSeq.  A sketch that
        # is a VIEW of a leaf block costs nothing by itself (the block is what occupies memory).
        self._lru: "OrderedDict[tuple, object]" = OrderedDict()
        self._cost: Dict[tuple, int] = {}
        self._bytes = 0
        self.pair_table = None   # cardinalities of every two-leaf union, filled by one batched K6 job (pair_unions)
        self.exact_pair_table = None   # exact counts of every leaf and two-leaf union (exact_pair_cards, remember=True)
        self.exact_family_table = None   # the genome sets of a running exact hill-climb, counted per k (exact_family)
        self.stats = {"leaf_passes": 0, "union_launches": 0, "files_written": 0, "files_read": 0, "exact_calls": 0,
                      "exact_family_jobs": 0}
        self.exact_workers = None   # set by start_exact_workers() for `--exact` under torchrun
        self.stream_stats: List[dict] = []   # per streamed FASTA: stage times (read, blake2b, GPU span, wall)

    # ------------------------------------------------------------------ cache plumbing
    def _put(self, key: tuple, value, cost: int) -> None:
        if key in self._lru:
            self._bytes -= self._cost.pop(key)
            del self._lru[key]
        self._lru[key] = value
        self._cost[key] = int(cost)
        self._bytes += int(cost)
        while self._bytes > self.cache_bytes and len(self._lru) > 1:
            old, gone = self._lru.popitem(last=False)
            self._bytes -= self._cost.pop(old)
            if old[0] == "leaf":       # the per-k sketches that are views of this block would keep it in HBM, uncounted
                for path in gone.get("views", ()):
                    self.forget(path)

    def _get(self, key: tuple):
        value = self._lru.get(key)
        if value is not None:
            self._lru.move_to_end(key)
        return value

    def _remember(self, path: str, regs: torch.Tensor, view_of_block: bool = False) -> None:
        self._put(("sketch", path), regs, 0 if view_of_block else regs.numel())

    def registers(self, path: str) -> torch.Tensor:
        """Device registers of the sketch stored at `path` (HBM cache, else read the file).  The
        returned tensor stays valid for as long as the caller holds it, whatever the cache evicts."""
        t = self._get(("sketch", path))
        if t is None:
            with timing.span("read_sketch_files"):
                try:
                    regs, _p, _ = hllfile.read_hll(path)
                    t = torch.from_numpy(regs).to(self.engine.device)
                except hllfile.StubSketch as stub:       # union marker: rebuild from its members
                    t = self.engine.union([self.registers(m) for m in stub.members])
            self.stats["files_read"] += 1
            self._remember(path, t)
        return t

    def forget(self, path: str) -> None:
        key = ("sketch", path)
        if key in self._lru:
            del self._lru[key]
            self._bytes -= self._cost.pop(key)

    def _write(self, path: str, regs: torch.Tensor, p: int, card: float, leaf: bool, members=None) -> None:
        with timing.span("write_sketch_files"):
            os.makedirs(os.path.dirname(path), exist_ok=True)
            if leaf or self.union_files == "full" or not members:
                hllfile.write_hll(path, regs.cpu().numpy(), p, card, self.hll_compresslevel)
            else:
                hllfile.write_stub(path, p, card, members)
        self.stats["files_written"] += 1

    # ------------------------------------------------------------------ dashing sketch
    def _pack_text(self, text):
        """K1, with the FASTQ detour: the packer only reports a line beginning with '+'; the text is
        then rewritten record by record the way kseq reads it (host side) and packed again."""
        from .engine import FastqInput
        try:
            return self.engine.pack(text).check()
        except FastqInput:
            return self.engine.pack(self.engine.fastq_to_fasta(text)).check()

    def packed(self, fasta: str):
        seq = self._get(("packed", fasta))
        if seq is None:
            seq = self._pack_text(read_fasta_bytes(fasta))
            self._put(("packed", fasta), seq, seq.codes.numel() + seq.invalid.numel())
        return seq

    def leaf_sketches(self, fasta: str, ks: Sequence[int], p: int, canon: bool, out_paths: Dict[int, str],
                      split: Optional[Tuple[int, int]] = None) -> Dict[int, float]:
        """Sketch `fasta` for every k in `ks` (one fused pass), write each sketch to out_paths[k]
        and return {k: cardinality}.  With prefetch_all_k the pass covers k = 1..32 once and later
        requests for other k of the same FASTA are served from HBM.

        split=(rank, world): a COLLECTIVE call -- every rank sketches its part of the file
        (dist.split_fasta), the registers are max-reduced over the ranks, every rank gets the
        cardinalities of the whole file and rank 0 writes the sketch files (SURVEY.md 8e, fewer
        genomes than GPUs)."""
        need = [int(k) for k in ks]
        ent = self._leaf_entry(fasta, need, p, canon, split)
        out = {}
        for k in need:
            i = ent["ks"][k]
            card = float(ent["cards"][i])
            ent.setdefault("views", set()).add(out_paths[k])     # (first: the next line may evict the block itself)
            self._remember(out_paths[k], ent["regs"][i], view_of_block=True)
            if split is None or split[0] == 0:
                self._write(out_paths[k], ent["regs"][i], p, card, leaf=True)
            out[k] = card
        return out

    def leaf_block(self, fasta: str, ks: Sequence[int], p: int, canon: bool,
                   out: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, np.ndarray]:
        """(registers [len(ks), 2^p] uint8 on the device, cardinalities [len(ks)]) of one FASTA, rows in the
        order of `ks`; nothing is named or written (`dashing hll` leaves no sketch behind:
        reference helpers/allpairs.py:32-35).  Same fused pass as leaf_sketches, for exactly these k; a
        block already in the HBM cache is used, a new one is not added to it (the caller keeps the
        registers: with `out` they are written straight into its [len(ks), 2^p] slice)."""
        need = [int(k) for k in ks]
        ent = self._leaf_entry(fasta, need, p, canon, None, all_k=False, keep=False)
        rows = [ent["ks"][k] for k in need]
        cards = np.asarray([float(ent["cards"][i]) for i in rows], dtype=np.float64)
        if out is not None and (tuple(out.shape) != (len(rows), 1 << p) or out.dtype != torch.uint8 or not out.is_contiguous()):
            raise ValueError(f"leaf_block: out must be a contiguous uint8 [{len(rows)}, {1 << p}] tensor, got {tuple(out.shape)}")
        if rows == list(range(ent["regs"].shape[0])):
            regs = ent["regs"] if out is None else out.copy_(ent["regs"])
        else:
            index = torch.as_tensor(rows, dtype=torch.int64, device=ent["regs"].device)
            regs = torch.index_select(ent["regs"], 0, index) if out is None else torch.index_select(ent["regs"], 0, index, out=out)
        return regs, cards

    def _leaf_entry(self, fasta: str, need: List[int], p: int, canon: bool, split: Optional[Tuple[int, int]],
                    all_k: Optional[bool] = None, keep: bool = True) -> dict:
        """The all-k block of one FASTA: {"regs": [nk, 2^p] device tensor, "cards": [nk], "ks": {k: row}},
        from the HBM cache or one fused pass (streamed above STREAM_MIN_BYTES).  all_k: sketch k = 1..32
        whatever is asked for (default: the store's prefetch_all_k); keep: remember a new block in the cache."""
        key = ("leaf", fasta, int(p), bool(canon))
        ent = self._get(key)
        if split is not None or ent is None or any(k not in ent["ks"] for k in need):
            all_k = self.prefetch_all_k if all_k is None else all_k
            run_ks = list(ALL_HLL_KS) if all_k else sorted(set(need) | set(ent["ks"] if ent else ()))
            streamed = None
            if split is None and os.path.getsize(fasta) >= STREAM_MIN_BYTES:
                streamed = self._stream_leaf(fasta, run_ks, p, canon)
            text = read_fasta_bytes(fasta) if streamed is None else None
            if split is not None:
                from dandd_b200 import dist as dd_dist
                run_ks = sorted(need)                      # identical on every rank, whatever each one has cached
                if b"\n+" in text or text[:1] == b"+":     # FASTQ: records as kseq reads them, then split
                    text = self.engine.fastq_to_fasta(text)
                text = dd_dist.split_fasta(text, split[1], only=split[0])[split[0]]
            if streamed is not None:
                regs, cards = streamed
            else:
                seq = self._pack_text(text)
                regs, cards = self.engine.sketch(seq, run_ks, p=p, canon=canon)
                if split is not None:
                    dd_dist.union_over_ranks(regs)
                    cards = self.engine.cards(regs, p)
                cards = cards.cpu().numpy()
            ent = {"regs": regs, "cards": cards, "ks": {k: i for i, k in enumerate(run_ks)}}
            if keep:
                self._put(key, ent, regs.numel())
            self.stats["leaf_passes"] += 1
        return ent

    def warm_leaf(self, fasta: str, p: int, canon: bool) -> None:
        """Sketch a large FASTA for all k NOW and keep the block in HBM, without naming or writing
        anything: lets the caller start the GPU work before the file's blake2b name (which the sketch
        database paths need, and which takes seconds for a multi-GB file) has been computed."""
        key = ("leaf", fasta, int(p), bool(canon))
        if not self.prefetch_all_k or self._get(key) is not None or not os.path.isfile(fasta) \
                or os.path.getsize(fasta) < STREAM_MIN_BYTES:
            return
        run_ks = list(ALL_HLL_KS)
        streamed = self._stream_leaf(fasta, run_ks, p, canon)
        if streamed is not None:
            regs, cards = streamed
            self._put(key, {"regs": regs, "cards": cards, "ks": {k: i for i, k in enumerate(run_ks)}}, regs.numel())
            self.stats["leaf_passes"] += 1

    def _stream_leaf(self, fasta, run_ks, p, canon):
        """Large FASTA: disk (or the prefetched bytes) -> pinned ring -> H2D -> K1 -> K2 in 64 MiB chunks,
        the blake2b name computed from the same chunks (dandd_b200/streaming.py).  None if the text is
        FASTQ (the whole-file path then rewrites it first)."""
        from . import streaming
        from .engine import FastqInput
        text = ingest.fasta_bytes(fasta) if ingest.is_prefetched(fasta) else None
        try:
            regs, cards, digest, stats = streaming.sketch_file(self.engine, fasta, run_ks, p, canon, text=text,
                                                               want_digest=not ingest.has_digest(fasta))
        except FastqInput:
            return None
        if digest:
            ingest.set_digest(fasta, digest)
        self.stream_stats.append(stats)
        for key in ("read_s", "blake2b_s", "inflate_s", "gpu_span_s", "wall_s"):
            if key in stats:
                timing.add("stream_" + key, stats[key])
        return regs, cards

    # ------------------------------------------------------------------ dashing union (+ card)
    def union_sketches(self, members_by_k: Dict[int, List[str]], p: int, out_paths: Dict[int, str]) -> Dict[int, float]:
        """For every k: union of the sketches stored at members_by_k[k]; written to out_paths[k];
        returns {k: cardinality}.  One launch for all k."""
        out = {}
        for k in sorted(members_by_k):   # cells a batched pair job (pair_unions) has already evaluated
            card = self._pair_lookup(members_by_k[k], p)
            if card is not None:
                out[k] = self.materialize_union(out_paths[k], p, card, members_by_k[k])
        ks = sorted(k for k in members_by_k if k not in out)
        if not ks:
            return out
        width = max(len(members_by_k[k]) for k in ks)
        tensors = [[self.registers(pth) for pth in members_by_k[k]] for k in ks]
        ptrs = np.zeros((len(ks), width), dtype=np.int64)
        for i, row in enumerate(tensors):
            for j, t in enumerate(row):
                ptrs[i, j] = t.data_ptr()
        with timing.span("union_gpu"):
            cards, unions = self.engine.union_sets(ptrs, p, final_only=True, materialize=True)
            self.stats["union_launches"] += 1
            cards = cards.cpu().numpy().reshape(len(ks))
        for i, k in enumerate(ks):
            regs = unions[i, 0]
            self._remember(out_paths[k], regs)
            self._write(out_paths[k], regs, p, float(cards[i]), leaf=False, members=list(members_by_k[k]))
            out[k] = float(cards[i])
        return out

    def union_many(self, jobs: Sequence[Tuple[Dict[int, List[str]], Dict[int, str]]], p: int,
                   chunk_bytes: int = 4 << 30) -> List[Dict[int, float]]:
        """union_sketches for MANY nodes at once (every inner node of a tree x every k): jobs[i] =
        (members_by_k, out_paths).  The (node, k) cells are grouped by member count (powers of two, so the
        pointer tables stay dense) and each group goes to the device as one launch -- or a few, when full
        union files are wanted and the materialised unions of a group exceed chunk_bytes.  Returns one
        {k: cardinality} per job; every out_path exists afterwards."""
        cells = [(i, k, list(members[k])) for i, (members, _) in enumerate(jobs) for k in sorted(members)]
        out: List[Dict[int, float]] = [dict() for _ in jobs]
        groups: Dict[int, list] = {}
        for cell in cells:
            groups.setdefault(max(1, len(cell[2]) - 1).bit_length(), []).append(cell)
        want_regs = self.union_files == "full"
        m = 1 << p
        for _, group in sorted(groups.items()):
            step = max(1, chunk_bytes // m) if want_regs else len(group)
            for g0 in range(0, len(group), step):
                part = group[g0:g0 + step]
                width = max(len(c[2]) for c in part)
                held = [[self.registers(pth) for pth in c[2]] for c in part]
                ptrs = np.zeros((len(part), width), dtype=np.int64)
                for r, row in enumerate(held):
                    ptrs[r, :len(row)] = [t.data_ptr() for t in row]
                with timing.span("union_gpu"):
                    res = self.engine.union_sets(ptrs, p, final_only=True, materialize=want_regs)
                    cards, unions = (res if want_regs else (res, None))
                    cards = cards.cpu().numpy().reshape(len(part))
                self.stats["union_launches"] += 1
                for r, (i, k, members) in enumerate(part):
                    path = jobs[i][1][k]
                    card = float(cards[r])
                    if want_regs:
                        self._remember(path, unions[r, 0])
                        self._write(path, unions[r, 0], p, card, leaf=False, members=members)
                    else:
                        self._write(path, None, p, card, leaf=False, members=members)
                    out[i][k] = card
                del held
        return out

    def prefix_unions(self, leaf_paths_by_k: Dict[int, List[str]], orderings: Sequence[Sequence[int]], p: int,
                      out_paths: Dict[tuple, str] = None, chunk_bytes: int = 4 << 30) -> np.ndarray:
        """Cardinalities of every prefix union: [n_orderings, n_steps, nk] for the k values (sorted)
        of leaf_paths_by_k, each listing the leaf sketches in genome-index order.  A running max per
        (ordering, k): n sketch reads instead of the n(n+1)/2 of re-unioning every prefix.
        out_paths maps (ordering index, step index, k) -> file path for the prefix unions that must
        also exist as sketch files; those are materialised (chunk_bytes of HBM at a time) and
        written once per distinct path."""
        ks = sorted(leaf_paths_by_k)
        orderings = np.asarray(orderings, dtype=np.int64)
        n_ord, n_steps = orderings.shape
        m = 1 << p
        # hold every leaf tensor for the duration of the call: a cache miss further down this list may
        # evict (and free) sketches whose addresses are already in the table
        held = [[self.registers(pth) for pth in leaf_paths_by_k[k]] for k in ks]
        base = np.array([[t.data_ptr() for t in row] for row in held], dtype=np.int64)  # [nk, n]
        # rows are laid out [ordering-chunk][k][ordering] at launch time: sets that read the same
        # sketches (same k, different ordering) are adjacent, which is what keeps them in L2
        ptrs = np.zeros((n_ord, len(ks), n_steps), dtype=np.int64)
        for i in range(len(ks)):
            ptrs[:, i, :] = np.where(orderings >= 0, base[i][np.clip(orderings, 0, None)], 0)
        out = np.empty((n_ord, n_steps, len(ks)), dtype=np.float64)
        want_files = bool(out_paths)
        per_ord = len(ks) * n_steps * m
        step_ords = max(1, chunk_bytes // per_ord) if want_files else n_ord
        written = set()
        for o0 in range(0, n_ord, step_ords):
            o1 = min(n_ord, o0 + step_ords)
            block = np.ascontiguousarray(ptrs[o0:o1].transpose(1, 0, 2)).reshape(len(ks) * (o1 - o0), n_steps)  # [k][o]
            if want_files:
                cards, unions = self.engine.union_sets(block, p, final_only=False, materialize=True)
                unions = unions.view(len(ks), o1 - o0, n_steps, m).transpose(0, 1)   # -> [o][k][step][m]
            else:
                cards = self.engine.union_sets(block, p, final_only=False)
            self.stats["union_launches"] += 1
            cards = cards.cpu().numpy().reshape(len(ks), o1 - o0, n_steps).transpose(1, 0, 2)   # [o][k][step]
            out[o0:o1] = cards.transpose(0, 2, 1)
            if want_files:
                for o in range(o0, o1):
                    for st in range(n_steps):
                        for i, k in enumerate(ks):
                            path = out_paths.get((o, st, k))
                            if path and path not in written:
                                written.add(path)
                                members = [leaf_paths_by_k[k][g] for g in orderings[o][:st + 1] if g >= 0]
                                self._write(path, unions[o - o0, i, st], p, float(cards[o - o0, i, st]), leaf=False,
                                            members=members)
        del held   # every launch above was followed by a device->host read of its results, so nothing still uses them
        return out

    # ------------------------------------------------------------------ all pairs (K6)
    def pair_unions(self, leaf_paths_by_k: Dict[int, List[str]], p: int, tile_pairs: int = 1 << 16,
                    remember: bool = True) -> np.ndarray:
        """Cardinality of the union of EVERY unordered pair of leaves, for every k: [n(n-1)/2, nk], pairs
        in the order (0,1), (0,2) .. (n-2,n-1), k sorted.  leaf_paths_by_k[k] lists the leaf sketches in
        leaf-index order.  The sketches are transposed into bit planes ONCE; the pair list then goes
        through K6 in tiles.  With `remember` the table also answers later union_sketches() calls for
        two-leaf unions (`dandd kij` builds one SubSpider per pair: reference lib/huffman_dandd.py:666-695)."""
        ks = sorted(leaf_paths_by_k)
        n = len(leaf_paths_by_k[ks[0]])
        m = 1 << p
        eng = self.engine
        regs = torch.empty((n, len(ks), m), dtype=torch.uint8, device=eng.device)
        for i, k in enumerate(ks):
            for g, pth in enumerate(leaf_paths_by_k[k]):
                regs[g, i].copy_(self.registers(pth))
        iu = np.triu_indices(n, 1)
        pairs = np.stack(iu, axis=1).astype(np.int32)
        out = self.pair_cards(regs, pairs, p, tile_pairs)
        if remember:
            self.pair_table = {"p": int(p), "n": n, "col": {k: i for i, k in enumerate(ks)}, "cards": out,
                               "leaf": {pth: (g, k) for k in ks for g, pth in enumerate(leaf_paths_by_k[k])}}
        return out

    def pair_cards(self, regs: torch.Tensor, pairs, p: int, tile_pairs: int = 1 << 16) -> np.ndarray:
        """card(A u B) for the listed pairs (int [t, 2] genome indices into regs [n, nk, 2^p], on the device)
        at every k: float64 [t, nk] on the host.  The sketches are transposed into bit planes once, the
        pair list goes through K6 in tiles (reference helpers/allpairs.py:360-370 runs one
        `dashing hll A B` -- two FASTA passes -- per pair and k)."""
        eng = self.engine
        n, nk = int(regs.shape[0]), int(regs.shape[1])
        pairs = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
        out = np.empty((pairs.shape[0], nk), dtype=np.float64)
        if not pairs.shape[0]:
            return out
        planes = eng.to_planes(regs, p) if p >= 12 else None
        for t0 in range(0, pairs.shape[0], tile_pairs):
            tile = pairs[t0:t0 + tile_pairs]
            if planes is not None:
                cards = eng.pairwise_cards(None, tile, p, planes=planes, n_genomes=n, nk=nk)
            else:
                cards = eng.pairwise_cards(regs, tile, p)
            out[t0:t0 + tile.shape[0]] = cards.cpu().numpy()
            self.stats["union_launches"] += 1
        return out

    def _pair_lookup(self, members: Sequence[str], p: int):
        """Cardinality of the union of two leaf sketches if the last pair_unions() job covered it."""
        tab = self.pair_table
        if tab is None or len(members) != 2 or tab["p"] != int(p):
            return None
        a, b = tab["leaf"].get(members[0]), tab["leaf"].get(members[1])
        if a is None or b is None or a[1] != b[1] or a[0] == b[0]:
            return None
        i, j = (a[0], b[0]) if a[0] < b[0] else (b[0], a[0])
        n = tab["n"]
        return float(tab["cards"][i * n - i * (i + 1) // 2 + (j - i - 1), tab["col"][a[1]]])

    def materialize_union(self, path: str, p: int, card: float, members) -> float:
        """A union whose cardinality a batched job already produced is asked for as a FILE: write the
        marker (or, with DANDD_B200_UNION_FILES=full, build the registers from the members) -- no
        estimator run.  The marker holds p, the cardinality and the member paths; registers() rebuilds
        the union from them on demand."""
        if self.pair_union_files == "full":
            regs = self.engine.union([self.registers(mb) for mb in members])
            self._remember(path, regs)
            self._write(path, regs, p, card, leaf=False, members=list(members))
        else:
            with timing.span("write_union_markers"):
                try:
                    hllfile.write_stub(path, p, card, list(members))
                except FileNotFoundError:
                    os.makedirs(os.path.dirname(path), exist_ok=True)
                    hllfile.write_stub(path, p, card, list(members))
            self.stats["files_written"] += 1
        return float(card)

    # ------------------------------------------------------------------ dashing card
    def card_of_file(self, path: str, p: int = None) -> float:
        regs = self.registers(path)
        pp = int(regs.numel()).bit_length() - 1
        return float(self.engine.cards(regs.view(1, -1), pp)[0])

    # ------------------------------------------------------------------ kmc / kmc_tools
    def exact_count(self, fastas: Sequence[str], k: int, canon: bool) -> int:
        """Number of distinct (canonical) k-mers in the union of the FASTAs (KMC semantics)."""
        known = self._exact_from_table(fastas, k, canon)
        if known is None:
            known = self._exact_from_family(fastas, k, canon)
        if known is not None:
            return known
        return self.exact_prefix_counts(fastas, k, canon)[-1]

    @contextmanager
    def exact_family(self, genomes: Sequence[str], canon: bool, sets=(), orderings=()):
        """While open, exact_count answers every genome of `genomes`, every set of `sets` (index lists into
        genomes: tree nodes) and every prefix of every ordering of `orderings` (index sequences: progressive
        orderings) from one family job per k (Engine.exact_family_counts: K7 lists + one K8 launch, the singles from
        the list-node counter), run the first time any of them is asked for at that k and kept as a few integers per
        (row, k).  For a caller that knows WHICH sets it will count but not at which k (the exact hill-climb).
        Another set, another `canon`, a k outside 1..256 or an engine without the job keep the per-union path."""
        genomes = [str(f) for f in genomes]
        n = len(genomes)
        sets = [[int(g) for g in s] for s in sets]
        orderings = [[int(g) for g in o] for o in orderings]
        ranks = np.full((len(sets) + len(orderings), n), 0xFFFF, dtype=np.uint16)
        cells = {frozenset([f]): ("single", g, 0) for g, f in reversed(list(enumerate(genomes)))}
        for r, members in enumerate(sets):
            ranks[r, members] = 0
            if members:
                cells.setdefault(frozenset(genomes[g] for g in members), ("row", r, 1))
        for o, order in enumerate(orderings):
            r = len(sets) + o
            ranks[r, order[::-1]] = np.arange(len(order), dtype=np.uint16)[::-1]   # a genome listed twice keeps its first place
            for i in range(1, len(order) + 1):
                cells.setdefault(frozenset(genomes[g] for g in order[:i]), ("row", r, i))
        family = {"genomes": genomes, "canon": bool(canon), "ranks": ranks, "cells": cells, "counts": {}}
        outer, self.exact_family_table = getattr(self, "exact_family_table", None), family
        try:
            yield family
        finally:
            self.exact_family_table = outer

    def _exact_from_family(self, fastas, k, canon):
        fam = getattr(self, "exact_family_table", None)
        if fam is None or fam["canon"] != bool(canon) or not 1 <= int(k) <= EXACT_MAX_K \
                or not hasattr(self.engine, "exact_family_counts"):
            return None
        cell = fam["cells"].get(frozenset(fastas))
        if cell is None:
            return None
        got = fam["counts"].get(int(k))
        if got is None:
            self.stats["exact_calls"] += 1
            self.stats["exact_family_jobs"] += 1
            workers = self.exact_workers
            if workers is not None and workers.active:
                got = workers.family_counts(fam["genomes"], fam["ranks"], int(k), fam["canon"])
            else:
                got = self._family_shard(fam["genomes"], fam["ranks"], int(k), fam["canon"], None)
            fam["counts"][int(k)] = got
        singles, hist = got
        kind, r, i = cell
        return int(singles[r]) if kind == "single" else int(hist[r, :i].sum())

    def _family_shard(self, fastas, ranks, k, canon, shard):
        """Engine.exact_family_counts on this process's key range `shard` (None: all keys), as int64."""
        singles, hist = self.engine.exact_family_counts([self.packed(f) for f in fastas], int(k), bool(canon), ranks, shard=shard)
        return np.asarray(singles, dtype=np.int64), np.asarray(hist, dtype=np.int64)

    def exact_prefix_counts(self, fastas: Sequence[str], k: int, canon: bool) -> List[int]:
        self.stats["exact_calls"] += 1
        if self.exact_workers is not None:
            return self.exact_workers.counts(list(fastas), int(k), bool(canon))
        return self._exact_shard_counts(fastas, k, canon, None)

    def exact_pair_cards(self, fastas: Sequence[str], ks: Sequence[int], canon: bool, shard: Optional[Tuple[int, int]] = None,
                         remember: bool = False) -> Tuple[np.ndarray, np.ndarray]:
        """Exact counts of every FASTA and of the union of every pair, at every k: (singles [n, nk],
        unions [n(n-1)/2, nk]) float64, pairs (0,1), (0,2) .. (n-2,n-1).  One batched device job per k
        (K7: every genome read once per k, |A u B| = |A| + |B| - |A n B| in integers).  shard=(rank, world):
        this rank's key range only; the ranks' results add up to the whole counts.  An engine without
        the batched job answers pair by pair through exact_count.  With `remember`, later exact_count
        calls for one or two of these FASTAs at these k are answered from the table."""
        n, ks = len(fastas), [int(k) for k in ks]
        singles = np.zeros((n, len(ks)), dtype=np.int64)
        unions = np.zeros((n * (n - 1) // 2, len(ks)), dtype=np.int64)
        batched = getattr(self.engine, "exact_pair_intersections", None)
        if batched is None:
            if shard is not None and shard[0] != 0:     # (the per-pair path counts whole sets: rank 0 holds them)
                return singles.astype(np.float64), unions.astype(np.float64)
            for c, k in enumerate(ks):
                singles[:, c] = [self.exact_count([f], k, canon) for f in fastas]
                unions[:, c] = [self.exact_count([fastas[a], fastas[b]], k, canon) for a, b in zip(*np.triu_indices(n, 1))]
        else:
            seqs = [self.packed(f) for f in fastas]
            iu = np.triu_indices(n, 1)
            for c, k in enumerate(ks):
                self.stats["exact_calls"] += 1
                singles[:, c] = [self.engine.exact_counts([s], k, canon, shard=shard)[0] for s in seqs]
                inter = batched(seqs, k, canon, singles[:, c].tolist(), shard=shard).astype(np.int64)
                unions[:, c] = singles[iu[0], c] + singles[iu[1], c] - inter
        if remember:
            self.exact_pair_table = {"n": n, "canon": bool(canon), "col": {k: c for c, k in enumerate(ks)},
                                     "row": {f: g for g, f in enumerate(fastas)}, "singles": singles, "unions": unions}
        return singles.astype(np.float64), unions.astype(np.float64)

    def exact_prefix_cards(self, fastas: Sequence[str], orderings, ks: Sequence[int], canon: bool,
                           shard: Optional[Tuple[int, int]] = None, singles=None) -> np.ndarray:
        """Exact counts of every prefix union of every ordering, at every k: int64 [n_orderings, n, nk], cell
        [o, i - 1, c] = |fastas[orderings[o][0]] u .. u fastas[orderings[o][i - 1]]| at ks[c] (an ordering shorter
        than n repeats its full union).  One batched device job per k (K7 lists + K8 first-rank histograms: every
        FASTA read once per k, whatever the number of orderings).  singles [n, nk]: exact counts of the single
        FASTAs if the caller has them on record (they size the job), else they are counted.  shard=(rank, world):
        this rank's key range only.  An engine without the batched job counts ordering by ordering."""
        n, ks = len(fastas), [int(k) for k in ks]
        orderings = [[int(g) for g in o] for o in orderings]
        out = np.zeros((len(orderings), n, len(ks)), dtype=np.int64)
        if not hasattr(self.engine, "exact_first_rank_hist"):
            for c, k in enumerate(ks):
                for o, order in enumerate(orderings):
                    if order:
                        got = self.exact_prefix_counts([fastas[g] for g in order], k, canon)
                        out[o, :len(got), c] = got
                        out[o, len(got):, c] = got[-1]
            return out
        ranks = np.full((len(orderings), n), 0xFFFF, dtype=np.uint16)
        for o, order in enumerate(orderings):
            ranks[o, order[::-1]] = np.arange(len(order), dtype=np.uint16)[::-1]   # a genome listed twice keeps its first place
        hist = self._rank_hists(fastas, ranks, ks, canon, shard, singles)
        return np.cumsum(hist, axis=2).transpose(1, 2, 0).copy()

    def exact_union_cards(self, fastas: Sequence[str], sets, ks: Sequence[int], canon: bool,
                          shard: Optional[Tuple[int, int]] = None, singles=None) -> np.ndarray:
        """Exact count of the union of every set of FASTAs (sets: lists of indices into fastas) at every k:
        int64 [n_sets, nk].  One batched device job per k, as exact_prefix_cards; an engine without it counts
        set by set."""
        n, ks = len(fastas), [int(k) for k in ks]
        sets = [[int(g) for g in s] for s in sets]
        if not hasattr(self.engine, "exact_first_rank_hist"):
            return np.array([[self.exact_count([fastas[g] for g in s], k, canon) if s else 0 for k in ks] for s in sets],
                            dtype=np.int64).reshape(len(sets), len(ks))
        ranks = np.full((len(sets), n), 0xFFFF, dtype=np.uint16)
        for r, members in enumerate(sets):
            ranks[r, members] = 0
        hist = self._rank_hists(fastas, ranks, ks, canon, shard, singles)
        return hist[:, :, 0].T.copy() if n else np.zeros((len(sets), len(ks)), dtype=np.int64)

    def _rank_hists(self, fastas, ranks, ks, canon, shard, singles) -> np.ndarray:
        """First-rank histograms int64 [nk, R, n], one engine job per k; all ranks helping under `tree --exact`
        with several ranks (dist.ExactWorkers), else this process's key range `shard` (None: all keys)."""
        self.stats["exact_calls"] += len(ks)
        workers = self.exact_workers
        if shard is None and workers is not None and workers.active:
            return workers.rank_hists(list(fastas), ranks, list(ks), bool(canon), singles)
        return self._rank_hists_shard(fastas, ranks, ks, canon, singles, shard)

    def _rank_hists_shard(self, fastas, ranks, ks, canon, singles, shard) -> np.ndarray:
        seqs = [self.packed(f) for f in fastas]
        out = np.zeros((len(ks), ranks.shape[0], len(fastas)), dtype=np.int64)
        for c, k in enumerate(ks):
            s = None if singles is None else [int(v) for v in np.asarray(singles)[:, c]]
            out[c] = self.engine.exact_first_rank_hist(seqs, int(k), bool(canon), ranks, singles=s, shard=shard).astype(np.int64)
        return out

    def exact_spectrum(self, fastas: Sequence[str], ks: Sequence[int], canon: bool,
                       shard: Optional[Tuple[int, int]] = None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """The sharing spectrum of the FASTAs at every k: (hist, singles, priv), int64 [nk, n] each; hist[c, i - 1] =
        distinct k-mers held by exactly i of the FASTAs at ks[c], singles[c, g] = |fastas[g]|, priv[c, g] = k-mers only
        fastas[g] holds.  One engine job per k (Engine.exact_spectrum: K7 lists + K9).  shard=(rank, world): this
        rank's key range only; the ranks' results add up.  There is no per-union fallback: the spectrum has no cheap
        equivalent in union counts."""
        if not hasattr(self.engine, "exact_spectrum"):
            raise RuntimeError("the exact sharing spectrum needs an engine with the spectrum job (Engine.exact_spectrum)")
        n, ks = len(fastas), [int(k) for k in ks]
        seqs = [self.packed(f) for f in fastas]
        out = np.zeros((3, len(ks), n), dtype=np.int64)
        for c, k in enumerate(ks):
            self.stats["exact_calls"] += 1
            out[:, c] = [np.asarray(a, dtype=np.int64) for a in self.engine.exact_spectrum(seqs, k, bool(canon), shard=shard)]
        return out[0], out[1], out[2]

    def leave_out_cards(self, regs: torch.Tensor, group, n_groups: int, p: int,
                        shard: Optional[Tuple[int, int]] = None) -> Tuple[np.ndarray, np.ndarray]:
        """HLL cardinalities of the union of all genomes of regs [n, nk, 2^p] and of the union without each group
        (group: n ids in [0, n_groups)): float64 [nk] and [nk, n_groups].  One K10 read of the registers, then the MLE
        of the nk (1 + n_groups) histograms; the histograms are the ones the per-union K3 path builds for the same
        members, so the estimates are the same floats.  shard=(rank, world): this rank takes an equal slice of every
        k's register range and one all_reduce(SUM) adds the histograms of all ranks (every rank holds all of regs)."""
        from dandd_b200 import dist as dd_dist
        nk, m = int(regs.shape[1]), 1 << p
        vec = m // 16
        rank, world = shard if shard is not None else (0, 1)
        span = (vec * rank // world * 16, vec * (rank + 1) // world * 16)
        hist = self.engine.leave_out_hist(regs, group, n_groups, p, reg_range=span)
        self.stats["union_launches"] += 1
        if world > 1:
            hist = dd_dist.sum_counts(hist)
        cards = self.engine.mle(hist, p).cpu().numpy().reshape(nk, 1 + int(n_groups))
        return cards[:, 0].copy(), cards[:, 1:].copy()

    def greedy_order(self, regs: torch.Tensor, ks: Sequence[int], p: int, steps: int, order: str = "max", first=(),
                     shard: Optional[Tuple[int, int]] = None, budget: Optional[int] = None):
        """Greedy ordering of the genomes of regs [n, nk, 2^p]: step t adds the genome g not chosen yet whose union with
        the running union U has the largest (order="max") or smallest ("min") delta = max_k card_k / k, the lowest
        index winning a tie; the genomes of `first` take the first steps as given.  Returns (order int64 [steps],
        cards float64 [steps, nk] of U after each step, stats).  card_k(U u g) is the MLE of the histogram of max(U, g),
        the histogram K3 builds for the same members, so the floats are those of a progressive replay of the order.

        Every step runs K11 over the remaining candidates: dense (every register) until the live registers (g > U)
        fit in 4-byte entries within `budget` (default: half of the free device memory) and take well under the
        dense step's bytes, then one compaction and sparse steps over the live entries to the end; both give the
        same histograms.  shard=(rank, world): rank r evaluates the candidates g = r (mod world), one
        all_reduce(SUM) of the [n, nk] cards per step adds the ranks' rows, and every rank makes the same pick."""
        if not hasattr(self.engine, "greedy_dense_hist"):
            raise RuntimeError("the greedy ordering needs an engine with the K11 step (Engine.greedy_dense_hist)")
        from dandd_b200 import dist as dd_dist
        n, nk, m = (int(x) for x in regs.shape)
        first = [int(g) for g in first]
        assert m == 1 << p and order in ("max", "min") and len(first) <= steps <= n and len(set(first)) == len(first)
        rank, world = shard if shard is not None else (0, 1)
        dev = regs.device
        if budget is None:
            budget = self.engine._pairs_budget()
        kdiv = torch.as_tensor(np.asarray(ks, dtype=np.float64), device=dev)
        union = torch.zeros((nk, m), dtype=torch.uint8, device=dev)
        _, uhist = self.engine.cards_hist(union, p)
        cards = torch.empty((steps, nk), dtype=torch.float64, device=dev)
        chosen = torch.zeros(n, dtype=torch.bool, device=dev)
        left, picks, sparse = list(range(n)), [], None
        stats = {"switch_step": None, "live": [], "dense_steps": 0, "sparse_steps": 0}
        for t in range(steps):
            mine = [g for g in left if g % world == rank]
            if t < len(first):
                pick_d = torch.tensor(first[t], device=dev)
                live_left = torch.zeros((), dtype=torch.int64, device=dev)
            else:
                full = torch.zeros((n, nk), dtype=torch.float64, device=dev)
                live_left = torch.zeros((), dtype=torch.int64, device=dev)
                if mine:
                    if sparse is None:
                        hist, live = self.engine.greedy_dense_hist(regs, union, uhist, mine, p)
                        stats["dense_steps"] += 1
                    else:
                        hist, live = self.engine.greedy_sparse_hist(sparse, union, uhist, mine, p)
                        stats["sparse_steps"] += 1
                    rows = torch.as_tensor(np.asarray(mine, dtype=np.int64), device=dev)
                    full[rows] = self.engine.mle(hist, p)
                if world > 1:
                    full = dd_dist.sum_counts(full)
                pick_d = greedy_pick(full, kdiv, chosen, order)
                if mine:
                    live_left = live.to(torch.int64).sum() - (live.to(torch.int64) * (rows == pick_d)[:, None]).sum()
            union = torch.maximum(union, regs.index_select(0, pick_d.view(1))[0])
            chosen.index_fill_(0, pick_d.view(1), True)
            ucards, uhist = self.engine.cards_hist(union, p)
            cards[t] = ucards
            pick, live_total = (int(x) for x in torch.stack([pick_d.to(torch.int64), live_left]).cpu())   # the one read
            picks.append(pick)
            left.remove(pick)
            stats["live"].append(live_total if t >= len(first) else -1)
            rest = [g for g in mine if g != pick]
            if (sparse is None and t >= len(first) and t + 1 < steps and rest and 4 * live_total < budget
                    and SPARSE_CROSS * 4 * live_total <= len(rest) * nk * m):
                # the dense step's live counts bound the live registers of the grown union: segment capacities
                counts = np.zeros((n, nk), dtype=np.int64)
                counts[mine] = live.cpu().numpy()
                counts[pick] = 0
                off = np.concatenate([[0], np.cumsum(counts.reshape(-1))])
                sparse = self.engine.greedy_compact(regs, union, rest, off, p)
                stats["switch_step"] = t + 1
        self.stats["union_launches"] += steps
        return np.asarray(picks, dtype=np.int64), cards.cpu().numpy(), stats

    def exact_greedy_order(self, fastas: Sequence[str], ks: Sequence[int], canon: bool, steps: int, order: str = "max",
                           first=(), shard: Optional[Tuple[int, int]] = None):
        """The greedy ordering of greedy_order by exact counts: step t adds the FASTA whose union with the ones chosen
        so far has the largest (order="max") or smallest ("min") delta = max_k |U u g|_k / k, the lowest index winning
        a tie; `first` takes the first steps as given.  Returns (order int64 [steps], cards int64 [steps, nk] of U
        after each step, stats {"index_bytes": per k, "distinct_keys": per k, |union of all FASTAs|}).

        A cover index per k (Engine.exact_cover_index, K12) is built first and held on the device for the call:
        |U u g| = |U| + |A_g| - lost[g], lost[g] = |A_g n U|.  Every step computes the [n, nk] candidate counts on the
        device, picks, reads the pick (the one device->host read) and runs one K12 step over every k, which adds the
        keys the pick covers to lost.  shard=(rank, world): this rank's key range; one all_reduce(SUM) of the
        candidate counts per step adds the ranks' shares (every key belongs to one rank, so |U|, |A_g| and lost[g] all
        add), and every rank makes the same pick."""
        if not hasattr(self.engine, "exact_cover_index"):
            raise RuntimeError("the exact greedy ordering needs an engine with the K12 cover index (Engine.exact_cover_index)")
        from dandd_b200 import dist as dd_dist
        n, ks = len(fastas), [int(k) for k in ks]
        first = [int(g) for g in first]
        assert order in ("max", "min") and len(first) <= steps <= n and len(set(first)) == len(first)
        world = shard[1] if shard is not None else 1
        dev = self.engine.device
        seqs = [self.packed(f) for f in fastas]
        indices, held = [], 0
        try:
            with timing.span("exact_cover_index"):
                for k in ks:
                    try:
                        ix = self.engine.exact_cover_index(seqs, k, bool(canon), shard=shard)
                    except torch.OutOfMemoryError as err:
                        raise RuntimeError("the exact greedy index does not fit the device: out of memory at k=%d with %d "
                                           "bytes of index held for the k before it; use fewer k or more ranks"
                                           % (k, held)) from err
                    indices.append(ix)
                    held += ix["bytes"]
                    self.stats["exact_calls"] += 1
            kdiv = torch.as_tensor(np.asarray(ks, dtype=np.float64), device=dev)
            singles = torch.as_tensor(np.stack([ix["singles"].astype(np.int64) for ix in indices], axis=1), device=dev)
            lost = torch.zeros((len(ks), n), dtype=torch.int64, device=dev)
            union = torch.zeros(len(ks), dtype=torch.int64, device=dev)
            cards = torch.empty((steps, len(ks)), dtype=torch.int64, device=dev)
            chosen = torch.zeros(n, dtype=torch.bool, device=dev)
            picks = []
            for t in range(steps):
                mine = union + singles - lost.T                      # [n, nk]: this rank's share of |U u g|
                full = dd_dist.sum_counts(mine.clone()) if world > 1 else mine
                if t < len(first):
                    pick_d = torch.tensor(first[t], device=dev)
                else:
                    pick_d = greedy_pick(full.to(torch.float64), kdiv, chosen, order)
                cards[t] = full.index_select(0, pick_d.view(1))[0]
                union = mine.index_select(0, pick_d.view(1))[0]
                chosen.index_fill_(0, pick_d.view(1), True)
                picks.append(int(pick_d))                            # the one read
                if t + 1 < steps:
                    self.engine.exact_cover_step(indices, picks[-1], lost)
            keys = torch.as_tensor(np.asarray([ix["keys"] for ix in indices], dtype=np.int64), device=dev)
            if world > 1:
                keys = dd_dist.sum_counts(keys)
            stats = {"index_bytes": [int(ix["bytes"]) for ix in indices], "distinct_keys": keys.cpu().numpy().tolist()}
            return np.asarray(picks, dtype=np.int64), cards.cpu().numpy(), stats
        finally:
            indices.clear()                                          # the index lives for this call only

    def exact_leave_out(self, fastas: Sequence[str], ks: Sequence[int], canon: bool, group, n_groups: int,
                        shard: Optional[Tuple[int, int]] = None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Exact counts of the union of the FASTAs and of the union without each group (group: one id in [0, n_groups)
        per FASTA), and of every FASTA alone: int64 [nk], [nk, n_groups] and [nk, n].  One engine job per k: with one
        FASTA per group the sharing-spectrum job (K9; without g = union - keys only g holds), else one first-rank job
        (K8) whose row g ranks group g's members 1 and every other FASTA 0 (without g = bin 0, its novel keys bin 1).
        shard=(rank, world): this rank's key range only; the ranks' results add up."""
        n, ks, n_groups = len(fastas), [int(k) for k in ks], int(n_groups)
        group = np.asarray(group, dtype=np.int64)
        seqs = [self.packed(f) for f in fastas]
        union = np.zeros(len(ks), dtype=np.int64)
        without = np.zeros((len(ks), n_groups), dtype=np.int64)
        singles = np.zeros((len(ks), n), dtype=np.int64)
        singleton = n_groups == n and len(set(group.tolist())) == n
        ranks = (group[None, :] == np.arange(n_groups)[:, None]).astype(np.uint16)
        for c, k in enumerate(ks):
            self.stats["exact_calls"] += 1
            if singleton:
                hist, singles[c], priv = (np.asarray(a, dtype=np.int64) for a in
                                          self.engine.exact_spectrum(seqs, k, bool(canon), shard=shard))
                union[c] = hist.sum()
                without[c, group] = union[c] - priv
            else:
                s, hist = self.engine.exact_family_counts(seqs, k, bool(canon), ranks, shard=shard)
                singles[c] = np.asarray(s, dtype=np.int64)
                hist = np.asarray(hist, dtype=np.int64)
                without[c] = hist[:, 0]
                union[c] = hist[0, 0] + hist[0, 1]
        return union, without, singles

    def exact_query_cards(self, ref_fastas: Sequence[str], query_fastas: Sequence[str], ks: Sequence[int], canon: bool,
                          shard: Optional[Tuple[int, int]] = None):
        """Exact counts of query FASTAs against a collection of reference FASTAs at every k, int64: (ref_single [nk, R],
        query_single [nk, Q], union_R [nk] = |U_R|, with_q [nk, Q] = |U_R u A_q|, pair_union [nk, Q, R] = |A_q u A_r|),
        U_R the union of the references.  One engine job per k (Engine.exact_query_counts: K7 lists + K13).
        shard=(rank, world): this rank's key range only; the ranks' results add up.  There is no per-union fallback:
        it would cost Q (R + 1) union counts per k."""
        if not hasattr(self.engine, "exact_query_counts"):
            raise RuntimeError("exact query counts need an engine with the query job (Engine.exact_query_counts)")
        R, Q, ks = len(ref_fastas), len(query_fastas), [int(k) for k in ks]
        seqs = [self.packed(f) for f in list(ref_fastas) + list(query_fastas)]
        singles = np.zeros((len(ks), R + Q), dtype=np.int64)
        union = np.zeros(len(ks), dtype=np.int64)
        with_q = np.zeros((len(ks), Q), dtype=np.int64)
        pair = np.zeros((len(ks), Q, R), dtype=np.int64)
        for c, k in enumerate(ks):
            self.stats["exact_calls"] += 1
            s, inter, shared, union[c] = self.engine.exact_query_counts(seqs, R, k, bool(canon), shard=shard)
            singles[c] = np.asarray(s, dtype=np.int64)
            with_q[c] = union[c] + singles[c, R:] - np.asarray(shared, dtype=np.int64)
            pair[c] = singles[c, R:, None] + singles[c, None, :R] - np.asarray(inter, dtype=np.int64)
        return singles[:, :R].copy(), singles[:, R:].copy(), union, with_q, pair

    def query_cards(self, regs: torch.Tensor, n_refs: int, p: int, shard: Optional[Tuple[int, int]] = None):
        """HLL cardinalities of query_cards' quantities from regs [R + Q, nk, 2^p] (references first, then queries):
        (ref_single [nk, R], query_single [nk, Q], union_R [nk], with_q [nk, Q], pair_union [nk, Q, R]) float64.  The
        union of the references and its histogram come from K3 and K4; card(max(U_R, q)) for every query from one K11
        dense step with the queries as candidates; the Q x R pair cards from pair_cards (K6).  The histograms are the
        ones the per-union K3 path builds for the same members, so the estimates are the same floats.
        shard=(rank, world): rank r takes the queries q = r (mod world), and one all_reduce(SUM) adds the ranks' rows
        (a row no rank owns is 0.0; rank 0 gives the references' rows); every rank holds all of regs."""
        from dandd_b200 import dist as dd_dist
        n, nk = int(regs.shape[0]), int(regs.shape[1])
        R = int(n_refs)
        Q = n - R
        rank, world = shard if shard is not None else (0, 1)
        mine = [q for q in range(Q) if q % world == rank]
        eng, dev = self.engine, regs.device
        union = eng.union([regs[r] for r in range(R)])
        ucards, uhist = eng.cards_hist(union, p)
        singles = eng.cards(regs, p)
        # [union_R | ref singles | query singles | with_q | pair cards], float64 [nk, 1 + R + 2Q + QR] on the device
        out = torch.zeros((nk, 1 + R + 2 * Q + Q * R), dtype=torch.float64, device=dev)
        if rank == 0:
            out[:, 0] = ucards
            out[:, 1:1 + R] = singles[:R].T
        if mine:
            rows = torch.as_tensor(np.asarray(mine, dtype=np.int64), device=dev)
            out[:, 1 + R + rows] = singles[R + rows].T
            hist, _ = eng.greedy_dense_hist(regs, union, uhist, [R + q for q in mine], p)
            out[:, 1 + R + Q + rows] = eng.mle(hist, p).T
            pairs = np.array([(r, R + q) for q in mine for r in range(R)], dtype=np.int64)
            cells = np.array([q * R + r for q in mine for r in range(R)], dtype=np.int64)
            got = torch.as_tensor(self.pair_cards(regs, pairs, p), device=dev)
            out[:, 1 + R + 2 * Q + torch.as_tensor(cells, device=dev)] = got.T
        self.stats["union_launches"] += 2
        if world > 1:
            out = dd_dist.sum_counts(out)
        out = out.cpu().numpy()
        return (out[:, 1:1 + R].copy(), out[:, 1 + R:1 + R + Q].copy(), out[:, 0].copy(), out[:, 1 + R + Q:1 + R + 2 * Q].copy(),
                out[:, 1 + R + 2 * Q:].reshape(nk, Q, R).copy())

    def _exact_from_table(self, fastas, k, canon):
        tab = getattr(self, "exact_pair_table", None)
        if tab is None or tab["canon"] != bool(canon) or int(k) not in tab["col"] or not 1 <= len(fastas) <= 2:
            return None
        rows = [tab["row"].get(f) for f in fastas]
        if None in rows:
            return None
        c = tab["col"][int(k)]
        if len(rows) == 1 or rows[0] == rows[1]:
            return int(tab["singles"][rows[0], c])
        i, j = sorted(rows)
        n = tab["n"]
        return int(tab["unions"][i * n - i * (i + 1) // 2 + (j - i - 1), c])

    def _exact_shard_counts(self, fastas, k, canon, shard):
        return self.engine.exact_counts([self.packed(f) for f in fastas], int(k), canon, shard=shard)

    def start_exact_workers(self):
        """Multi-rank exact mode (dandd_b200.dist.ExactWorkers): rank 0 keeps going, the others serve."""
        from dandd_b200 import dist as dd_dist
        self.exact_workers = dd_dist.ExactWorkers(self._exact_shard_counts, self._rank_hists_shard, self._family_shard)
        return self.exact_workers


import threading as _threading  # noqa: E402

_store = None
_store_lock = _threading.Lock()
_bound_threads = set()


def get_store():
    """The process-wide store.  Thread-safe: the command line starts it on a background thread (CUDA
    start-up takes seconds) while the main thread joins the process group."""
    global _store
    if _store is None:
        with _store_lock:
            if _store is None:
                from dandd_b200 import _startup
                if _startup.TRIM_REQUESTED:          # command-line start-up trim, see _startup.py
                    _startup.trim_torch_cuda_init()
                with timing.span("engine_start"):    # CUDA context + library load (torch itself was imported with this module)
                    _store = GpuSketchStore()
                timing.mark("engine_ready")
    ident = _threading.get_ident()
    if ident not in _bound_threads and hasattr(getattr(_store, "engine", None), "bind_thread"):
        _store.engine.bind_thread()                  # the store may have been started on another thread
        _bound_threads.add(ident)
    return _store


def set_store(store) -> None:
    """Install another store (a different device; the test-suite installs an oracle-backed double
    here to exercise the host logic on machines without a GPU)."""
    global _store
    _store = store
