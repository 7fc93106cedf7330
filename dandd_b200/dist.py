"""Multi-GPU sharding of the hot path (SURVEY.md 8e): one process per GPU (torchrun), genomes
sharded across ranks, no collective on the sketching itself.  The path has exactly one exchange
step -- merging register arrays -- and HLL merge is an exact, associative, commutative, idempotent
max, so the results are bit-identical to a single-GPU run:

    union_over_ranks   all_reduce(MAX, uint8)  over [nk][2^p]      (the union sketch of the job)
    gather_registers   all_gather              of [n_local][nk][2^p] (every rank gets every leaf:
                                               progressive orderings / pair tiles are then split
                                               across ranks with no further communication)
    sum_counts         all_reduce(SUM, int64)  for key-range-sharded exact counts

Backend: NCCL over NVLink on GPUs, gloo in the CPU tests (tests/test_dist.py, world_size 2).
The payloads are tiny next to NVLink bandwidth (<= 31 MiB per genome), so plain collectives on the
compute stream are the right tool; there is no compute kernel to fuse them into."""
import os
from typing import List

import numpy as np
import torch
import torch.distributed as dist


def init(backend: str = None) -> (int, int):
    """Initialise the default process group from the torchrun environment (no-op if world is 1).

    backend=None (the command line): the default group is gloo -- it is up in a fraction of a second
    and all the command line exchanges through it are small Python objects (cardinalities, names);
    creating NCCL communicators for 8 ranks costs seconds, so the NCCL group that carries REGISTER
    tensors (union_over_ranks / gather_registers) is created on first use only (tensor_group()).
    backend="nccl" (bench.py, tools/): NCCL from the start, eagerly bound to LOCAL_RANK's GPU."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1 and not dist.is_initialized():
        backend = backend or "gloo"
        kwargs = {}
        if backend == "nccl":
            kwargs["device_id"] = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
            # object collectives pick torch's CURRENT device; a rank that never touched its GPU (everything
            # cached) would otherwise run them on device 0
            torch.cuda.set_device(kwargs["device_id"])
        dist.init_process_group(backend, **kwargs)
    return rank, world


def world() -> (int, int):
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


from .shard import shard_by_size  # noqa: E402,F401  (re-exported: the table every rank computes)


_nccl_group = None


def tensor_group(t: torch.Tensor):
    """The process group for a collective on tensor `t`: the default group, or -- CUDA tensor while
    the default group is gloo -- an NCCL group over all ranks, created the first time it is needed
    (a collective call itself: every rank reaches it, because every rank enters the same tensor
    collective)."""
    global _nccl_group
    if not t.is_cuda or dist.get_backend() == "nccl":
        return None
    if _nccl_group is None:
        torch.cuda.set_device(t.device)
        _nccl_group = dist.new_group(backend="nccl")
    return _nccl_group


def union_over_ranks(regs: torch.Tensor) -> torch.Tensor:
    """In-place register-wise max over all ranks (uint8 tensor of any shape): NCCL MAX all-reduce
    over NVLink for device tensors."""
    _, n = world()
    if n > 1:
        dist.all_reduce(regs, op=dist.ReduceOp.MAX, group=tensor_group(regs))
    return regs


def gather_registers(local: torch.Tensor, owners: List[List[int]]) -> torch.Tensor:
    """local: [n_local, nk, m] registers of this rank's genomes (in the order of owners[rank]).
    Returns [n_total, nk, m] in global genome order on every rank."""
    rank, n = world()
    total = sum(len(o) for o in owners)
    if n == 1:
        return local
    nk, m = local.shape[1], local.shape[2]
    width = max(len(o) for o in owners)
    padded = torch.zeros((width, nk, m), dtype=local.dtype, device=local.device)
    padded[:local.shape[0]] = local
    bucket = [torch.empty_like(padded) for _ in range(n)]
    dist.all_gather(bucket, padded, group=tensor_group(padded))
    out = torch.empty((total, nk, m), dtype=local.dtype, device=local.device)
    for r, idxs in enumerate(owners):
        for j, g in enumerate(idxs):
            out[g] = bucket[r][j]
    return out


def gather_cards(local: torch.Tensor, owners: List[List[int]]) -> torch.Tensor:
    """Same for the [n_local, nk] float64 cardinalities."""
    return gather_registers(local.unsqueeze(-1), owners).squeeze(-1)


def sum_counts(counts: torch.Tensor) -> torch.Tensor:
    _, n = world()
    if n > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=tensor_group(counts))
    return counts


def split_work(n_items: int) -> range:
    """Contiguous slice of n_items (orderings, pair tiles) owned by this rank."""
    rank, n = world()
    lo = (n_items * rank) // n
    hi = (n_items * (rank + 1)) // n
    return range(lo, hi)


# ---- one genome over several ranks -------------------------------------------------------------------
def split_fasta(text, nparts: int, overlap_symbols: int = 255, only: int = None, min_grain: int = 4096) -> List[bytes]:
    """Cut ONE FASTA text into `nparts` FASTA texts whose sketches merge to the sketch of the whole
    (SURVEY.md 8e, "genomes < GPUs"): register-wise max for HLL, set union for exact counts.

    k-mers never span records, so whole records can go anywhere; a record larger than its fair
    share is cut inside its sequence body and every later piece starts `overlap_symbols` symbols
    early (>= k-1 for every k <= 256 by default) behind a synthetic header line, so each k-mer of the
    record lies wholly inside at least one piece.  Seeing a k-mer twice is harmless for a max / a
    set.  Pieces are assigned to parts largest-first; a part may be empty.  `only=r` materialises
    part r alone (the others come back as None) -- a rank needs just its own bytes.  Records are not
    cut into pieces smaller than `min_grain` bytes."""
    raw = text.tobytes() if isinstance(text, np.ndarray) else bytes(text) if not isinstance(text, bytes) else text
    buf = np.frombuffer(raw, dtype=np.uint8)
    n = len(raw)
    nparts = max(1, int(nparts))
    if nparts == 1 or n == 0:
        return [raw] + [b""] * (nparts - 1)
    # records: the FIRST '>' / '@' of the file wherever it is (kseq skips to the first marker and takes
    # it as a header line, SURVEY.md A.1), afterwards every '>' / '@' at a line start.  (FASTQ text --
    # a line beginning with '+' -- must be rewritten with Engine.fastq_to_fasta before it gets here.)
    starts = []
    for mark in (b">", b"@"):
        at = raw.find(mark)                                          # (single-byte find runs at memchr speed)
        while at >= 0:
            starts.append(at)
            at = raw.find(mark, at + 1)
    starts.sort()
    starts = [at for i, at in enumerate(starts) if i == 0 or raw[at - 1] == 10]
    if not starts:                                                   # no record at all: nothing is sequence
        return [raw] + [b""] * (nparts - 1)
    bounds = starts + [n]
    total = n - starts[0]
    target = max(1, -(-total // nparts))
    pieces = []                                                      # (begin, end, needs_header)
    for a, b in zip(bounds[:-1], bounds[1:]):
        nl = raw.find(b"\n", a, b)
        body = nl + 1 if nl >= 0 else b                              # first byte after the header line
        grain = max(target // 4, min_grain)                          # pieces of a quarter share balance well
        if b - a <= grain + grain // 4 or body >= b:
            pieces.append((a, b, False))
            continue
        ncut = -(-(b - body) // grain)
        cuts = [body + (b - body) * i // ncut for i in range(1, ncut)]
        prev = a
        for c in cuts:
            pieces.append((prev, c, prev != a))
            # step back over at least overlap_symbols sequence bytes (newlines / CRs do not count)
            # ... and never start on a '>', '@' or '+' (junk inside a sequence line): behind the synthetic
            # header it would sit at a line start and turn the rest of its line into a header / quality
            back, span, need = c, 2 * overlap_symbols + 64, overlap_symbols
            while True:
                lo = max(body, c - span)
                seg = buf[lo:c]
                is_sym = (seg != 10) & (seg != 13)
                have = int(is_sym.sum())
                if have >= need:
                    idx = np.flatnonzero(is_sym)
                    at = lo + int(idx[have - need])
                    if buf[at] in (62, 64, 43) and at > body:
                        need += 1
                        continue
                    back = at
                    break
                if lo == body:
                    back = body
                    break
                span *= 2
            prev = back
        pieces.append((prev, b, True))
    order = sorted(range(len(pieces)), key=lambda i: (-(pieces[i][1] - pieces[i][0]), i))
    load = [0] * nparts
    owned = [[] for _ in range(nparts)]
    for i in order:
        r = min(range(nparts), key=lambda j: (load[j], j))
        owned[r].append(i)
        load[r] += pieces[i][1] - pieces[i][0]
    out = []
    view = memoryview(raw)
    for r in range(nparts):
        if only is not None and r != only:
            out.append(None)
            continue
        chunks = []
        for i in sorted(owned[r]):
            a, b, hdr = pieces[i]
            if hdr:
                chunks.append(b">part\n")
            chunks.append(view[a:b])
            if b > a and raw[b - 1] != 10:
                chunks.append(b"\n")                                 # keep the next header at a line start
        out.append(b"".join(chunks))
    return out


# ---- rank 0 drives, the other ranks serve (exact mode from the command line) -----------------------
def broadcast_object(obj, src: int = 0):
    """Small Python object from rank `src` to everyone; returns it on every rank."""
    _, n = world()
    if n < 2:
        return obj
    box = [obj]
    dist.broadcast_object_list(box, src=src)
    return box[0]


class ExactWorkers:
    """`dandd tree --exact` under torchrun: rank 0 runs the (inherently sequential) tree logic; every
    exact count it needs is announced to the other ranks, all ranks insert their key range of the
    k-mer set (`shard=(rank, world)`) and the counts are summed.  Ranks > 0 sit in serve() until
    rank 0 calls stop().  Three kinds of request: the progressive counts of one FASTA list at one k ("exact"),
    the first-rank histograms of a rank table at several k ("hist", GpuSketchStore.exact_union_cards), and the
    single counts + first-rank histograms of a registered family at one k ("family", GpuSketchStore.exact_family)."""

    def __init__(self, counter, hists=None, family=None):
        self.counter = counter          # callable(fastas, k, canon, shard) -> list of progressive counts (this rank's shard)
        self.hists = hists              # callable(fastas, ranks, ks, canon, singles, shard) -> int64 [nk, R, n] (this rank's shard)
        self.family = family            # callable(fastas, ranks, k, canon, shard) -> (int64 [n], int64 [R, n]) (this rank's shard)
        self.rank, self.world = world()
        self.active = self.world > 1

    def counts(self, fastas, k, canon):
        """Called on rank 0: progressive distinct counts of the union of fastas[:i+1], all ranks helping."""
        if not self.active:
            return self.counter(fastas, k, canon, None)
        broadcast_object(("exact", list(fastas), int(k), bool(canon)))
        return self._collective(fastas, k, canon)

    def _collective(self, fastas, k, canon):
        mine = torch.tensor(self.counter(fastas, k, canon, (self.rank, self.world)), dtype=torch.int64)
        if dist.get_backend() == "nccl":
            mine = mine.cuda()
        return [int(v) for v in sum_counts(mine).cpu().tolist()]

    def rank_hists(self, fastas, ranks, ks, canon, singles=None):
        """Called on rank 0: first-rank histograms int64 [nk, R, n], every rank running its key range."""
        if not self.active:
            return self.hists(fastas, ranks, ks, canon, singles, None)
        broadcast_object(("hist", list(fastas), ranks, list(ks), bool(canon), singles))
        return self._hist_collective(fastas, ranks, ks, canon, singles)

    def _hist_collective(self, fastas, ranks, ks, canon, singles):
        mine = torch.from_numpy(np.ascontiguousarray(self.hists(fastas, ranks, ks, canon, singles, (self.rank, self.world)),
                                                     dtype=np.int64))
        if dist.get_backend() == "nccl":
            mine = mine.cuda()
        return sum_counts(mine).cpu().numpy()

    def family_counts(self, fastas, ranks, k, canon):
        """Called on rank 0: (singles int64 [n], first-rank histograms int64 [R, n]) at k, every rank running its key
        range; one all_reduce of [n + R n] adds them up."""
        if not self.active:
            return self.family(fastas, ranks, k, canon, None)
        broadcast_object(("family", list(fastas), ranks, int(k), bool(canon)))
        return self._family_collective(fastas, ranks, k, canon)

    def _family_collective(self, fastas, ranks, k, canon):
        singles, hist = self.family(fastas, ranks, k, canon, (self.rank, self.world))
        mine = torch.from_numpy(np.concatenate([np.asarray(singles, dtype=np.int64).reshape(-1),
                                                np.asarray(hist, dtype=np.int64).reshape(-1)]))
        if dist.get_backend() == "nccl":
            mine = mine.cuda()
        total = sum_counts(mine).cpu().numpy()
        n = len(fastas)
        return total[:n], total[n:].reshape(len(ranks), n)

    def serve(self) -> int:
        """Ranks > 0: answer requests until rank 0 says stop; returns how many were served."""
        served = 0
        while True:
            req = broadcast_object(None)
            if not req or req[0] == "stop":
                return served
            if req[0] == "hist":
                self._hist_collective(*req[1:])
            elif req[0] == "family":
                self._family_collective(*req[1:])
            else:
                self._collective(req[1], req[2], req[3])
            served += 1

    def stop(self) -> None:
        if self.active and self.rank == 0:
            broadcast_object(("stop",))
        self.active = False
