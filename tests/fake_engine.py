"""FakeEngine: a CPU double of dandd_b200.engine.Engine for the `-m "not gpu"` tests.

TEST INFRASTRUCTURE.  It answers the engine-level calls of dandd_b200/store.py from the CPU oracle on
torch CPU tensors, so that the REAL GpuSketchStore -- cache and eviction, pointer tables built from
`data_ptr()`, grouping and chunking of batched union jobs, layout transposes of the prefix-union
results, pair-table index arithmetic, marker files -- runs in a container without a GPU
(tests/test_store_cpu.py).  The product never imports this module; on the GPU box the same scenarios
run on the real engine (tests/test_host_gpu.py, tests/test_allpairs_gpu.py)."""
import ctypes

import numpy as np
import torch

from dandd_b200.engine import Engine, FastqInput
from oracle import pyoracle as orc


class FakePacked:
    """What Engine.pack returns, as far as the store looks at it."""

    def __init__(self, text: bytes):
        self.text = text
        self.codes = torch.zeros(max(1, len(text) // 4), dtype=torch.uint8)      # (sizes only matter for the cache budget)
        self.invalid = torch.zeros(max(1, len(text) // 8), dtype=torch.uint8)
        self._sym = None

    def check(self):
        # the packer reports a line that begins with '+' (FASTQ) instead of packing it
        if self.text[:1] == b"+" or b"\n+" in self.text:
            raise FastqInput("FASTQ text (a line begins with '+')")
        return self

    @property
    def sym(self):
        if self._sym is None:
            self._sym = orc.fasta_symbols(self.check().text)
        return self._sym

    @property
    def nsym(self):
        return int(self.sym.size)


def _at(address: int, nbytes: int) -> np.ndarray:
    """The bytes a device pointer table entry points at (CPU tensors: real host addresses)."""
    return np.frombuffer(ctypes.string_at(int(address), nbytes), dtype=np.uint8)


class FakeEngine:
    polyt_sentinel = False
    fastq_to_fasta = staticmethod(Engine.fastq_to_fasta)        # host-side code of the real library

    def __init__(self):
        self.device = torch.device("cpu")
        self.calls = {"pack": 0, "sketch": 0, "union_sets": 0, "pairwise_cards": 0, "to_planes": 0, "exact_counts": 0}

    def bind_thread(self):
        pass

    def pack(self, text, **_):
        self.calls["pack"] += 1
        return FakePacked(bytes(text))

    def sketch(self, seq, ks, p=20, canon=True, **_):
        self.calls["sketch"] += 1
        regs = np.stack([orc.hll_sketch(seq.sym, int(k), p, canon) for k in ks])
        return torch.from_numpy(regs), torch.tensor([orc.card(r, p) for r in regs], dtype=torch.float64)

    def cards(self, regs, p):
        flat = regs.contiguous().view(-1, 1 << p).numpy()
        return torch.tensor([orc.card(r, p) for r in flat], dtype=torch.float64).view(regs.shape[:-1])

    def union(self, sketches):
        return torch.from_numpy(orc.union_max([s.numpy() for s in sketches]).copy())

    def union_sets(self, member_ptrs, p, final_only=True, materialize=False):
        """Engine.union_sets: running max over each row of ADDRESSES (0 = skip), cardinality per step."""
        self.calls["union_sets"] += 1
        ptrs = np.ascontiguousarray(member_ptrs, dtype=np.int64)
        n_sets, n_steps = ptrs.shape
        m = 1 << p
        osteps = 1 if final_only else n_steps
        cards = torch.zeros((n_sets, osteps), dtype=torch.float64)
        unions = torch.zeros((n_sets, osteps, m), dtype=torch.uint8)
        for s in range(n_sets):
            run = np.zeros(m, dtype=np.uint8)
            for st in range(n_steps):
                if ptrs[s, st]:
                    run = np.maximum(run, _at(ptrs[s, st], m))
                if not final_only or st == n_steps - 1:
                    o = 0 if final_only else st
                    cards[s, o] = orc.card(run, p)
                    unions[s, o] = torch.from_numpy(run.copy())
        return (cards, unions) if materialize else cards

    def to_planes(self, regs, p, out=None):
        self.calls["to_planes"] += 1
        assert p >= 12, "bit planes need p >= 12 (dd_to_planes)"
        return regs.contiguous().view(-1, 1 << p).clone()      # opaque to the store; pairwise_cards reads it back

    def pairwise_cards(self, regs, pairs, p, planes=None, n_genomes=None, nk=None, out=None):
        self.calls["pairwise_cards"] += 1
        if planes is not None:
            regs = planes.view(n_genomes, nk, 1 << p)
        h = regs.numpy()
        pairs = np.asarray(pairs).reshape(-1, 2)
        cards = torch.zeros((len(pairs), h.shape[1]), dtype=torch.float64)
        for j, (a, b) in enumerate(pairs):
            for i in range(h.shape[1]):
                cards[j, i] = orc.card(np.maximum(h[a, i], h[b, i]), p)
        return cards

    def mle(self, hist, p):
        flat = hist.reshape(-1, 64).numpy()
        return torch.tensor([orc.ertl_mle(row.astype(np.uint32), p) for row in flat], dtype=torch.float64).view(hist.shape[:-1])

    def exact_counts(self, seqs, k, canon=True, capacity=None, shard=None):
        self.calls["exact_counts"] += 1
        if shard is not None and shard[0] != 0:      # (the oracle has no key-range filter: rank 0 counts everything)
            return [0] * len(seqs)
        return [orc.exact_count([s.sym for s in seqs[:i + 1]], int(k), canon) for i in range(len(seqs))]


LIST_JOBS = ("exact_pair_intersections", "exact_first_rank_hist", "exact_family_counts", "exact_spectrum")


def _absent(job):
    def get(self):
        raise AttributeError(job)
    return property(get)


class ListJobEngine(FakeEngine):
    """FakeEngine plus the jobs Engine runs over the K7 co-occurrence lists (LIST_JOBS), all read off one table of
    which genomes hold each distinct k-mer, from oracle k-mer sets (rank 0 holds every key, as in
    FakeEngine.exact_counts).  Records the genome count of every per-union count and the k of every family job."""

    def __init__(self):
        super().__init__()
        self.calls.update(dict.fromkeys(LIST_JOBS, 0))
        self.union_sizes = []           # len(seqs) of every exact_counts call
        self.family_ks = []             # k of every exact_family_counts call
        self._held = {}

    @classmethod
    def only(cls, *jobs):
        """This double offering only the list jobs `jobs`.  The store takes a job's batched path when its engine has
        the method (hasattr), else the per-union path: the other jobs are hidden as an engine without them lacks them."""
        hidden = {job: _absent(job) for job in LIST_JOBS if job not in jobs}
        return type("%s.only(%s)" % (cls.__name__, ", ".join(jobs)), (cls,), hidden)

    def exact_counts(self, seqs, k, canon=True, capacity=None, shard=None):
        self.union_sizes.append(len(seqs))
        return super().exact_counts(seqs, k, canon, capacity, shard)

    def _holders(self, seqs, k, canon):
        """bool [distinct k-mers of seqs, n]: which genomes hold each k-mer.  Cached per (seqs, k, canon); the cache
        keeps the seqs, so their ids stay theirs."""
        key = (tuple(id(s) for s in seqs), int(k), bool(canon))
        if key not in self._held:
            sets = [np.unique(orc.kmers(s.sym, int(k), canon)) for s in seqs]
            keys, row = np.unique(np.concatenate([np.zeros(0, np.uint64)] + sets), return_inverse=True)
            held = np.zeros((keys.size, len(seqs)), dtype=bool)
            held[row, np.repeat(np.arange(len(seqs)), [a.size for a in sets])] = True
            self._held[key] = (list(seqs), held)
        return self._held[key][1]

    def _first_rank(self, held, ranks):
        """hist uint64 [R, n]: hist[r][m] = k-mers whose least rank over their holders is m under row r."""
        n = held.shape[1]
        hist = np.zeros(ranks.shape, dtype=np.uint64)
        for r, row in enumerate(ranks):
            m = np.where(held, row, 0xFFFF).min(axis=1)
            hist[r] = np.bincount(m[m < n], minlength=n)
        return hist

    def exact_pair_intersections(self, seqs, k, canon=True, singles=None, shard=None):
        self.calls["exact_pair_intersections"] += 1
        n = len(seqs)
        if shard is not None and shard[0] != 0:
            return np.zeros(n * (n - 1) // 2, dtype=np.uint64)
        held = self._holders(seqs, k, canon).astype(np.uint64)
        assert singles is None or list(singles) == held.sum(axis=0).tolist()
        return (held.T @ held)[np.triu_indices(n, 1)]

    def exact_first_rank_hist(self, seqs, k, canon, ranks, singles=None, shard=None, passes=None):
        self.calls["exact_first_rank_hist"] += 1
        ranks = np.asarray(ranks, dtype=np.uint16).reshape(-1, len(seqs))
        if shard is not None and shard[0] != 0:
            return np.zeros(ranks.shape, dtype=np.uint64)
        held = self._holders(seqs, k, canon)
        assert singles is None or list(singles) == held.sum(axis=0).tolist()
        return self._first_rank(held, ranks)

    def exact_family_counts(self, seqs, k, canon, ranks, shard=None, passes=None):
        from dandd_b200.engine import length_bounds
        self.calls["exact_family_counts"] += 1
        self.family_ks.append(int(k))
        n = len(seqs)
        ranks = np.asarray(ranks, dtype=np.uint16).reshape(-1, n)
        if shard is not None and shard[0] != 0:
            return np.zeros(n, dtype=np.uint64), np.zeros(ranks.shape, dtype=np.uint64)
        held = self._holders(seqs, k, canon)
        singles = held.sum(axis=0).astype(np.uint64)
        assert all(b >= c for b, c in zip(length_bounds([s.nsym for s in seqs], k), singles))   # the job is never undersized
        return singles, self._first_rank(held, ranks)

    def exact_spectrum(self, seqs, k, canon, shard=None, passes=None):
        self.calls["exact_spectrum"] += 1
        n = len(seqs)
        if shard is not None and shard[0] != 0:
            return tuple(np.zeros(n, dtype=np.uint64) for _ in range(3))
        held = self._holders(seqs, k, canon)
        holders = held.sum(axis=1)
        hist = np.bincount(holders, minlength=n + 1)[1:].astype(np.uint64)
        return hist, held.sum(axis=0).astype(np.uint64), held[holders == 1].sum(axis=0).astype(np.uint64)
