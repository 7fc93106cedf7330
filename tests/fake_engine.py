"""FakeEngine: a CPU double of dandd_b200.engine.Engine for the `-m "not gpu"` tests.

TEST INFRASTRUCTURE.  It answers every engine-level call of dandd_b200/store.py (tests/test_store_cpu.py checks that
none is missing) from the CPU oracle on torch CPU tensors, so that the REAL GpuSketchStore -- cache and eviction,
pointer tables built from `data_ptr()`, grouping and chunking of batched union jobs, layout transposes of the
prefix-union results, pair-table index arithmetic, marker files, the batched exact jobs -- runs in a container without
a GPU.  The kernels it stands in for are restated in numpy by the module functions below; each is checked against
brute force in the test module of its feature.  The product never imports this module; on the GPU box the same
scenarios run on the real engine (tests/test_host_gpu.py, tests/test_allpairs_gpu.py)."""
import ctypes
import math
from collections import Counter

import numpy as np
import torch

from dandd_b200.engine import Engine, FastqInput, length_bounds
from oracle import pyoracle as orc

BINS = 64


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


# ---------------------------------------------------------------- numpy restatements of the kernels
def kmer_keys(sym, k: int, canon: bool = True) -> np.ndarray:
    """The distinct (canonical) k-mers of a symbol stream, any k in 1..256: oracle u64 codes up to k = 32, above that
    rows of k symbols as bytes (canonical: the smaller of the k-mer and its reverse complement in A<C<G<T order)."""
    if k <= 32:
        return np.unique(orc.kmers(sym, k, canon))
    sym = np.asarray(sym, dtype=np.uint8)
    win = np.lib.stride_tricks.sliding_window_view(sym, k) if sym.size >= k else np.zeros((0, k), np.uint8)
    win = win[(win <= 3).all(axis=1)]
    if canon:
        rc = 3 - win[:, ::-1]
        diff = win != rc
        at = diff.argmax(axis=1)
        rows = np.arange(win.shape[0])
        win = np.where((rc[rows, at] < win[rows, at])[:, None], rc, win)
    return np.unique(np.ascontiguousarray(win).view(np.dtype((np.void, k))).reshape(-1))


def hist_of(regs) -> np.ndarray:
    """int64 [..., 64]: the register histogram of every row of regs [..., 2^p] (values clamped at 63)."""
    regs = np.asarray(regs)
    flat = regs.reshape(-1, regs.shape[-1])
    out = np.stack([np.bincount(np.minimum(r, BINS - 1), minlength=BINS) for r in flat]) if flat.shape[0] else np.zeros((0, BINS))
    return out.reshape(tuple(regs.shape[:-1]) + (BINS,)).astype(np.int64)


def dense_rule(regs, union, uhist, cand):
    """K11 dense step.  (hist [C, nk, 64], live [C, nk]): hist(U) plus -1 at U[j] and +1 at g[j] for every register
    where g > U."""
    regs, union = np.asarray(regs).astype(np.int64), np.asarray(union).astype(np.int64)
    nk = union.shape[0]
    hist = np.zeros((len(cand), nk, BINS), dtype=np.int64)
    live = np.zeros((len(cand), nk), dtype=np.int64)
    for c, g in enumerate(cand):
        for k in range(nk):
            up = regs[g, k] > union[k]
            hist[c, k] = uhist[k]
            np.subtract.at(hist[c, k], union[k][up], 1)
            np.add.at(hist[c, k], regs[g, k][up], 1)
            live[c, k] = up.sum()
    return hist, live


def compact_rule(regs, union, cand, seg_off):
    """K11 compaction.  The sparse state: entries `j << 6 | value` of every live register in segment g * nk + k, within
    capacity."""
    regs, union = np.asarray(regs).astype(np.int64), np.asarray(union).astype(np.int64)
    n, nk, _ = regs.shape
    seg_off = np.asarray(seg_off, dtype=np.int64)
    entries = np.zeros(int(seg_off[-1]), dtype=np.int64)
    seg_len = np.zeros(n * nk, dtype=np.int64)
    for g in cand:
        for k in range(nk):
            s = g * nk + k
            j = np.nonzero(regs[g, k] > union[k])[0]
            cap = seg_off[s + 1] - seg_off[s]
            entries[seg_off[s]:seg_off[s] + min(cap, j.size)] = ((j << 6) | regs[g, k][j])[:cap]
            seg_len[s] = j.size
    return {"entries": entries, "seg_off": seg_off, "seg_len": seg_len, "nk": nk}


def sparse_rule(state, union, uhist, cand):
    """K11 sparse step: drop the entries with value <= U[k][j], keep the rest in place, count their pairs."""
    union = np.asarray(union).astype(np.int64)
    nk = state["nk"]
    hist = np.zeros((len(cand), nk, BINS), dtype=np.int64)
    live = np.zeros((len(cand), nk), dtype=np.int64)
    for c, g in enumerate(cand):
        for k in range(nk):
            s = g * nk + k
            off = state["seg_off"][s]
            n_len = min(state["seg_len"][s], state["seg_off"][s + 1] - off)
            seg = state["entries"][off:off + n_len]
            v, j = seg & 63, seg >> 6
            keep = v > union[k][j]
            state["entries"][off:off + keep.sum()] = seg[keep]
            state["seg_len"][s] = live[c, k] = keep.sum()
            hist[c, k] = uhist[k]
            np.subtract.at(hist[c, k], union[k][j[keep]], 1)
            np.add.at(hist[c, k], v[keep], 1)
    return hist, live


def emit_rule(held, rng):
    """K12 emit.  The index of one part from its holder matrix held bool [keys, n], as K7 + K12 build it: genomes push
    one node per key they hold, one genome after another (in any order within a genome), and keys take ids in any
    order.  Returns {"offsets", "holders", "key_of_node", "node_start", "n_keys", "n_nodes", "covered"}."""
    n_keys, n = held.shape
    node_key, node_genome, node_start = [], [], [0]
    for g in range(n):
        keys = np.flatnonzero(held[:, g])
        node_key += rng.permutation(keys).tolist()
        node_genome += [g] * keys.size
        node_start.append(len(node_key))
    node_key, node_genome = np.asarray(node_key, dtype=np.int64), np.asarray(node_genome, dtype=np.int64)
    slot_to_id = rng.permutation(n_keys)                     # the reservation order of the occupied slots
    key_of_node = slot_to_id[node_key] if node_key.size else node_key
    order = np.argsort(key_of_node, kind="stable")
    counts = np.bincount(key_of_node, minlength=n_keys)
    offsets = np.concatenate([[0], np.cumsum(counts)])
    return {"offsets": offsets, "holders": node_genome[order], "key_of_node": key_of_node,
            "node_start": np.asarray(node_start, dtype=np.int64), "n_keys": n_keys, "n_nodes": node_key.size,
            "covered": np.zeros(n_keys, dtype=bool)}


def step_rule(part, genome, lost):
    """K12 step.  Genome `genome` joins the union: its keys not covered yet are covered, and each adds 1 to lost[h] of
    every holder h."""
    for node in range(part["node_start"][genome], part["node_start"][genome + 1]):
        key = part["key_of_node"][node]
        if part["covered"][key]:
            continue
        part["covered"][key] = True
        for h in part["holders"][part["offsets"][key]:part["offsets"][key + 1]]:
            lost[h] += 1


def brute_hist(regs, group, n_groups, begin=0, end=None):
    """K10.  int64 [nk, 1 + G, 64]: row 0 the histogram of the union of all genomes, row 1 + g of the union of every
    genome outside group g (explicit maxima; no genome left: all zeros), registers [begin, end) of every k."""
    regs = np.asarray(regs)[:, :, begin:end]
    group = np.asarray(group)
    n, nk, m = regs.shape
    out = np.zeros((nk, 1 + n_groups, BINS), dtype=np.int64)
    for g in range(-1, n_groups):
        keep = group != g
        u = regs[keep].max(axis=0) if keep.any() else np.zeros((nk, m), dtype=np.uint8)
        for c in range(nk):
            out[c, 1 + g] = np.bincount(np.minimum(u[c], BINS - 1), minlength=BINS)
    return out


def spectrum_numpy(regs, begin=0, end=None) -> np.ndarray:
    """K14.  int64 [nk, 64, n]: entry (k, v, c - 1) = registers of [begin, end) where exactly c genomes hold a value >= v
    (values clamped at 63), from regs [n, nk, 2^p]."""
    x = np.minimum(np.asarray(regs)[:, :, begin:end], BINS - 1).astype(np.int16)
    n, nk, _ = x.shape
    out = np.zeros((nk, BINS, n), dtype=np.int64)
    for k in range(nk):
        for v in range(1, BINS):
            c = (x[:, k, :] >= v).sum(axis=0)
            out[k, v] = np.bincount(c, minlength=n + 1)[1:]
    return out


def ertl_mle_float(c, p: int) -> float:
    """oracle/ref_numpy.ertl_mle_py with float counts: the same steps, every count a Python float."""
    q = 64 - p
    m = float(1 << p)
    c = [float(v) for v in c] + [0.0] * (q + 2 - len(c))
    if c[q + 1] == m:
        return math.inf
    kmin = next(j for j in range(q + 2) if c[j])
    kmax = next(j for j in range(q + 1, -1, -1) if c[j])
    kminp, kmaxp = max(1, kmin), min(q, kmax)
    z = 0.0
    for j in range(kmaxp, kminp - 1, -1):
        z = 0.5 * z + c[j]
    z = math.ldexp(z, -kminp)
    cp = c[q + 1] + (c[kmaxp] if q >= 1 else 0.0)
    a = z + c[0]
    mp_ = m - c[0]
    b = z + math.ldexp(c[q + 1], -q)
    x = mp_ / (0.5 * b + a) if b <= 1.5 * a else mp_ / b * math.log1p(b / a)
    gprev, dx, relerr = 0.0, x, 1e-2 / math.sqrt(m)
    while dx > x * relerr:
        kap = math.frexp(x)[1]
        xp = math.ldexp(x, -max(kmaxp + 1, kap + 2))
        xp2 = xp * xp
        h = xp - xp2 / 3.0 + (xp2 * xp2) * (1.0 / 45.0 - xp2 / 472.5)
        for _ in range(kap, kmaxp - 1, -1):
            hp = 1.0 - h
            h = (xp + h * hp) / (xp + hp)
            xp += xp
        g = cp * h
        for j in range(kmaxp - 1, kminp - 1, -1):
            hp = 1.0 - h
            h = (xp + h * hp) / (xp + hp)
            xp += xp
            g += c[j] * h
        g += x * a
        dx = dx * (g - mp_) / (gprev - g) if (gprev < g <= mp_) else 0.0
        x += dx
        gprev = g
    return x * m


def _i32(a) -> torch.Tensor:
    return torch.from_numpy(np.asarray(a).astype(np.int32))


# ---------------------------------------------------------------- the double
class FakeEngine:
    """Every list job (K7-K9, K12, K13) is read off one table of which genomes hold each distinct k-mer, from oracle k-mer
    sets; a job given a shard other than rank 0's returns zeros (the oracle has no key-range filter: rank 0 holds every
    key).  Records the calls per method (`calls`), the genome count of every per-union count (`union_sizes`) and the k
    of every family job (`family_ks`).  `passes`: key-range parts of each cover index."""
    polyt_sentinel = False
    fastq_to_fasta = staticmethod(Engine.fastq_to_fasta)        # host-side code of the real library
    passes = 1

    def __init__(self):
        self.device = torch.device("cpu")
        self.calls = Counter()
        self.union_sizes = []
        self.family_ks = []
        self._held = {}

    def bind_thread(self):
        pass

    def _pairs_budget(self):
        return 1 << 40

    # ------------------------------------------------ sketches and HLL unions
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

    def cards_hist(self, regs, p):
        h = _i32(hist_of(regs.numpy()))
        return self.mle(h, p), h

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
        flat = hist.reshape(-1, BINS).numpy()
        return torch.tensor([orc.ertl_mle(row.astype(np.uint32), p) for row in flat], dtype=torch.float64).view(hist.shape[:-1])

    def mle_f64(self, hist, p):
        flat = hist.reshape(-1, BINS).numpy()
        return torch.tensor([ertl_mle_float(row.tolist(), p) for row in flat], dtype=torch.float64).view(hist.shape[:-1])

    def leave_out_hist(self, regs, group, n_groups, p, reg_range=None, out=None):
        self.calls["leave_out_hist"] += 1
        begin, end = reg_range if reg_range is not None else (0, 1 << p)
        assert begin % 16 == 0 and end % 16 == 0
        got = _i32(brute_hist(regs.numpy(), group, n_groups, begin, end))
        return got if out is None else out.add_(got)

    def register_spectrum(self, regs, p, reg_range=None, out=None):
        self.calls["register_spectrum"] += 1
        begin, end = reg_range if reg_range is not None else (0, 1 << p)
        assert begin % 16 == 0 and end % 16 == 0 and regs.shape[2] == 1 << p
        got = _i32(spectrum_numpy(regs.numpy(), begin, end))
        return got if out is None else out.add_(got)

    def greedy_dense_hist(self, regs, union, union_hist, cand, p):
        self.calls["greedy_dense"] += 1
        h, live = dense_rule(regs.numpy(), union.numpy(), union_hist.numpy(), list(cand))
        return _i32(h), _i32(live)

    def greedy_compact(self, regs, union, cand, seg_off, p):
        self.calls["greedy_compact"] += 1
        return compact_rule(regs.numpy(), union.numpy(), list(cand), seg_off)

    def greedy_sparse_hist(self, state, union, union_hist, cand, p):
        self.calls["greedy_sparse"] += 1
        h, live = sparse_rule(state, union.numpy(), union_hist.numpy(), list(cand))
        return _i32(h), _i32(live)

    # ------------------------------------------------ exact k-mer sets
    def exact_counts(self, seqs, k, canon=True, capacity=None, shard=None):
        self.calls["exact_counts"] += 1
        self.union_sizes.append(len(seqs))
        if shard is not None and shard[0] != 0:
            return [0] * len(seqs)
        return [orc.exact_count([s.sym for s in seqs[:i + 1]], int(k), canon) for i in range(len(seqs))]

    def _holders(self, seqs, k, canon):
        """bool [distinct k-mers of seqs, n]: which genomes hold each k-mer.  Cached per (seqs, k, canon); the cache
        keeps the seqs, so their ids stay theirs."""
        key = (tuple(id(s) for s in seqs), int(k), bool(canon))
        if key not in self._held:
            sets = [kmer_keys(s.sym, int(k), canon) for s in seqs]
            keys, row = np.unique(np.concatenate(sets) if sets else np.zeros(0, np.uint64), return_inverse=True)
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

    def exact_query_counts(self, seqs, n_refs, k, canon, shard=None, passes=None):
        self.calls["exact_query_counts"] += 1
        R, Q = int(n_refs), len(seqs) - int(n_refs)
        assert R >= 1 and Q >= 1
        if shard is not None and shard[0] != 0:
            return np.zeros(R + Q, np.uint64), np.zeros((Q, R), np.uint64), np.zeros(Q, np.uint64), 0
        held = self._holders(seqs, k, canon).astype(np.uint64)
        in_refs = held[:, :R].max(axis=1)
        return held.sum(axis=0), held[:, R:].T @ held[:, :R], held[:, R:].T @ in_refs, int(in_refs.sum())

    def exact_cover_index(self, seqs, k, canon, shard=None, passes=None):
        self.calls["exact_cover_index"] += 1
        held = self._holders(seqs, k, canon)
        if shard is not None and shard[0] != 0:
            held = held[:0]
        rng = np.random.default_rng(int(k))
        parts = [emit_rule(held[np.arange(held.shape[0]) % self.passes == p], rng) for p in range(self.passes)]
        return {"k": int(k), "n": len(seqs), "parts": parts, "singles": held.sum(axis=0).astype(np.uint64),
                "keys": int(held.shape[0]), "bytes": int(6 * held.sum() + 5 * held.shape[0])}

    def exact_cover_step(self, indices, genome, lost):
        self.calls["exact_cover_step"] += 1
        view = lost.numpy()
        for c, ix in enumerate(indices):
            for part in ix["parts"]:
                step_rule(part, genome, view[c])
