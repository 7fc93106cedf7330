"""QueryFakeEngine: ListJobEngine plus the engine calls of `helpers/query.py`, for the CPU tests and as the CPU run the GPU
tests compare the helper against.  Engine.exact_query_counts is restated from Python k-mer sets; Engine.cards_hist and
Engine.greedy_dense_hist from explicit register maxima and the oracle MLE."""
import numpy as np
import torch

from oracle import pyoracle as orc
from tests.fake_engine import ListJobEngine

BINS = 64


def hist_of(regs: np.ndarray) -> np.ndarray:
    """int64 [..., 64]: the register histogram of every row of regs [..., 2^p]."""
    flat = np.asarray(regs).reshape(-1, regs.shape[-1])
    out = np.stack([np.bincount(np.minimum(r, BINS - 1), minlength=BINS) for r in flat]) if flat.shape[0] else np.zeros((0, BINS))
    return out.reshape(tuple(regs.shape[:-1]) + (BINS,)).astype(np.int64)


class QueryFakeEngine(ListJobEngine):

    def exact_query_counts(self, seqs, n_refs, k, canon, shard=None, passes=None):
        self.calls["exact_query_counts"] = self.calls.get("exact_query_counts", 0) + 1
        R, Q = int(n_refs), len(seqs) - int(n_refs)
        assert R >= 1 and Q >= 1
        if shard is not None and shard[0] != 0:      # (rank 0 holds every key, as in FakeEngine.exact_counts)
            return np.zeros(R + Q, np.uint64), np.zeros((Q, R), np.uint64), np.zeros(Q, np.uint64), 0
        sets = [set(orc.kmers(s.sym, int(k), canon).tolist()) for s in seqs]
        union = set().union(*sets[:R])
        inter = [[len(sets[R + q] & sets[r]) for r in range(R)] for q in range(Q)]
        shared = [len(sets[R + q] & union) for q in range(Q)]
        return (np.array([len(s) for s in sets], np.uint64), np.array(inter, np.uint64).reshape(Q, R),
                np.array(shared, np.uint64), len(union))

    def cards_hist(self, regs, p):
        h = torch.from_numpy(hist_of(regs.numpy()).astype(np.int32))
        return self.mle(h, p), h

    def greedy_dense_hist(self, regs, union, union_hist, cand, p):
        self.calls["greedy_dense"] = self.calls.get("greedy_dense", 0) + 1
        r, u = regs.numpy(), union.numpy()
        hist = np.stack([hist_of(np.maximum(u, r[g])) for g in cand])
        live = np.stack([(r[g] > u).sum(axis=-1) for g in cand])
        return torch.from_numpy(hist.astype(np.int32)), torch.from_numpy(live.astype(np.int32))
