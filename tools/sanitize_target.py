#!/usr/bin/env python
"""A small pass through every kernel family, for compute-sanitizer (SURVEY.md section 5):
    compute-sanitizer --tool memcheck  python tools/sanitize_target.py
    compute-sanitizer --tool racecheck python tools/sanitize_target.py
K1 (general + fast tiles, chunked), K2 (persistent small-k bitmap path, static k sets, generic mask,
floor schedule, the rank-1 sink kernel with and without a small-k launch beside it), finalize, K3 byte + bit-plane kernels with the identical-prefix table, K4, K5 (bitmap,
64-bit and 128-bit hash sets), K6, K7 lists with K8 first-rank histograms (shared and global counters), the
poly-T pass.  Results are compared with the oracle so that a
"clean" run is also a correct one."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pyoracle as orc  # noqa: E402
from tests.util import adversarial_fasta, kseq_fasta, mutate, random_bases, to_fasta  # noqa: E402


def main():
    import torch
    from dandd_b200.engine import Engine
    eng = Engine(0)
    rng = np.random.default_rng(0)
    txt = adversarial_fasta(rng, n=60000) + kseq_fasta(rng, n=40000) + to_fasta([(b"body", random_bases(rng, 200000))], width=80)
    sym = orc.fasta_symbols(txt)
    p = 12
    for chunk in (None, 16384 + 16):
        seq = eng.pack(txt, chunk_bytes=chunk)
        assert seq.nsym == sym.size
    for ks in ([2, 3, 5, 9, 10, 17, 32], list(range(10, 33)), list(range(2, 33)), list(range(1, 33))):
        regs, cards = eng.sketch(seq, ks, p=p)
        for i in (0, len(ks) - 1):
            assert np.array_equal(regs[i].cpu().numpy(), orc.hll_sketch(sym, ks[i], p)), ks[i]
    regs, _ = eng.sketch(seq, list(range(10, 33)), p=16)     # rank-1 sink: whole stream before the first cut
    assert np.array_equal(regs[0].cpu().numpy(), orc.hll_sketch(sym, 10, 16))
    assert np.array_equal(regs[22].cpu().numpy(), orc.hll_sketch(sym, 32, 16))
    regs, _ = eng.sketch(seq, list(range(2, 33)), p=8, ranges=[(0, 5000), (5000, sym.size)], floor_every=4096)   # floor path on
    assert np.array_equal(regs[10].cpu().numpy(), orc.hll_sketch(sym, 12, 8))
    hregs, hcards = eng.sketch_fasta_host(txt, [11, 21], p=p)
    assert np.array_equal(hregs[1], orc.hll_sketch(sym, 21, p))
    # K3 / K4 / K6
    anc = random_bases(rng, 30000)
    ks = [12, 20, 31]
    sk = torch.stack([eng.sketch(eng.pack(to_fasta([(b"g", mutate(rng, anc, sub=0.05))])), ks, p=p)[0] for _ in range(6)]).contiguous()
    h = sk.cpu().numpy()
    orders = [[0, 1, 2, 3, 4, 5], [5, 4, 3, 2, 1, 0], [2, -1, 2, 0, 1, 5], [0, 1, 2, 3, 4, 5]]
    a = eng.prefix_union_cards(sk, orders, p).cpu().numpy()
    b, un = eng.prefix_union_cards(sk, orders, p, materialize=True)
    assert np.allclose(a, b.cpu().numpy(), rtol=1e-12)
    assert np.array_equal(un[1, 5].cpu().numpy(), h.max(axis=0))
    planes = eng.to_planes(sk, p)
    pairs = [(x, y) for x in range(6) for y in range(x + 1, 6)]
    c = eng.pairwise_cards(None, pairs, p, planes=planes, n_genomes=6, nk=len(ks)).cpu().numpy()
    assert abs(c[0, 0] - orc.card(np.maximum(h[0, 0], h[1, 0]), p)) <= 1e-9 * c[0, 0]
    assert np.array_equal(eng.union([sk[i] for i in range(6)]).cpu().numpy(), h.max(axis=0))
    eng.cards(sk, p)
    # K5
    for k in (5, 12, 21, 32, 40, 64):
        got = eng.exact_counts([seq], k)
        assert got == [orc.exact_count([sym], k)] if k <= 32 else got[0] > 0, k
    # K7 lists + K8 first-rank histograms: prefix unions of two orderings and one set, on both counter paths
    texts = [to_fasta([(b"g", mutate(rng, anc, sub=0.05))]) for _ in range(4)]
    gseqs = [eng.pack(t) for t in texts]
    gsyms = [orc.fasta_symbols(t) for t in texts]
    ranks = np.array([[0, 1, 2, 3], [3, 2, 1, 0], [0, 0xFFFF, 0, 0xFFFF]], dtype=np.uint16)
    for k in (12, 21, 40):
        for reps in (1, 2000):   # 3 rows: counters in shared memory; 6000 rows: global atomics
            hist = eng.exact_first_rank_hist(gseqs, k, True, np.tile(ranks, (reps, 1)))[:3].astype(np.int64)
            if k <= 32:
                assert hist[0].cumsum().tolist() == [orc.exact_count(gsyms[:i + 1], k) for i in range(4)], k
                assert hist[1].cumsum()[-1] == orc.exact_count(gsyms, k) and hist[2, 0] == orc.exact_count(gsyms[::2], k), k
    # A.6 pass
    eng.polyt_sentinel = True
    t2 = to_fasta([(b"t", np.full(300, ord("T"), dtype=np.uint8))])
    s2 = eng.pack(t2)
    assert s2.nsym == 301
    eng.polyt_sentinel = False
    torch.cuda.synchronize()
    print("sanitize target: all paths ran and matched the oracle")


if __name__ == "__main__":
    main()
