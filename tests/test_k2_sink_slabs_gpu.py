"""K2 rank-1 sink slabs and the all-valid warp path (-m gpu): each sink CTA stores its bitmap to its own slab,
a later launch into the same workspace starts from it, and finalize ORs a k's slabs.  Warps whose 32 words hold
no break take an unrolled symbol loop; all others the per-symbol path.  Every case is checked against the
oracle and between dd_set_option("sketch_sink") on and off."""
import numpy as np
import pytest
import torch

from oracle import pyoracle as orc
from tests.test_k2_sink_gpu import _end, _raw_ws, _sched, oracle_regs, set_sink, sketch_both
from tests.util import random_bases, to_fasta

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    return Engine(0)


def sink_slices(nk_sink):
    """CTAs per k of a p = 20 sink launch: one 128 KiB bitmap per SM, the SMs shared among the k values."""
    return max(1, torch.cuda.get_device_properties(0).multi_processor_count // nk_sink)


def broken_genome(seed, n, nk_sink):
    """n bases in one record with N runs (symbol = base index + 1, after the record's break) at code-word edges,
    at the sink's slice edges and inside warp tiles, and a second record (one more break) near the middle."""
    rng = np.random.default_rng(seed)
    s = random_bases(rng, n).copy()
    slices = sink_slices(nk_sink)
    per = -(-((n + 2 + 15) // 16) // slices)           # words per slice of the whole stream
    breaks = []
    for c in range(1, slices):                          # slice edges, and a symbol either side
        breaks += [c * per * 16 + d for d in (-1, 0, 1)]
    for t in range(0, n, 37 * 512):                     # one warp tile (512 symbols) in 37: word edges and inside
        breaks.append(t + int(rng.choice([0, 15, 16, 17, 100 + int(rng.integers(0, 300))])))
    for b in breaks:
        if 1 <= b <= n:
            run = int(rng.integers(1, 40))
            s[b - 1:min(n, b - 1 + run)] = ord("N")
    half = n // 2
    return to_fasta([(b"a", s[:half]), (b"b", s[half:])], width=80)


@pytest.mark.parametrize("canon", [True, False])
def test_breaks_at_word_slice_and_tile_edges(eng, canon):
    """p = 20, k = 10..32: all-valid and per-symbol warps in one launch give the oracle's registers."""
    ks = list(range(10, 33))
    txt = broken_genome(21, 4_000_000, len(ks))
    sym = orc.fasta_symbols(txt)
    assert (sym == 4).sum() > 1000
    want = oracle_regs(sym, ks, 20, canon)
    (r_on, c_on), (r_off, c_off) = sketch_both(eng, eng.pack(txt), ks, 20, canon)
    assert np.array_equal(r_on, r_off)
    assert np.array_equal(c_on, c_off)
    for i, k in enumerate(ks):
        assert np.array_equal(r_on[i], want[i]), (k, canon)


@pytest.mark.parametrize("pieces", [2, 3])
def test_successive_sink_launches_accumulate_in_the_slabs(eng, pieces):
    """p = 20: 2 or 3 scheduled calls into one workspace, each long enough for the sink (slices x 2^18 symbols)
    and all before the first cut, so every launch after the first starts from the slabs of the one before."""
    from dandd_b200._lib import check
    p = 20
    ks = list(range(10, 33))
    kmask = sum(1 << (k - 1) for k in ks)
    rng = np.random.default_rng(30 + pieces)
    txt = to_fasta([(b"g", random_bases(rng, 5_000_000))], width=80)
    sym = orc.fasta_symbols(txt)
    assert sym.size // pieces >= sink_slices(len(ks)) << (p - 2)
    cuts = [sym.size * i // pieces for i in range(pieces + 1)]
    seq = eng.pack(txt)
    out = []
    for on in (1, 0):
        set_sink(eng, on)
        try:
            ws, wsb = _raw_ws(eng, len(ks), p)
            check(eng.lib.dd_sketch_begin(ws.data_ptr(), wsb, len(ks), p, eng.stream), "dd_sketch_begin")
            for b, e in zip(cuts, cuts[1:]):
                _sched(eng, seq, ws, wsb, b, e, b, kmask, p)
            out.append(_end(eng, ws, wsb, len(ks), p))
        finally:
            set_sink(eng, 1)
    assert np.array_equal(out[0], out[1])
    for i, w in enumerate(oracle_regs(sym, ks, p)):
        assert np.array_equal(out[0][i], w), ks[i]


def test_eleven_k_values(eng):
    """k = 10..20 at p = 20: another slice count than the 23 k of the benchmark."""
    ks = list(range(10, 21))
    assert sink_slices(len(ks)) != sink_slices(23)
    txt = broken_genome(22, 4_000_000, len(ks))
    want = oracle_regs(orc.fasta_symbols(txt), ks, 20)
    (r_on, c_on), (r_off, c_off) = sketch_both(eng, eng.pack(txt), ks, 20)
    assert np.array_equal(r_on, r_off)
    assert np.array_equal(c_on, c_off)
    for i, k in enumerate(ks):
        assert np.array_equal(r_on[i], want[i]), k
