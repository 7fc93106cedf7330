"""K2 rank-1 sink (-m gpu): pieces before the first floor cut sketch their k >= 10 with one k per CTA and
absorb rank-1 updates in a shared-memory bitmap; every register reads max(accumulator, bit).  Each case
is checked against the oracle and between dd_set_option("sketch_sink") on and off."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from oracle import pyoracle as orc
from tests.util import mutate, random_bases, to_fasta

pytestmark = pytest.mark.gpu
THREADS = max(1, min(32, (os.cpu_count() or 2) - 1))


@pytest.fixture(scope="module")
def eng():
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    return Engine(0)


def set_sink(eng, on):
    from dandd_b200._lib import check
    check(eng.lib.dd_set_option(b"sketch_sink", int(on)), "dd_set_option")


def sketch_both(eng, seq, ks, p, canon=True):
    """(regs, cards) with the sink on and with it off, on the host."""
    out = []
    for on in (1, 0):
        set_sink(eng, on)
        try:
            regs, cards = eng.sketch(seq, ks, p=p, canon=canon)
            out.append((regs.cpu().numpy(), cards.cpu().numpy()))
        finally:
            set_sink(eng, 1)
    return out


def oracle_regs(sym, ks, p, canon=True):
    with ThreadPoolExecutor(THREADS) as ex:
        return list(ex.map(lambda k: orc.hll_sketch(sym, k, p, canon), ks))


def genome(seed, n):
    rng = np.random.default_rng(seed)
    return to_fasta([(b"g", mutate(rng, random_bases(rng, n)))], width=80)


@pytest.mark.parametrize("canon", [True, False])
def test_config2_genome_every_k(eng, canon):
    """A config-2 genome (5 Mbp, p = 20, k = 10..32): registers bit-exact, histograms and cardinalities equal."""
    txt = genome(7, 5_000_000)
    ks = list(range(10, 33))
    want = oracle_regs(orc.fasta_symbols(txt), ks, 20, canon)
    (r_on, c_on), (r_off, c_off) = sketch_both(eng, eng.pack(txt), ks, 20, canon)
    assert np.array_equal(r_on, r_off)
    assert np.array_equal(c_on, c_off)
    for i, k in enumerate(ks):
        assert np.array_equal(r_on[i], want[i]), (k, canon)
        assert np.array_equal(orc.hist(r_on[i], 20), orc.hist(want[i], 20)), k


@pytest.mark.parametrize("p", [12, 16, 18, 20, 21])
def test_precisions(eng, p):
    """p = 20 is the largest bitmap; p = 21 takes the plain kernel and must be exact as well."""
    txt = genome(100 + p, 3_000_000)
    ks = list(range(10, 33))
    check_ks = [10, 11, 16, 17, 21, 31, 32]
    want = oracle_regs(orc.fasta_symbols(txt), check_ks, p)
    (r_on, c_on), (r_off, c_off) = sketch_both(eng, eng.pack(txt), ks, p)
    assert np.array_equal(r_on, r_off)
    assert np.array_equal(c_on, c_off)
    for k, w in zip(check_ks, want):
        assert np.array_equal(r_on[k - 10], w), (k, p)


@pytest.mark.parametrize("canon", [True, False])
def test_mixed_small_and_large_k(eng, canon):
    """k = 2..32 in one call: the presence-bitmap kernel takes k <= 9, the sink k >= 10, one workspace."""
    txt = genome(11, 2_000_000)
    ks = list(range(2, 33))
    check_ks = [2, 5, 9, 10, 12, 20, 32]
    want = oracle_regs(orc.fasta_symbols(txt), check_ks, 16, canon)
    (r_on, _), (r_off, _) = sketch_both(eng, eng.pack(txt), ks, 16, canon)
    assert np.array_equal(r_on, r_off)
    for k, w in zip(check_ks, want):
        assert np.array_equal(r_on[k - 2], w), (k, canon)


def _raw_ws(eng, nk, p):
    wsb = eng.lib.dd_sketch_workspace_bytes(nk, p)
    return torch.empty(wsb, dtype=torch.uint8, device=eng.device), wsb


def _sched(eng, seq, ws, wsb, begin, end, seen_before, kmask, p, canon=1):
    from dandd_b200._lib import check
    check(eng.lib.dd_sketch_update_sched(seq.codes.data_ptr(), seq.invalid.data_ptr(), None, begin, end, 0, seen_before, kmask, p,
                                         canon, ws.data_ptr(), wsb, eng.stream), "dd_sketch_update_sched")


def _end(eng, ws, wsb, nk, p):
    from dandd_b200._lib import check
    regs = torch.empty((nk, 1 << p), dtype=torch.uint8, device=eng.device)
    check(eng.lib.dd_sketch_end(ws.data_ptr(), wsb, nk, p, regs.data_ptr(), None, None, eng.stream), "dd_sketch_end")
    return regs.cpu().numpy()


def test_floor_refresh_sees_the_sink_bits(eng):
    """p = 12, 100 k symbols: the first cut (65 536) falls inside the call, so one refresh publishes the
    floors of the first 65 536 symbols -- computed from max(accumulator, bit).  A register that holds only
    rank-1 hits lives in the sink alone; without the bits that k's floor would read 0."""
    from dandd_b200._lib import check
    p, n, cut = 12, 100_000, 16 << 12
    ks = list(range(10, 33))
    kmask = sum(1 << (k - 1) for k in ks)
    for seed in range(40):       # a seed where some k's first-cut sketch has min(register) = 1
        rng = np.random.default_rng(seed)
        txt = to_fasta([(b"c", random_bases(rng, n))], width=80)
        sym = orc.fasta_symbols(txt)
        first = oracle_regs(sym[:cut], ks, p)
        mins = [int(r.min()) for r in first]
        if 1 in mins:
            break
    assert 1 in mins
    seq = eng.pack(txt)
    ws, wsb = _raw_ws(eng, len(ks), p)
    check(eng.lib.dd_sketch_begin(ws.data_ptr(), wsb, len(ks), p, eng.stream), "dd_sketch_begin")
    _sched(eng, seq, ws, wsb, 0, sym.size, 0, kmask, p)
    regs = _end(eng, ws, wsb, len(ks), p)
    floors = ws[:32].cpu().numpy()
    want = oracle_regs(sym, ks, p)
    for i, k in enumerate(ks):
        assert int(floors[k - 1]) == mins[i], k
        assert np.array_equal(regs[i], want[i]), k


def test_successive_sched_calls_share_the_sink(eng):
    """Three calls before the first cut (p = 18: 4.2 M symbols) with seen_before > 0 into one workspace, so
    the workspace bitmap collects bits across calls, then one call across the cut."""
    from dandd_b200._lib import check
    p = 18
    txt = genome(5, 6_000_000)
    sym = orc.fasta_symbols(txt)
    seq = eng.pack(txt)
    ks = list(range(10, 33))
    kmask = sum(1 << (k - 1) for k in ks)
    cuts = [0, 1_300_000, 2_700_000, 4_000_000, sym.size]
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
    check_ks = [10, 14, 21, 32]
    for k, w in zip(check_ks, oracle_regs(sym, check_ks, p)):
        assert np.array_equal(out[0][k - 10], w), k


def test_host_buffer_over_32_mib(eng):
    """dd_sketch_fasta_host on 40 Mbp at p = 16: 32 MiB text chunks, the first cut inside the first chunk."""
    txt = genome(9, 40_000_000)
    sym = orc.fasta_symbols(txt)
    ks = list(range(10, 33))
    got = []
    for on in (1, 0):
        set_sink(eng, on)
        try:
            got.append(eng.sketch_fasta_host(txt, ks, p=16))
        finally:
            set_sink(eng, 1)
    assert np.array_equal(got[0][0], got[1][0])
    assert np.array_equal(got[0][1], got[1][1])
    check_ks = [10, 13, 21, 32]
    for k, w in zip(check_ks, oracle_regs(sym, check_ks, 16)):
        assert np.array_equal(got[0][0][k - 10], w), k


@pytest.mark.parametrize("kind", ["empty", "all_n", "short"])
def test_degenerate_streams(eng, kind):
    """No symbols; only breaks; and a stream whose text is long (the grid is sized from the text bytes, so
    the sink runs) but whose few symbols fill less than one CTA's slice."""
    rng = np.random.default_rng(3)
    if kind == "empty":
        txt = b">e\n"
    elif kind == "all_n":
        txt = to_fasta([(b"n", np.full(200_000, ord("N"), dtype=np.uint8))], width=80)
    else:
        txt = b">" + b"h" * 400_000 + b"\n" + to_fasta([(b"s", random_bases(rng, 3000))], width=80)
    ks = list(range(2, 33))
    sym = orc.fasta_symbols(txt)
    (r_on, c_on), (r_off, c_off) = sketch_both(eng, eng.pack(txt), ks, 12)
    assert np.array_equal(r_on, r_off)
    assert np.array_equal(c_on, c_off)
    for k, w in zip(ks, oracle_regs(sym, ks, 12)):
        assert np.array_equal(r_on[k - 2], w), k
