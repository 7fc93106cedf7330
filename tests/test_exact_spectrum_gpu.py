"""K9 on the device: the exact sharing spectrum over the K7 lists (dandd_b200.engine exact_spectrum) against oracle k-mer
sets -- histogram of sharing counts, private counts, singles; passes and shards; both counter placements; overflow;
n = 2 against K7; and growth.tsv against `progressive --ksweep` over all n! orderings on the real engine."""
import csv
import itertools
import math
import os
import pickle
import random

import numpy as np
import pytest

from tests.test_exact_pairs_gpu import _genomes
from tests.test_exact_sets_gpu import _holders

pytestmark = pytest.mark.gpu

KS = [1, 5, 12, 16, 17, 31, 32, 33, 64, 65, 100, 256]


@pytest.fixture(scope="module")
def eng():
    from dandd_b200 import build
    build.build()
    from dandd_b200.engine import Engine
    return Engine(0)


@pytest.fixture(scope="module")
def packed(eng):
    texts = _genomes()
    return texts, [eng.pack(t).check() for t in texts]


def _want(held):
    """(hist, priv) of a [n_keys, n] holder matrix."""
    n = held.shape[1]
    c = held.sum(axis=1)
    hist = np.bincount(c, minlength=n + 1)[1:n + 1]
    priv = held[c == 1].sum(axis=0)
    return hist.tolist(), priv.tolist()


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("k", KS)
def test_spectrum_equals_the_oracle_sets(eng, packed, k, canon):
    """(k = 32 and 64 --no-canon: the poly-T runs make the all-ones key, which lives in the extra slot.  The genomes
    include an identical pair and one without k-mers above k = 4.)"""
    texts, seqs = packed
    held, singles = _holders(texts, k, canon)
    hist, got_singles, priv = eng.exact_spectrum(seqs, k, canon)
    assert hist.dtype == got_singles.dtype == priv.dtype == np.uint64 and hist.shape == (len(seqs),)
    want_hist, want_priv = _want(held)
    assert hist.astype(np.int64).tolist() == want_hist
    assert priv.astype(np.int64).tolist() == want_priv
    assert got_singles.astype(np.int64).tolist() == singles
    if k > 4:
        assert singles[5] == 0 and priv[0] == priv[4] == 0          # the empty genome; the identical pair


@pytest.mark.parametrize("k", [12, 33, 99])
def test_passes_and_shards_add_up(eng, packed, k):
    texts, seqs = packed
    one = eng.exact_spectrum(seqs, k, True, passes=1)
    for passes in (2, 3):
        got = eng.exact_spectrum(seqs, k, True, passes=passes)
        assert eng.last_pair_plan["passes"] == passes
        assert [a.tolist() for a in got] == [a.tolist() for a in one]
    parts = [eng.exact_spectrum(seqs, k, True, shard=(r, 2)) for r in range(2)]
    assert all(p[1].sum() > 0 for p in parts)                         # both halves hold keys
    assert [(a + b).tolist() for a, b in zip(*parts)] == [a.tolist() for a in one]
    held, singles = _holders(texts, k, True)
    assert one[0].astype(np.int64).tolist() == _want(held)[0] and one[1].astype(np.int64).tolist() == singles


@pytest.mark.parametrize("k", [9, 21, 70])
def test_shared_and_global_counters_agree(eng, packed, k):
    """Calling the ABI entry on one job's lists: n = 7 (shared memory, with and without the private counts) and the
    same genomes as the first 7 of n = 20000 (2n u32 > 96 KiB: global atomics; n alone = 78 KiB: shared again)."""
    import torch
    from dandd_b200._lib import check
    texts, seqs = packed
    want_hist, want_priv = _want(_holders(texts, k, True)[0])
    lib, st = eng.lib, eng.stream
    n, cap, nodes = len(seqs), 1 << 16, 40000
    ws = torch.empty(lib.dd_exact_pairs_workspace_bytes(k, cap, nodes, n), dtype=torch.uint8, device=eng.device)
    check(lib.dd_exact_pairs_begin(ws.data_ptr(), ws.numel(), k, cap, nodes, n, st))
    for g, s in enumerate(seqs):
        check(lib.dd_exact_pairs_insert_shard(s.codes.data_ptr(), s.invalid.data_ptr(), 0, s.nsym, k, 1, g, ws.data_ptr(),
                                              ws.numel(), cap, nodes, n, 0, 1, st))
    for width, with_priv in [(n, True), (n, False), (20000, True), (20000, False)]:
        out = torch.zeros(2 * width, dtype=torch.int64, device=eng.device)
        check(lib.dd_exact_occupancy_hist(ws.data_ptr(), ws.numel(), k, cap, nodes, n, width, out.data_ptr(),
                                          out.data_ptr() + 8 * width if with_priv else None, st))
        got = out.cpu().numpy()
        assert got[:n].tolist() == want_hist and not got[n:width].any()
        assert got[width:width + n].tolist() == (want_priv if with_priv else [0] * n) and not got[width + n:].any()
    # genome indices >= n_genomes are neither counted nor used as addresses: the first 3 genomes alone
    out = torch.zeros(6, dtype=torch.int64, device=eng.device)
    check(lib.dd_exact_occupancy_hist(ws.data_ptr(), ws.numel(), k, cap, nodes, n, 3, out.data_ptr(), out.data_ptr() + 24, st))
    want3 = _want(_holders(texts[:3], k, True)[0])
    assert out.cpu().tolist() == want3[0] + want3[1]


def test_pair_intersection_is_h2(eng, packed):
    texts, seqs = packed
    for k in (11, 21, 40, 90):
        for a, b in [(0, 1), (0, 4), (2, 3)]:
            inter = eng.exact_pairs_sparse([seqs[a], seqs[b]], k, True, _holders([texts[a], texts[b]], k, True)[1])
            assert int(eng.exact_spectrum([seqs[a], seqs[b]], k, True)[0][1]) == int(inter[0])


def test_overflow_raises(eng, packed):
    from dandd_b200._lib import DandDError
    from dandd_b200 import engine as E
    _, seqs = packed
    real = E.length_bounds
    E.length_bounds = lambda nsyms, k, world=1: [1] * len(nsyms)
    try:
        with pytest.raises(DandDError, match="overflow"):
            eng.exact_spectrum(seqs, 21, True)
    finally:
        E.length_bounds = real


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
def test_growth_equals_the_mean_over_all_orderings(tmp_path, canon):
    """The CPU test's comparison on the real engine: 5 genomes, every ordering through `progressive --ksweep`."""
    from dandd_b200 import store as ddstore
    from dandd_b200.helpers import spectrum
    from tests.host_harness import read_csv, run_dandd
    from tests.util import make_dataset
    tmp, ngen, lo, hi = str(tmp_path), 5, 3, 12
    data = os.path.join(tmp, "data")
    make_dataset(data, ngen, 3000, seed=31)
    flags = [] if canon else ["--no-canon"]
    with open(os.path.join(tmp, "all.pickle"), "wb") as fh:
        pickle.dump(set(itertools.permutations(range(ngen))), fh)
    st = ddstore.GpuSketchStore()
    ddstore.set_store(st)
    try:
        random.seed(3)
        run_dandd(["tree", "-d", data, "-s", "ex", "-o", os.path.join(tmp, "out"), "--exact"] + flags)
        run_dandd(["progressive", "-d", os.path.join(tmp, "out", "ex_%d_kmc_dtree.pickle" % ngen), "-o", os.path.join(tmp, "out"),
                   "--ksweep", "--mink", str(lo), "--maxk", str(hi), "-r", os.path.join(tmp, "all.pickle"), "-n", "120"])
        spectrum.go(["-d", data, "--mink", str(lo), "--maxk", str(hi), "--name", os.path.join(tmp, "spec")] + flags)
    finally:
        ddstore.set_store(None)
    summary = [f for f in os.listdir(os.path.join(tmp, "out")) if f.endswith("summary.csv")]
    sums = {}
    for row in read_csv(os.path.join(tmp, "out", summary[0])):
        sums.setdefault((int(row["ngen"]), int(row["kval"])), []).append(float(row["card"]))
    with open(os.path.join(tmp, "spec", "growth.tsv"), newline="") as fh:
        growth = list(csv.DictReader(fh, delimiter="\t"))
    assert len(growth) == ngen * (hi - lo + 1)
    for row in growth:
        cards = sums[(int(row["ngen"]), int(row["k"]))]
        assert len(cards) == math.factorial(ngen)
        assert float(row["mean_card"]) == pytest.approx(sum(cards) / len(cards), rel=1e-12)
