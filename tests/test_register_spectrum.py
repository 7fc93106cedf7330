"""The HLL register sharing spectrum and its all-orderings mean growth curve (helpers/spectrum.py --tool dashing, K14) on
the CPU: hit_weights against mean_growth; the command line end to end through the real store on an engine double that
counts T with numpy from the oracle's registers, against brute-force averages over every m-subset of `np.maximum`
unions; refusals; the default tool's output unchanged; two gloo ranks; the ABI entries."""
import csv
import itertools
import os
import re
import socket

import numpy as np
import pytest

from dandd_b200 import store as ddstore
from dandd_b200.helpers import spectrum
from tests.fake_engine import ListJobEngine
from tests.register_spectrum_engine import BINS, RegisterSpectrumFakeEngine, ertl_mle_float, spectrum_numpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read_tsv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


def _parent_mean_growth(hist):
    """mean_growth as it stood before hit_weights was factored out of it, verbatim."""
    h = np.asarray(hist, dtype=np.float64)
    n = len(h)
    card, core = np.zeros(n), np.zeros(n)
    c = np.arange(n, dtype=np.float64)
    for m in range(1, n + 1):
        miss = np.concatenate([[1.0], np.maximum(np.cumprod((n - c[:-1] - m) / (n - c[:-1])), 0.0)])
        hit = np.cumsum(miss * (m / (n - c)))
        card[m - 1] = float(np.dot(h, hit))
        top = np.arange(n, m, -1, dtype=np.float64)
        hold = np.cumprod(np.concatenate([[1.0], (top - m) / top]))[::-1]
        core[m - 1] = float(np.dot(h[m - 1:], hold))
    return card, core


# ---------------------------------------------------------------- weights
@pytest.mark.parametrize("n", [1, 2, 3, 7, 30, 257, 1000])
def test_hit_weights_reproduce_mean_growth(n):
    rng = np.random.default_rng(n)
    w = spectrum.hit_weights(n)
    assert w.shape == (n, n) and w.dtype == np.float64
    assert np.all(w[:, n - 1] == 1.0)
    for hist in (rng.integers(0, 10 ** 6, n), rng.integers(0, 3, n)):
        card, core = spectrum.mean_growth(hist)
        want_card, want_core = _parent_mean_growth(hist)
        assert np.array_equal(card, want_card) and np.array_equal(core, want_core)       # bit for bit
    for c in sorted({1, n // 2 + 1, n}):                 # a unit spectrum reads one row of the weights, exactly
        unit = np.zeros(n, dtype=np.int64)
        unit[c - 1] = 1
        assert np.array_equal(spectrum.mean_growth(unit)[0], w[c - 1])


# ---------------------------------------------------------------- the mean histogram
def _brute_mean_hist(regs, m):
    """float64 [nk, 64]: the histogram of max over an m-subset, averaged over every m-subset (integer sums, one
    division)."""
    n, nk, _ = regs.shape
    total = np.zeros((nk, BINS), dtype=np.int64)
    subsets = list(itertools.combinations(range(n), m))
    for s in subsets:
        u = np.minimum(regs[list(s)].max(axis=0), BINS - 1)
        for k in range(nk):
            total[k] += np.bincount(u[k], minlength=BINS)
    return total / len(subsets)


def _assert_bins_close(got, want, p):
    # relative per bin; a bin whose true mean is 0 is the difference of two means of up to 2^p registers
    assert np.all(np.abs(got - want) <= 1e-12 * np.maximum(want, 1.0) + 4 * 2.0 ** -52 * 2 ** p), np.abs(got - want).max()


@pytest.mark.parametrize("n", [1, 2, 5, 9])
def test_mean_histogram_equals_the_average_over_every_subset(n):
    import torch
    p = 8
    rng = np.random.default_rng(40 + n)
    regs = rng.geometric(0.45, (n, 3, 1 << p)).astype(np.uint8)
    regs[:, 1] = np.minimum(regs[:, 1], 2)                    # many ties
    regs[0, 2, :7] = 80                                       # values >= 64 are clamped
    spec = torch.from_numpy(spectrum_numpy(regs))
    assert np.array_equal(spec[:, 1:].sum(axis=2).numpy(),
                          [[(np.minimum(regs[:, k].max(axis=0), 63) >= v).sum() for v in range(1, BINS)] for k in range(3)])
    hist = ddstore.mean_prefix_hist(spec, p).numpy()
    assert hist.shape == (3, n, BINS)
    for m in range(1, n + 1):
        _assert_bins_close(hist[:, m - 1], _brute_mean_hist(regs, m), p)
    union = np.minimum(regs.max(axis=0), 63)
    assert np.array_equal(hist[:, n - 1], [np.bincount(u, minlength=BINS) for u in union])    # m = n: the union, exactly


# ---------------------------------------------------------------- the command line
def _run(argv, engine=RegisterSpectrumFakeEngine):
    st = ddstore.GpuSketchStore(engine=engine())
    ddstore.set_store(st)
    try:
        return spectrum.go(argv), st
    finally:
        ddstore.set_store(None)


def _syms(fastas):
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    return [orc.fasta_symbols(_read_fasta(f)) for f in fastas]


@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
def test_dashing_against_oracle_registers(tmp_path, canon):
    from oracle import pyoracle as orc
    from tests.util import make_dataset
    p, n = 10, 6
    fastas = make_dataset(str(tmp_path / "data"), n, 1500, seed=8)
    names = [os.path.basename(f) for f in fastas]
    name = str(tmp_path / "run")
    argv = ["-d", str(tmp_path / "data"), "--tool", "dashing", "--mink", "4", "--maxk", "9", "--registers", str(p), "--name", name]
    if not canon:
        argv.append("--no-canon")
    (spec, single, cards), st = _run(argv)
    ks = list(range(4, 10))
    assert st.engine.calls["register_spectrum"] == 1 and spec.dtype == np.int64 and spec.shape == (len(ks), BINS, n)
    syms = _syms(fastas)
    regs = np.stack([np.stack([orc.hll_sketch(s, k, p, canon) for k in ks]) for s in syms])        # [n, nk, 2^p]
    assert np.array_equal(spec, spectrum_numpy(regs))
    hist = ddstore.mean_prefix_hist(__import__("torch").from_numpy(spec), p).numpy()
    for m in range(1, n + 1):
        _assert_bins_close(hist[:, m - 1], _brute_mean_hist(regs, m), p)
    for c in range(len(ks)):
        assert cards[c, n - 1] == orc.card(orc.union_max(list(regs[:, c])), p)                   # the union's card, exactly
        for m in range(n):
            assert cards[c, m] == pytest.approx(ertl_mle_float(hist[c, m].tolist(), p), rel=0, abs=0)
        assert single[:, c].tolist() == [orc.card(r, p) for r in regs[:, c]]
    assert np.all(np.diff(cards, axis=1) >= 0)                # the mean union only grows
    assert sorted(os.listdir(name)) == ["delta.tsv", "genomes.tsv", "growth.tsv", "registers.tsv"]
    rows = _read_tsv(os.path.join(name, "registers.tsv"))
    want = [(k, v, g + 1, int(spec[c, v, g])) for c, k in enumerate(ks) for v, g in zip(*np.nonzero(spec[c]))]
    assert [(int(r["k"]), int(r["value"]), int(r["genomes"]), int(r["registers"])) for r in rows] == want
    assert all(int(r["registers"]) > 0 and int(r["value"]) >= 1 for r in rows)
    rows = _read_tsv(os.path.join(name, "genomes.tsv"))
    assert [(int(r["k"]), r["name"]) for r in rows] == [(k, x) for k in ks for x in names]
    assert [r["card"] for r in rows] == [repr(float(single[g, c])) for c in range(len(ks)) for g in range(n)]
    rows = _read_tsv(os.path.join(name, "growth.tsv"))
    assert list(rows[0]) == ["k", "ngen", "mean_card", "mean_delta_pos"]
    assert [(int(r["k"]), int(r["ngen"])) for r in rows] == [(k, m) for k in ks for m in range(1, n + 1)]
    assert [r["mean_card"] for r in rows] == [repr(float(x)) for x in cards.reshape(-1)]
    assert [float(r["mean_delta_pos"]) for r in rows] == [float(cards[c, m]) / k for c, k in enumerate(ks) for m in range(n)]
    delta, best = spectrum.delta_of_mean(ks, cards)
    rows = _read_tsv(os.path.join(name, "delta.tsv"))
    assert [(int(r["ngen"]), r["delta"], int(r["k"])) for r in rows] == \
        [(m + 1, repr(float(d)), int(b)) for m, (d, b) in enumerate(zip(delta, best))]


def test_dashing_identical_genomes(tmp_path):
    """Three copies of one FASTA: every register has one level with c = n, so every mean histogram is the genome's own
    and every mean card its card."""
    from oracle import pyoracle as orc
    from tests.util import make_dataset
    data = tmp_path / "data"
    src = make_dataset(str(data), 1, 3000, seed=4)[0]
    for i in (1, 2):
        (data / ("g%d.fasta" % i)).write_bytes(open(src, "rb").read())
    (spec, single, cards), _ = _run(["-d", str(data), "--tool", "dashing", "--mink", "5", "--maxk", "7", "--registers", "9",
                                     "--name", str(tmp_path / "run")])
    assert np.all(spec[:, :, :2] == 0)
    for c, k in enumerate([5, 6, 7]):
        own = orc.card(orc.hll_sketch(_syms([src])[0], k, 9, True), 9)
        assert cards[c].tolist() == [own] * 3 and single[:, c].tolist() == [own] * 3


# ---------------------------------------------------------------- refusals and the default tool
@pytest.mark.parametrize("argv,match", [
    (["--maxk", "33"], "--maxk 33 is outside 1..32 for dashing"),
    (["--mink", "0"], "--mink 0 is outside 1..32 for dashing"),
    (["--registers", "4"], "--registers 4 is outside 5..26"),
    (["--registers", "27"], "--registers 27 is outside 5..26"),
    ([], None),
])
def test_refusals(tmp_path, argv, match):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 2, 800, seed=2)
    name = str(tmp_path / "run")
    if match is None:                                        # an existing --name
        os.makedirs(name)
        with pytest.raises(RuntimeError, match="already exists"):
            _run(["-d", data, "--tool", "dashing", "--name", name])
        return
    with pytest.raises(RuntimeError, match=match):
        _run(["-d", data, "--tool", "dashing", "--name", name] + argv)
    assert not os.path.exists(name)


def test_kmc_takes_k_above_32_and_ignores_registers(tmp_path):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 2, 800, seed=2)
    engine = ListJobEngine.only("exact_spectrum")
    _run(["-d", data, "--mink", "40", "--maxk", "41", "--registers", "4", "--name", str(tmp_path / "run")], engine=engine)
    assert sorted(os.listdir(str(tmp_path / "run"))) == ["delta.tsv", "genomes.tsv", "growth.tsv", "spectrum.tsv"]


def test_default_tool_is_the_exact_one(tmp_path):
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    fastas = make_dataset(data, 4, 1500, seed=6)
    engine = ListJobEngine.only("exact_spectrum")
    common = ["-d", data, "--mink", "3", "--maxk", "8", "--no-canon"]
    plain, kmc, direct = str(tmp_path / "plain"), str(tmp_path / "kmc"), str(tmp_path / "direct")
    _run(common + ["--name", plain], engine=engine)
    _run(common + ["--tool", "kmc", "--name", kmc], engine=engine)
    os.makedirs(direct)
    st = ddstore.GpuSketchStore(engine=engine())
    hist, singles, priv = st.exact_spectrum(sorted(fastas), list(range(3, 9)), False)
    spectrum.write_outputs(direct, [os.path.basename(f) for f in sorted(fastas)], list(range(3, 9)), hist, singles, priv)
    for fn in ("spectrum.tsv", "genomes.tsv", "growth.tsv", "delta.tsv"):
        text = open(os.path.join(plain, fn), "rb").read()
        assert text == open(os.path.join(kmc, fn), "rb").read() == open(os.path.join(direct, fn), "rb").read(), fn
    assert sorted(os.listdir(plain)) == ["delta.tsv", "genomes.tsv", "growth.tsv", "spectrum.tsv"]


# ---------------------------------------------------------------- two ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_worker(rank, world, port, argv):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    _run(argv)


def test_two_ranks_write_what_one_writes(tmp_path):
    import torch.multiprocessing as mp
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 5, 1200, seed=6)
    common = ["-d", data, "--tool", "dashing", "--mink", "3", "--maxk", "8", "--registers", "9"]
    two, one = str(tmp_path / "two"), str(tmp_path / "one")
    mp.spawn(_rank_worker, args=(2, _free_port(), common + ["--name", two]), nprocs=2, join=True)
    _run(common + ["--name", one])
    for fn in ("registers.tsv", "genomes.tsv", "growth.tsv", "delta.tsv"):
        assert open(os.path.join(two, fn), "rb").read() == open(os.path.join(one, fn), "rb").read(), fn


# ---------------------------------------------------------------- ABI
def test_entries_are_declared():
    from dandd_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dandd_b200.h")).read()
    assert re.search(r"DD_API\s+int\s+dd_register_spectrum\s*\(", header)
    assert re.search(r"DD_API\s+size_t\s+dd_register_spectrum_workspace_bytes\s*\(", header)
    assert re.search(r"DD_API\s+int\s+dd_mle_from_hist_f64\s*\(", header)
    assert len(_lib.SIGNATURES["dd_register_spectrum"][1]) == 10
    assert len(_lib.SIGNATURES["dd_register_spectrum_workspace_bytes"][1]) == 2
    assert len(_lib.SIGNATURES["dd_mle_from_hist_f64"][1]) == 5
    integration = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert re.search(r"\| `dd_register_spectrum_workspace_bytes`, `dd_register_spectrum` \|", integration)
    assert re.search(r"\| `dd_mle_from_hist_f64` \|", integration)
    assert _lib.ABI_VERSION == 2


def test_entries_are_exported_and_check_arguments():
    """Arguments refused before any CUDA call (these run without a device)."""
    import subprocess
    from dandd_b200 import build, _lib
    build.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(ROOT, "dandd_b200", "libdandd_b200.so")], text=True)
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    assert {"dd_register_spectrum", "dd_register_spectrum_workspace_bytes", "dd_mle_from_hist_f64"} <= exported
    lib = _lib.load()
    ws = lib.dd_register_spectrum_workspace_bytes(3, 2)
    assert ws == 2 * 64 * 3 * 4
    assert lib.dd_register_spectrum_workspace_bytes(0, 2) == 0 and lib.dd_register_spectrum_workspace_bytes(65536, 1) == 0
    assert lib.dd_register_spectrum_workspace_bytes(3, 0) == 0
    before = lib.dd_kernel_launches()
    R, S, W = 1 << 20, 1 << 21, 1 << 22                       # (never dereferenced: every call below is refused)

    def call(regs=R, n=3, nk=2, p=10, b=0, e=1024, spec=S, wsp=W, wsb=ws):
        return lib.dd_register_spectrum(regs, n, nk, p, b, e, spec, wsp, wsb, None)

    assert call(regs=None) == -1 and call(spec=None) == -1 and call(wsp=None) == -1
    assert call(p=4) == -1 and call(p=27) == -1
    assert call(nk=0) == -1 and call(nk=65536) == -1
    assert call(n=0) == -1 and call(n=65536) == -1 and b"n_genomes" in lib.dd_last_error()
    assert call(nk=40000, n=1000) == -1 and b"too many" in lib.dd_last_error()
    assert call(b=8) == -1 and call(e=1000) == -1 and call(e=1040) == -1 and call(b=32, e=16) == -1
    assert b"register range" in lib.dd_last_error()
    assert call(regs=R + 8) == -1 and call(spec=S + 2) == -1 and call(wsp=W + 2) == -1
    assert call(wsb=ws - 1) == -3
    assert lib.dd_mle_from_hist_f64(None, 2, 10, 1 << 20, None) == -1
    assert lib.dd_mle_from_hist_f64(1 << 20, 2, 4, 1 << 21, None) == -1
    assert lib.dd_mle_from_hist_f64(1 << 20, -1, 10, 1 << 21, None) == -1
    assert lib.dd_mle_from_hist_f64(None, 0, 10, None, None) == 0
    assert lib.dd_kernel_launches() == before
