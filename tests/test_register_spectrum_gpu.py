"""K14 (dd_register_spectrum) and dd_mle_from_hist_f64 on the device: the spectrum against torch counts bit for bit
on random and adversarial registers, both table placements, register ranges and repeated calls that add up; row m = n
against the K3 union and K4; the f64 MLE against the u32 one and against a float-count transcription of the oracle's
MLE; the command line on the real engine against oracle registers and against the exact mode's mean curve; refusals."""
import csv
import os

import numpy as np
import pytest
import torch

from tests.register_spectrum_engine import ertl_mle_float

pytestmark = pytest.mark.gpu
BINS = 64


@pytest.fixture(scope="module")
def eng():
    from dandd_b200.engine import get_engine
    return get_engine()


def brute(regs, begin=0, end=None):
    """int64 [nk, 64, n] on the device: registers of [begin, end) where exactly c genomes are >= v (clamped at 63)."""
    x = torch.clamp(regs[:, :, begin:end], max=BINS - 1)
    n, nk, _ = x.shape
    out = torch.zeros((nk, BINS, n), dtype=torch.int64, device=regs.device)
    rowid = torch.arange(nk, device=regs.device)[:, None] * (n + 1)
    for v in range(1, BINS):
        c = (x >= v).sum(dim=0)                                                  # [nk, m]
        out[:, v] = torch.bincount((rowid + c).flatten(), minlength=nk * (n + 1)).view(nk, n + 1)[:, 1:]
    return out


def make_regs(n, nk, p, seed, dev, kind="random"):
    g = torch.Generator(device=dev).manual_seed(seed)
    m, top = 1 << p, 64 - p + 1
    if kind == "zeros":
        return torch.zeros((n, nk, m), dtype=torch.uint8, device=dev)
    if kind == "equal":
        return torch.full((n, nk, m), 7, dtype=torch.uint8, device=dev)
    if kind == "saturated":
        return torch.full((n, nk, m), top, dtype=torch.uint8, device=dev)
    if kind == "clamped":                                   # bytes 0..255: values >= 64 count as 63
        return torch.randint(0, 256, (n, nk, m), generator=g, dtype=torch.uint8, device=dev)

    def geo(*shape):                                        # HLL ranks: P(x = j) = 2^-j, at most 64 - p + 1
        u = torch.rand(shape, generator=g, device=dev)
        return torch.clamp(torch.floor(-torch.log2(1.0 - u)) + 1, max=top).to(torch.uint8)
    # HLL-like: clusters of near-copies, exact duplicates, an all-zero genome and the largest value a register holds
    roots = geo(max(1, n // 8), nk, m)
    regs = roots[torch.randint(0, roots.shape[0], (n,), generator=g, device=dev)]
    change = torch.rand((n, nk, m), generator=g, device=dev) < 0.1
    regs = torch.where(change, geo(n, nk, m), regs)
    regs[torch.rand((n, nk, m), generator=g, device=dev) < 0.002] = top
    if n > 2:
        regs[n - 1] = regs[0]
        regs[n // 2] = 0
    return regs.contiguous()


# (n, nk, p): n <= 128 keeps the whole [64][n] table in shared memory, n >= 129 the c = n and c = 1 columns
SHAPES = [(1, 3, 12), (2, 2, 20), (3, 5, 14), (12, 23, 12), (13, 4, 20), (100, 3, 14), (128, 2, 12), (129, 2, 12),
          (1000, 2, 12), (1000, 1, 20), (1000, 3, 14)]


@pytest.mark.parametrize("n,nk,p", SHAPES)
def test_spectrum_equals_brute_force(eng, n, nk, p):
    regs = make_regs(n, nk, p, seed=n * 100 + nk * 10 + p, dev=eng.device)
    got = eng.register_spectrum(regs, p)
    want = brute(regs)
    assert torch.equal(got.long(), want)
    assert bool((got[:, 0] == 0).all())
    m = 1 << p
    cuts = [0, (m // 3) // 16 * 16, (2 * m // 3) // 16 * 16, m]              # three slices add up to the whole
    acc = torch.zeros_like(got)
    for b, e in zip(cuts, cuts[1:]):
        eng.register_spectrum(regs, p, reg_range=(b, e), out=acc)
        assert torch.equal(eng.register_spectrum(regs, p, reg_range=(b, e)).long(), brute(regs, b, e))
    assert torch.equal(acc, got)
    eng.register_spectrum(regs, p, out=acc)                                   # a repeated call adds again
    assert torch.equal(acc.long(), 2 * want)


@pytest.mark.parametrize("kind", ["zeros", "equal", "saturated", "clamped"])
@pytest.mark.parametrize("n,p", [(1, 12), (3, 14), (13, 12), (200, 12), (5, 20)])
def test_adversarial_registers(eng, kind, n, p):
    regs = make_regs(n, 2, p, seed=n + p, dev=eng.device, kind=kind)
    assert torch.equal(eng.register_spectrum(regs, p).long(), brute(regs))


@pytest.mark.parametrize("n,nk,p", [(1, 2, 12), (5, 3, 14), (13, 2, 20), (300, 2, 12)])
def test_last_row_is_the_union(eng, n, nk, p):
    """m = n: the mean histogram is the union's histogram (K3 + K4) and its card the union's, bit for bit; each row
    v of T sums to the union's registers >= v."""
    from dandd_b200 import store as ddstore
    regs = make_regs(n, nk, p, seed=7 * n + p, dev=eng.device)
    regs[0, 0, :5] = 200                                                      # clamped as hist_kernel clamps
    spec = eng.register_spectrum(regs, p)
    union = regs.amax(dim=0).contiguous()
    cards, hist = eng.cards_hist(union, p)
    ge = torch.flip(torch.cumsum(torch.flip(hist.long(), [1]), 1), [1])      # registers >= v
    assert torch.equal(spec.long().sum(dim=2)[:, 1:], ge[:, 1:])
    mean = ddstore.mean_prefix_hist(spec, p)
    assert torch.equal(mean[:, n - 1], hist.double())
    st = ddstore.GpuSketchStore(engine=eng)
    t, mean_cards = st.register_spectrum_cards(regs, p)
    assert np.array_equal(t, spec.long().cpu().numpy())
    assert np.array_equal(mean_cards[:, n - 1], cards.cpu().numpy())
    assert np.array_equal(mean_cards, eng.mle_f64(mean, p).cpu().numpy())


@pytest.mark.parametrize("p", [10, 14, 18])
def test_mle_f64_on_integer_histograms_is_the_u32_mle(eng, p):
    regs = make_regs(40, 3, p, seed=p, dev=eng.device)
    hist = eng.cards_hist(regs, p)[1].view(-1, BINS)
    extra = torch.zeros((3, BINS), dtype=torch.int32, device=eng.device)
    extra[0, 0] = 1 << p                                    # empty sketch
    extra[1, 64 - p + 1] = 1 << p                           # every register saturated
    extra[2, 1], extra[2, 0] = 1, (1 << p) - 1              # one register set
    hist = torch.cat([hist, extra]).contiguous()
    a = eng.mle(hist, p).cpu().numpy()
    b = eng.mle_f64(hist.double(), p).cpu().numpy()
    assert np.array_equal(a, b)
    assert a[-3] == 0.0 and np.isinf(a[-2])


@pytest.mark.parametrize("p", [10, 14, 20])
def test_mle_f64_on_fractional_histograms(eng, p):
    from dandd_b200 import store as ddstore
    regs = make_regs(9, 2, p, seed=p + 1, dev=eng.device)
    mean = ddstore.mean_prefix_hist(eng.register_spectrum(regs, p), p)
    rng = np.random.default_rng(p)
    noise = torch.as_tensor(rng.uniform(0.0, 3.0, (4, 20)), device=eng.device)          # odd fractions in bins 1..20
    extra = torch.zeros((4, BINS), dtype=torch.float64, device=eng.device)
    extra[:, 1:21] = noise
    extra[:, 0] = float(1 << p) - extra.sum(dim=1)
    hist = torch.cat([mean.view(-1, BINS), extra]).contiguous()
    got = eng.mle_f64(hist, p).cpu().numpy()
    for row, x in zip(hist.cpu().numpy(), got):
        assert x == pytest.approx(ertl_mle_float(row.tolist(), p), rel=1e-12)


def test_refusals_leave_the_table_alone(eng):
    from dandd_b200._lib import DandDError
    regs = make_regs(4, 2, 10, seed=4, dev=eng.device)
    out = torch.full((2, BINS, 4), 7, dtype=torch.int32, device=eng.device)
    before = eng.lib.dd_kernel_launches()
    for rng in [(8, 64), (0, 1040), (64, 32)]:
        with pytest.raises(DandDError, match="register range"):
            eng.register_spectrum(regs, 10, reg_range=rng, out=out)
    with pytest.raises(DandDError, match="p=4"):
        eng.register_spectrum(regs[:, :, :16].contiguous(), 4)
    torch.cuda.synchronize()
    assert eng.lib.dd_kernel_launches() == before
    assert bool((out == 7).all())


def _read_tsv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


def test_command_line_on_the_engine(tmp_path):
    """helpers/spectrum.py --tool dashing on synthetic FASTAs: T from the oracle's registers, the m = n card the
    oracle's union card; and on mutated copies of one ancestor the mean curve within 5 standard errors of the HLL
    (1.04 / sqrt(2^p)) of the exact mode's mean curve on the same FASTAs."""
    from dandd_b200 import store as ddstore
    from dandd_b200.helpers import spectrum
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    from tests.register_spectrum_engine import spectrum_numpy
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    n, p, lo, hi = 7, 14, 12, 18
    fastas = make_dataset(data, n, 30000, seed=21)
    st = ddstore.GpuSketchStore()
    ddstore.set_store(st)
    try:
        hll, exact = str(tmp_path / "hll"), str(tmp_path / "exact")
        spec, single, cards = spectrum.go(["-d", data, "--tool", "dashing", "--mink", str(lo), "--maxk", str(hi),
                                           "--registers", str(p), "--name", hll])
        spectrum.go(["-d", data, "--mink", str(lo), "--maxk", str(hi), "--name", exact])
    finally:
        ddstore.set_store(None)
    ks = list(range(lo, hi + 1))
    syms = [orc.fasta_symbols(_read_fasta(f)) for f in fastas]
    regs = np.stack([np.stack([orc.hll_sketch(s, k, p, True) for k in ks]) for s in syms])
    assert np.array_equal(spec, spectrum_numpy(regs))
    for c in range(len(ks)):                        # the oracle's MLE is the sequential form: rounding only
        assert cards[c, n - 1] == pytest.approx(orc.card(orc.union_max(list(regs[:, c])), p), rel=1e-9)
        assert single[:, c] == pytest.approx([orc.card(r, p) for r in regs[:, c]], rel=1e-9)
    got = {(r["k"], r["ngen"]): float(r["mean_card"]) for r in _read_tsv(os.path.join(hll, "growth.tsv"))}
    want = {(r["k"], r["ngen"]): float(r["mean_card"]) for r in _read_tsv(os.path.join(exact, "growth.tsv"))}
    assert got.keys() == want.keys() and len(got) == len(ks) * n
    tol = 5 * 1.04 / np.sqrt(1 << p)
    for key, x in got.items():
        assert abs(x - want[key]) <= tol * want[key], (key, x, want[key])
