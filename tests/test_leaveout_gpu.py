"""K10 (dd_leave_out_hist) on the device: histograms against torch brute force bit for bit, register ranges that add
up, both counter placements, the cards against the per-union K3 path, refusals, and the leave-out command line on
the real engine against the per-union path and oracle k-mer sets."""
import csv
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
BINS = 64


@pytest.fixture(scope="module")
def eng():
    from dandd_b200.engine import get_engine
    return get_engine()


def make_regs(n, nk, p, seed, dev):
    """HLL-like registers, values 0 .. 64 - p + 1: clusters of near-copies (ties with the leader), exact duplicates
    and an all-zero genome."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    m = 1 << p
    top = 64 - p + 1
    geo = lambda *shape: torch.clamp(torch.distributions.Geometric(0.5).sample(shape).to(torch.int64) + 1, max=top)  # noqa: E731
    torch.manual_seed(seed)
    roots = geo(max(1, n // 8), nk, m)
    regs = roots[torch.randint(0, roots.shape[0], (n,), generator=g)].clone()
    change = torch.rand((n, nk, m), generator=g) < 0.1
    regs[change] = geo(int(change.sum()))
    regs[torch.rand((n, nk, m), generator=g) < 0.002] = top                   # the largest value a register can hold
    if n > 2:
        regs[n - 1] = regs[0]
        regs[n // 2] = 0
    return regs.to(torch.uint8).to(dev).contiguous()


def brute(regs, group, n_groups, begin=0, end=None):
    """int64 [nk, 1 + G, 64] by explicit maxima on the device."""
    regs = regs[:, :, begin:end]
    n, nk, m = regs.shape
    group = torch.as_tensor(group, device=regs.device)
    out = torch.zeros((nk, 1 + n_groups, BINS), dtype=torch.int64, device=regs.device)
    rowid = torch.arange(nk, device=regs.device)[:, None] * BINS
    for g in range(-1, n_groups):
        keep = group != g
        u = regs[keep].amax(dim=0) if bool(keep.any()) else torch.zeros((nk, m), dtype=torch.uint8, device=regs.device)
        out[:, 1 + g] = torch.bincount((rowid + u.long()).flatten(), minlength=nk * BINS).view(nk, BINS)
    return out


def groups_for(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "one":
        return np.zeros(n, dtype=np.int32), 1
    if kind == "two":
        g = rng.integers(0, 2, n).astype(np.int32)
        g[:2] = [1, 0]
        return g, 2
    if kind == "each":
        return rng.permutation(n).astype(np.int32), n
    G = int(rng.integers(1, n + 1))
    g = np.concatenate([np.arange(G), rng.integers(0, G, n - G)]).astype(np.int32)
    rng.shuffle(g)
    return g, G


# (n, nk, p): every n, nk and p of the checklist; G = n = 400 counts corrections by global atomics, the rest in
# shared memory
SHAPES = [(2, 31, 20), (3, 23, 18), (3, 1, 10), (40, 23, 14), (40, 1, 20), (400, 1, 18), (400, 31, 10), (400, 7, 14)]


@pytest.mark.parametrize("kind", ["one", "two", "each", "random"])
@pytest.mark.parametrize("n,nk,p", SHAPES)
def test_histograms_equal_brute_force(eng, n, nk, p, kind):
    regs = make_regs(n, nk, p, seed=n * 1000 + nk * 10 + p, dev=eng.device)
    group, G = groups_for(kind, n, seed=n + p)
    got = eng.leave_out_hist(regs, group, G, p)
    want = brute(regs, group, G)
    assert torch.equal(got.long(), want)
    # the same histograms from three register ranges added into one buffer
    m = 1 << p
    cuts = [0, (m // 3) // 16 * 16, (2 * m // 3) // 16 * 16, m]
    acc = torch.zeros_like(got)
    for b, e in zip(cuts, cuts[1:]):
        eng.leave_out_hist(regs, group, G, p, reg_range=(b, e), out=acc)
        assert torch.equal(eng.leave_out_hist(regs, group, G, p, reg_range=(b, e)).long(), brute(regs, group, G, b, e))
    assert torch.equal(acc, got)


@pytest.mark.parametrize("n_groups,placement", [(192, "shared"), (193, "global")])
def test_counter_placements_meet(eng, n_groups, placement):
    """The largest G counted in shared memory (48 KiB of counters) and the smallest counted by global atomics."""
    regs = make_regs(200, 3, 12, seed=n_groups, dev=eng.device)
    group = np.concatenate([np.arange(n_groups), np.arange(200 - n_groups) % n_groups]).astype(np.int32)
    np.random.default_rng(3).shuffle(group)
    assert torch.equal(eng.leave_out_hist(regs, group, n_groups, 12).long(), brute(regs, group, n_groups))


@pytest.mark.parametrize("p", [10, 14])
def test_cards_equal_the_per_union_path(eng, p):
    """The MLE of the K10 rows equals Engine.union_sets over the same members (same histogram, same kernel): ==."""
    n, nk = 9, 5
    regs = make_regs(n, nk, p, seed=p, dev=eng.device)
    group = np.array([2, 0, 1, 2, 3, 0, 3, 1, 2], dtype=np.int32)
    G = 4
    cards = eng.mle(eng.leave_out_hist(regs, group, G, p), p).cpu().numpy()
    m = 1 << p
    base = regs.data_ptr()
    table = np.zeros((nk * (1 + G), n), dtype=np.int64)
    for c in range(nk):
        for r in range(1 + G):
            members = [i for i in range(n) if r == 0 or group[i] != r - 1]
            table[c * (1 + G) + r, :len(members)] = [base + (i * nk + c) * m for i in members]
    want = eng.union_sets(table, p, final_only=True).cpu().numpy().reshape(nk, 1 + G)
    torch.cuda.synchronize()
    assert np.array_equal(cards, want)


def test_refusals_leave_the_histograms_alone(eng):
    from dandd_b200._lib import DandDError
    regs = make_regs(4, 2, 10, seed=4, dev=eng.device)
    out = torch.full((2, 3, BINS), 7, dtype=torch.int32, device=eng.device)
    before = eng.lib.dd_kernel_launches()
    for group, G, rng, match in [([0, 1, 2, 1], 2, None, "group 2 outside"), ([0, -1, 1, 1], 2, None, "group -1 outside"),
                                 ([0, 1, 0, 1], 2, (8, 64), "register range"), ([0, 1, 0, 1], 2, (0, 1040), "register range"),
                                 ([0, 1, 0, 1], 2, (64, 32), "register range"), ([0, 0, 0, 0], 5, None, "n_groups")]:
        with pytest.raises(DandDError, match=match):
            eng.leave_out_hist(regs, group, G, 10, reg_range=rng, out=out if G == 2 else None)
    torch.cuda.synchronize()
    assert eng.lib.dd_kernel_launches() == before
    assert bool((out == 7).all())


def _read_tsv(path):
    with open(path, newline="") as fh:
        return list(csv.DictReader(fh, delimiter="\t"))


@pytest.mark.parametrize("tool", ["dashing", "kmc"])
def test_command_line_on_the_engine(tmp_path, tool):
    """helpers/leaveout.py on synthetic FASTAs: dashing cards equal the per-union path (Engine.union_sets over the
    leaf sketches of the other genomes), kmc counts equal oracle k-mer sets."""
    from dandd_b200 import store as ddstore
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    fastas = make_dataset(data, 6, 20000, seed=12)
    names = [os.path.basename(f) for f in fastas]
    groups = tmp_path / "groups.tsv"
    labels_of = ["a", "b", "a", "c", "b", "c"]
    groups.write_text("".join("%s\t%s\n" % x for x in zip(names, labels_of)))
    st = ddstore.GpuSketchStore()
    ddstore.set_store(st)
    p, ks = 14, list(range(8, 16))
    try:
        _check_runs(tmp_path, st, tool, data, fastas, names, labels_of, str(groups), p, ks)
    finally:
        ddstore.set_store(None)


def _check_runs(tmp_path, st, tool, data, fastas, names, labels_of, groups, p, ks):
    from dandd_b200.helpers import leaveout
    from oracle import pyoracle as orc
    from tests.oracle_store import _read_fasta
    for grouped in (False, True):
        name = str(tmp_path / ("run%d" % grouped))
        argv = ["-d", data, "--tool", tool, "--mink", "8", "--maxk", "15", "--registers", str(p), "--name", name]
        labels = ["a", "b", "c"] if grouped else names
        group = [labels.index(x) for x in labels_of] if grouped else list(range(6))
        union, without = leaveout.go(argv + (["--groups", groups] if grouped else []))
        if tool == "dashing":
            regs = torch.stack([st.leaf_block(f, ks, p, True)[0] for f in fastas]).contiguous()
            nk, m, base = len(ks), 1 << p, regs.data_ptr()
            for g in range(-1, len(labels)):
                members = [i for i in range(6) if group[i] != g]
                table = np.array([[base + (i * nk + c) * m for i in members] for c in range(nk)], dtype=np.int64)
                want = st.engine.union_sets(table, p, final_only=True).cpu().numpy().reshape(nk)
                assert np.array_equal(union if g < 0 else without[:, g], want), g
        else:
            syms = [orc.fasta_symbols(_read_fasta(f)) for f in fastas]
            for c, k in enumerate(ks):
                sets = [set(orc.kmers(s, k, True).tolist()) for s in syms]
                assert union[c] == len(set().union(*sets))
                for g in range(len(labels)):
                    assert without[c, g] == len(set().union(*[s for s, x in zip(sets, group) if x != g])), (k, g)
        rows = _read_tsv(os.path.join(name, "without.tsv"))
        assert len(rows) == len(ks) * len(labels)
