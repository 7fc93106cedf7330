"""K12 on the device: the cover index emitted from the K7 lists against oracle holder sets (keys, holders, each genome's
node range), the step against the numpy restatement with both counter placements, whole exact greedy orders against a
per-step K8 order (store.exact_union_cards), and the `greedy.py --tool kmc` output replayed by `dandd tree --exact` +
`progressive --ksweep -r` on the real engine."""
import collections
import os
import pickle

import numpy as np
import pytest

from tests.test_exact_greedy import _read_tsv, emit_rule, step_rule
from tests.test_exact_pairs_gpu import _genomes
from tests.test_exact_sets_gpu import _holders

pytestmark = pytest.mark.gpu


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


def _host(part):
    return {"offsets": part["offsets"].cpu().numpy().view(np.uint32).astype(np.int64),
            "holders": part["holders"].cpu().numpy().view(np.uint16).astype(np.int64)[:part["n_nodes"]],
            "key_of_node": part["key_of_node"].cpu().numpy().view(np.uint32).astype(np.int64)[:part["n_nodes"]],
            "node_start": part["node_start"].astype(np.int64), "n_keys": part["n_keys"], "n_nodes": part["n_nodes"],
            "covered": np.zeros(part["n_keys"], dtype=bool)}


@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("canon", [True, False], ids=["canon", "nocanon"])
@pytest.mark.parametrize("k", [5, 12, 16, 17, 31, 32, 33, 64, 65, 127])
def test_emit_equals_the_oracle_holder_sets(eng, packed, k, canon, passes):
    """(k = 32 and 64 --no-canon: the all-ones key lives in the extra slot.  The genomes include an identical pair and
    one without k-mers above k = 4.)"""
    texts, seqs = packed
    held, singles = _holders(texts, k, canon)
    ix = eng.exact_cover_index(seqs, k, canon, passes=passes)
    assert len(ix["parts"]) == passes == eng.last_pair_plan["passes"]
    assert ix["keys"] == held.shape[0] and ix["singles"].astype(np.int64).tolist() == singles
    got = collections.Counter()
    for part in map(_host, ix["parts"]):
        off = part["offsets"]
        assert off[0] == 0 and (np.diff(off) >= 1).all() and off[-1] == part["n_nodes"]
        assert part["node_start"][-1] == part["n_nodes"] and (np.diff(part["node_start"]) >= 0).all()
        spans = [tuple(sorted(part["holders"][off[i]:off[i + 1]].tolist())) for i in range(part["n_keys"])]
        got.update(spans)
        for g in range(len(seqs)):        # genome g's node range is its key list: the keys whose span holds g
            keys = part["key_of_node"][part["node_start"][g]:part["node_start"][g + 1]]
            assert sorted(keys.tolist()) == [i for i, s in enumerate(spans) if g in s]
    assert got == collections.Counter(tuple(np.flatnonzero(row).tolist()) for row in held)
    assert ix["bytes"] == sum(4 * (p["n_keys"] + 1) + 6 * max(p["n_nodes"], 1) + max(p["n_keys"], 1) for p in ix["parts"])


def _upload(eng, part):
    import torch
    dev = eng.device
    return {"offsets": torch.from_numpy(part["offsets"].astype(np.int32)).to(dev),
            "holders": torch.from_numpy(part["holders"].astype(np.uint16).view(np.int16)).to(dev),
            "key_of_node": torch.from_numpy(part["key_of_node"].astype(np.int32)).to(dev),
            "covered": torch.zeros(max(part["n_keys"], 1), dtype=torch.uint8, device=dev),
            "n_keys": part["n_keys"], "n_nodes": part["n_nodes"], "node_start": part["node_start"].astype(np.uint64)}


@pytest.mark.parametrize("n", [40, 20000], ids=["shared", "global"])
def test_step_equals_the_restatement(eng, n):
    """Synthetic indices of two k with two parts each, uploaded; n = 20000 takes the 64-bit global counters (n u32 >
    48 KiB), n = 40 the shared ones.  Every step's lost equals the restatement's, and that is |A_h n U|."""
    import torch
    rng = np.random.default_rng(n)
    helds, host, dev = [], [], []
    for c in range(2):
        held = rng.random((3000, n)) < (3.0 / n if n > 100 else 0.2)
        held[5] = True                                                    # a key every genome holds
        held = held[held.any(axis=1)]
        helds.append(held)
        split = [held[i::2] for i in range(2)]
        host.append([emit_rule(h, rng) for h in split])
        dev.append({"n": n, "parts": [_upload(eng, p) for p in host[-1]]})
    lost = torch.zeros((2, n), dtype=torch.int64, device=eng.device)
    want = np.zeros((2, n), dtype=np.int64)
    union = [np.zeros(h.shape[0], dtype=bool) for h in helds]
    for g in rng.permutation(n)[:12]:
        eng.exact_cover_step(dev, int(g), lost)
        for c in range(2):
            for p in host[c]:
                step_rule(p, int(g), want[c])
            union[c] |= helds[c][:, g]
            assert want[c].tolist() == (helds[c] & union[c][:, None]).sum(axis=0).tolist()
        assert np.array_equal(lost.cpu().numpy(), want)


def _k8_greedy(store, fastas, ks, steps, order):
    """The greedy order by per-step K8 union counts of every (chosen + candidate) set."""
    picks, cards = [], []
    for t in range(steps):
        cand = [g for g in range(len(fastas)) if g not in picks]
        got = store.exact_union_cards(fastas, [picks + [g] for g in cand], ks, True)
        d = [max(got[i, c] / k for c, k in enumerate(ks)) for i in range(len(cand))]
        best = d.index(max(d) if order == "max" else min(d))
        picks.append(cand[best])
        cards.append(got[best])
    return picks, np.asarray(cards, dtype=np.int64)


@pytest.fixture(scope="module")
def eight(tmp_path_factory):
    from tests.util import make_dataset
    d = tmp_path_factory.mktemp("eight")
    return make_dataset(str(d / "a"), 5, 20000, seed=12, prefix="a") + make_dataset(str(d / "b"), 3, 20000, seed=13, prefix="b")


@pytest.mark.parametrize("order", ["max", "min"])
def test_whole_order_equals_the_k8_order(eng, eight, order):
    from dandd_b200 import store as ddstore
    st = ddstore.GpuSketchStore(engine=eng)
    ks = list(range(10, 33))
    got, cards, stats = st.exact_greedy_order(eight, ks, True, len(eight), order=order)
    want, want_cards = _k8_greedy(st, eight, ks, len(eight), order)
    assert got.tolist() == want and np.array_equal(cards, want_cards)
    assert stats["distinct_keys"] == cards[-1].tolist() and len(stats["index_bytes"]) == len(ks)
    one = st.exact_greedy_order(eight, ks, True, 4, order=order, first=[want[2]])
    assert one[0].tolist()[0] == want[2]


def test_helper_output_replays_exactly(tmp_path):
    from dandd_b200 import store as ddstore
    from dandd_b200.helpers import greedy
    from tests.host_harness import read_csv, run_dandd
    from tests.util import make_dataset
    data = str(tmp_path / "data")
    make_dataset(data, 5, 3000, seed=23)
    name, out = str(tmp_path / "run"), str(tmp_path / "out")
    lo, hi = 4, 40
    st = ddstore.GpuSketchStore()
    ddstore.set_store(st)
    try:
        greedy.go(["-d", data, "--tool", "kmc", "--mink", str(lo), "--maxk", str(hi), "--name", name])
        run_dandd(["tree", "-d", data, "-s", "ex", "-o", out, "--exact"])
        run_dandd(["progressive", "-d", os.path.join(out, "ex_5_kmc_dtree.pickle"), "-o", out, "--ksweep",
                   "--mink", str(lo), "--maxk", str(hi), "-r", os.path.join(name, "ordering.pickle")])
    finally:
        ddstore.set_store(None)
    growth = _read_tsv(os.path.join(name, "growth.tsv"))
    summary = [f for f in os.listdir(out) if f.endswith("summary.csv")]
    replay = {(int(r["ngen"]), int(r["kval"])): float(r["card"]) for r in read_csv(os.path.join(out, summary[0]))}
    assert len(growth) == len(replay) == 5 * (hi - lo + 1)
    for r in growth:
        assert int(r["card"]) == replay[(int(r["ngen"]), int(r["k"]))], r
    with open(os.path.join(name, "ordering.pickle"), "rb") as fh:
        assert len(next(iter(pickle.load(fh)))) == 5
