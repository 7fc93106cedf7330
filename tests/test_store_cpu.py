"""The REAL dandd_b200.store.GpuSketchStore on the CPU: its engine is replaced by the oracle-backed
double of tests/fake_engine.py, everything above it -- cache and eviction, pointer tables, batched
union jobs, prefix-union layouts, the pair table, marker files, the all-pairs driver -- is the shipped
code, run through the same drop-in scenarios and reference goldens as on the GPU
(tests/test_host_gpu.py, tests/test_allpairs_gpu.py)."""
import os

import numpy as np
import pytest

from dandd_b200 import hllfile
from dandd_b200 import store as ddstore
from oracle import pyoracle as orc
from tests import allpairs_cases, host_cases
from tests.fake_engine import FakeEngine
from tests.util import make_dataset


@pytest.fixture()
def real_store():
    st = ddstore.GpuSketchStore(engine=FakeEngine())
    ddstore.set_store(st)
    yield st
    ddstore.set_store(None)


def test_tree_hillclimb_one_pass_per_fasta(tmp_path, real_store):
    host_cases.scenario_tree_hillclimb(str(tmp_path))
    assert real_store.stats["leaf_passes"] == 5 and real_store.engine.calls["sketch"] == 5


def test_rerun_is_fully_cached(tmp_path, real_store):
    host_cases.scenario_rerun_is_fully_cached(str(tmp_path), real_store)


def test_ksweep_and_progressive(tmp_path, real_store):
    host_cases.scenario_ksweep_and_progressive(str(tmp_path))


def test_progressive_hillclimb_and_kij(tmp_path, real_store):
    host_cases.scenario_progressive_hillclimb_and_kij(str(tmp_path))


def test_tree_nchildren(tmp_path, real_store):
    host_cases.scenario_tree_nchildren(str(tmp_path))


def test_tree_exact(tmp_path, real_store):
    host_cases.scenario_tree_exact(str(tmp_path))


def test_option_coverage(tmp_path, real_store):
    host_cases.scenario_option_coverage(str(tmp_path))


def test_stub_union_files(tmp_path, real_store):
    real_store.union_files = "stub"
    host_cases.scenario_tree_hillclimb(str(tmp_path))


@pytest.mark.parametrize("budget", [0, 3 << 20])
def test_results_do_not_depend_on_the_cache_budget(tmp_path, budget):
    """A byte budget that holds almost nothing: blocks and sketches are evicted all the time (views with
    their block), evicted sketches come back from their files, and every table still equals the golden."""
    st = ddstore.GpuSketchStore(engine=FakeEngine(), cache_bytes=budget)
    ddstore.set_store(st)
    try:
        host_cases.scenario_ksweep_and_progressive(str(tmp_path))
    finally:
        ddstore.set_store(None)
    assert st.stats["files_read"] > 0 and st._bytes <= max(budget, 1 << 20) and set(st._cost) == set(st._lru)


def test_pair_table_serves_two_leaf_unions(tmp_path):
    """tests/test_gpu_round2.py::test_store_pair_table_serves_two_leaf_unions on the CPU double."""
    rng = np.random.default_rng(40)
    ks, p, n = [14, 15, 16], 12, 5
    regs = rng.integers(0, 30, (n, len(ks), 1 << p), dtype=np.uint8)
    store = ddstore.GpuSketchStore(engine=FakeEngine(), union_files="stub")
    leaf_paths = {k: [] for k in ks}
    for g in range(n):
        for i, k in enumerate(ks):
            path = str(tmp_path / f"k{k}" / f"g{g}.hll")
            os.makedirs(os.path.dirname(path), exist_ok=True)
            hllfile.write_hll(path, regs[g, i], p, 0.0)
            leaf_paths[k].append(path)
    table = store.pair_unions(leaf_paths, p, tile_pairs=4)                   # 10 pairs in three tiles
    assert table.shape == (n * (n - 1) // 2, len(ks)) and store.engine.calls["to_planes"] == 1
    assert store.engine.calls["pairwise_cards"] == 3
    launches = store.stats["union_launches"]
    out = {k: str(tmp_path / f"u{k}.hll") for k in ks}
    got = store.union_sketches({k: [leaf_paths[k][3], leaf_paths[k][1]] for k in ks}, p, out)   # order reversed on purpose
    assert store.stats["union_launches"] == launches
    for i, k in enumerate(ks):
        assert got[k] == orc.card(np.maximum(regs[1, i], regs[3, i]), p)
        assert os.path.getsize(out[k]) > 0
        assert np.array_equal(store.registers(out[k]).numpy(), np.maximum(regs[1, i], regs[3, i]))   # the marker rebuilds
    store.union_sketches({14: leaf_paths[14][:3]}, p, {14: str(tmp_path / "u3.hll")})            # three members: a launch
    assert store.stats["union_launches"] == launches + 1
    # pair_cards on an explicit pair list, bytes path (p < 12 has no bit planes)
    small = np.ascontiguousarray(regs[:, :, :1 << 10])
    import torch
    cards = store.pair_cards(torch.from_numpy(small), [(0, 4), (2, 1)], 10)
    assert cards.shape == (2, 3) and cards[1, 2] == orc.card(np.maximum(small[2, 2], small[1, 2]), 10)
    assert store.engine.calls["to_planes"] == 1                               # unchanged
    assert store.pair_cards(torch.from_numpy(small), np.zeros((0, 2)), 10).shape == (0, 3)


def test_leaf_block_rows_follow_the_request_and_skip_the_cache(tmp_path, real_store):
    inputs = make_dataset(str(tmp_path / "d"), 2, 6000, seed=5)
    import torch
    sym = orc.fasta_symbols(open(inputs[0], "rb").read())
    regs, cards = real_store.leaf_block(inputs[0], [21, 9, 15], 10, False)
    for row, k in enumerate([21, 9, 15]):
        assert np.array_equal(regs[row].numpy(), orc.hll_sketch(sym, k, 10, False)) and cards[row] == orc.card(regs[row].numpy(), 10)
    assert len(real_store._lru) == 0 and real_store.stats["files_written"] == 0
    out = torch.zeros((2, 3, 1 << 10), dtype=torch.uint8)
    real_store.leaf_block(inputs[0], [9, 15, 21], 10, False, out=out[1])         # sorted request: straight copy into the slice
    assert np.array_equal(out[1, 2].numpy(), orc.hll_sketch(sym, 21, 10, False)) and not out[0].any()
    # a block the tree commands left in the cache is reused (all 32 k: rows are picked by index)
    paths = {k: str(tmp_path / "db" / f"k{k}.hll") for k in (9, 15)}
    real_store.leaf_sketches(inputs[0], [9, 15], 10, False, paths)
    passes = real_store.stats["leaf_passes"]
    with pytest.raises(ValueError, match="out must be"):
        real_store.leaf_block(inputs[0], [15, 9], 10, False, out=out[0])            # three rows offered for two k
    real_store.leaf_block(inputs[0], [15, 9], 10, False, out=out[0, :2])
    assert real_store.stats["leaf_passes"] == passes and np.array_equal(out[0, 0].numpy(), orc.hll_sketch(sym, 15, 10, False))
    assert np.array_equal(hllfile.read_hll(paths[9])[0], out[0, 1].numpy())


@pytest.mark.parametrize("name", sorted(allpairs_cases.gold_cases()))
def test_allpairs_tables(tmp_path, real_store, name):
    table = allpairs_cases.scenario_gold(str(tmp_path), name)
    assert real_store.stats["leaf_passes"] == len(table.names) and real_store.stats["files_written"] == 0
    assert real_store.engine.calls["pairwise_cards"] == 1


def test_allpairs_exact(tmp_path, real_store):
    allpairs_cases.scenario_exact(
        str(tmp_path), lambda fastas, k: orc.exact_count([orc.fasta_symbols(open(f, "rb").read()) for f in fastas], k, True))


def test_engine_and_double_have_everything_the_store_reads():
    """Every attribute the store reads off its engine (`self.engine.X`, `_store.engine.X`, `eng.X`) exists on Engine (a
    class attribute or one its methods set on self) and on FakeEngine: the store calls the engine's jobs without probing
    for them, and the CPU tests run the paths the device runs."""
    import ast
    import inspect
    from dandd_b200.engine import Engine
    used = {node.attr for node in ast.walk(ast.parse(inspect.getsource(ddstore))) if isinstance(node, ast.Attribute)
            and (isinstance(node.value, ast.Attribute) and node.value.attr == "engine"
                 or isinstance(node.value, ast.Name) and node.value.id == "eng")}
    on_self = {node.attr for node in ast.walk(ast.parse(inspect.getsource(Engine)))
               if isinstance(node, ast.Attribute) and isinstance(node.ctx, ast.Store) and isinstance(node.value, ast.Name)
               and node.value.id == "self"}
    assert {"exact_pair_intersections", "exact_family_counts", "greedy_dense_hist", "device"} <= used
    assert sorted(a for a in used if not hasattr(Engine, a) and a not in on_self) == []
    fake = FakeEngine()
    assert sorted(a for a in used if not hasattr(fake, a)) == []


# ---- the streaming branch of the store (files above STREAM_MIN_BYTES) on CPU doubles -----------------------
class _OracleLib:
    """The slice of the C ABI that dandd_b200/streaming.py drives, answered by the oracle: the text given to
    dd_pack_fasta is accumulated, dd_sketch_end writes the oracle's registers, histogram-free cardinalities
    and the FASTQ flag where the real library would."""

    def __init__(self, real):
        self.real, self.fed, self.kmask, self.canon = real, [], 0, True

    def dd_pack_codes_bytes(self, n):
        return 64

    dd_pack_invalid_bytes = dd_pack_codes_bytes

    def dd_pack_workspace_bytes(self, n):
        return 64

    def dd_sketch_workspace_bytes(self, nk, p):
        return 64

    def dd_pack_reset(self, codes, cb, invalid, ib, state, st):
        import ctypes
        self.fed, self.state = [], state
        ctypes.memset(state, 0, 32)
        return 0

    def dd_sketch_begin(self, *a):
        return 0

    def dd_fasta_first_record_host(self, ptr, n):
        return self.real.dd_fasta_first_record_host(ptr, n)

    def dd_pack_fasta(self, d_text, ln, *rest):
        import ctypes
        self.fed.append(ctypes.string_at(d_text, ln))
        return 0

    def dd_sketch_update_sched(self, codes, invalid, state, a, b, ln, seen, kmask, p, canon, *rest):
        self.kmask, self.canon = kmask, bool(canon)
        return 0

    def dd_sketch_end(self, ws, wsb, nk, p, regs, hist, cards, st):
        import ctypes
        text = b"".join(self.fed)
        if text[:1] == b"+" or b"\n+" in text:                      # DD_PACK_FLAG_FASTQ in dd_pack_state.reserved
            (ctypes.c_uint64 * 4).from_address(self.state)[3] = 2
            return 0
        sym = orc.fasta_symbols(text)
        ks = [k for k in range(1, 33) if (self.kmask >> (k - 1)) & 1]
        assert len(ks) == nk
        for i, k in enumerate(ks):
            r = orc.hll_sketch(sym, k, p, self.canon)
            ctypes.memmove(regs + (i << p), r.ctypes.data, 1 << p)
            (ctypes.c_double * nk).from_address(cards)[i] = orc.card(r, p)
        return 0

    def dd_last_error(self):
        return b"oracle lib"


def test_store_streams_large_fastas_on_cpu(tmp_path, monkeypatch):
    """tests/test_gpu_round2.py::test_store_streams_large_fastas on CPU doubles: above the size threshold
    leaf_sketches / warm_leaf take dandd_b200/streaming.py (ring, readers, in-order feed), the digest
    reaches the naming layer, FASTQ falls back to the whole-file detour."""
    import hashlib
    import types
    import torch
    from dandd_b200 import _lib, ingest, streaming
    from dandd_b200._lib import DD_PACK_FLAG_FASTQ
    from tests.test_streaming_host import _FakeCuda
    from tests.util import kseq_fasta, random_bases, to_fasta
    assert DD_PACK_FLAG_FASTQ == 2
    fake_torch = types.SimpleNamespace(cuda=_FakeCuda, empty=torch.empty, Tensor=torch.Tensor, uint8=torch.uint8,
                                       int32=torch.int32, float64=torch.float64)
    monkeypatch.setattr(streaming, "torch", fake_torch)
    monkeypatch.setattr(streaming, "_Ring", lambda chunk, pin=True, _R=streaming._Ring: _R(chunk, pin=False))
    monkeypatch.setattr(streaming, "_rings", {})
    monkeypatch.setattr(ddstore, "STREAM_MIN_BYTES", 1 << 20)
    monkeypatch.setattr(ingest, "_jobs", {})
    eng = FakeEngine()
    eng.lib = _OracleLib(_lib.load())
    scratch = {}

    def grow_only_buffer(nbytes, tag):                      # Engine._buf
        if tag not in scratch or scratch[tag].numel() < nbytes:
            scratch[tag] = torch.empty(max(int(nbytes), 256), dtype=torch.uint8)
        return scratch[tag]
    eng._buf = grow_only_buffer
    rng = np.random.default_rng(78)
    texts = {"a.fa": to_fasta([(b"a", random_bases(rng, 2_500_000))], width=80),
             "q.fq": kseq_fasta(rng, n=1_500_000, fastq=True)}
    st = ddstore.GpuSketchStore(engine=eng, prefetch_all_k=False)
    for name, txt in texts.items():
        path = tmp_path / name
        path.write_bytes(txt)
        out = {k: str(tmp_path / "db" / f"k{k}" / (name + ".hll")) for k in (12, 31)}
        cards = st.leaf_sketches(str(path), [12, 31], 14, True, out)
        sym = orc.fasta_symbols(txt)
        for k in (12, 31):
            want = orc.hll_sketch(sym, k, 14)
            assert np.array_equal(hllfile.read_hll(out[k])[0], want), (name, k)
            assert cards[k] == orc.card(want, 14)
        assert ingest.digest(str(path)) == hashlib.blake2b(txt).hexdigest()
    assert len(st.stream_stats) == 1 and st.stream_stats[0]["chunks"] >= 1      # the FASTA streamed; the FASTQ took the detour
    assert eng.calls["pack"] == 2                                               # (FASTQ: flagged, rewritten, packed again)
    # warm_leaf: the all-k pass of a large fresh FASTA before anything is named or written
    big = tmp_path / "w.fa"
    big.write_bytes(to_fasta([(b"w", random_bases(rng, 1_400_000))], width=60))
    st2 = ddstore.GpuSketchStore(engine=eng)
    st2.warm_leaf(str(big), 12, True)
    assert st2.stats["leaf_passes"] == 1 and st2.stats["files_written"] == 0
    out = {k: str(tmp_path / "db2" / f"k{k}.hll") for k in (9, 32)}
    got = st2.leaf_sketches(str(big), [9, 32], 12, True, out)
    assert st2.stats["leaf_passes"] == 1                                        # served from the warmed block
    wsym = orc.fasta_symbols(big.read_bytes())
    assert got[32] == orc.card(orc.hll_sketch(wsym, 32, 12), 12)
    assert np.array_equal(hllfile.read_hll(out[9])[0], orc.hll_sketch(wsym, 9, 12))
