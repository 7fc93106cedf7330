#!/usr/bin/env python
"""bench.py -- Gbp/s sketched (all k) on the BASELINE.json config-2 workload.

Workload (SURVEY.md 8d, config 2), per GPU: 12 synthetic 5 Mbp bacterial-like genomes (mutated
copies of one random ancestor, 80-column FASTA), k = 10..32 (23 k values), p = 20 registers,
leaf sketches + leaf cardinalities + progressive unions over 30 orderings with the cardinality of
every prefix union.  One "step" = one full pass of that hot path over the rank's 12 genomes.
At N > 1 every rank owns its own 12 genomes (weak scaling, no data-path collective for the
sketching); the one real exchange step of the path -- the union sketch over every genome of the
job -- is an NCCL MAX all-reduce of the [23][2^20] register array, inside the timed step.

  value : whole-job bases / step time, FASTA text already resident in HBM
  e2e   : same, through the host-buffer C-ABI call (dd_sketch_fasta_host) from pinned host
          memory, H2D copy and D2H of the cardinalities inside the timed region
  roofline / cpu_baseline : see DESIGN.md "Measurement"

--config 3 switches the workload to BASELINE.json configs[2] (one 3.1 Gbp human-scale assembly per GPU,
k = 2..32, all-gather of the registers, prefix unions of the identity ordering); the default stays
config 2, the configuration that fits one GPU and that the metric is quoted on.

--impl reference times the CPU path the reference drives (one single-threaded `dashing sketch`
per (genome, k), floor(0.95*cores) at a time -- lib/huffman_dandd.py:217) using the oracle port,
because neither Dashing nor GNU parallel exists here (see oracle/dandd_oracle.c header).

--dump-outputs DIR writes what the last step of each timed loop computed (leaf and prefix-union
cardinalities, a fixed sample of the registers) as DIR/<name>.npy.  The inputs are generated from
fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

# Rank 0 prints exactly ONE JSON line on stdout.  Libraries chat on fd 1 too (NCCL prints its version
# banner there), so fd 1 is pointed at stderr for the whole run and the line goes to the saved fd.
_STDOUT_FD = None


def _claim_stdout():
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_STDOUT_FD if _STDOUT_FD is not None else 1, data)

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_GENOMES = 12
GENOME_BP = 5_000_000
KS = list(range(10, 33))
P = 20
N_ORDERINGS = 30
LINE = 80
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


# ------------------------------------------------------------------------------------ synthetic data
def make_genomes(seed, n_genomes=N_GENOMES, bp=GENOME_BP):
    """Ancestor + mutated copies: 1 % substitutions, 0.1 % 1-10 bp indels (SURVEY.md 8d config 2)."""
    rng = np.random.default_rng(seed)
    anc = ACGT[rng.integers(0, 4, bp)]
    texts = []
    for g in range(n_genomes):
        r = np.random.default_rng(seed * 1000 + g + 1)
        s = anc.copy()
        hit = r.random(s.size) < 0.01
        s[hit] = ACGT[r.integers(0, 4, int(hit.sum()))]
        sites = np.flatnonzero(r.random(s.size) < 0.001)
        pieces, pos = [], 0
        for at in sites:
            if at < pos:
                continue
            pieces.append(s[pos:at])
            ln = int(r.integers(1, 11))
            if r.random() < 0.5:
                pieces.append(ACGT[r.integers(0, 4, ln)])
                pos = at
            else:
                pos = min(s.size, at + ln)
        pieces.append(s[pos:])
        s = np.concatenate(pieces)
        nfull = s.size // LINE
        body = np.empty((nfull, LINE + 1), dtype=np.uint8)
        body[:, :LINE] = s[:nfull * LINE].reshape(nfull, LINE)
        body[:, LINE] = 10
        text = b">genome%d seed%d\n" % (g, seed) + body.tobytes() + s[nfull * LINE:].tobytes() + b"\n"
        texts.append((text, int(s.size)))
    return texts


def make_orderings(n, count, seed):
    rng = np.random.default_rng(seed)
    return np.stack([rng.permutation(n) for _ in range(count)]).astype(np.int32)


# ------------------------------------------------------------------------------------- clock sampler
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region through in-process NVML
    (nvidia_ml_py).  Spawning nvidia-smi instead stalls kernel launches for tens of milliseconds on
    these boxes -- it inflated a 15 ms step to 47 ms -- so the handle is opened before warm-up and
    each sample is two cheap NVML queries."""

    def __init__(self, index=0, period=0.01):
        super().__init__(daemon=True)
        self.samples, self.stop_flag, self.period = [], False, period
        self.active = False
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = str(e)

    def run(self):
        if self.h is None:
            return
        nv = self.nv
        while not self.stop_flag:
            if self.active:
                try:
                    self.samples.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)),
                                         int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
                except Exception:  # noqa: BLE001
                    pass
            time.sleep(self.period)

    def summary(self):
        if self.h is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        nv = self.nv
        sm = sorted(s[0] for s in self.samples)
        bits = 0
        for _, r in self.samples:
            bits |= r
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": [n for n, b in names.items() if bits & b],
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------- CPU arm
def cpu_sketch_sample(texts, ks, p, threads):
    """The reference's CPU topology on the oracle port: one single-threaded sketch+card job per
    (genome, k), `threads` jobs in flight.  Returns (seconds, bases)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as orc
    orc.lib()
    jobs = [(t, k) for (t, _) in texts for k in ks]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(lambda j: orc.sketch_fasta(j[0], j[1], p)[1], jobs))
    return time.perf_counter() - t0, sum(n for _, n in texts)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = max(1, int(cores * 0.95))
    if args.config == 3:
        return run_reference_config3(args, threads)
    texts = make_genomes(seed=2, n_genomes=N_GENOMES)   # one whole step of leaf sketches: ~10-20 s of CPU work
    for _ in range(min(args.warmup, 1)):
        cpu_sketch_sample(texts[:1], KS[:min(len(KS), threads)], P, threads)
    secs = []
    for _ in range(args.steps):
        dt, bases = cpu_sketch_sample(texts, KS, P, threads)
        secs.append(dt)
    ms = 1e3 * sum(secs) / len(secs)
    value = bases / (ms / 1e3) / 1e9
    sample = (f"{N_GENOMES} genomes x 5 Mbp x 23 k (k=10..32), p=20, one single-threaded oracle job per (genome,k), "
              f"{threads} in flight (leaf sketches + cardinalities only; the reference's union / card processes are not timed)")
    line = {"impl": "reference", "metric": "Gbp/s sketched (all k)", "value": value, "unit": "Gbp/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "Gbp/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(n_gpus):
    return {"workload": "config 2: 12 synthetic 5 Mbp genomes per GPU (1% subst + 0.1% indels), k=10..32 (23 k), "
                        "p=20, leaf sketches + cardinalities + progressive unions over 30 orderings",
            "genomes_per_gpu": N_GENOMES, "genome_bp": GENOME_BP, "k_min": KS[0], "k_max": KS[-1], "registers_log2": P,
            "orderings": N_ORDERINGS, "parallelism": f"genomes sharded over {n_gpus} GPU(s)",
            "l2_policy": "per-step working set (60 MB text + 276 MiB registers + 46 MiB accumulators re-zeroed per "
                         "genome) exceeds the 126 MB L2; no explicit flush"}


# ----------------------------------------------------------------------------------------- GPU arm
def bind_to_gpu_numa_node(local_rank):
    """Pin this rank to the CPU cores of its GPU's NUMA node before any pinned host buffer exists, so
    that the per-step host->device copies do not cross sockets (at N=8 half the ranks otherwise do).
    Best effort: returns the node, or None when the topology cannot be read."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local_rank)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:           # nvml pads the domain to 8 hex digits, sysfs uses 4
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            # virtualised hosts hide the PCI NUMA node; NVML still knows which CPUs sit next to the GPU
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1} & os.sched_getaffinity(0)
            if cpus and len(cpus) < len(os.sched_getaffinity(0)):
                os.sched_setaffinity(0, cpus)
                return "nvml:%d-cpus" % len(cpus)
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def _profile_json(name):
    try:
        with open(os.path.join(ROOT, "profiles", name)) as fh:
            return json.load(fh)
    except Exception:  # noqa: BLE001
        return {}


# ------------------------------------------------------------------------------------ --dump-outputs
DUMP_LIMIT_BYTES = 64 << 20
REGISTER_SAMPLE = 1 << 20


def register_sample(regs):
    """A fixed, seeded sample of a register array (12 x 23 x 2^20 bytes per step at config 2, too large to
    write whole), as float32: distinct positions, the same on every run, so two builds can be compared."""
    import torch
    idx = np.sort(np.random.default_rng(0).choice(regs.numel(), min(REGISTER_SAMPLE, regs.numel()), replace=False))
    return regs.reshape(-1)[torch.from_numpy(idx).to(regs.device)].float()


def write_outputs(directory, arrays):
    """Write each array (tensor or numpy) as <directory>/<name>.npy; float32 / float64 only, 64 MiB in all."""
    arrays = {name: a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a) for name, a in arrays.items()}
    bad = [name for name, a in arrays.items() if a.dtype not in (np.float32, np.float64)]
    total = sum(a.nbytes for a in arrays.values())
    if bad or total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes, non-float arrays {bad}")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(args):
    if args.config == 3:
        return run_ours_config3(args)
    import torch
    import torch.distributed as dist
    from dandd_b200 import build
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank == 0:
        build.build()
    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    torch.cuda.set_device(local)
    from dandd_b200 import dist as dd_dist
    if world > 1:
        dd_dist.init("nccl")
        dist.barrier()
    from dandd_b200.engine import Engine
    from dandd_b200._lib import check
    eng = Engine(local)
    if os.environ.get("DD_K_PER_PASS"):
        check(eng.lib.dd_set_option(b"sketch_k_per_pass", int(os.environ["DD_K_PER_PASS"])), "dd_set_option")
    dev = eng.device
    nk, m = len(KS), 1 << P

    texts = make_genomes(seed=2 + rank)
    bases = sum(n for _, n in texts)
    d_texts = [torch.from_numpy(np.frombuffer(t, dtype=np.uint8).copy()).to(dev) for t, _ in texts]
    pinned = []
    for t, _ in texts:
        h = torch.empty(len(t), dtype=torch.uint8).pin_memory()
        h.copy_(torch.from_numpy(np.frombuffer(t, dtype=np.uint8).copy()))
        pinned.append(h)
    orders = make_orderings(N_GENOMES, N_ORDERINGS, seed=2)
    regs = torch.empty((N_GENOMES, nk, m), dtype=torch.uint8, device=dev)
    leaf_hist = torch.empty((N_GENOMES, nk, 64), dtype=torch.int32, device=dev)
    leaf_cards_host = torch.empty((N_GENOMES, nk), dtype=torch.float64).pin_memory()
    NS = int(os.environ.get("DD_BENCH_STREAMS", "2"))   # genomes in flight
    side = [torch.cuda.Stream(device=dev) for _ in range(NS)]
    k2_events = []

    def step_resident(time_k2=False):
        """pack + all-k sketch + leaf cards for every genome, progressive prefix-union cards,
        (N>1) all-reduce MAX of the rank's full union + its cardinalities."""
        main = torch.cuda.current_stream()
        for s_ in side:
            s_.wait_stream(main)
        for g, dt in enumerate(d_texts):
            with torch.cuda.stream(side[g % NS]):   # several genomes in flight: pack/finalize of one overlap K2 of another
                seq = eng.pack(dt, start=0, ws_tag=f"pack{g % NS}")
                if time_k2:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    eng._k2_events = (e0, e1)
                eng.sketch(seq, KS, p=P, out=regs[g], hist_out=leaf_hist[g], ws_tag=f"sketch{g % NS}")
                if time_k2:
                    k2_events.append(eng._k2_events)
                    eng._k2_events = None
        for s_ in side:
            main.wait_stream(s_)
        leaf_cards = eng.mle(leaf_hist, P)          # one estimator launch for all 12 x 23 leaf sketches
        return leaf_cards, progressive_and_union()

    def progressive_and_union():
        """K3/K4 over the rank's genomes; at N>1 the one exchange step of the path: the union sketch
        of the whole job = MAX all-reduce of the rank unions, then its cardinalities."""
        prog = eng.prefix_union_cards(regs, orders, P)
        full = None
        if world > 1:
            full = dd_dist.union_over_ranks(eng.union([regs[g] for g in range(N_GENOMES)]))
            full = eng.cards(full, P)
        return prog, full

    def step_e2e():
        """The same step through the host-buffer C ABI: FASTA in pinned host memory -> H2D ->
        K1 -> K2 -> K4, registers stay in HBM, every cardinality comes back to the host."""
        out = []
        main = torch.cuda.current_stream()
        for s_ in side:
            s_.wait_stream(main)
        for g, h in enumerate(pinned):
            with torch.cuda.stream(side[g % NS]):      # several files in flight: copies overlap kernels
                eng.sketch_fasta_host(h, KS, p=P, want_regs=False, out_dev=regs[g], cards_out=leaf_cards_host[g],
                                      ws_tag=f"host{g % NS}", sync=False)
        for s_ in side:
            main.wait_stream(s_)
        out.append(leaf_cards_host)
        prog, full = progressive_and_union()
        out.append(prog.cpu())
        if full is not None:
            out.append(full.cpu())
        return out

    def breakdown():
        """DD_BENCH_BREAKDOWN=1: per-rank wall/GPU time of each phase of one step (diagnostics)."""
        def phase(fn):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            return out, round(e0.elapsed_time(e1), 3), round((time.perf_counter() - t0) * 1e3, 3)

        def sketch_all():
            for g, dt in enumerate(d_texts):
                eng.sketch(eng.pack(dt, start=0), KS, p=P, out=regs[g], hist_out=leaf_hist[g])
        rep = {"rank": rank}
        _, rep["sketch_gpu_ms"], rep["sketch_wall_ms"] = phase(sketch_all)
        _, rep["mle_gpu_ms"], rep["mle_wall_ms"] = phase(lambda: eng.mle(leaf_hist, P))
        _, rep["prefix_gpu_ms"], rep["prefix_wall_ms"] = phase(lambda: eng.prefix_union_cards(regs, orders, P))
        if world > 1:
            full, rep["union_gpu_ms"], rep["union_wall_ms"] = phase(lambda: eng.union([regs[g] for g in range(N_GENOMES)]))
            _, rep["allreduce_gpu_ms"], rep["allreduce_wall_ms"] = phase(lambda: dd_dist.union_over_ranks(full))
            _, rep["cards_gpu_ms"], rep["cards_wall_ms"] = phase(lambda: eng.cards(full, P))
        print("BREAKDOWN " + json.dumps(rep), file=sys.stderr, flush=True)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), res

    # K2 timing hook: events recorded right around dd_sketch_update on the launching stream
    orig_update = eng._update_from_state

    def hooked(seq, kmask, p, canon, ws, st):
        ev = getattr(eng, "_k2_events", None)
        if ev:
            ev[0].record()
        orig_update(seq, kmask, p, canon, ws, st)
        if ev:
            ev[1].record()
    eng._update_from_state = hooked

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    if world > 1:
        # NCCL builds channels lazily over its first calls; keep that out of the timed region
        warm = torch.zeros((nk, m), dtype=torch.uint8, device=dev)
        for _ in range(8):
            dd_dist.union_over_ranks(warm)
        for _ in range(2):
            step_resident()
    if os.environ.get("DD_BENCH_BREAKDOWN"):
        breakdown()
        breakdown()
    sampler.active = True
    launches0 = eng.lib.dd_kernel_launches()
    ms_step, res = timed(lambda: step_resident(time_k2=True), args.steps)
    launches_timed = eng.lib.dd_kernel_launches() - launches0     # counted inside the library, not a formula
    sampler.active = False
    outputs = {}
    if args.dump_outputs:     # the last timed step's results, taken before the serialized K2 pass below rewrites regs
        leaf_cards, (prog, full) = res
        outputs = {"leaf_cards": leaf_cards, "prefix_union_cards": prog, "registers_sample": register_sample(regs)}
        if full is not None:
            outputs["union_cards"] = full
    # K2's own duration: with several streams in flight the per-launch events above include time shared
    # with the other stream's kernels, so the roofline uses a serialized pass over the same 12
    # genomes taken right after the timed region (same clocks, L2 displaced by the other genomes).
    k2_overlapped_ms = [a.elapsed_time(b) for a, b in k2_events]
    k2_events.clear()
    packed = [eng.pack(dt, start=0) for dt in d_texts]
    for rep in range(2):
        for g, seq in enumerate(packed):
            eng._k2_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            eng.sketch(seq, KS, p=P, out=regs[g], hist_out=leaf_hist[g])
            if rep == 1:
                k2_events.append(eng._k2_events)
            eng._k2_events = None
    torch.cuda.synchronize()
    k2_ms = [a.elapsed_time(b) for a, b in k2_events]
    del packed
    for _ in range(max(args.warmup, 3)):
        step_e2e()
    sampler.active = True
    ms_e2e, res_e2e = timed(step_e2e, args.steps)
    sampler.stop_flag = True
    if args.dump_outputs:
        outputs.update(zip(("e2e_leaf_cards", "e2e_prefix_union_cards", "e2e_union_cards"), res_e2e))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)

    total_bases = bases * world  # every rank holds the same number of genomes; sizes differ by < 0.1 %
    value = total_bases / (ms_step / 1e3) / 1e9
    e2e_value = total_bases / (ms_e2e / 1e3) / 1e9

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    try:   # DRAM bytes per K2 launch from the committed `ncu --set full` capture of this same command
        traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_k2_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        traffic = None
    k2_avg_ms = sum(k2_ms) / len(k2_ms)
    bases_per_launch = bases / N_GENOMES
    achieved = bases_per_launch * 1.0 / (k2_avg_ms / 1e3) / 1e9          # 1.0 algorithmic byte per input base
    clocks = sampler.summary()
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    int_peak = 148 * 128 * sm_mhz * 1e6                                    # lane-instructions / s
    sass = _profile_json("r02_k2_sass.json")
    instr_per_update = float(sass.get("instr_per_update_k10_32", 43.0))   # counted from the committed SASS listing
    int_frac = (bases_per_launch * nk * instr_per_update / (k2_avg_ms / 1e3)) / int_peak
    # what actually binds K2 at this size: one scattered 4-byte reduction per (base, k) into the L2-resident table
    red = _profile_json("r02_red_ceiling.json")
    red_rate = bases_per_launch * nk / (k2_avg_ms / 1e3) / 1e9            # G reductions / s
    red_ceiling = red.get("ceiling_f16x2_64mib")

    cores = os.cpu_count() or 1
    threads = max(1, int(cores * 0.95))
    cpu_dt, cpu_bases = cpu_sketch_sample(texts, KS, P, threads)           # the step's 12 genomes: ~10-20 s of CPU work
    cpu_value = cpu_bases / cpu_dt / 1e9
    line = {
        "metric": "Gbp/s sketched (all k)", "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config(world),
        "e2e": {"value": e2e_value, "unit": "Gbp/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(sum(len(t) for t, _ in texts)) + int(orders.nbytes),
                "d2h_bytes_per_step": N_GENOMES * nk * 8 + N_ORDERINGS * N_GENOMES * nk * 8 + (nk * 8 if world > 1 else 0),
                "host_numa_node": numa_node,   # N>1: each rank is bound to the cores of its GPU's NUMA node
                "note": "dd_sketch_fasta_host_async per genome from pinned memory (%d files in flight on as many streams) + " % NS +
                        "progressive unions; every cardinality is copied back to the host, registers stay in HBM"},
        "gpu_launches": int(launches_timed),
        "clocks": clocks,
        "roofline": {"kernel": "sketch_allk_kernel", "bound": "hbm", "achieved": achieved, "peak": hbm_peak,
                     "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                     "traffic_source": "profiles/r02_sketch_allk_cfg2_ncu.md (dram__bytes_read+write per launch, ncu --set full of this command)",
                     "algorithmic_bytes_per_launch": bases_per_launch * 1.0,
                     "peak_source": "MEASURED_PEAKS.json (burst copy)" if peaks else "fallback 6650 GB/s",
                     "algorithmic_bytes_per_base": 1.0, "launch_ms": k2_avg_ms,
                     "share_of_step": sum(k2_ms) / ms_step,
                     "launch_ms_overlapped": sum(k2_overlapped_ms) / len(k2_overlapped_ms),
                     "int32_issue": {"instr_per_update": instr_per_update, "updates_per_base": nk,
                                     "frac_of_issue_peak": int_frac, "sm_mhz": sm_mhz,
                                     "source": "profiles/r02_k2_sass.json"},
                     "red_rate": {"achieved_g_per_s": red_rate, "ceiling_g_per_s": red_ceiling,
                                  "red_rate_frac": (red_rate / red_ceiling) if red_ceiling else None,
                                  "source": "profiles/r02_red_ceiling.json (experiments/red_ceiling.cu on a B200 of this pool)"},
                     "note": "K2 is INT32-issue / L2-scattered-update bound, not HBM bound (SURVEY.md 8d); both fractions reported"},
        "cpu_baseline": {"value": cpu_value, "unit": "Gbp/s", "cores": threads, "kind": "port",
                         "sample": f"{N_GENOMES} genomes x 5 Mbp x 23 k, p=20, one single-threaded oracle job per (genome,k), "
                                   f"{threads} in flight ({cpu_dt:.2f} s wall; leaf sketches + cardinalities only)"},
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------ config 3 arms
KS3 = list(range(2, 33))
CPU_SAMPLE_BASES_3 = 256_000_000


def human_like_sample(bases, seed=3):
    """numpy stand-in for tools/synth.synth_fasta (24 records, ~1 % N runs, 50 % lower case, 80 columns),
    used for the CPU arm's bounded sample."""
    rng = np.random.default_rng(seed)
    out = []
    per = bases // 24 // LINE * LINE
    for r in range(24):
        b = ACGT[rng.integers(0, 4, per)]
        b = np.where(rng.random(per) < 0.5, b | 0x20, b).astype(np.uint8)
        for st in rng.integers(0, max(1, per - 1000), max(1, per // 100000)):
            b[st:st + 1000] = ord("N")
        body = np.empty((per // LINE, LINE + 1), dtype=np.uint8)
        body[:, :LINE] = b.reshape(-1, LINE)
        body[:, LINE] = 10
        out.append(b">chr%d synthetic length=%d\n" % (r + 1, per) + body.tobytes())
    return b"".join(out), per * 24


def cpu_sample_config3(text, bases, threads):
    """One single-threaded oracle sketch job per k (the reference's `parallel ... ::: k` topology), all 31 k."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as orc
    sym = orc.fasta_symbols(text)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(lambda k: orc.card(orc.hll_sketch(sym, k, P), P), KS3))
    return time.perf_counter() - t0, bases


def workload_config3(n_gpus, bases):
    return {"workload": f"config 3: one synthetic human-scale assembly of {bases / 1e9:.2f} Gbp per GPU (24 records, ~1% N runs, "
                        "50% soft-masked; copies 0.1% substitutions apart), k=2..32 (31 k), p=20, leaf sketch + cardinalities, "
                        "all-gather of the registers, prefix unions of the identity ordering",
            "genomes_per_gpu": 1, "genome_bp": int(bases), "k_min": 2, "k_max": 32, "registers_log2": P,
            "parallelism": f"one genome per GPU over {n_gpus} GPU(s)",
            "l2_policy": "per-step working set (3.1 GB text, 1.2 GB packed stream) exceeds the 126 MB L2; no explicit flush"}


def run_reference_config3(args, threads):
    text, bases = human_like_sample(CPU_SAMPLE_BASES_3)
    secs = [cpu_sample_config3(text, bases, threads)[0] for _ in range(max(1, args.steps))]
    ms = 1e3 * sum(secs) / len(secs)
    value = bases / (ms / 1e3) / 1e9
    sample = (f"{bases / 1e6:.0f} Mbp sample of one human-like genome x 31 k (k=2..32), p=20, one single-threaded oracle job "
              f"per k, {threads} in flight; Gbp/s is size-independent for this path, so the sample stands for the 3.1 Gbp genome")
    emit({"impl": "reference", "metric": "Gbp/s sketched (all k)", "value": value, "unit": "Gbp/s", "n_gpus": args.gpus,
          "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config3(args.gpus, args.bases),
          "cpu_baseline": {"value": value, "unit": "Gbp/s", "cores": threads, "kind": "port", "sample": sample},
          "e2e": {"value": value, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


def run_ours_config3(args):
    import torch
    import torch.distributed as dist
    from dandd_b200 import build
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank == 0:
        build.build()
    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    torch.cuda.set_device(local)
    from dandd_b200 import dist as dd_dist
    if world > 1:
        dd_dist.init("nccl")
        dist.barrier()
    from dandd_b200.engine import Engine
    from tools.synth import mutate_text, synth_fasta
    eng = Engine(local)
    dev = eng.device
    nk, m, bases = len(KS3), 1 << P, int(args.bases)
    text = synth_fasta(bases, 24, seed=3, device=dev)
    if rank:
        text = mutate_text(text, 0.001, 3 + rank)
    pinned = torch.empty(text.numel(), dtype=torch.uint8).pin_memory()
    pinned.copy_(text)
    torch.cuda.synchronize()
    regs = torch.empty((1, nk, m), dtype=torch.uint8, device=dev)
    hist = torch.empty((nk, 64), dtype=torch.int32, device=dev)
    cards_host = torch.empty(nk, dtype=torch.float64).pin_memory()
    owners = [[r] for r in range(world)]
    order = [list(range(world))]
    k2_events = []

    orig_update = eng._update_from_state

    def hooked(seq, kmask, p, canon, ws, st):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_update(seq, kmask, p, canon, ws, st)
        e1.record()
        k2_events.append((e0, e1))
    eng._update_from_state = hooked

    def unions():
        """the one exchange step: every rank gets every leaf (NCCL all-gather), then the prefix unions"""
        allr = dd_dist.gather_registers(regs, owners) if world > 1 else regs
        return eng.prefix_union_cards(allr, order, P)

    def step_resident():
        seq = eng.pack(text, start=0)
        eng.sketch(seq, KS3, p=P, out=regs[0], hist_out=hist)
        return eng.mle(hist, P), unions()

    def step_e2e():
        eng.sketch_fasta_host(pinned, KS3, p=P, want_regs=False, out_dev=regs[0], cards_out=cards_host, sync=False)
        prog = unions().cpu()
        torch.cuda.synchronize()
        return cards_host, prog

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), res

    sampler = ClockSampler(local, period=0.05)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    k2_events.clear()
    sampler.active = True
    launches0 = eng.lib.dd_kernel_launches()
    ms_step, res = timed(step_resident, args.steps)
    launches_timed = eng.lib.dd_kernel_launches() - launches0
    sampler.active = False
    outputs = {}
    if args.dump_outputs:     # the last timed step's results, taken before the e2e steps below rewrite regs
        outputs = {"leaf_cards": res[0], "prefix_union_cards": res[1], "registers_sample": register_sample(regs)}
    k2_ms = [a.elapsed_time(b) for a, b in k2_events]
    for _ in range(max(args.warmup, 3)):
        step_e2e()
    sampler.active = True
    ms_e2e, res_e2e = timed(step_e2e, args.steps)
    sampler.stop_flag = True
    if args.dump_outputs:
        outputs.update(e2e_leaf_cards=res_e2e[0], e2e_prefix_union_cards=res_e2e[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    total_bases = bases * world
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    k2_avg = sum(k2_ms) / len(k2_ms)
    achieved = bases * 1.0 / (k2_avg / 1e3) / 1e9
    clocks = sampler.summary()
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    sass = _profile_json("r02_k2_sass.json")
    ipu = float(sass.get("instr_per_update_k2_32_floor", 38.0))
    int_frac = (bases * nk * ipu / (k2_avg / 1e3)) / (148 * 128 * sm_mhz * 1e6)
    threads = max(1, int((os.cpu_count() or 1) * 0.95))
    sample_text = text[: CPU_SAMPLE_BASES_3 * 81 // 80 + 4096].cpu().numpy().tobytes()
    sample_text = sample_text[:sample_text.rfind(b"\n") + 1]
    sample_bases = int(np.isin(np.frombuffer(sample_text, dtype=np.uint8) & 0xDF, [65, 67, 71, 84, 78]).sum())   # letters, N included
    cpu_dt, _ = cpu_sample_config3(sample_text, sample_bases, threads)
    cpu_value = sample_bases / cpu_dt / 1e9
    emit({
        "metric": "Gbp/s sketched (all k)", "value": total_bases / (ms_step / 1e3) / 1e9, "unit": "Gbp/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config3(world, bases),
        "e2e": {"value": total_bases / (ms_e2e / 1e3) / 1e9, "unit": "Gbp/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(text.numel()), "d2h_bytes_per_step": nk * 8 + world * nk * 8, "host_numa_node": numa_node,
                "note": "dd_sketch_fasta_host_async from pinned memory (32 MiB chunks, copies double-buffered against K1+K2), "
                        "register all-gather, prefix unions; every cardinality is copied back to the host"},
        "gpu_launches": int(launches_timed), "clocks": clocks,
        "roofline": {"kernel": "sketch_allk_kernel", "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": None, "algorithmic_bytes_per_launch": bases * 1.0,
                     "algorithmic_bytes_per_base": 1.0, "launch_ms": k2_avg,
                     "launch_note": "one genome's K2 work: the sketch launches between the floor schedule's cuts plus the refreshes",
                     "share_of_step": k2_avg / ms_step,
                     "peak_source": "MEASURED_PEAKS.json (burst copy)" if peaks else "fallback 6650 GB/s",
                     "int32_issue": {"instr_per_update": ipu, "updates_per_base": nk, "frac_of_issue_peak": int_frac, "sm_mhz": sm_mhz,
                                     "source": "profiles/r02_k2_sass.json"},
                     "note": "K2 is ALU-issue bound at this size (SURVEY.md 8d), not HBM bound; both fractions reported"},
        "cpu_baseline": {"value": cpu_value, "unit": "Gbp/s", "cores": threads, "kind": "port",
                         "sample": f"{sample_bases / 1e6:.0f} Mbp of this rank's genome x 31 k, one single-threaded oracle job per k, "
                                   f"{threads} in flight ({cpu_dt:.2f} s wall)"},
    })
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3],
                    help="BASELINE.json workload: 2 = 12 x 5 Mbp per GPU (default, the metric's configuration), "
                         "3 = one 3.1 Gbp assembly per GPU, k = 2..32")
    ap.add_argument("--bases", type=float, default=3.1e9, help="config 3: bases per genome")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy: "
                         "float64 cardinalities and a fixed sample of the registers as float32 (rank 0).  Only with "
                         "--impl ours: it compares builds of this project, and the CPU arm keeps no results")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
