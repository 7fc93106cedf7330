#!/usr/bin/env python
"""Wall time of the UNMODIFIED reference command line on the config-2 inputs with the CPU oracle
behind stand-in `dashing` / `parallel` executables (oracle/shims) -- the "reference-equivalent CPU
proxy" of SURVEY.md 8(d): same process topology as the reference (one single-threaded process per
(file, k), floor(0.95 * cores) at a time, genomes sequential, one `dashing union` + `dashing card`
process per prefix union).  Needs DANDD_REFERENCE to name a checkout of the reference; the
result is committed under profiles/.   usage: reference_cli_cpu_time.py [n_orderings] [out.json]"""
import json
import os
import pickle
import random
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import pyoracle  # noqa: E402
from tests.util import reference_path  # noqa: E402

REF = reference_path("lib")


def main():
    if not REF:
        sys.exit("set DANDD_REFERENCE to a checkout of the reference")
    n_ord = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    out_json = sys.argv[2] if len(sys.argv) > 2 else None
    cores = os.cpu_count() or 1
    jobs = max(1, int(cores * 0.95))
    work = tempfile.mkdtemp(prefix="dd_refcli_")
    rep = {"cores": cores, "parallel_jobs": jobs, "orderings": n_ord,
           "what": "unmodified reference lib/dandd + oracle-backed dashing/parallel stand-ins, config 2 (12 x 5 Mbp, k=10..32)"}
    try:
        bindir = os.path.join(work, "bin")
        pyoracle.install_shims(bindir)
        data = os.path.join(work, "fastas")
        os.makedirs(data)
        for i, (text, _) in enumerate(bench.make_genomes(seed=2)):
            with open(os.path.join(data, f"genome{i:02d}.fasta"), "wb") as fh:
                fh.write(text)
        random.seed(2)
        orderings = set()
        while len(orderings) < n_ord:
            orderings.add(tuple(random.sample(range(12), 12)))
        ofile = os.path.join(work, "orderings.pickle")
        with open(ofile, "wb") as fh:
            pickle.dump(orderings, fh)
        env = dict(os.environ, PATH=bindir + os.pathsep + os.environ["PATH"], PYTHONPATH=REF, PYTHONHASHSEED="0",
                   ORC_PARALLEL_JOBS=str(jobs))
        out = os.path.join(work, "out")
        sweep = ["--ksweep", "--mink", "10", "--maxk", "32"]

        def run(argv):
            t0 = time.perf_counter()
            subprocess.run([sys.executable, os.path.join(REF, "dandd")] + argv, check=True, env=env, stdout=subprocess.DEVNULL,
                           stderr=subprocess.DEVNULL)
            return time.perf_counter() - t0

        rep["tree_ksweep_s"] = run(["tree", "-d", data, "-s", "cfg2", "-k", "14", "-o", out] + sweep)
        print(json.dumps(rep), flush=True)
        dtree = os.path.join(out, "cfg2_12_dashing_dtree.pickle")
        rep["progressive_s"] = run(["progressive", "-d", dtree, "-r", ofile, "-o", out] + sweep)
    finally:
        shutil.rmtree(work, ignore_errors=True)
    print(json.dumps(rep))
    if out_json:
        with open(out_json, "w") as fh:
            json.dump(rep, fh, indent=1)


if __name__ == "__main__":
    main()
