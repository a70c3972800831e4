"""Build kernel rate by k list, two builds of the library side by side.

Times gp_build_run alone (the device timer of the kernel, stats()["build_kernel_ms"], after warm-up launches) on two
workloads -- configs[1] (5 Mbp draft, 30x reads, bsize 1) and a 10 Mbp / 40x / bsize-8 cut of configs[2] -- for the
k lists (32, 28, 24, 20), (31, 27, 23, 19) and (30, 26, 22, 18).  With --base-lib, every round runs that library and
the in-tree one in separate processes (GP_LIB_PATH), alternating which goes first, so that both see the same machine
state; lists the base library rejects are recorded as such.  Prints and writes one JSON document.

usage: python profiles/build_rate_by_k.py [--base-lib PATH] [--rounds 3] [--reps 10] [--out profiles/build_rate_by_k.json]
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LISTS = [(32, 28, 24, 20), (31, 27, 23, 19), (30, 26, 22, 18)]
WORKLOADS = {
    "config2_5mbp_30x_bsize1": dict(genome_len=5_000_000, coverage=30.0, bsize=1),
    "cut_10mbp_40x_bsize8": dict(genome_len=10_000_000, coverage=40.0, bsize=8),
}
SEED = 20250607
WARMUP = 2


def make_data(dirpath):
    """Seeded data sets and their batch plans, saved for the measuring processes."""
    import goldpolish_b200 as gp
    import sim
    for name, w in WORKLOADS.items():
        d = sim.simulate(genome_len=w["genome_len"], coverage=w["coverage"], seed=SEED)
        pl = gp.plan_batches(np.diff(d.contig_off), [d.contig_name(i) for i in range(d.n_contigs)],
                             [d.read_name(i) for i in range(d.n_reads)], d.read_phred, np.diff(d.read_off),
                             d.map_read, d.map_contig, bsize=w["bsize"], subsample_max_per_10kbp=40.0)
        np.savez(os.path.join(dirpath, name + ".npz"), read_seq=d.read_seq, read_off=d.read_off,
                 batch_entry_off=pl.batch_entry_off, entries=pl.entries)


def measure(dirpath, reps):
    """One library (GP_LIB_PATH or in-tree): build_kernel_ms of every launch, per workload and k list."""
    import goldpolish_b200 as gp
    out = {}
    for name in WORKLOADS:
        z = np.load(os.path.join(dirpath, name + ".npz"))
        for ks in LISTS:
            key = f"{name}/k{'-'.join(map(str, ks))}"
            try:
                ctx = gp.Context(ks=ks)
            except gp.GpError as e:
                out[key] = {"error": str(e)}
                continue
            with ctx:
                ctx.upload_reads(z["read_seq"], z["read_off"])
                try:
                    ctx.build_stage(z["batch_entry_off"], z["entries"])
                except gp.GpError as e:
                    out[key] = {"error": str(e)}
                    continue
                ms = []
                for i in range(WARMUP + reps):
                    ctx.build_run()
                    ctx.synchronize()
                    if i >= WARMUP:
                        ms.append(ctx.stats()["build_kernel_ms"])
                st = ctx.stats()
                out[key] = {"kmer_ops": int(st["kmer_ops"]), "build_kernel_ms": ms}
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except OSError:
        return "unknown"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def summary(runs):
    """Per library and point: the rate of every round (G k-mer ops/s over the mean kernel time of its launches)."""
    res = {}
    for lib, rounds in runs.items():
        for r in rounds:
            for key, v in r.items():
                e = res.setdefault(key, {}).setdefault(lib, {"round_gops": [], "launch_ms": []})
                if "error" in v:
                    e["error"] = v["error"]
                    continue
                e["round_gops"].append(v["kmer_ops"] / (np.mean(v["build_kernel_ms"]) * 1e-3) / 1e9)
                e["launch_ms"] += v["build_kernel_ms"]
                e["kmer_ops"] = v["kmer_ops"]
    for key, libs in res.items():
        for lib, e in libs.items():
            if e["round_gops"]:
                g = e["round_gops"]
                e.update(mean_gops=float(np.mean(g)), min_gops=float(min(g)), max_gops=float(max(g)),
                         spread_pct=float((max(g) - min(g)) / np.mean(g) * 100.0),
                         launch_ms_min=float(min(e["launch_ms"])), launch_ms_max=float(max(e["launch_ms"])))
            e.pop("launch_ms", None)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", default=None, help="another build of libgoldpolish_b200.so to compare with")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "build_rate_by_k.json"))
    ap.add_argument("--measure", default=None, help=argparse.SUPPRESS)  # (child process: data directory)
    a = ap.parse_args()
    if a.measure:
        print(json.dumps(measure(a.measure, a.reps)))
        return
    tmp = tempfile.mkdtemp(prefix="gp_rate_by_k_")
    try:
        t0 = time.time()
        make_data(tmp)
        libs = {"in_tree": None}
        if a.base_lib:
            libs["base"] = os.path.abspath(a.base_lib)
        runs = {lib: [] for lib in libs}
        order = list(libs)
        for r in range(a.rounds):
            for lib in (order if r % 2 == 0 else order[::-1]):
                env = dict(os.environ)
                env.pop("GP_LIB_PATH", None)
                if libs[lib]:
                    env["GP_LIB_PATH"] = libs[lib]
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--measure", tmp, "--reps", str(a.reps)],
                                   env=env, capture_output=True, text=True, check=True)
                runs[lib].append(json.loads(p.stdout.strip().splitlines()[-1]))
                print(f"round {r} {lib} done", file=sys.stderr, flush=True)
        doc = {"what": "build kernel alone (gp_build_run, device timer), G k-mer ops/s per round = kmer_ops / mean "
                       f"launch time of {a.reps} launches after {WARMUP} warm-up ones; rounds alternate the libraries",
               "card": card(), "workloads": WORKLOADS, "lists": LISTS, "rounds": a.rounds,
               "libraries": {k: (v or "in-tree") for k, v in libs.items()},
               "summary": summary(runs), "runs": runs, "wall_s": time.time() - t0}
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)
        print(json.dumps(doc["summary"], indent=1))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
