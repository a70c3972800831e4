"""What edit tracking (gp_config.track_edits) costs the polish, against the parent commit's library.

Per workload -- configs[1] (5 Mbp draft, 30x reads, bsize 1) and configs[2] (100 Mbp draft, 40x reads, bsize 8) -- and
per round, three arms run in one process, in an order that rotates from round to round: the base library (--base-lib,
tracking unknown to it), the in-tree library with tracking off, and the in-tree library with tracking on.  Each arm
builds the filters, polishes once to warm up, then times `reps` polishes: the edit kernel's device time
(stats()["edit_kernel_ms"], CUDA events around the kernel) and, with tracking on, the host clock around the first
polish_fetch_edits after each polish (the derivation kernels and scans, their synchronisations and the copy of the
records to the host).  Prints and writes one JSON document; the card's name and power limit are part of it.

usage: python profiles/edit_records_cost.py --base-lib PATH [--rounds 3] [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "config2_5mbp_30x_bsize1": dict(genome_len=5_000_000, coverage=30.0, bsize=1),
    "config3_100mbp_40x_bsize8": dict(genome_len=100_000_000, coverage=40.0, bsize=8),
}
SEED = 20250607


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def arm(gp, lib, d, pl, track, reps):
    gp.api._lib = lib  # Context binds the library loaded last
    ctx = gp.Context(track_edits=track)
    try:
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        edit_ms, fetch_ms, n_rec = [], [], 0
        for r in range(reps + 1):
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.polish_run()
            out, off, dropped = ctx.polish_fetch()
            ms = ctx.stats()["edit_kernel_ms"]
            if track:
                t0 = time.perf_counter()
                rec = ctx.polish_fetch_edits()
                t1 = time.perf_counter()
                n_rec = len(rec["pos"])
            if r:  # the first polish warms up
                edit_ms.append(ms)
                if track:
                    fetch_ms.append((t1 - t0) * 1e3)
        return dict(edit_kernel_ms=edit_ms, fetch_edits_ms=fetch_ms, records=n_rec, polished_bytes=int(off[-1]))
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "edit_records_cost.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    a = ap.parse_args()
    import goldpolish_b200 as gp
    import sim
    new = gp.load_library()

    class Tolerant:  # the base library lacks the entry points this change adds: their argtypes go nowhere
        def __init__(self, lib):
            self._lib = lib

        def __getattr__(self, n):
            try:
                return getattr(self._lib, n)
            except AttributeError:
                return types.SimpleNamespace()

    cdll = C.CDLL
    gp.api._lib = None
    os.environ["GP_LIB_PATH"] = os.path.abspath(a.base_lib)
    C.CDLL = lambda path: Tolerant(cdll(path))
    try:
        base = gp.load_library()
    finally:
        C.CDLL = cdll
        del os.environ["GP_LIB_PATH"]
    libs = {"base": (base, False), "tree_off": (new, False), "tree_on": (new, True)}
    doc = dict(card=card(), rounds=a.rounds, reps=a.reps, results={})
    for name in a.workloads.split(","):
        w = WORKLOADS[name]
        d = sim.simulate(genome_len=w["genome_len"], coverage=w["coverage"], seed=SEED)
        pl = gp.plan_batches(np.diff(d.contig_off), [d.contig_name(i) for i in range(d.n_contigs)],
                             [d.read_name(i) for i in range(d.n_reads)], d.read_phred, np.diff(d.read_off),
                             d.map_read, d.map_contig, bsize=w["bsize"], subsample_max_per_10kbp=40.0)
        res = {k: [] for k in libs}
        order = list(libs)
        for r in range(a.rounds):
            for k in order[r % 3:] + order[:r % 3]:
                lib, track = libs[k]
                res[k].append(arm(gp, lib, d, pl, track, a.reps))
                print(name, "round", r, k, json.dumps({x: res[k][-1][x] for x in ("edit_kernel_ms", "fetch_edits_ms")}),
                      flush=True)
        summ = {}
        for k, runs in res.items():
            med = [float(np.median(x["edit_kernel_ms"])) for x in runs]
            summ[k] = dict(edit_kernel_ms_median_per_round=med, edit_kernel_ms_min=min(min(x["edit_kernel_ms"]) for x in runs),
                           polished_bytes=runs[-1]["polished_bytes"])
            if k == "tree_on":
                summ[k]["fetch_edits_ms_median_per_round"] = [float(np.median(x["fetch_edits_ms"])) for x in runs]
                summ[k]["records"] = runs[-1]["records"]
        doc["results"][name] = dict(draft_bases=int(d.contig_off[-1]), contigs=int(d.n_contigs), summary=summ, runs=res)
        print(name, json.dumps(summ), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: v["summary"] for k, v in doc["results"].items()}))


if __name__ == "__main__":
    main()
