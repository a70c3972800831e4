"""What k-mer support (gp_config.kmer_support) costs the overlapped pass, against the parent commit's library.

Per workload -- configs[1] (5 Mbp draft, 30x reads, bsize 1) and configs[2] (100 Mbp draft, 40x reads, bsize 8) -- and
per round, three arms run in one process, in an order that rotates from round to round: the base library (--base-lib,
the option unknown to it), the in-tree library with the option off, and the in-tree library with it on.  Each arm
stages the work once, runs one gp_pipeline_run to warm up, then times `reps` of them as bench.py times a step (CUDA
events around pipeline_run on the context's stream), and records the edit kernel's device time (stats()).  After the
rounds one more pass of the "on" arm runs under torch.profiler (CUDA activities): the device time of the support
kernels (support_steps / support_count / support_popcount and the scan between them -- the only scan of a pass without
track_edits).  Prints and writes one JSON document; the card's name and power limit are part of it.

usage: python profiles/kmer_support_cost.py --base-lib PATH [--rounds 3] [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
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
SUPPORT_KERNELS = ("support_steps_kernel", "support_count_kernel", "support_popcount_kernel", "DeviceScan")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def staged(gp, lib, d, pl, on):
    import torch
    gp.api._lib = lib  # Context binds the library loaded last
    ctx = gp.Context(kmer_support=on) if on else gp.Context()
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.upload_reads(d.read_seq, d.read_off)
    ctx.build_stage(pl.batch_entry_off, pl.entries)
    ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
    return ctx, stream


def arm(gp, lib, d, pl, on, reps):
    import torch
    ctx, stream = staged(gp, lib, d, pl, on)
    try:
        step_ms, edit_ms = [], []
        for r in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.pipeline_run()
            e1.record(stream)
            e1.synchronize()
            if r:  # the first pass warms up
                step_ms.append(e0.elapsed_time(e1))
                edit_ms.append(ctx.stats()["edit_kernel_ms"])
        out, off, dropped = ctx.polish_fetch()
        res = dict(step_ms=step_ms, edit_kernel_ms=edit_ms, polished_bytes=int(off[-1]))
        if on:
            counts, bits = ctx.polish_fetch_support()
            tot = counts.sum(axis=0)
            res["kmers_per_k"] = tot[:, 0].tolist()
            res["support_totals"] = tot.tolist()
        return res
    finally:
        ctx.close()


def profiled_support(gp, lib, d, pl):
    """Device time of the support kernels in one overlapped pass, by torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctx, stream = staged(gp, lib, d, pl, True)
    try:
        ctx.pipeline_run()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.pipeline_run()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA and any(s in ev.name for s in SUPPORT_KERNELS):
                key = next(s for s in SUPPORT_KERNELS if s in ev.name)
                t = getattr(ev, "device_time", None)
                if t is None:
                    t = ev.cuda_time
                per.setdefault(key, [0.0, 0])
                per[key][0] += t / 1e3
                per[key][1] += 1
        return dict(kernels_ms={k: v[0] for k, v in per.items()}, launches={k: v[1] for k, v in per.items()},
                    total_ms=sum(v[0] for v in per.values()))
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kmer_support_cost.json"))
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
                lib, on = libs[k]
                res[k].append(arm(gp, lib, d, pl, on, a.reps))
                print(name, "round", r, k, json.dumps({x: res[k][-1][x] for x in ("step_ms", "edit_kernel_ms")}), flush=True)
        summ = {}
        for k, runs in res.items():
            summ[k] = dict(step_ms_median_per_round=[float(np.median(x["step_ms"])) for x in runs],
                           step_ms_min=min(min(x["step_ms"]) for x in runs),
                           edit_kernel_ms_median_per_round=[float(np.median(x["edit_kernel_ms"])) for x in runs],
                           polished_bytes=runs[-1]["polished_bytes"])
        summ["tree_on"]["support_kernels"] = profiled_support(gp, new, d, pl)
        summ["tree_on"]["support_totals_per_k"] = res["tree_on"][-1]["support_totals"]
        doc["results"][name] = dict(draft_bases=int(d.contig_off[-1]), contigs=int(d.n_contigs),
                                    batches=int(len(pl.batch_entry_off) - 1), summary=summ, runs=res)
        print(name, json.dumps(summ), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: v["summary"] for k, v in doc["results"].items()}))


if __name__ == "__main__":
    main()
