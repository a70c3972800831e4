"""What keeping the unsupported k-mer starts (the bitmap behind gp_polish_fetch_unsupported) costs the overlapped pass
with gp_config.kmer_support on, against the library before it (which counts support the same way, without the bitmap).

Per workload -- configs[1] (5 Mbp draft, 30x reads, bsize 1) and configs[2] (100 Mbp draft, 40x reads, bsize 8) -- and
per round, two arms run in one process, alternating, the first arm rotating from round to round: the base library
(--base-lib) and the in-tree library, both with kmer_support on.  Each arm stages the work once, runs one
gp_pipeline_run to warm up, then times `reps` of them as bench.py times a step (CUDA events around pipeline_run on the
context's stream).  After the timed passes the in-tree arm times its first polish_fetch_unsupported (host clock, the
derivation and the copy to the host) and records the run count.  Both arms' support counts and polished bytes are
compared.  After the rounds one more pass of each arm runs under torch.profiler (CUDA activities): the device time of
the support kernels, and of the derivation kernels at the first fetch.  Prints and writes one JSON document; the card's
name and power limit are part of it.

usage: python profiles/kmer_unsupported_cost.py --base-lib PATH [--rounds 3] [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
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
SUPPORT_KERNELS = ("support_steps_kernel", "support_count_kernel", "support_popcount_kernel")
DERIVE_KERNELS = ("unsupported_count_kernel", "unsupported_fill_kernel", "unsupported_off_kernel", "DeviceScan")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def staged(gp, lib, d, pl):
    import torch
    gp.api._lib = lib  # Context binds the library loaded last
    ctx = gp.Context(kmer_support=True)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.upload_reads(d.read_seq, d.read_off)
    ctx.build_stage(pl.batch_entry_off, pl.entries)
    ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
    return ctx, stream


def arm(gp, lib, d, pl, reps, runs):
    import torch
    ctx, stream = staged(gp, lib, d, pl)
    try:
        step_ms = []
        for r in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.pipeline_run()
            e1.record(stream)
            e1.synchronize()
            if r:  # the first pass warms up
                step_ms.append(e0.elapsed_time(e1))
        out, off, dropped = ctx.polish_fetch()
        counts, bits = ctx.polish_fetch_support()
        res = dict(step_ms=step_ms, polished_bytes=int(off[-1]),
                   polished_sha=hashlib.sha256(out[:int(off[-1])].tobytes()).hexdigest()[:16],
                   counts_sha=hashlib.sha256(counts.tobytes()).hexdigest()[:16],
                   support_totals=counts.sum(axis=0).tolist())
        if runs:
            t0 = time.perf_counter()
            u = ctx.polish_fetch_unsupported()
            res["first_fetch_unsupported_ms"] = (time.perf_counter() - t0) * 1e3
            res["runs"] = int(len(u["start"]))
            res["run_kmers"] = int(u["kmers"].astype(np.uint64).sum())
            res["run_bases"] = int((u["end"].astype(np.int64) - u["start"]).sum())
            t0 = time.perf_counter()
            ctx.polish_fetch_unsupported()
            res["cached_fetch_unsupported_ms"] = (time.perf_counter() - t0) * 1e3
        return res
    finally:
        ctx.close()


def profiled(gp, lib, d, pl, runs):
    """Device time of the support kernels in one overlapped pass (and of the derivation at the first fetch)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctx, stream = staged(gp, lib, d, pl)
    try:
        ctx.pipeline_run()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.pipeline_run()
            torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof2:
            ctx.polish_fetch()
            if runs:
                ctx.polish_fetch_unsupported()
            torch.cuda.synchronize()

        def sums(p, names):
            per = {}
            for ev in p.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA and any(s in ev.name for s in names):
                    key = next(s for s in names if s in ev.name)
                    t = getattr(ev, "device_time", None)
                    if t is None:
                        t = ev.cuda_time
                    per.setdefault(key, [0.0, 0])
                    per[key][0] += t / 1e3
                    per[key][1] += 1
            return dict(kernels_ms={k: v[0] for k, v in per.items()}, launches={k: v[1] for k, v in per.items()},
                        total_ms=sum(v[0] for v in per.values()))
        res = dict(support=sums(prof, SUPPORT_KERNELS))
        if runs:
            res["derive"] = sums(prof2, DERIVE_KERNELS)
        return res
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kmer_unsupported_cost.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    a = ap.parse_args()
    import goldpolish_b200 as gp
    import sim
    new = gp.load_library()

    class Tolerant:  # the base library lacks the entry point this change adds: its argtypes go nowhere
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
    libs = {"base": (base, False), "tree": (new, True)}
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
            for k in order[r % 2:] + order[:r % 2]:
                lib, runs = libs[k]
                res[k].append(arm(gp, lib, d, pl, a.reps, runs))
                print(name, "round", r, k, json.dumps({x: v for x, v in res[k][-1].items() if x != "support_totals"}), flush=True)
        summ = {}
        for k, rs in res.items():
            summ[k] = dict(step_ms_median_per_round=[float(np.median(x["step_ms"])) for x in rs],
                           step_ms_min=min(min(x["step_ms"]) for x in rs),
                           polished_bytes=rs[-1]["polished_bytes"])
            summ[k].update(profiled(gp, libs[k][0], d, pl, libs[k][1]))
        t = res["tree"]
        summ["tree"].update(first_fetch_unsupported_ms=[x["first_fetch_unsupported_ms"] for x in t],
                            cached_fetch_unsupported_ms=[x["cached_fetch_unsupported_ms"] for x in t],
                            runs=t[-1]["runs"], run_kmers=t[-1]["run_kmers"], run_bases=t[-1]["run_bases"])
        summ["same_output"] = all(x["polished_sha"] == res["base"][0]["polished_sha"] and x["counts_sha"] == res["base"][0]["counts_sha"]
                                  for x in res["base"] + res["tree"])
        summ["support_totals_per_k"] = res["tree"][-1]["support_totals"]
        summ["runs_kmers_equal_missing"] = t[-1]["run_kmers"] == int(sum(r[0] - r[1] + r[2] - r[3] for r in summ["support_totals_per_k"]))
        doc["results"][name] = dict(draft_bases=int(d.contig_off[-1]), contigs=int(d.n_contigs),
                                    batches=int(len(pl.batch_entry_off) - 1), summary=summ, runs=res)
        print(name, json.dumps(summ), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({k: v["summary"] for k, v in doc["results"].items()}))


if __name__ == "__main__":
    main()
