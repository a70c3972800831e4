#!/usr/bin/env python
"""bench.py -- polished Mbp/s of the GoldPolish hot path (filter build + 4 ntEdit rounds + guard).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|5] [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole workload: for every batch, build the 4 (counting filter,
filter) pairs from its mapped reads and run the k=32,28,24,20 ntEdit chain over its contigs, then the 0.75 guard.

Workloads (BASELINE.json `configs`, numbered from 0 there and from 1 in SURVEY.md):
  --config 3 (default)  configs[2] = SURVEY config 3: ONE synthetic 100 Mbp draft, 40x reads, bsize 8.  The same data set
                        on every rank; its batches are sharded over the N GPUs (longest-processing-time on read bases,
                        goldpolish_b200/shard.py), no collective in the data path, and rank 0 gathers the polished
                        records in batch order inside the end-to-end timed region: STRONG scaling.  BASELINE.json quotes
                        its metric ("polished Mbp/s at 1/2/4/8 B200") on this configuration, and it fits one GPU.
  --config 2            configs[1] = SURVEY config 2: 5 Mbp draft, 30x reads, bsize 1 (round 1's bench line); with N > 1
                        every rank polishes a private 5 Mbp data set (weak scaling of replicas).
  --config 5            configs[4] = SURVEY config 5 shape: every rank polishes a private rank-seeded 375 Mbp shard of a
                        3 Gbp draft (30x reads, ntLink-style mappings s=100 x=150, bsize 1), batches streamed through a
                        bounded filter pool.  Weak by construction; meant for --gpus 8.

`value`   : device-resident inputs (packed reads, staged contigs) -> kernels only.
`e2e`     : through the C ABI with HOST buffers: H2D of reads + packing, build, D2H of the filter payloads, H2D of
            contigs, polish, D2H of the polished sequences, the guard, and (N > 1) the gather on rank 0.
`--impl reference` : the reference's own sources (oracle/_ref, compiled from /root/reference) on the host cores,
            a bounded sample of the same workload.  That arm never imports goldpolish_b200.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "polished_mbp_per_s"
UNIT = "Mbp/s"
KS = [32, 28, 24, 20]
ALGO_BYTES_PER_KMER_OP = 256  # 8 random 32-byte sector touches, SURVEY.md §8(d)
BF_BYTES = 524288
SEED = 20250607

WORKLOADS = {
    2: dict(workload="configs[1] (SURVEY config 2): synthetic 5 Mbp draft (contigs ~lognormal median 7 kbp) + 30x simulated "
                     "ONT reads (5% error), PAF mappings s=40, bsize 1, k=32,28,24,20; N>1: one private data set per rank",
            genome_len=5_000_000, coverage=30.0, bsize=1, subsample_max=40.0, mx_max=150.0, mappings="paf",
            scaling="weak"),
    3: dict(workload="configs[2] (SURVEY config 3): ONE synthetic 100 Mbp draft (contigs ~lognormal median 7 kbp) + 40x "
                     "simulated ONT reads (5% error), PAF mappings s=40, bsize 8, k=32,28,24,20; batches sharded over the "
                     "N GPUs, polished records gathered on rank 0",
            genome_len=100_000_000, coverage=40.0, bsize=8, subsample_max=40.0, mx_max=150.0, mappings="paf",
            scaling="strong"),
    5: dict(workload="configs[4] (SURVEY config 5) shape: 3 Gbp draft as rank-seeded 375 Mbp shards, one per GPU, 30x "
                     "simulated ONT reads, ntLink-style mappings (s=100, x=150, minimizer filter), bsize 1, "
                     "k=32,28,24,20; filters streamed through a bounded pool",
            genome_len=375_000_000, coverage=30.0, bsize=1, subsample_max=100.0, mx_max=150.0, mappings="ntlink",
            scaling="weak"),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_JSON_FD = None


def own_stdout():
    """Keep stdout for the ONE JSON line: anything a library prints there (NCCL announces its version on stdout)
    goes to stderr instead."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def config_of(args) -> dict:
    """The `config` object of the JSON line: identical in both arms (what is measured, not how)."""
    w = WORKLOADS[args.config]
    read_bases = w["genome_len"] * w["coverage"]
    return {"workload": w["workload"], "genome_len": w["genome_len"], "coverage": w["coverage"], "bsize": w["bsize"],
            "subsample_max": w["subsample_max"], "mx_max": w["mx_max"], "mappings": w["mappings"], "ks": KS,
            "seed": SEED,
            "l2": "inputs larger than L2: a step streams ~%.0f MB of 2-bit packed reads + masks and %.2f GB of filter "
                  "payloads through the 126 MB L2 (the build kernel's own 80 MiB of timestamps are L2-resident by design)"
                  % (read_bases * 0.375 / 1e6, w["genome_len"] / 9200.0 / w["bsize"] * 4 * BF_BYTES / 1e9)}


def make_dataset(args, rank: int):
    import sim
    w = WORKLOADS[args.config]
    seed = SEED if w["scaling"] == "strong" else SEED + 1000003 * rank
    return sim.simulate(genome_len=w["genome_len"], coverage=w["coverage"], seed=seed)


def n_batches_of(d, bsize):
    return (d.n_contigs + bsize - 1) // bsize


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, device_index: int):
        self.path = tempfile.mktemp(prefix="gp_clocks_", suffix=".csv")
        self.proc = None
        self.idx = device_index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for ln in open(self.path):
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kmer_ops_per_launch):
    """DRAM bytes per launch of the build kernel: the committed `ncu --set full` capture
    (profiles/build_kernel_dram.json) gives bytes per k-mer op; scaled to the k-mer ops of this launch."""
    p = os.path.join(ROOT, "profiles", "build_kernel_dram.json")
    if os.path.exists(p):
        try:
            per_op = json.load(open(p)).get("dram_bytes_per_kmer_op")
            return None if per_op is None else per_op * kmer_ops_per_launch
        except Exception:
            return None
    return None


# ----------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own sources on the host cores (never imports goldpolish_b200)
# ----------------------------------------------------------------------------------------------
def sample_batches(args, d, threads: int) -> int:
    """How many leading batches one CPU step covers: about --ref-bases-per-core draft bases per host core."""
    w = WORKLOADS[args.config]
    nb_total = n_batches_of(d, w["bsize"])
    mean_batch = float(d.contig_off[-1]) / max(nb_total, 1)
    nb = int(round(threads * args.ref_bases_per_core / max(mean_batch, 1.0)))
    return max(min(nb_total, max(nb, threads, 8)), 1)


def reference_arm(args, rank, world):
    if rank != 0:
        return
    d = make_dataset(args, 0)
    w = WORKLOADS[args.config]
    nb_total = n_batches_of(d, w["bsize"])
    threads = os.cpu_count() or 1
    nb = sample_batches(args, d, threads)
    from oracle.ref_sample import ReferenceSample
    rs = ReferenceSample(WORKLOADS[args.config], d, range(nb), threads)
    try:
        times, res = [], None
        for it in range(args.warmup + args.steps):
            res = rs.run()
            if it >= args.warmup:
                times.append(res["seconds_build"] + res["seconds_edit"])
        t = float(np.mean(times))
        val = res["bases"] / 1e6 / t
        sample = (f"first {res['batches']} of {nb_total} batches ({res['bases']} of {int(d.contig_off[-1])} draft bases) per step; "
                  f"last step: build {res['seconds_build']:.2f}s + edit {res['seconds_edit']:.2f}s; "
                  f"steps min/mean/max {min(times):.2f}/{t:.2f}/{max(times):.2f}s; value = sample bases / mean step time")
        emit({
            "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
            "dtype": "u8/u64 integer", "data": "synthetic (seeded simulator, sim/gpsim.c)", "impl": "reference",
            "config": config_of(args),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": res["cores"], "kind": res["kind"], "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        })
        assert "goldpolish_b200" not in sys.modules, "the reference arm must not load the product"
    finally:
        rs.close()


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
class LocalShare:
    """This rank's part of the workload: its batches (global indices, ascending), their contigs and the reads their
    entries name, re-indexed into a rank-local read store."""

    def __init__(self, d, pl, my_batches, bsize):
        self.batches = np.asarray(my_batches, dtype=np.int64)
        if len(my_batches) == len(pl.batch_entry_off) - 1:  # the whole data set: nothing to cut out or re-index
            self.batch_entry_off, self.entries = pl.batch_entry_off, pl.entries
            self.read_off, self.read_seq, self.n_reads = d.read_off, d.read_seq, d.n_reads
            self.contigs = np.arange(d.n_contigs, dtype=np.int64)
            self.contig_off, self.contig_seq, self.contig_batch = d.contig_off, d.contig_seq, pl.contig_batch
            self.name_len = np.array([len(d.contig_name(int(c))) for c in self.contigs], dtype=np.int64)
            self.draft_bases = int(self.contig_off[-1])
            return
        off = pl.batch_entry_off.astype(np.int64)
        ent_idx = np.concatenate([np.arange(off[b], off[b + 1]) for b in my_batches]) if len(my_batches) else np.zeros(0, np.int64)
        ents = pl.entries[ent_idx]
        self.batch_entry_off = np.concatenate([[0], np.cumsum([off[b + 1] - off[b] for b in my_batches])]).astype(np.uint64)
        # local read store: reads in first-use order
        uniq, first = np.unique(ents["read_id"], return_index=True)
        order = uniq[np.argsort(first)]
        remap = np.full(d.n_reads, -1, dtype=np.int64)
        remap[order] = np.arange(len(order))
        self.entries = ents.copy()
        self.entries["read_id"] = remap[ents["read_id"]].astype(np.uint32)
        rl = np.diff(d.read_off)[order]
        self.read_off = np.concatenate([[0], np.cumsum(rl)]).astype(np.int64)
        self.read_seq = np.empty(int(self.read_off[-1]), dtype=np.uint8)
        for i, r in enumerate(order.tolist()):
            self.read_seq[self.read_off[i]:self.read_off[i + 1]] = d.read_seq[d.read_off[r]:d.read_off[r + 1]]
        self.n_reads = len(order)
        # local contigs, in global order
        self.contigs = np.concatenate([np.arange(b * bsize, min((b + 1) * bsize, d.n_contigs)) for b in my_batches]) \
            if len(my_batches) else np.zeros(0, np.int64)
        cl = np.diff(d.contig_off)[self.contigs]
        self.contig_off = np.concatenate([[0], np.cumsum(cl)]).astype(np.int64)
        self.contig_seq = np.empty(int(self.contig_off[-1]), dtype=np.uint8)
        for i, c in enumerate(self.contigs.tolist()):
            self.contig_seq[self.contig_off[i]:self.contig_off[i + 1]] = d.contig_seq[d.contig_off[c]:d.contig_off[c + 1]]
        local_batch_of = {int(b): i for i, b in enumerate(my_batches)}
        self.contig_batch = np.array([local_batch_of[int(c) // bsize] for c in self.contigs], dtype=np.uint32)
        self.name_len = np.array([len(d.contig_name(int(c))) for c in self.contigs], dtype=np.int64)
        self.draft_bases = int(self.contig_off[-1])


def apply_guard(share, out, off, dropped, guard_fn):
    """scripts/goldpolish-ntedit:31-40 per batch: bytes(last _edited.fa) / bytes(batch.fa) < 0.75 (bc scale=4) -> the
    batch keeps its ORIGINAL records.  File sizes count '>' + name + '\\n' + sequence + '\\n' per record; a dropped
    record is absent from the output file.  Returns (out, off, dropped, rejected batch count); out/off are replaced
    only when a batch is rejected (rare)."""
    n = len(share.contigs)
    if n == 0:
        return out, off, dropped, 0
    if hasattr(out, "numpy"):
        out = out.numpy()
    in_len = np.diff(share.contig_off)
    out_len = np.diff(off.astype(np.int64))
    keep = dropped == 0
    in_sz = share.name_len + 3 + in_len
    out_sz = np.where(keep, share.name_len + 3 + out_len, 0)
    nb = len(share.batches)
    bi = np.zeros(nb, dtype=np.int64)
    bo = np.zeros(nb, dtype=np.int64)
    np.add.at(bi, share.contig_batch, in_sz)
    np.add.at(bo, share.contig_batch, out_sz)
    rejected = (bo * 10000) // np.maximum(bi, 1) < 7500
    n_rej = int(rejected.sum())
    if n_rej == 0:
        return out, off, dropped, 0
    assert all(bool(guard_fn(int(bi[b]), int(bo[b]))) for b in np.nonzero(rejected)[0][:4])  # same rule as the C ABI's
    rej_c = rejected[share.contig_batch]
    new_len = np.where(rej_c, in_len, np.where(keep, out_len, 0))
    new_off = np.concatenate([[0], np.cumsum(new_len)]).astype(np.uint64)
    new_out = np.empty(int(new_off[-1]), dtype=np.uint8)
    for i in range(n):
        src = share.contig_seq[share.contig_off[i]:share.contig_off[i + 1]] if rej_c[i] else out[int(off[i]):int(off[i + 1])]
        new_out[int(new_off[i]):int(new_off[i + 1])] = src
    new_dropped = np.where(rej_c, 0, dropped).astype(np.uint8)
    return new_out, new_off, new_dropped, n_rej


DUMP_SAMPLE_BASES = 4_000_000     # draft bases of the contigs whose polished bytes are written
DUMP_MAX_POLISHED = 8_000_000     # polished bytes written at most (32 MB as float32)
DUMP_FILTER_BATCHES = 3           # batches whose filter payloads are written (3 x 4 x 512 KiB: 25 MB as float32)


def dump_outputs(path, share, out, off, dropped, bfs=None):
    """Write what one pass of the timed path hands its caller, as .npy files of float32/float64 (under 64 MB in all):
      polished_len, dropped       per contig of the share: length of the polished record, 1 if it was dropped
      polished_sample             polished bytes of a seeded sample of contigs, concatenated in contig order
      polished_sample_contigs     the (global) contig indices of that sample
      filters_sample              [batches, k, BF_BYTES] filter payloads of a seeded sample of batches (when fetched)
      filters_sample_batches      the (global) batch indices of that sample
    The samples are drawn from SEED and the input sizes only, so two builds of the project write the same positions."""
    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(SEED)
    out = np.asarray(out)
    off = np.asarray(off, dtype=np.int64)
    n = len(share.contigs)
    order = rng.permutation(n)
    take = max(1, int(np.searchsorted(np.cumsum(np.diff(share.contig_off)[order]), DUMP_SAMPLE_BASES, side="right")))
    pick = np.sort(order[:take])
    sample = np.concatenate([out[off[c]:off[c + 1]] for c in pick] + [np.zeros(0, np.uint8)])[:DUMP_MAX_POLISHED]
    arrays = {"polished_len": np.diff(off).astype(np.float64), "dropped": np.asarray(dropped).astype(np.float32),
              "polished_sample": sample.astype(np.float32),
              "polished_sample_contigs": share.contigs[pick].astype(np.float64)}
    if bfs is not None:
        nb = len(share.batches)
        bsel = np.sort(rng.choice(nb, size=min(DUMP_FILTER_BATCHES, nb), replace=False))
        arrays["filters_sample"] = np.asarray(bfs)[bsel].astype(np.float32)
        arrays["filters_sample_batches"] = share.batches[bsel].astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    return arrays


def ours(args, rank, world, local_rank):
    import torch

    import goldpolish_b200 as gp
    from goldpolish_b200 import shard
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; goldpolish_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    w = WORKLOADS[args.config]
    strong = w["scaling"] == "strong"
    t0 = time.time()
    d = make_dataset(args, rank)
    clens, rlens = np.diff(d.contig_off), np.diff(d.read_off)
    pl = gp.plan_batches(clens, [d.contig_name(i) for i in range(d.n_contigs)],
                         [d.read_name(i) for i in range(d.n_reads)], d.read_phred, rlens, d.map_read, d.map_contig,
                         bsize=w["bsize"], subsample_max_per_10kbp=w["subsample_max"],
                         map_mx=d.map_mx if w["mappings"] == "ntlink" else None, mx_max_per_10kbp=w["mx_max"])
    nb_total = len(pl.batch_entry_off) - 1
    # sharding: batches are independent (private filters): LPT on read bases; every rank derives the same assignment
    if strong and world > 1:
        off = pl.batch_entry_off.astype(np.int64)
        ent_bases = rlens[pl.entries["read_id"]]
        csum = np.concatenate([[0], np.cumsum(ent_bases)])
        work = (csum[off[1:]] - csum[off[:-1]]) + 1
        assignment = shard.assign_batches(work.tolist(), world)
    else:
        assignment = None
    my_batches = assignment[rank] if assignment is not None else list(range(nb_total))
    sh = LocalShare(d, pl, my_batches, w["bsize"])
    n_batches = len(my_batches)
    log(f"[rank {rank}] data: {d.n_contigs} contigs / {int(d.contig_off[-1])} bp, {d.n_reads} reads / {int(d.read_off[-1])} bp, "
        f"{nb_total} batches; this rank: {n_batches} batches, {sh.draft_bases} draft bp, {sh.n_reads} reads / "
        f"{int(sh.read_off[-1])} bp, {len(sh.entries)} read entries ({time.time() - t0:.1f}s)")

    # pinned host buffers (e2e copies come from / go to these); the read set is page-locked in place
    def pin_in_place(a):
        t = torch.from_numpy(a)
        if a.nbytes and torch.cuda.cudart().cudaHostRegister(t.data_ptr(), a.nbytes, 0) != 0:
            return t.pin_memory()
        return t
    reads_h = pin_in_place(sh.read_seq)
    contigs_h = pin_in_place(sh.contig_seq)
    # config 5: 40 k batches x 2 MiB of filters per rank are not brought to the host (they feed the polish on the device;
    # only Sealer, out of scope, would read them) and live in a bounded pool that is reused wave after wave
    fetch_filters = args.config != 5
    bf_h = torch.empty((max(n_batches, 1) if fetch_filters else 1, 4, gp.BF_BYTES), dtype=torch.uint8).pin_memory()
    out_h = torch.empty(sh.draft_bases + sh.draft_bases // 4 + 65536, dtype=torch.uint8).pin_memory()

    ctx = gp.Context(device=local_rank, max_resident_filters=0 if fetch_filters else args.resident_filters)
    # a non-default torch stream: the library's kernels are launched on it so that the
    # torch.cuda.Event pair below brackets exactly the timed work
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.upload_reads(reads_h, sh.read_off)
    ctx.build_stage(sh.batch_entry_off, sh.entries)
    ctx.polish_stage(contigs_h, sh.contig_off, sh.contig_batch)

    # one step = filter build of every batch + the 4-round ntEdit chain over every contig, as one overlapped
    # pass (gp_pipeline_run: the edit kernel starts on a contig when its batch's filters are final); with
    # --separate the two stages run one after the other (gp_build_run, gp_polish_run)
    def step_resident():
        if args.separate:
            ctx.build_run()
            ctx.polish_run()
        else:
            ctx.pipeline_run()

    # ---- host gather in batch order (scripts/goldpolish-reaper:51-73): rank 0 receives every rank's polished
    # records over NCCL (device staging buffers), and lays them out in contig order ----
    gatherer = shard.RecordGather(clens, w["bsize"], assignment, rank, dist, device="cuda") if dist is not None and strong else None

    def gather(out, off, dropped):
        """-> (sequence bytes in contig order, per-contig lengths with 0 for dropped records) on rank 0, None elsewhere"""
        if gatherer is None:
            lens_local = np.where(dropped == 0, np.diff(off.astype(np.int64)), 0).astype(np.int64)
            return np.asarray(out[:int(off[-1])]), lens_local
        return gatherer(out, off, dropped)

    e2e_info = {}

    def step_e2e():
        ctx.upload_reads(reads_h, sh.read_off)
        ctx.build_stage(sh.batch_entry_off, sh.entries)
        ctx.polish_stage(contigs_h, sh.contig_off, sh.contig_batch)
        step_resident()
        if fetch_filters:
            ctx.build_fetch(out=bf_h)
        out, off, dropped = ctx.polish_fetch(out=out_h)
        out, off, dropped, n_rej = apply_guard(sh, out, off, dropped, gp.guard_rejects)
        e2e_info.update(rejected=n_rej, local=(out, off, dropped))
        return gather(out, off, dropped)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x: int) -> int:
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    # ---- device-resident timing ----
    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    barrier()
    ms_step = allmax(e0.elapsed_time(e1) / args.steps)
    clocks = sampler.stop()
    st = ctx.stats()  # of the last step
    build_kernel_ms_overlapped = st["build_kernel_ms"]  # device timer when overlapped with the edit kernel
    edit_kernel_ms = st["edit_kernel_ms"]
    launches_per_step = allsum(st["build_launches"] + st["polish_launches"])
    if args.dump_outputs and rank == 0:
        # the results of the last timed step, before any later pass overwrites them
        out_d, off_d, dropped_d = ctx.polish_fetch(out=out_h)
        dump_outputs(args.dump_outputs, sh, out_d, off_d, dropped_d, ctx.build_fetch(out=bf_h) if fetch_filters else None)
        log(f"[rank {rank}] outputs of the last timed step written to {args.dump_outputs}")
    # roofline leg: the dominant (build) kernel alone, CUDA events on the launching stream around each launch
    # (bounded filter pool: its waves run inside the pipelined pass only -- the kernel's in-step span stands in)
    if fetch_filters:
        ctx.build_run()
        alone = []
        for _ in range(args.steps):
            ctx.build_run()
            alone.append(ctx.stats()["build_kernel_ms"])
        build_kernel_ms = float(np.mean(alone))
    else:
        build_kernel_ms = float(build_kernel_ms_overlapped)
    total_bases = int(d.contig_off[-1]) if strong else allsum(sh.draft_bases)

    # ---- end to end through the C ABI with host buffers ----
    # the pinned destination of the filter payloads is named once: the build kernel writes each filter there as
    # it becomes final (gp_build_output_host), build_fetch then only synchronises
    if fetch_filters:
        ctx.build_output(bf_h)
    step_e2e()
    barrier()
    e2e_steps = args.steps
    t_e2e0 = time.perf_counter()
    for _ in range(e2e_steps):
        gathered = step_e2e()
    barrier()
    e2e_s = allmax((time.perf_counter() - t_e2e0) / e2e_steps)
    st2 = ctx.stats()
    if st2["polish_reruns"]:
        log(f"[rank {rank}] note: gp_polish_fetch re-ran the polish {st2['polish_reruns']} time(s) (buffer growth / watchdog); "
            "the timed steps include those re-runs")
    out_l, off_l, dropped_l = e2e_info["local"]
    h2d = allsum(int(sh.read_off[-1]) + (sh.n_reads + 1) * 8 * 2 + sh.n_reads * 4 + (n_batches + 1) * 8 + len(sh.entries) * 8
                 + n_batches * 4 * 4 + sh.draft_bases + (len(sh.contigs) + 1) * 8 * 3 + len(sh.contigs) * 8)
    d2h = allsum((n_batches * 4 * gp.BF_BYTES if fetch_filters else 0) + int(off_l[-1]) + len(sh.contigs) * 5 + 4)
    rejected = allsum(e2e_info["rejected"])
    gathered_sha = None
    if rank == 0:
        seqs, lens_all = gathered
        hsh = hashlib.sha256()
        hsh.update(np.ascontiguousarray(lens_all, dtype=np.int64).tobytes())
        hsh.update(np.ascontiguousarray(seqs).tobytes())
        gathered_sha = hsh.hexdigest()

    if rank == 0:
        peaks, peak_src = measured_peaks()
        kops = st["kmer_ops"]
        ops_per_s = kops / (build_kernel_ms * 1e-3) if build_kernel_ms > 0 else 0.0
        achieved = ops_per_s * ALGO_BYTES_PER_KMER_OP / 1e9
        kname = {1: "gp::build_filters_kernel (one warp per stream, counters in HBM)",
                 2: "gp::build_filters_levels_kernel (level-synchronous rounds, timestamps in L2)"}.get(st["build_kernel"], "?")
        read_bases_local = int(np.diff(sh.read_off)[sh.entries["read_id"]].sum())
        hashing_gbs = read_bases_local * 4 * 0.375 / (build_kernel_ms * 1e-3) / 1e9 if build_kernel_ms > 0 else 0.0
        roof = {"bound": "hbm", "achieved": achieved, "peak": float(peaks["hbm_gbs"]), "unit": "GB/s",
                "frac": achieved / float(peaks["hbm_gbs"]), "traffic": ncu_traffic(kops),
                "traffic_source": "profiles/build_kernel_dram.json (ncu dram__bytes_read+write per k-mer op) x k-mer ops of this launch",
                "kernel": kname, "kernel_ms": build_kernel_ms, "kmer_ops_per_launch": kops,
                "algorithmic_bytes_per_kmer_op": ALGO_BYTES_PER_KMER_OP, "peak_source": peak_src,
                "kmer_ops_per_s": ops_per_s, "streams_in_flight": st["build_slots"],
                "kernel_ms_inside_step": build_kernel_ms_overlapped, "edit_kernel_ms": edit_kernel_ms,
                "frac_of_hbm_copy_peak": achieved / float(peaks["hbm_gbs"]), "hbm_copy_peak_gbs": float(peaks["hbm_gbs"]),
                # the sequential side of the same kernel: every entry's read is streamed once per k, 2 bits per base
                # + 1 mask bit per base; three orders of magnitude below the copy peak -- the kernel lives on random
                # 32-byte-sector touches, not on this stream
                "hashing_stream_gbs": hashing_gbs, "hashing_stream_frac_of_hbm_copy_peak": hashing_gbs / float(peaks["hbm_gbs"]),
                "overlap": (f"edit kernel runs beside the build kernel on {st2['edit_sms']} SMs of its own (its span includes waiting for filters)"
                            if st2.get("edit_sms") else "edit kernel runs beside the build kernel, sharing its SMs (its span includes waiting for filters)") if not args.separate
                           else "none (--separate)"}
        if args.roof:
            # measured random-access roofs (sector touches / s), same access shapes as the kernels:
            #   hbm : private 10 MiB counter regions per warp (the one-warp-per-stream kernel's mix)
            #   l2_ld / l2_red : random 4-byte loads / atomicMin over one shared 40 MiB array
            #   l2_mix : rounds of 4 loads alternating with rounds of 4 atomicMin in the same launch (they overlap)
            # a k-mer op needs at least 4 loads + 4 atomics -> ops/s roof = 1 / (4/ld + 4/red); the overlapped
            # variant (l2_mix / 8) is the higher roof
            try:
                r = {}
                for name, mode, region in (("hbm", "0", gp.CBF_BYTES), ("l2_ld", "5", 4096), ("l2_red", "4", 4096), ("l2_mix", "3", 4096)):
                    os.environ["GP_ROOF_MODE"] = mode
                    r[name], _ = ctx.roof_microbench(148 * 24, 4000 if mode != "0" else 2000, region)
                os.environ.pop("GP_ROOF_MODE", None)
                roof["random_access_roof_sectors_per_s"] = r
                if st["build_kernel"] == 2:
                    ops_roof = 1.0 / (4.0 / r["l2_ld"] + 4.0 / r["l2_red"])
                    roof["bound"] = "l2_random_access"
                    roof["peak_source"] = ("measured live: gp_roof_microbench, random 4-byte loads and atomicMin over one 40 MiB array in "
                                           "L2 (the kernel's access shape); peak = 1 / (4/loads_per_s + 4/atomics_per_s) k-mer ops/s x 256 B")
                else:
                    ops_roof = r["hbm"] / 8.0
                    roof["bound"] = "hbm_random_access"
                    roof["peak_source"] = "measured live: gp_roof_microbench, private 10 MiB counter regions in HBM; peak = sectors_per_s / 8 x 256 B"
                roof["peak"] = ops_roof * ALGO_BYTES_PER_KMER_OP / 1e9
                roof["frac"] = ops_per_s / ops_roof if ops_roof else None
                roof["random_access_roof_kmer_ops_per_s"] = ops_roof
                roof["frac_of_random_access_roof"] = roof["frac"]
                roof["overlapped_roof_kmer_ops_per_s"] = r["l2_mix"] / 8.0
                roof["frac_of_overlapped_roof"] = ops_per_s / (r["l2_mix"] / 8.0) if r["l2_mix"] else None
                # against the HBM random-access roof the north star names (8 touches per op at the HBM sector rate):
                # above 1 because the level-synchronous kernel keeps the touched state in L2
                roof["frac_of_hbm_random_access_roof"] = ops_per_s * 8.0 / r["hbm"] if r["hbm"] else None
            except Exception as e:  # measurement aid only
                roof["random_access_roof_error"] = str(e)
        cpu, parity = None, None
        if args.cpu_baseline and world == 1:
            rs = None
            try:
                threads = os.cpu_count() or 1
                nb = sample_batches(args, d, threads)
                from oracle.ref_sample import ReferenceSample
                rs = ReferenceSample(w, d, range(nb), threads)
                r = rs.run()
                tt = r["seconds_build"] + r["seconds_edit"]
                cpu = {"value": r["bases"] / 1e6 / tt, "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                       "sample": f"first {r['batches']} of {nb_total} batches ({r['bases']} of {int(d.contig_off[-1])} draft bases), "
                                 f"one pass: build {r['seconds_build']:.2f}s + edit {r['seconds_edit']:.2f}s"}
                if r["kind"] in ("reference", "port"):
                    # parity at the benched size: what the reference's own code wrote for the sampled batches against
                    # what the GPU produced for the same batches in the timed end-to-end step
                    bf_np = bf_h.numpy()
                    bf_equal, fasta_equal, n_rec = (True if fetch_filters else None), True, 0
                    bs = w["bsize"]
                    for b in range(r["batches"]):
                        if fetch_filters and not np.array_equal(rs.filters(b), bf_np[b]):
                            bf_equal = False
                            log(f"PARITY: filter payloads of batch {b} differ from the reference")
                        ours_recs = []
                        for c in range(b * bs, min((b + 1) * bs, d.n_contigs)):
                            if not dropped_l[c]:
                                ours_recs.append((d.contig_name(c), np.asarray(out_l[int(off_l[c]):int(off_l[c + 1])]).tobytes()))
                        ref_recs = rs.polished(b)
                        n_rec += len(ref_recs)
                        if ours_recs != ref_recs:
                            fasta_equal = False
                            log(f"PARITY: polished records of batch {b} differ from the reference")
                    parity = {"batches": r["batches"], "records": n_rec, "bf_equal": bf_equal, "fasta_equal": fasta_equal,
                              "against": ("oracle/_ref (the reference's own serve_batch + ntEdit chain + guard)" if r["kind"] == "reference"
                                          else "oracle/gp_oracle.c (C restatement; oracle/_ref is not built on this machine)") + " on the same batches"}
            except Exception as e:
                cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "error", "sample": str(e)}
            finally:
                if rs is not None:
                    rs.close()
        line = {
            "metric": METRIC, "value": total_bases / 1e6 / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": w["scaling"], "vs_baseline": None, "dtype": "u8/u64 integer",
            "data": "synthetic (seeded simulator, sim/gpsim.c)",
            "config": config_of(args),
            "detail": {"total_draft_bases": total_bases, "batches_total": nb_total, "batches_rank0": n_batches,
                       "draft_bases_rank0": sh.draft_bases, "guard_rejected_batches": rejected,
                       "parallelism": (f"batches of one data set sharded over {world} GPU(s) by LPT on read bases, no collective in "
                                       "the data path; rank 0 gathers the polished records (NCCL gather of device staging "
                                       "buffers + host layout in contig order) inside the e2e step") if strong else
                                      f"{world} independent data sets, one per GPU, no collective",
                       "gathered_sha256": gathered_sha},
            "clocks": clocks,
            "e2e": {"value": total_bases / 1e6 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                    "includes": "H2D reads+pack, H2D contigs, build + polish, " + ("D2H filter payloads, " if fetch_filters else "") + "D2H polished, guard"
                                + (", gather on rank 0" if strong and world > 1 else "")},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roof,
            "cpu_baseline": cpu,
            "parity": parity,
            "stats": {k: st2[k] for k in ("kmer_ops", "serial_kmers", "triggers", "edits", "masked", "rollbacks",
                                          "build_ms", "polish_ms", "pack_ms", "build_kernel_ms", "edit_kernel_ms", "polish_reruns", "edit_sms")},
        }
        emit(line)
        if parity is not None and (parity["bf_equal"] is False or not parity["fasta_equal"]):
            ctx.close()
            raise SystemExit("bench.py: PARITY FAILURE against the reference on the sampled batches (see stderr)")
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(WORKLOADS))
    ap.add_argument("--genome-len", type=int, default=None, help="override the workload's draft size (experiments)")
    ap.add_argument("--coverage", type=float, default=None)
    ap.add_argument("--bsize", type=int, default=None, help="contigs per batch (parity/scale experiments)")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-roof", dest="roof", action="store_false")
    ap.add_argument("--ref-bases-per-core", type=float, default=76000.0,
                    help="draft bases per host core in one CPU step (reference arm / cpu_baseline sample)")
    ap.add_argument("--resident-filters", type=int, default=4096,
                    help="config 5: batches whose filters are resident at once (8 GiB of pool at 4096)")
    ap.add_argument("--separate", action="store_true", help="build, then polish (no overlap of the two kernels)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0's share; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none to write")
    w = WORKLOADS[args.config]
    if args.genome_len is not None:
        w["genome_len"] = args.genome_len
    if args.coverage is not None:
        w["coverage"] = args.coverage
    if args.bsize is not None:
        w["bsize"] = args.bsize
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "ours":
        log("bench.py: note: timing rules ask for >= 3 warm-up steps")
    own_stdout()
    if args.impl == "reference":
        reference_arm(args, rank, world)
    else:
        ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
