"""Runs of unsupported k-mers on the device (gp_polish_fetch_unsupported, Context(kmer_support=True)): every (contig,
record, k) equals the numpy restatement of tests/test_kmer_unsupported.py on the draft and on the polished record, for
two k lists, at bsize 1 and 8, through gp_polish, gp_pipeline_run (every filter resident, and a 2-batch pool whose
filters are gone before the fetch) and on loaded filters; per-run kmers sum to kmers - present of
polish_fetch_support; the mask / to-upper pass, a dropped contig and the re-run after buffer growth change nothing; the
fetch order does not matter; at config-2 size the option changes no polished byte, flag, stat or edit record; both
tools' BEDs; the error paths."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_gpu_edit_records import BIN, ENV, ODD, _bf_files, _fasta
from test_gpu_kmer_support import restated as restated_counts
from test_kmer_unsupported import unsupported_bed, unsupported_runs
from util import KS, dataset, plan

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gp():
    import goldpolish_b200
    return goldpolish_b200


def _run(gp, d, pl, ks, path, fetch_first=None, **kw):
    """(filters, runs dict, counts, polished bytes, offsets, dropped, stats)"""
    with gp.Context(ks=ks, kmer_support=True, **kw) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        if path == "polish":
            bfs = ctx.build_filters(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.polish_run()
        elif path == "loaded":
            with gp.Context(ks=ks) as other:
                other.upload_reads(d.read_seq, d.read_off)
                bfs = other.build_filters(pl.batch_entry_off, pl.entries)
            ctx.load_filters(bfs)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.polish_run()
        else:
            ctx.build_stage(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            pinned = None
            if kw.get("max_resident_filters"):
                import torch
                pinned = torch.empty((len(pl.batch_entry_off) - 1, len(ks), gp.BF_BYTES), dtype=torch.uint8).pin_memory()
                ctx.build_output(pinned)
            ctx.pipeline_run()
            bfs = ctx.build_fetch(out=pinned)
            bfs = bfs.numpy().copy() if pinned is not None else bfs
        if fetch_first == "polish":
            out, off, dropped = ctx.polish_fetch()
            runs = ctx.polish_fetch_unsupported()
        else:
            runs = ctx.polish_fetch_unsupported()
            out, off, dropped = ctx.polish_fetch()
        counts, _ = ctx.polish_fetch_support()
        st = ctx.stats()
    return bfs, runs, counts, out, off, dropped, st


def device_runs(r, c, rec, j):
    off = r["run_off"]
    i = (c * 2 + rec) * r["offsets"].shape[2] + j
    a, b = int(off[i]), int(off[i + 1])
    return list(zip(r["start"][a:b].tolist(), r["end"][a:b].tolist(), r["kmers"][a:b].tolist()))


def check(d, pl, ks, res, sample=1):
    bfs, r, counts, out, off, dropped, _ = res
    assert r["offsets"].shape == (d.n_contigs, 2, len(ks))
    assert np.array_equal(r["offsets"].ravel(), r["run_off"][:-1]) and int(r["run_off"][-1]) == len(r["start"])
    if sample == 1:
        assert np.array_equal(counts, restated_counts(d, pl, bfs, ks, out, off, dropped))
    n = 0
    for c in range(0, d.n_contigs, sample):
        b = int(pl.contig_batch[c])
        pol = None if dropped[c] else out[int(off[c]):int(off[c + 1])].tobytes()
        for j, k in enumerate(ks):
            for rec, seq in ((0, d.contig(c)), (1, pol)):
                got = device_runs(r, c, rec, j)
                assert got == unsupported_runs(seq, bfs[b, j], k), (c, rec, k)
                n += len(got)
    # per-run kmers sum to the support counts' missing k-mers, for every (contig, record, k)
    sums = np.add.reduceat(np.append(r["kmers"].astype(np.uint64), 0), r["run_off"][:-1].astype(np.int64))
    sums[np.diff(r["run_off"]) == 0] = 0
    sums = sums.reshape(d.n_contigs, 2, len(ks))
    assert np.array_equal(sums[:, 0], counts[:, :, 0] - counts[:, :, 1])
    assert np.array_equal(sums[:, 1], counts[:, :, 2] - counts[:, :, 3])
    assert n > 0
    return r


CASES = [(ks, bsize, path) for ks in (KS, ODD) for bsize in (1, 8) for path in ("polish", "pipeline")]


@pytest.mark.parametrize("ks,bsize,path", CASES)
def test_device_runs_equal_the_restatement(gp, ks, bsize, path):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=bsize)
    check(d, pl, ks, _run(gp, d, pl, ks, path))


def test_two_batch_filter_pool(gp):
    """The filters of every wave but the last are gone when the runs are derived: they come from the bitmap."""
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    assert len(pl.batch_entry_off) - 1 > 2
    check(d, pl, KS, _run(gp, d, pl, KS, "pipeline", max_resident_filters=2))


def test_loaded_filters(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=8)
    check(d, pl, ODD, _run(gp, d, pl, ODD, "loaded"))


def _same(a, b):
    return all(np.array_equal(a[key], b[key]) for key in ("run_off", "start", "end", "kmers"))


@pytest.mark.parametrize("path", ["polish", "pipeline"])
def test_mask_and_to_upper_change_nothing(gp, path):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    base = _run(gp, d, pl, KS, path)
    for prep_mode in (1, 2):
        res = _run(gp, d, pl, KS, path, prep_mode=prep_mode, prep_k=KS[0], to_upper=1)
        assert _same(res[1], base[1]), prep_mode


def test_dropped_contig(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    cut = int(np.median(np.diff(d.contig_off)))  # the shorter half is dropped at the first round
    res = _run(gp, d, pl, KS, "polish", min_contig_len=cut)
    r, dropped = res[1], res[5]
    assert dropped.any() and not dropped.all()
    seg = np.diff(r["run_off"]).reshape(d.n_contigs, 2, len(KS))
    assert (seg[dropped == 1][:, 1] == 0).all()
    assert seg[dropped == 1][:, 0].sum() > 0  # their draft runs are still reported
    check(d, pl, KS, res)


@pytest.mark.parametrize("path,resident", [("polish", 0), ("pipeline", 0), ("pipeline", 2)])
def test_rerun_after_buffer_growth(gp, path, resident, monkeypatch):
    """GP_POLISH_CAPS makes edited contigs outgrow their buffers: the re-run (polish_launch over resident filters, or a
    whole new gp_pipeline_run pass with a 2-batch pool) grows the bitmap with the buffers and reports the final records."""
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    base = _run(gp, d, pl, KS, path, max_resident_filters=resident)
    monkeypatch.setenv("GP_POLISH_CAPS", "16,64")
    for first in ("unsupported", "polish"):
        res = _run(gp, d, pl, KS, path, fetch_first=first, max_resident_filters=resident)
        assert res[6]["polish_reruns"] >= 1
        assert _same(res[1], base[1]), first
        check(d, pl, KS, res)


def test_fetch_order_does_not_matter(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    got = []
    for order in (("unsupported", "support", "edits", "polish"), ("polish", "edits", "support", "unsupported"),
                  ("edits", "unsupported", "polish", "support")):
        with gp.Context(kmer_support=True, track_edits=True) as ctx:
            ctx.upload_reads(d.read_seq, d.read_off)
            ctx.build_stage(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.pipeline_run()
            r = {}
            for what in order:
                if what == "unsupported":
                    r[what] = ctx.polish_fetch_unsupported()
                elif what == "support":
                    r[what] = ctx.polish_fetch_support()[0]
                elif what == "edits":
                    r[what] = ctx.polish_fetch_edits()["pos"]
                else:
                    r[what] = ctx.polish_fetch()[1]
            r["again"] = ctx.polish_fetch_unsupported()
        got.append(r)
    for r in got:
        assert _same(r["unsupported"], got[0]["unsupported"]) and _same(r["again"], r["unsupported"])
        assert np.array_equal(r["support"], got[0]["support"]) and np.array_equal(r["edits"], got[0]["edits"])
        assert np.array_equal(r["polish"], got[0]["polish"])


# k-mer support counts of this config-2 set (5 Mbp draft, 30x, bsize 1, default k chain) summed over the contigs, per k:
# draft k-mers, draft present, polished k-mers, polished present -- as the library before the runs were added reported
# them (profiles/kmer_support_cost.json, support_totals_per_k of config2_5mbp_30x_bsize1).  Keeping the bitmap must not
# move a count.
CONFIG2_TOTALS = [[4981268, 2977398, 4981810, 3881947], [4983608, 3012210, 4984142, 3805672],
                  [4985948, 3143665, 4986474, 3838017], [4988288, 3354589, 4988806, 3951737]]


def test_config2_size(gp):
    d = dataset(genome_len=5_000_000)
    pl = plan(d, bsize=1)
    runs = []
    for on in (False, True):
        with gp.Context(kmer_support=on, track_edits=True) as ctx:
            ctx.upload_reads(d.read_seq, d.read_off)
            ctx.build_stage(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.pipeline_run()
            bfs = ctx.build_fetch()
            out, off, dropped = ctx.polish_fetch()
            ed = ctx.polish_fetch_edits()
            r = ctx.polish_fetch_unsupported() if on else None
            counts = ctx.polish_fetch_support()[0] if on else None
            runs.append((out[:int(off[-1])].copy(), off, dropped, ctx.stats(), ed, r, counts, bfs))
    (o0, f0, d0, s0, e0, _, _, _), (o1, f1, d1, s1, e1, r, counts, bfs) = runs
    assert np.array_equal(o0, o1) and np.array_equal(f0, f1) and np.array_equal(d0, d1)
    for key in ("kmer_ops", "serial_kmers", "triggers", "edits", "masked", "rollbacks", "polish_reruns", "build_launches",
                "polish_launches"):
        assert s0[key] == s1[key], key
    for key in e0:
        assert np.array_equal(e0[key], e1[key]), key
    assert np.array_equal(counts.sum(axis=0), np.array(CONFIG2_TOTALS, dtype=np.uint64))
    check(d, pl, KS, (bfs, r, counts, o1, f1, d1, s1), sample=max(1, d.n_contigs // 16))


def test_error_paths(gp):
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    l = gp.load_library()
    with gp.Context() as ctx:  # the option off
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        with pytest.raises(gp.GpError) as e:
            ctx.polish_fetch_unsupported()
        assert e.value.code == -5
    with gp.Context(kmer_support=True) as ctx:
        with pytest.raises(gp.GpError) as e:  # before any polish
            ctx.polish_fetch_unsupported()
        assert e.value.code == -5
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        with pytest.raises(gp.GpError) as e:  # filters, but no polish yet
            ctx.polish_fetch_unsupported()
        assert e.value.code == -5
        ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        r = ctx.polish_fetch_unsupported()
        total = len(r["start"])
        assert total > 1
        off = np.zeros_like(r["run_off"])
        need = np.zeros(1, dtype=np.uint64)
        buf = np.zeros(total, dtype=gp.api.UNSUPPORTED_DTYPE)
        # a short cap: GP_ERR_ARG, the total in needed, the offsets filled
        assert l.gp_polish_fetch_unsupported(ctx._h, off.ctypes.data, buf.ctypes.data, total - 1, need.ctypes.data) == -1
        assert int(need[0]) == total and np.array_equal(off, r["run_off"])
        assert l.gp_polish_fetch_unsupported(ctx._h, None, None, 0, need.ctypes.data) == -1  # nowhere for the offsets
        assert l.gp_polish_fetch_unsupported(ctx._h, off.ctypes.data, buf.ctypes.data, total, need.ctypes.data) == 0
        assert np.array_equal(buf["start"], r["start"]) and np.array_equal(buf["kmers"], r["kmers"])
        ctx.prep(d.contig_seq, d.contig_off, 0, 0, 1)  # gp_prep is no polish: nothing to report after it
        with pytest.raises(gp.GpError) as e:
            ctx.polish_fetch_unsupported()
        assert e.value.code == -5


# ---- the drop-in tools -------------------------------------------------------------------------------------------------
NAMES = ["mixed_dense", "subs", "short_80bp", "lowercase"]


def _tool_want(bfs, ks, names, records):
    """The BED from the restatement: runs of every record present in `records` against the single batch's filters."""
    payload = [np.fromfile(p, dtype=np.uint8)[-524288:] for p in bfs]
    runs = [[unsupported_runs(None if records.get(n) is None else records[n].encode(), payload[j], k) for j, k in enumerate(ks)]
            for n in names]
    return unsupported_bed(names, ks, runs, emit=[records.get(n) is not None for n in names])


def test_ntedit_gr_kmer_bed():
    import json
    from util import GOLDEN
    cli = json.load(open(os.path.join(GOLDEN, "ntedit_cli.json")))
    w = tempfile.mkdtemp()
    try:
        g, bfs = _bf_files(w)
        fa = os.path.join(w, "in.fa")
        with open(fa, "w") as f:
            f.write(cli["input_fasta"])
            for n in NAMES:
                f.write(f">{n} a comment\n{g['cases'][n]['draft']}\n")
        bed = os.path.join(w, "runs.bed")
        subprocess.check_call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-d5", "-i5", "-m1", "-X0.5",
                               "-Y0.5", "-b", os.path.join(w, "out"), "-t1", "-a1", "--kmer-bed", bed], env=ENV)
        names = list(_fasta(fa))
        edited = _fasta(os.path.join(w, "out_edited.fa"))  # the emitted records (-a1 soft-masking hashes alike)
        want = _tool_want(bfs[:1], KS[:1], names, edited)
        assert want and open(bed, "rb").read() == want
    finally:
        shutil.rmtree(w, ignore_errors=True)


def test_goldpolish_ntedit_kmer_bed_and_guard():
    w = tempfile.mkdtemp()
    try:
        g, bfs = _bf_files(w)
        base = os.path.join(w, "batch")
        with open(base + ".fa", "w") as f:
            for n in NAMES:
                f.write(f">{n} some comment\n{g['cases'][n]['draft']}\n")
        out = os.path.join(w, "batch.ntedited.fa")
        env = dict(ENV, GP_KMER_BED="1")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out],
                              env=env, stdout=subprocess.DEVNULL)
        chain = {n: g["cases"][n]["chain"] for n in NAMES}
        assert chain["short_80bp"] is None
        assert open(out + ".kmer_unsupported.bed", "rb").read() == _tool_want(bfs, KS, NAMES, chain)
        assert not os.path.exists(out + ".kmer_qv.tsv")
        # a batch the 0.75 guard rejects: the runs of the input it keeps
        base2 = os.path.join(w, "tiny")
        tiny = {f"t{i}": g["truth"][i * 90:i * 90 + 90] for i in range(6)}
        tiny["keep"] = g["truth"][:150]
        tiny["err"] = g["truth"][200:260] + "A" + g["truth"][261:400]  # a substitution the reads do not support
        with open(base2 + ".fa", "w") as f:
            for n, s in tiny.items():
                f.write(f">{n}\n{s}\n")
        out2 = os.path.join(w, "tiny.ntedited.fa")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base2, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out2],
                              env=env, stdout=subprocess.DEVNULL)
        assert os.readlink(out2) == base2 + ".fa"
        assert open(out2 + ".kmer_unsupported.bed", "rb").read() == _tool_want(bfs, KS, list(tiny), tiny)
        out3 = os.path.join(w, "batch3.ntedited.fa")  # without the variable no BED is written
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out3],
                              env=ENV, stdout=subprocess.DEVNULL)
        assert not os.path.exists(out3 + ".kmer_unsupported.bed")
    finally:
        shutil.rmtree(w, ignore_errors=True)
