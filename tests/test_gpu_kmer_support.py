"""k-mer support on the device (gp_polish_fetch_support, Context(kmer_support=True)): every (contig, k) count equals the
numpy restatement of tests/test_kmer_support.py on the draft and on the polished record, for two k lists, at bsize 1 and
8, through gp_polish, gp_pipeline_run (every filter resident, and a 2-batch pool) and on loaded filters; the mask /
to-upper pass, a dropped contig and the re-run after buffer growth change nothing; filter_bits_set is the payloads'
popcount; the option changes no polished byte, flag, stat or edit record; both tools' TSVs; the error paths."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_gpu_edit_records import BIN, ENV, ODD, _bf_files, _fasta
from test_kmer_support import kmer_qv_tsv, support
from util import KS, dataset, plan

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gp():
    import goldpolish_b200
    return goldpolish_b200


def _run(gp, d, pl, ks, path, fetch_first=None, **kw):
    """(filters, counts, bits, polished bytes, offsets, dropped, stats)"""
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
            counts, bits = ctx.polish_fetch_support()
        else:
            counts, bits = ctx.polish_fetch_support()
            out, off, dropped = ctx.polish_fetch()
        st = ctx.stats()
    return bfs, counts, bits, out, off, dropped, st


def restated(d, pl, bfs, ks, out, off, dropped):
    want = np.zeros((d.n_contigs, len(ks), 4), dtype=np.uint64)
    for c in range(d.n_contigs):
        b = int(pl.contig_batch[c])
        pol = None if dropped[c] else out[int(off[c]):int(off[c + 1])].tobytes()
        for j, k in enumerate(ks):
            want[c, j, :2] = support(d.contig(c), bfs[b, j], k)
            want[c, j, 2:] = support(pol, bfs[b, j], k)
    return want


def popcounts(bfs):
    return np.unpackbits(np.ascontiguousarray(bfs), axis=-1).sum(axis=-1).astype(np.uint64)


def check(d, pl, ks, res):
    bfs, counts, bits, out, off, dropped, _ = res
    want = restated(d, pl, bfs, ks, out, off, dropped)
    for c in range(d.n_contigs):
        assert np.array_equal(counts[c], want[c]), f"contig {c}: {counts[c].tolist()} != {want[c].tolist()}"
    assert np.array_equal(bits, popcounts(bfs))
    assert (counts[:, :, 0] > counts[:, :, 1]).any()  # the drafts have k-mers the reads do not support


CASES = [(ks, bsize, path) for ks in (KS, ODD) for bsize in (1, 8) for path in ("polish", "pipeline")]


@pytest.mark.parametrize("ks,bsize,path", CASES)
def test_device_counts_equal_the_restatement(gp, ks, bsize, path):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=bsize)
    check(d, pl, ks, _run(gp, d, pl, ks, path))


def test_two_batch_filter_pool(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    assert len(pl.batch_entry_off) - 1 > 2
    check(d, pl, KS, _run(gp, d, pl, KS, "pipeline", max_resident_filters=2))


def test_loaded_filters(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=8)
    check(d, pl, ODD, _run(gp, d, pl, ODD, "loaded"))


@pytest.mark.parametrize("path", ["polish", "pipeline"])
def test_mask_and_to_upper_change_no_count(gp, path):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    base = _run(gp, d, pl, KS, path)
    for prep_mode in (1, 2):
        res = _run(gp, d, pl, KS, path, prep_mode=prep_mode, prep_k=KS[0], to_upper=1)
        assert np.array_equal(res[1], base[1]) and np.array_equal(res[2], base[2]), prep_mode


def test_dropped_contig(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    lens = np.diff(d.contig_off)
    cut = int(np.median(lens))  # the shorter half is dropped at the first round
    res = _run(gp, d, pl, KS, "polish", min_contig_len=cut)
    _, counts, _, _, _, dropped, _ = res
    assert dropped.any() and not dropped.all()
    assert (counts[dropped == 1][:, :, 2:] == 0).all()
    assert (counts[dropped == 1][:, :, 0] > 0).all()
    check(d, pl, KS, res)


@pytest.mark.parametrize("path,resident", [("polish", 0), ("pipeline", 0), ("pipeline", 2)])
def test_rerun_after_buffer_growth(gp, path, resident, monkeypatch):
    """GP_POLISH_CAPS makes edited contigs outgrow their buffers: the re-run (polish_launch over resident filters, or a
    whole new gp_pipeline_run pass with a 2-batch pool) must count every contig from its final record."""
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    base = _run(gp, d, pl, KS, path, max_resident_filters=resident)
    monkeypatch.setenv("GP_POLISH_CAPS", "16,64")
    for first in ("support", "polish"):
        res = _run(gp, d, pl, KS, path, fetch_first=first, max_resident_filters=resident)
        assert res[6]["polish_reruns"] >= 1
        assert np.array_equal(res[1], base[1]) and np.array_equal(res[2], base[2]), first
        assert np.array_equal(res[4], base[4]) and np.array_equal(res[3][:int(res[4][-1])], base[3][:int(base[4][-1])])


def test_fetch_order_does_not_matter(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    got = []
    for order in (("support", "edits", "polish"), ("polish", "edits", "support"), ("edits", "support", "polish")):
        with gp.Context(kmer_support=True, track_edits=True) as ctx:
            ctx.upload_reads(d.read_seq, d.read_off)
            ctx.build_stage(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.pipeline_run()
            r = {}
            for what in order:
                if what == "support":
                    r[what] = ctx.polish_fetch_support()
                elif what == "edits":
                    r[what] = ctx.polish_fetch_edits()["pos"]
                else:
                    r[what] = ctx.polish_fetch()[1]
            r["again"] = ctx.polish_fetch_support()
        got.append(r)
    for r in got:
        assert np.array_equal(r["support"][0], got[0]["support"][0]) and np.array_equal(r["support"][1], got[0]["support"][1])
        assert np.array_equal(r["again"][0], r["support"][0])
        assert np.array_equal(r["edits"], got[0]["edits"]) and np.array_equal(r["polish"], got[0]["polish"])


def test_option_changes_nothing_else_at_config2_size(gp):
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
            sup = ctx.polish_fetch_support() if on else None
            runs.append((out[:int(off[-1])].copy(), off, dropped, ctx.stats(), ed, sup, bfs))
    (o0, f0, d0, s0, e0, _, _), (o1, f1, d1, s1, e1, sup, bfs) = runs
    assert np.array_equal(o0, o1) and np.array_equal(f0, f1) and np.array_equal(d0, d1)
    for key in ("kmer_ops", "serial_kmers", "triggers", "edits", "masked", "rollbacks", "polish_reruns", "build_launches",
                "polish_launches"):
        assert s0[key] == s1[key], key
    for key in e0:
        assert np.array_equal(e0[key], e1[key]), key
    counts, bits = sup
    assert np.array_equal(bits, popcounts(bfs))
    # polishing raises the share of supported k-mers over the whole assembly
    tot = counts.sum(axis=0)
    assert (tot[:, 1] / tot[:, 0] < tot[:, 3] / tot[:, 2]).all()
    for c in range(0, d.n_contigs, max(1, d.n_contigs // 8)):  # a sample of contigs against the restatement
        b = int(pl.contig_batch[c])
        pol = None if d1[c] else o1[int(f1[c]):int(f1[c + 1])].tobytes()
        for j, k in enumerate(KS):
            assert tuple(counts[c, j]) == support(d.contig(c), bfs[b, j], k) + support(pol, bfs[b, j], k), (c, k)


def test_error_paths(gp):
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    with gp.Context() as ctx:  # the option off
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        with pytest.raises(gp.GpError) as e:
            ctx.polish_fetch_support()
        assert e.value.code == -5
    with gp.Context(kmer_support=True) as ctx:
        with pytest.raises(gp.GpError) as e:  # before any polish
            ctx.polish_fetch_support()
        assert e.value.code == -5
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        with pytest.raises(gp.GpError) as e:  # filters, but no polish yet
            ctx.polish_fetch_support()
        assert e.value.code == -5
        ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        counts, bits = ctx.polish_fetch_support()
        l = gp.load_library()
        assert l.gp_polish_fetch_support(ctx._h, None, None) == -1  # contigs, but nowhere to put their counts
        again = np.zeros_like(counts)
        assert l.gp_polish_fetch_support(ctx._h, again.ctypes.data, None) == 0 and np.array_equal(again, counts)
        ctx.prep(d.contig_seq, d.contig_off, 0, 0, 1)  # gp_prep is no polish: nothing to report after it
        with pytest.raises(gp.GpError) as e:
            ctx.polish_fetch_support()
        assert e.value.code == -5


# ---- the drop-in tools -------------------------------------------------------------------------------------------------
NAMES = ["mixed_dense", "subs", "short_80bp", "lowercase"]


def _tool_want(g, bfs, ks, names, seqs, polished, polished_is_draft=False):
    """The TSV from the restatement: counts of every record against the single batch's filters."""
    import oracle.oracle_lib  # noqa: F401
    payload = [np.fromfile(p, dtype=np.uint8)[-524288:] for p in bfs]
    counts = np.zeros((len(names), len(ks), 4), dtype=np.uint64)
    for c, n in enumerate(names):
        for j, k in enumerate(ks):
            counts[c, j, :2] = support(seqs[n].encode(), payload[j], k)
            counts[c, j, 2:] = support(None if polished.get(n) is None else polished[n].encode(), payload[j], k)
    bits = popcounts(np.stack(payload))[None, :]
    return kmer_qv_tsv(names, ks, counts, bits, polished_is_draft)


def test_ntedit_gr_kmer_qv():
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
        tsv = os.path.join(w, "qv.tsv")
        subprocess.check_call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-d5", "-i5", "-m1", "-X0.5",
                               "-Y0.5", "-b", os.path.join(w, "out"), "-t1", "-a1", "--kmer-qv", tsv], env=ENV)
        drafts = _fasta(fa)
        edited = _fasta(os.path.join(w, "out_edited.fa"))  # -a1 output: the soft-masking does not change the hashes
        want = _tool_want(g, bfs[:1], KS[:1], list(drafts), drafts, edited)
        assert open(tsv, "rb").read() == want
    finally:
        shutil.rmtree(w, ignore_errors=True)


def test_goldpolish_ntedit_kmer_qv_and_guard():
    w = tempfile.mkdtemp()
    try:
        g, bfs = _bf_files(w)
        base = os.path.join(w, "batch")
        with open(base + ".fa", "w") as f:
            for n in NAMES:
                f.write(f">{n} some comment\n{g['cases'][n]['draft']}\n")
        out = os.path.join(w, "batch.ntedited.fa")
        env = dict(ENV, GP_KMER_QV="1")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out],
                              env=env, stdout=subprocess.DEVNULL)
        drafts = {n: g["cases"][n]["draft"] for n in NAMES}
        chain = {n: g["cases"][n]["chain"] for n in NAMES}
        assert chain["short_80bp"] is None
        assert open(out + ".kmer_qv.tsv", "rb").read() == _tool_want(g, bfs, KS, NAMES, drafts, chain)
        # a batch the 0.75 guard rejects: the polished columns describe the input it keeps
        base2 = os.path.join(w, "tiny")
        tiny = {f"t{i}": g["truth"][i * 90:i * 90 + 90] for i in range(6)}
        tiny["keep"] = g["truth"][:150]
        with open(base2 + ".fa", "w") as f:
            for n, s in tiny.items():
                f.write(f">{n}\n{s}\n")
        out2 = os.path.join(w, "tiny.ntedited.fa")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base2, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out2],
                              env=env, stdout=subprocess.DEVNULL)
        assert os.readlink(out2) == base2 + ".fa"
        assert open(out2 + ".kmer_qv.tsv", "rb").read() == _tool_want(g, bfs, KS, list(tiny), tiny, {}, polished_is_draft=True)
        out3 = os.path.join(w, "batch3.ntedited.fa")  # without the variable no TSV is written
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out3],
                              env=ENV, stdout=subprocess.DEVNULL)
        assert not os.path.exists(out3 + ".kmer_qv.tsv")
    finally:
        shutil.rmtree(w, ignore_errors=True)
