"""The polish re-run after buffer growth: GP_POLISH_CAPS gives every contig a few bytes of slack and a few rope nodes, so
that an edited contig outgrows its device buffers, the kernel flags it, and gp_polish_fetch doubles the buffers and
polishes again (from the resident filters, or as a whole new gp_pipeline_run pass when the filter pool holds one wave).
The records equal the C restatement's and the edit records the numpy restatement's; stats and flags equal a run without
the knob; four doublings that do not suffice end in GP_ERR_OVERFLOW, and the tools write the same files."""
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_edit_records import chain_with_origins, derive_records
from test_gpu_edit_records import BIN, ENV, ODD, _bf_files, device_records
from util import KS, dataset, ol, oracle_build, plan

pytestmark = pytest.mark.gpu

# "16,": any contig whose k chain grows it by more than 16 bytes (plus the 16-byte rounding) overflows once; ",64": the
# most edited contig (about 180 edits at k = 32) needs more than 128 nodes, i.e. at least two doublings
BYTES, NODES, BOTH = "16,", ",64", "16,64"


@pytest.fixture(scope="module")
def gp():
    import goldpolish_b200
    return goldpolish_b200


@functools.lru_cache(maxsize=None)
def _ref():
    """Data set, plan, restatement filters, and per contig the restatement's polished record (None: dropped) and the
    longest length along its k chain."""
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    bfs = oracle_build(d, pl)
    want, longest = [], []
    for c in range(d.n_contigs):
        cur, top = d.contig(c), len(d.contig(c))
        for ki, k in enumerate(KS):
            cur, _ = ol.ntedit_contig(cur, bfs[int(pl.contig_batch[c])].bfs[ki], k)
            if cur is None:
                break
            top = max(top, len(cur))
        want.append(cur)
        longest.append(top)
    return d, pl, want, longest


def byte_reruns(d, longest, extra):
    """Doublings until the k chain of every contig fits cap = (len + extra) << g, rounded up to 16 (polish_layout)."""
    g = 0
    while any(((((len(d.contig(c)) + extra) << g) + 15) & ~15) < longest[c] for c in range(d.n_contigs)):
        g += 1
    return g


def check_records(d, want, out, off, dropped):
    for c in range(d.n_contigs):
        got = out[int(off[c]):int(off[c + 1])].tobytes()
        if want[c] is None:
            assert dropped[c] == 1 and got == b"", c
        else:
            assert dropped[c] == 0 and got == want[c], f"contig {c} differs from the restatement"


STAT_KEYS = ("triggers", "edits", "masked", "rollbacks")


@pytest.mark.parametrize("caps", [BYTES, NODES])
def test_polish_regrows_and_matches(gp, caps, monkeypatch):
    d, pl, want, longest = _ref()
    with gp.Context() as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        out0, off0, dr0 = ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        st0 = ctx.stats()
        assert st0["polish_reruns"] == 0
        monkeypatch.setenv("GP_POLISH_CAPS", caps)
        out, off, dropped = ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        st = ctx.stats()
    check_records(d, want, out, off, dropped)
    assert np.array_equal(dropped, dr0) and np.array_equal(off, off0)
    if caps == BYTES:
        assert byte_reruns(d, longest, 16) == 1
        assert st["polish_reruns"] == 1
    else:
        assert 2 <= st["polish_reruns"] <= 4
    for key in STAT_KEYS:  # the counters of the overflowed pass do not add up with those of the re-run
        assert st[key] == st0[key], key


@pytest.mark.parametrize("resident", [0, 2])
def test_pipeline_regrows_by_either_route(gp, resident, monkeypatch):
    """Every filter resident: the re-run is polish_launch over the resident filters.  A 2-batch pool: the re-run is a
    whole new gp_pipeline_run pass, payloads streamed to page-locked memory again.  Then a pass without the knob on the
    same context (which reads the edit kernel's error word of the overflowed pass) neither re-runs nor changes a byte."""
    import torch
    d, pl, want, _ = _ref()
    nb = len(pl.batch_entry_off) - 1
    with gp.Context() as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        bfs = ctx.build_filters(pl.batch_entry_off, pl.entries)
        ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        st0 = ctx.stats()
    monkeypatch.setenv("GP_POLISH_CAPS", BOTH)
    with gp.Context(max_resident_filters=resident) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        pinned = torch.zeros((nb, len(KS), gp.BF_BYTES), dtype=torch.uint8).pin_memory()
        ctx.build_output(pinned)
        ctx.build_stage(pl.batch_entry_off, pl.entries)
        ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
        ctx.pipeline_run()
        out, off, dropped = ctx.polish_fetch()
        got = ctx.build_fetch(out=pinned).numpy().copy()
        st = ctx.stats()
        reruns = st["polish_reruns"]
        assert reruns >= 1
        assert np.array_equal(got, bfs)
        check_records(d, want, out, off, dropped)
        for key in STAT_KEYS:
            assert st[key] == st0[key], key
        monkeypatch.delenv("GP_POLISH_CAPS")
        pinned.zero_()
        ctx.pipeline_run()
        out2, off2, dropped2 = ctx.polish_fetch()
        assert ctx.stats()["polish_reruns"] == reruns
        assert np.array_equal(ctx.build_fetch(out=pinned).numpy(), bfs)
        assert np.array_equal(off2, off) and np.array_equal(dropped2, dropped)
        assert np.array_equal(out2[:int(off2[-1])], out[:int(off[-1])])
        ctx.build_output(None)


_restated = {}


def _records_want(d, pl, bfs, ks):
    if ks not in _restated:
        rows = []
        for c in range(d.n_contigs):
            out, origin = chain_with_origins(d.contig(c), [bfs[pl.contig_batch[c], ki] for ki in range(len(ks))], ks)
            rows.append(None if out is None else derive_records(d.contig(c), out, origin))
        _restated[ks] = rows
    return _restated[ks]


@pytest.mark.parametrize("edits_first", [True, False])
@pytest.mark.parametrize("route", ["polish", "pipeline", "pipeline_pool"])
@pytest.mark.parametrize("ks", [KS, ODD])
def test_edit_records_across_reruns(gp, ks, route, edits_first, monkeypatch):
    """track_edits: the re-run happens inside polish_fetch_edits (called first) or inside polish_fetch (called first);
    either way the records equal the restatement record for record."""
    import torch
    d, pl, _, _ = _ref()
    nb = len(pl.batch_entry_off) - 1
    monkeypatch.setenv("GP_POLISH_CAPS", BOTH)
    with gp.Context(ks=ks, track_edits=True, max_resident_filters=2 if route == "pipeline_pool" else 0) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        if route == "polish":
            bfs = ctx.build_filters(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.polish_run()
        else:
            pinned = torch.zeros((nb, len(ks), gp.BF_BYTES), dtype=torch.uint8).pin_memory()
            ctx.build_output(pinned)
            ctx.build_stage(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.pipeline_run()
            bfs = ctx.build_fetch(out=pinned).numpy().copy()
        if edits_first:
            rec = ctx.polish_fetch_edits()
            reruns = ctx.stats()["polish_reruns"]
            out, off, dropped = ctx.polish_fetch()
        else:
            out, off, dropped = ctx.polish_fetch()
            reruns = ctx.stats()["polish_reruns"]
            rec = ctx.polish_fetch_edits()
        assert reruns >= 1 and ctx.stats()["polish_reruns"] == reruns
        if route != "polish":
            ctx.build_output(None)
    want = _records_want(d, pl, bfs, ks)
    got = device_records(rec, d.n_contigs)
    for c in range(d.n_contigs):
        if want[c] is None:
            assert dropped[c] and got[c] == [], c
        else:
            assert not dropped[c] and got[c] == want[c], f"contig {c}: device records differ from the restatement"
    assert sum(len(g) for g in got) > 0


def test_mask_and_to_upper_across_rerun(gp, monkeypatch):
    d, pl, _, _ = _ref()
    with gp.Context(prep_mode=1, prep_k=32, to_upper=1) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        out0, off0, dr0 = ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        out0 = out0[:int(off0[-1])].copy()
        monkeypatch.setenv("GP_POLISH_CAPS", BOTH)
        out, off, dropped = ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        assert ctx.stats()["polish_reruns"] >= 1
    assert np.array_equal(off, off0) and np.array_equal(dropped, dr0)
    assert np.array_equal(out[:int(off[-1])], out0)


def test_overflow_after_four_doublings(gp, monkeypatch):
    """One rope node per contig: 16 after four doublings are too few for the edited contigs.  Every fetch says so
    (and re-runs nothing more); after the knob is gone a new polish_stage starts again from the default layout."""
    d, pl, want, _ = _ref()
    with gp.Context(track_edits=True) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        monkeypatch.setenv("GP_POLISH_CAPS", ",1")
        ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
        ctx.polish_run()
        for fetch in (ctx.polish_fetch, ctx.polish_fetch, ctx.polish_fetch_edits):
            with pytest.raises(gp.GpError) as e:
                fetch()
            assert e.value.code == -6
            assert ctx.stats()["polish_reruns"] == 4
        monkeypatch.delenv("GP_POLISH_CAPS")
        ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
        ctx.polish_run()
        out, off, dropped = ctx.polish_fetch()
        assert ctx.stats()["polish_reruns"] == 4
        check_records(d, want, out, off, dropped)


def _tool_outputs(caps):
    """ntedit-gr --vcf --bed and goldpolish-ntedit (GP_EDITS_VCF=1, GP_FLAGGED_BED) on the golden ntEdit cases: the
    bytes of every file they write."""
    import json
    from util import GOLDEN
    env = dict(ENV)
    env.pop("GP_POLISH_CAPS", None)
    if caps:
        env["GP_POLISH_CAPS"] = caps
    w = tempfile.mkdtemp()
    try:
        g, bfs = _bf_files(w)
        cli = json.load(open(os.path.join(GOLDEN, "ntedit_cli.json")))
        names = ["mixed_dense", "subs", "short_80bp", "lowercase"]
        fa = os.path.join(w, "in.fa")
        with open(fa, "w") as f:
            f.write(cli["input_fasta"])
            for n in names:
                f.write(f">{n} a comment\n{g['cases'][n]['draft']}\n")
        subprocess.check_call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-d5", "-i5", "-m1", "-X0.5", "-Y0.5",
                               "-b", os.path.join(w, "out"), "-t1", "-a1", "--vcf", os.path.join(w, "gr.vcf"),
                               "--bed", os.path.join(w, "gr.bed")], env=env, stdout=subprocess.DEVNULL)
        base = os.path.join(w, "batch")
        with open(base + ".fa", "w") as f:
            for n in names:
                f.write(f">{n} some comment\n{g['cases'][n]['draft']}\n")
        out = os.path.join(w, "batch.ntedited.fa")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out],
                              env=dict(env, GP_EDITS_VCF="1", GP_FLAGGED_BED=os.path.join(w, "chain.bed")),
                              stdout=subprocess.DEVNULL)
        files = {}
        for name in ("out_edited.fa", "gr.vcf", "gr.bed", "batch.ntedited.fa", "batch.ntedited.fa.edits.vcf", "chain.bed"):
            with open(os.path.join(w, name), "rb") as f:
                files[name] = f.read()
        return files
    finally:
        shutil.rmtree(w, ignore_errors=True)


def test_tools_write_the_same_files():
    plain, small = _tool_outputs(None), _tool_outputs("16,8")
    assert plain.keys() == small.keys()
    for name in plain:
        assert small[name] == plain[name], name
    assert plain["gr.vcf"].count(b"\n") > 10 and plain["batch.ntedited.fa.edits.vcf"].count(b"\n") > 10
