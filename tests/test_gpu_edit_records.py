"""Edit records on the device (gp_polish_fetch_edits, Context(track_edits=True)): record for record against the numpy
restatement over ntEdit's C restatement with origins, through gp_polish and gp_pipeline_run and with a 2-batch filter
pool; tracking changes no polished byte; the records replay to the polished records at config-2 size; the VCF of
ntedit-gr --vcf and goldpolish-ntedit (GP_EDITS_VCF=1); the error paths."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_edit_records import TYPES, _up, chain_with_origins, derive_records, replay
from util import GOLDEN, KS, ROOT, dataset, ol, plan

pytestmark = pytest.mark.gpu

ODD = (31, 27, 23, 19)
BIN = os.path.join(ROOT, "goldpolish_b200", "bin")
ENV = dict(os.environ, GP_QUIET="1")


@pytest.fixture(scope="module")
def gp():
    import goldpolish_b200
    return goldpolish_b200


def device_records(rec, n_contigs):
    """Per contig: [(pos, REF, ALT, TYPE)] from polish_fetch_edits' arrays."""
    off, al = rec["offsets"], rec["alleles"]
    out = []
    for c in range(n_contigs):
        rows = []
        for r in range(int(off[c]), int(off[c + 1])):
            a, rl, xl = int(rec["allele_off"][r]), int(rec["ref_len"][r]), int(rec["alt_len"][r])
            rows.append((int(rec["pos"][r]), al[a:a + rl].tobytes().decode(), al[a + rl:a + rl + xl].tobytes().decode(),
                         TYPES[int(rec["type"][r])]))
        out.append(rows)
    return out


_want_cache = {}


def _restated(d, pl, bfs, ks, bsize):
    key = (ks, bsize)
    if key not in _want_cache:
        want = []
        for c in range(d.n_contigs):
            draft = d.contig(c)
            out, origin = chain_with_origins(draft, [bfs[pl.contig_batch[c], ki] for ki in range(len(ks))], ks)
            want.append(None if out is None else derive_records(draft, out, origin))
        _want_cache[key] = want
    return _want_cache[key]


def _run(gp, d, pl, ks, path, track=True, **kw):
    with gp.Context(ks=ks, track_edits=track, **kw) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        if path == "polish":
            bfs = ctx.build_filters(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            ctx.polish_run()
        else:
            ctx.build_stage(pl.batch_entry_off, pl.entries)
            ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
            pinned = None
            if kw.get("max_resident_filters"):  # a pool of fewer batches than the call: payloads go to page-locked memory
                import torch
                pinned = torch.empty((len(pl.batch_entry_off) - 1, len(ks), gp.BF_BYTES), dtype=torch.uint8).pin_memory()
                ctx.build_output(pinned)
            ctx.pipeline_run()
            bfs = ctx.build_fetch(out=pinned)
            bfs = bfs.numpy() if pinned is not None else bfs
        rec = ctx.polish_fetch_edits() if track else None
        out, off, dropped = ctx.polish_fetch()
        st = ctx.stats()
    return bfs, rec, out, off, dropped, st


CASES = [(ks, bsize, path) for ks in (KS, ODD) for bsize in (1, 8) for path in ("polish", "pipeline")]


@pytest.mark.parametrize("ks,bsize,path", CASES)
def test_device_records_equal_the_restatement(gp, ks, bsize, path):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=bsize)
    bfs, rec, out, off, dropped, _ = _run(gp, d, pl, ks, path)
    want = _restated(d, pl, bfs, ks, bsize)
    got = device_records(rec, d.n_contigs)
    for c in range(d.n_contigs):
        if want[c] is None:
            assert dropped[c] and got[c] == [], c
        else:
            assert got[c] == want[c], f"contig {c}: device records differ from the restatement"
    assert sum(len(g) for g in got) > 0


def test_two_batch_filter_pool(gp):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    assert len(pl.batch_entry_off) - 1 > 2
    bfs, rec, out, off, dropped, _ = _run(gp, d, pl, KS, "pipeline", max_resident_filters=2)
    want = _restated(d, pl, bfs, KS, 1)
    got = device_records(rec, d.n_contigs)
    for c in range(d.n_contigs):
        assert got[c] == (want[c] or []), c


@pytest.mark.parametrize("path", ["polish", "pipeline"])
def test_tracking_changes_no_polished_byte(gp, path):
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    _, _, out1, off1, dr1, st1 = _run(gp, d, pl, ODD, path, track=True)
    _, _, out0, off0, dr0, st0 = _run(gp, d, pl, ODD, path, track=False)
    assert np.array_equal(off1, off0) and np.array_equal(dr1, dr0)
    assert np.array_equal(out1[:int(off1[-1])], out0[:int(off0[-1])])
    for key in ("triggers", "edits", "masked", "rollbacks", "kmer_ops"):
        assert st1[key] == st0[key], key


def test_config2_size_records_replay(gp):
    d = dataset(genome_len=5_000_000)
    pl = plan(d, bsize=1)
    _, rec, out, off, dropped, st = _run(gp, d, pl, KS, "pipeline")
    got = device_records(rec, d.n_contigs)
    edited = 0
    for c in range(d.n_contigs):
        if dropped[c]:
            assert got[c] == []
            continue
        assert replay(d.contig(c), got[c]) == _up(out[int(off[c]):int(off[c + 1])].tobytes()).tobytes(), c
        edited += bool(got[c])
    assert edited > 0 and st["edits"] > 0


def test_error_paths(gp):
    with pytest.raises(gp.GpError) as e:
        gp.Context(track_edits=True, prep_mode=2, prep_k=32)
    assert e.value.code == -1
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    with gp.Context() as ctx:  # tracking off
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        with pytest.raises(gp.GpError) as e:
            ctx.polish_fetch_edits()
        assert e.value.code == -5
    with gp.Context(track_edits=True) as ctx:
        with pytest.raises(gp.GpError) as e:  # before any polish
            ctx.polish_fetch_edits()
        assert e.value.code == -5
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_filters(pl.batch_entry_off, pl.entries, fetch=False)
        ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        full = ctx.polish_fetch_edits()
        n_rec, n_bytes = len(full["pos"]), len(full["alleles"])
        assert n_rec > 0
        off = np.zeros(d.n_contigs + 1, dtype=np.uint64)
        need = np.zeros(2, dtype=np.uint64)
        recs = np.zeros(n_rec, dtype=gp.api.EDIT_DTYPE)
        al = np.zeros(n_bytes, dtype=np.uint8)
        l = gp.load_library()
        for cap_r, cap_a in ((0, 0), (n_rec - 1, n_bytes), (n_rec, n_bytes - 1)):
            need[:] = 0
            rc = l.gp_polish_fetch_edits(ctx._h, off.ctypes.data, recs.ctypes.data, cap_r, al.ctypes.data, cap_a,
                                         need.ctypes.data)
            assert rc == -1 and need.tolist() == [n_rec, n_bytes]
        assert np.array_equal(off, full["offsets"])
        rc = l.gp_polish_fetch_edits(ctx._h, off.ctypes.data, recs.ctypes.data, n_rec, al.ctypes.data, n_bytes,
                                     need.ctypes.data)
        assert rc == 0 and np.array_equal(recs["pos"], full["pos"]) and np.array_equal(al, full["alleles"])


# ---- the drop-in tools -------------------------------------------------------------------------------------------------
def parse_vcf(path):
    contigs, recs = [], {}
    with open(path) as f:
        lines = f.read().splitlines()
    assert lines[0] == "##fileformat=VCFv4.2" and "##source=goldpolish_b200" in lines
    assert any(ln.startswith("##INFO=<ID=TYPE,") for ln in lines)
    assert "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO" in lines
    for ln in lines:
        if ln.startswith("##contig=<ID="):
            name, length = ln[len("##contig=<ID="):-1].split(",length=")
            contigs.append((name, int(length)))
        elif not ln.startswith("#"):
            chrom, pos, ident, ref, alt, qual, filt, info = ln.split("\t")
            assert ident == "." and qual == "." and filt == "PASS" and info.startswith("TYPE=")
            recs.setdefault(chrom, []).append((int(pos) - 1, ref, alt, info[5:]))
    for rows in recs.values():
        assert [r[0] for r in rows] == sorted(r[0] for r in rows)
    return contigs, recs


def _fasta(path):
    recs, name = {}, None
    for ln in open(path).read().splitlines():
        if ln.startswith(">"):
            name = ln[1:].split()[0]
            recs[name] = ""
        elif name is not None:
            recs[name] += ln
    return recs


def _bf_files(w):
    import json
    g = json.load(open(os.path.join(GOLDEN, "ntedit_cases.json")))
    fs = ol.FilterSet(KS)
    for _ in range(5):
        fs.add_read(g["truth"].encode(), 4)
    paths = []
    for i, k in enumerate(KS):
        p = os.path.join(w, f"k{k}.bf")
        with open(p, "wb") as f:
            f.write(f'[BTLKmerBloomFilter_v6]\nbytes = 524288\nhash_fn = "ntHash_v2"\nhash_num = 4\nk = {k}\n[HeaderEnd]\n'.encode())
            f.write(b"\n  <binary data>\n" + b"\n" * 48)
            f.write(fs.bfs[i].tobytes())
        paths.append(p)
    return g, paths


def test_ntedit_gr_vcf():
    import json
    cli = json.load(open(os.path.join(GOLDEN, "ntedit_cli.json")))
    w = tempfile.mkdtemp()
    try:
        g, bfs = _bf_files(w)
        fa = os.path.join(w, "in.fa")
        names = ["mixed_dense", "subs", "short_80bp", "lowercase"]
        with open(fa, "w") as f:
            f.write(cli["input_fasta"])
            for n in names:
                f.write(f">{n} a comment\n{g['cases'][n]['draft']}\n")
        vcf = os.path.join(w, "edits.vcf")
        subprocess.check_call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-d5", "-i5", "-m1", "-X0.5",
                               "-Y0.5", "-b", os.path.join(w, "out"), "-t1", "-a1", "--vcf", vcf], env=ENV)
        drafts = _fasta(fa)
        edited = _fasta(os.path.join(w, "out_edited.fa"))
        contigs, recs = parse_vcf(vcf)
        assert contigs == [(n, len(s)) for n, s in drafts.items()]
        assert set(recs) <= set(edited) and recs
        for name, seq in edited.items():
            assert replay(drafts[name].encode(), recs.get(name, [])) == seq.upper().encode(), name
    finally:
        shutil.rmtree(w, ignore_errors=True)


def test_goldpolish_ntedit_vcf_and_guard():
    w = tempfile.mkdtemp()
    try:
        g, bfs = _bf_files(w)
        names = ["mixed_dense", "subs", "short_80bp", "lowercase"]
        base = os.path.join(w, "batch")
        with open(base + ".fa", "w") as f:
            for n in names:
                f.write(f">{n} some comment\n{g['cases'][n]['draft']}\n")
        out = os.path.join(w, "batch.ntedited.fa")
        env = dict(ENV, GP_EDITS_VCF="1")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out],
                              env=env, stdout=subprocess.DEVNULL)
        contigs, recs = parse_vcf(out + ".edits.vcf")
        assert [c for c, _ in contigs] == names
        assert "short_80bp" not in recs and recs
        for n in names:
            if g["cases"][n]["chain"] is not None:
                assert replay(g["cases"][n]["draft"].encode(), recs.get(n, [])) == g["cases"][n]["chain"].upper().encode(), n
        # a batch the 0.75 guard rejects: its output is the input, and the VCF holds the header only
        base2 = os.path.join(w, "tiny")
        with open(base2 + ".fa", "w") as f:
            for i in range(6):
                f.write(f">t{i}\n{g['truth'][i * 90:i * 90 + 90]}\n")
            f.write(f">keep\n{g['truth'][:150]}\n")
        out2 = os.path.join(w, "tiny.ntedited.fa")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base2, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out2],
                              env=env, stdout=subprocess.DEVNULL)
        assert os.readlink(out2) == base2 + ".fa"
        contigs, recs = parse_vcf(out2 + ".edits.vcf")
        assert len(contigs) == 7 and recs == {}
        # without the variable no VCF is written
        out3 = os.path.join(w, "batch3.ntedited.fa")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out3],
                              env=ENV, stdout=subprocess.DEVNULL)
        assert not os.path.exists(out3 + ".edits.vcf")
    finally:
        shutil.rmtree(w, ignore_errors=True)
