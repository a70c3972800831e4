"""k values that are not multiples of 4, on the device, through the C ABI and the drop-in tools: the hashes of every k in
4..32, filter bits and counter bytes for k lists that mix residues mod 4, the overlapped pipeline, the edit kernel
chained over such lists, and the FIFO server / goldpolish-polish-batch / goldpolish-ntedit flow at -k 31 27 23 19."""
import os
import shutil
import subprocess
import threading

import numpy as np
import pytest

from test_any_k import random_read
from util import ROOT, dataset, ol, plan

pytestmark = pytest.mark.gpu

LISTS = [(31, 27, 25, 21), (30, 26, 22, 18), (29, 23, 17, 5), (32, 25, 20, 13)]
ODD = (31, 27, 23, 19)  # 31, 27, 23 cover every residue mod 3 (the edit kernel's sample sets)
BIN = os.path.join(ROOT, "goldpolish_b200", "bin")
ENV = dict(os.environ, GP_QUIET="1")


@pytest.fixture(scope="module")
def gp():
    import goldpolish_b200
    return goldpolish_b200


def _oracle_filters(d, pl, ks):
    out = []
    for b in range(len(pl.batch_entry_off) - 1):
        fs = ol.FilterSet(ks)
        for e in range(int(pl.batch_entry_off[b]), int(pl.batch_entry_off[b + 1])):
            fs.add_read(d.read(int(pl.entries[e]["read_id"])), int(pl.entries[e]["kmer_threshold"]))
        out.append(fs)
    return out


def _chain(seq, bfs, ks, **opts):
    """ntEdit chained over the k list (scripts/goldpolish-ntedit:20-29) by the C restatement; None when dropped"""
    cur, rollbacks = seq, 0
    for bf, k in zip(bfs, ks):
        cur, st = ol.ntedit_contig(cur, bf, k, **opts)
        if cur is None:
            return None, rollbacks
        rollbacks += st["rollbacks"]
    return cur, rollbacks


def test_debug_nthash_every_k(gp):
    """h0..h3 and valid positions of every k in 4..32 as the build kernels' device code computes them, on reads with
    lower-case bases, N runs and other non-ACGT bytes, against the C restatement."""
    rng = np.random.default_rng(404)
    seqs = [random_read(rng, int(n)) for n in (4, 5, 31, 33, 64, 65, 97, 300, 1000)]
    data = np.frombuffer(b"".join(seqs), dtype=np.uint8)
    off = np.cumsum([0] + [len(s) for s in seqs]).astype(np.uint64)
    n = 0
    with gp.Context() as ctx:
        ctx.upload_reads(data, off)
        for k in range(4, 33):
            for i, s in enumerate(seqs):
                pos, hs = ctx.debug_nthash(i, k)
                want_pos, want_hs = ol.nthash_all(s, k)
                assert np.array_equal(pos, want_pos), (k, i)
                assert np.array_equal(hs, want_hs), (k, i)
                n += len(want_pos)
    assert n > 10000


@pytest.mark.parametrize("algo", ["l", "s"])
@pytest.mark.parametrize("ks", LISTS)
@pytest.mark.parametrize("size", ["bsize1", "bsize8_loaded"])
def test_filters_and_counters_match_oracle(gp, ks, algo, size, monkeypatch):
    """Filter bits AND counter bytes of every batch, level-synchronous and in-order kernels.  The bsize-8 cut loads
    the counting filters far beyond one touch per counter, where an order-free update would differ."""
    monkeypatch.setenv("GP_BUILD_KERNEL", algo)
    d = dataset(genome_len=60000) if size == "bsize1" else dataset(genome_len=300000, coverage=40.0)
    pl = plan(d, bsize=1 if size == "bsize1" else 8)
    ref = _oracle_filters(d, pl, ks)
    with gp.Context(ks=ks, keep_counters=1) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        bfs = ctx.build_filters(pl.batch_entry_off, pl.entries)
        assert ctx.stats()["kmer_ops"] == sum(fs.ops for fs in ref)
        for b, fs in enumerate(ref):
            for ki, k in enumerate(ks):
                assert np.array_equal(bfs[b, ki], fs.bfs[ki]), f"BF differs: batch {b} k={k}"
                assert np.array_equal(ctx.fetch_cbf(b, ki), fs.cbfs[ki]), f"CBF differs: batch {b} k={k}"


@pytest.mark.parametrize("resident", [0, 2])
def test_pipeline_matches_separate_calls_and_oracle(gp, resident):
    """gp_pipeline_run at -k 31 27 23 19 with all filters resident and with a 2-batch pool (several waves, every
    batch holding contigs; the payloads arrive in a page-locked buffer) gives the filters and records of
    gp_build_run + gp_polish_run and of the oracle."""
    import torch
    d = dataset(genome_len=150000)
    pl = plan(d, bsize=4)
    with gp.Context(ks=ODD) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        bfs = ctx.build_filters(pl.batch_entry_off, pl.entries)
        out, off, dropped = ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        out = out[:int(off[-1])].copy()
    nb = len(pl.batch_entry_off) - 1
    assert nb > 2 * 2
    pinned = torch.zeros((nb, len(ODD), gp.BF_BYTES), dtype=torch.uint8).pin_memory()
    with gp.Context(ks=ODD, max_resident_filters=resident) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        ctx.build_stage(pl.batch_entry_off, pl.entries)
        ctx.build_output(pinned)
        ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
        ctx.pipeline_run()
        if resident:
            assert ctx.stats()["build_launches"] == (nb + resident - 1) // resident
        bfs2 = ctx.build_fetch(out=pinned).numpy()
        out2, off2, dropped2 = ctx.polish_fetch()
    assert np.array_equal(bfs, bfs2)
    assert np.array_equal(off, off2) and np.array_equal(dropped, dropped2)
    assert np.array_equal(out, out2[:int(off2[-1])])
    ref = _oracle_filters(d, pl, ODD)
    for b, fs in enumerate(ref):
        for ki in range(len(ODD)):
            assert np.array_equal(bfs[b, ki], fs.bfs[ki]), (b, ki)
    for c in range(d.n_contigs):
        want, _ = _chain(d.contig(c), [bfs[pl.contig_batch[c], ki] for ki in range(len(ODD))], ODD)
        got = out[int(off[c]):int(off[c + 1])].tobytes()
        assert (want is None and dropped[c]) or (not dropped[c] and got == want), c


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_polish_chain_matches_oracle(gp, mode):
    """Every contig polished over -k 31 27 23 19 (each residue mod 3), in modes 0/1/2, against ntEdit's C restatement
    chained over the same filters; the data set holds contigs that take the low-complexity rollback."""
    d = dataset(genome_len=400000)
    pl = plan(d, bsize=1)
    with gp.Context(ks=ODD, mode=mode) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        bfs = ctx.build_filters(pl.batch_entry_off, pl.entries)
        out, off, dropped = ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        st = ctx.stats()
    rollbacks = 0
    for c in range(d.n_contigs):
        want, rb = _chain(d.contig(c), [bfs[pl.contig_batch[c], ki] for ki in range(len(ODD))], ODD, mode=mode)
        rollbacks += rb
        got = out[int(off[c]):int(off[c + 1])].tobytes()
        if want is None:
            assert dropped[c] == 1 and got == b"", c
        else:
            assert dropped[c] == 0 and got == want, f"contig {c} (mode {mode}) differs from the oracle"
    assert st["edits"] > 0
    assert rollbacks > 0 and st["rollbacks"] > 0


def _parse_bf(path):
    data = open(path, "rb").read()
    hdr_end = data.index(b"[HeaderEnd]\n")
    fields = dict(ln.split(" = ") for ln in data[:hdr_end].decode().splitlines()[1:] if " = " in ln)
    return fields, data[len(data) - int(fields["bytes"]):]


def _restated_flow(records, bf_paths, ks):
    """scripts/goldpolish-ntedit:20-40 by the C restatement: the k chain over the .bf files (records < 100 bp dropped),
    then the 0.75 guard on the file sizes.  Returns the text of the file the flow keeps."""
    bfs = [np.frombuffer(_parse_bf(p)[1], dtype=np.uint8) for p in bf_paths]
    text_in, kept = "", []
    for name, seq in records:
        text_in += f">{name}\n{seq.decode()}\n"
        cur, _ = _chain(seq, bfs, ks)
        if cur is not None:
            kept.append(f">{name}\n{cur.decode()}\n")
    text_out = "".join(kept)
    return text_in if ol.lib().gpo_guard_rejects(len(text_in), len(text_out)) else text_out


def test_dropin_tools_at_odd_k(tmp_path):
    """goldpolish-index -> goldpolish-targeted-bfs ... 31 27 23 19 -> goldpolish-polish-batch (fused @polish and
    @prep -k31), and goldpolish-ntedit over the served .bf files: header k, payloads and records against the oracle."""
    import sim
    from oracle import mask_oracle as mo
    from oracle import ref_driver as rd
    w = str(tmp_path)
    d = sim.simulate(write_dir=w, genome_len=60000, seed=31)
    reads = os.path.join(w, "reads.fq" if d.fastq else "reads.fa")
    draft = os.path.join(w, "draft.fa")
    for f in (draft, reads):
        subprocess.check_call([os.path.join(BIN, "goldpolish-index"), f, f + ".index"], env=ENV)
    pl = plan(d, bsize=2)
    ref = _oracle_filters(d, pl, ODD)
    bdir = os.path.join(w, "bfs")
    with rd.BfServer(bdir, draft, draft + ".index", os.path.join(w, "mappings.paf"), reads, reads + ".index", threads=2,
                     ks=ODD, binary=os.path.join(BIN, "goldpolish-targeted-bfs"), env=ENV) as srv:
        for b in range(min(3, len(pl.batch_entry_off) - 1)):
            cs = [int(c) for c in np.nonzero(pl.contig_batch == b)[0]]
            ids = [d.contig_name(c) for c in cs]
            records = [(d.contig_name(c), d.contig(c)) for c in cs]
            # plain protocol: the served .bf files
            paths = srv.build(f"p{b}", ids)
            for ki, k in enumerate(ODD):
                fields, payload = _parse_bf(paths[k])
                assert int(fields["k"]) == k
                assert np.array_equal(np.frombuffer(payload, dtype=np.uint8), ref[b].bfs[ki]), (b, k)
            expected = _restated_flow(records, [paths[k] for k in ODD], ODD)
            # goldpolish-ntedit over those files
            plain = os.path.join(w, f"plain{b}")
            os.makedirs(plain)
            with open(os.path.join(plain, "batch.fa"), "w") as f:
                f.writelines(f">{n}\n{s.decode()}\n" for n, s in records)
            out = os.path.join(plain, "batch.ntedited.fa")
            subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), os.path.join(plain, "batch"),
                                   " ".join(paths[k] for k in ODD), " ".join(map(str, ODD)), "0.5", "0.5", "1", out],
                                  env=ENV, stdout=subprocess.DEVNULL)
            assert open(out).read() == expected, b
            # goldpolish-polish-batch, fused with the server
            fused = os.path.join(w, f"fused{b}")
            os.makedirs(fused)
            shutil.copy(os.path.join(plain, "batch.fa"), os.path.join(fused, "batch.fa"))
            with open(os.path.join(fused, "seq_ids"), "w") as f:
                f.write("\n".join(ids) + "\n")
            done_pipe = os.path.join(fused, "polishing_done")
            os.mkfifo(done_pipe)
            name = f"f{b}"
            with open(os.path.join(bdir, "batch_name_input"), "w") as f:
                f.write(name + "\n")
            with open(os.path.join(bdir, "batch_target_ids_input_ready")) as f:
                f.read()
            got_done = []
            t = threading.Thread(target=lambda: got_done.append(open(done_pipe).read()))
            t.start()
            subprocess.check_call([os.path.join(BIN, "goldpolish-polish-batch"), "batch.fa", bdir, w, "pre", "4"] +
                                  [f"-k{k}" for k in ODD] + [f"-b{name}-k{k}.bf" for k in ODD] +
                                  ["--seq-ids", "seq_ids", "--bfs-ids-pipe", f"{name}-target_ids_input",
                                   "--bfs-ready-pipe", f"{name}-bfs_ready", "--batch-done-pipe", done_pipe, "-t", "1"],
                                  cwd=fused, env=dict(ENV, GP_POLISH_BATCH_STOP_AFTER="ntedit",
                                                      PATH=BIN + os.pathsep + os.environ.get("PATH", "")))
            t.join(timeout=60)
            assert got_done and got_done[0].strip() == "1"
            assert open(os.path.join(fused, "batch.ntedited.fa")).read() == expected, b
            lines = expected.split("\n")
            want = "".join(h + "\n" + mo.mask(q, ODD[0]) + "\n" for h, q in zip(lines[0::2], lines[1::2]) if h)
            assert open(os.path.join(fused, "batch.ntedited.prepd.fa")).read() == want, b
            assert not any(os.path.exists(os.path.join(bdir, f"{name}-k{k}.bf")) for k in ODD)
