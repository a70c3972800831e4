"""The C++ drop-in tools (goldpolish_b200/host): index builder on CPU; FIFO server, ntedit-gr and
goldpolish-ntedit on the GPU, all against golden vectors minted from the reference's binaries."""
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

from util import GOLDEN, KS, ROOT, ol, sha

BIN = os.path.join(ROOT, "goldpolish_b200", "bin")
ENV = dict(os.environ, GP_QUIET="1")


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def _tmp():
    return tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)


def test_index_tool_matches_reference_index():
    import sim
    g = _load("filters.json")
    for case in g["cases"]:
        with _tmp() as w:
            d = sim.simulate(write_dir=w, **case["sim"])
            reads = os.path.join(w, "reads.fq" if d.fastq else "reads.fa")
            subprocess.check_call([os.path.join(BIN, "goldpolish-index"), reads, reads + ".idx"], env=ENV)
            got = sha("".join(sorted(open(reads + ".idx").readlines())).encode())
            assert got == case["reads_index_sha256"], case["name"]


def test_server_slab_reader_fetches_the_reads_the_index_names():
    """SeqIndex::read_many (the server's slab reader: all host cores pread the reads of a slab into place) returns the
    sequence line of every id, in the order asked, for FASTQ and FASTA, whatever the slab size and thread count --
    what the reference's SeqIndex::get_seq<1> returns one read at a time (src/seqindex.hpp:59-102)."""
    import sim
    rng = np.random.default_rng(5)
    for fastq in (1, 0):
        with _tmp() as w:
            d = sim.simulate(write_dir=w, genome_len=400000, coverage=12.0, seed=77, fastq=fastq)
            reads = os.path.join(w, "reads.fq" if d.fastq else "reads.fa")
            subprocess.check_call([os.path.join(BIN, "goldpolish-index"), reads, reads + ".idx"], env=ENV)
            ids = rng.permutation(d.n_reads)[: d.n_reads // 2].tolist() + [3, 3, 0]      # scrambled, with repeats
            with open(os.path.join(w, "ids"), "w") as f:
                f.write("".join(d.read_name(i) + "\n" for i in ids))
            want = b"".join(d.read(i) + b"\n" for i in ids)
            for slab, threads in ((1, 1), (200000, 3), (5 << 20, 8), (64 << 20, 0)):
                got = subprocess.check_output([os.path.join(BIN, "gp-host-check"), "reads", reads, reads + ".idx",
                                               os.path.join(w, "ids"), str(slab), str(threads)], env=ENV)
                assert got == want, (fastq, slab, threads)


def _parse_bf(path):
    data = open(path, "rb").read()
    hdr_end = data.index(b"[HeaderEnd]\n")
    fields = dict(ln.split(" = ") for ln in data[:hdr_end].decode().splitlines()[1:] if " = " in ln)
    n = int(fields["bytes"])
    return fields, data[len(data) - n:]


@pytest.mark.gpu
def test_fifo_server_matches_reference_server():
    import sim
    from oracle import ref_driver as rd
    g = _load("filters.json")
    jobs = [(c, "mappings.paf", 150.0, 40.0) for c in g["cases"][:2]] + [(g["ntlink"], "mappings.tsv", g["ntlink"]["mx_max"], g["ntlink"]["subsample_max"])]
    assert g["cases"][0].get("sam_equals_paf")
    jobs.append((g["cases"][0], "mappings.sam", 150.0, 40.0))
    for case, mapfile, mx_max, sub in jobs:
        with _tmp() as w:
            d = sim.simulate(write_dir=w, **case["sim"])
            reads = os.path.join(w, "reads.fq" if d.fastq else "reads.fa")
            if mapfile.endswith(".sam"):
                import importlib.util
                spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
                mg = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mg)
                mg.write_sam(d, os.path.join(w, mapfile))
            for f in (os.path.join(w, "draft.fa"), reads):
                subprocess.check_call([os.path.join(BIN, "goldpolish-index"), f, f + ".index"], env=ENV)
            bs = case["bsize"]
            with rd.BfServer(os.path.join(w, "bfs"), os.path.join(w, "draft.fa"), os.path.join(w, "draft.fa.index"),
                             os.path.join(w, mapfile), reads, reads + ".index", mx_max=mx_max, subsample_max=sub,
                             threads=2, binary=os.path.join(BIN, "goldpolish-targeted-bfs"), env=ENV) as srv:
                for b, rec in enumerate(case["batches"]):
                    ids = [d.contig_name(c) for c in range(b * bs, min((b + 1) * bs, d.n_contigs))]
                    paths = srv.build(str(b), ids)
                    got = []
                    for k in KS:
                        fields, pay = _parse_bf(paths[k])
                        assert int(fields["k"]) == k and int(fields["hash_num"]) == 4 and int(fields["bytes"]) == 524288
                        got.append(sha(pay))
                    assert got == rec["server_bf_sha256"], (case["name"], b)
                    # the per-batch pipes are gone, as after the reference's serve_batch (:144-145)
                    assert not os.path.exists(os.path.join(w, "bfs", f"{b}-bfs_ready"))
            assert not os.path.exists(os.path.join(w, "bfs", "batch_name_input"))


def _truth_bf_files(w):
    g = _load("ntedit_cases.json")
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
    return g, fs, paths


@pytest.mark.gpu
def test_ntedit_gr_cli_matches_reference_binary():
    cli = _load("ntedit_cli.json")
    with _tmp() as w:
        _, _, bfs = _truth_bf_files(w)
        fa = os.path.join(w, "in.fa")
        open(fa, "w").write(cli["input_fasta"])
        subprocess.check_call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-d5", "-i5", "-m1", "-X0.5",
                               "-Y0.5", "-b", os.path.join(w, "out"), "-t1", "-a1"], env=ENV)
        assert open(os.path.join(w, "out_edited.fa")).read() == cli["edited_fasta"]
        # -x/-y threshold form with ntEdit's own defaults, and a mode-2 / custom-limit run
        subprocess.check_call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-b", os.path.join(w, "xy"), "-t1"], env=ENV)
        assert open(os.path.join(w, "xy_edited.fa")).read() == cli["edited_fasta_defaults_xy"]
        subprocess.check_call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-b", os.path.join(w, "xy2"), "-x4", "-y6",
                               "-m2", "-i2", "-d3", "-z200", "-a1", "-t1"], env=ENV)
        assert open(os.path.join(w, "xy2_edited.fa")).read() == cli["edited_fasta_x4_y6_m2_i2_d3_z200_a1"]
        # error behaviour of ntedit.cpp:346-353,1944-1947: unreadable file / malformed option -> exit 1
        assert subprocess.call([os.path.join(BIN, "ntedit-gr"), "-f", fa + ".missing", "-r", bfs[0]], env=ENV,
                               stderr=subprocess.DEVNULL) == 1
        assert subprocess.call([os.path.join(BIN, "ntedit-gr"), "-f", fa, "-r", bfs[0], "-d", "5x"], env=ENV,
                               stderr=subprocess.DEVNULL) == 1


@pytest.mark.gpu
def test_goldpolish_ntedit_chain_and_guard():
    with _tmp() as w:
        g, fs, bfs = _truth_bf_files(w)
        names = ["mixed_dense", "subs", "short_80bp", "lowercase"]
        base = os.path.join(w, "batch")
        with open(base + ".fa", "w") as f:
            for n in names:
                f.write(f">{n} some comment\n{g['cases'][n]['draft']}\n")
        out = os.path.join(w, "batch.ntedited.fa")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out],
                              env=ENV, stdout=subprocess.DEVNULL)
        want = "".join(f">{n} some comment\n{g['cases'][n]['chain']}\n" for n in names if g["cases"][n]["chain"] is not None)
        assert os.path.islink(out)
        assert os.path.basename(os.readlink(out)) == "batch.k32.X0.5.Y0.5_edited.k28.X0.5.Y0.5_edited.k24.X0.5.Y0.5_edited.k20.X0.5.Y0.5_edited.fa"
        assert open(out).read() == want
        # guard: a batch whose records are mostly dropped (< 100 bp) falls back to the original file
        base2 = os.path.join(w, "tiny")
        with open(base2 + ".fa", "w") as f:
            for i in range(6):
                f.write(f">t{i}\n{g['truth'][i * 90:i * 90 + 90]}\n")
            f.write(f">keep\n{g['truth'][:150]}\n")
        out2 = os.path.join(w, "tiny.ntedited.fa")
        subprocess.check_call([os.path.join(BIN, "goldpolish-ntedit"), base2, " ".join(bfs), "32 28 24 20", "0.5", "0.5", "1", out2],
                              env=ENV, stdout=subprocess.DEVNULL)
        assert os.readlink(out2) == base2 + ".fa"


def _odd_files(w):
    """FASTA / FASTQ files that stress the line arithmetic of src/seqindex.cpp:12-66."""
    import random
    rnd = random.Random(11)
    files = {}
    recs = []
    for i in range(3000):
        n = rnd.choice([1, 2, 5, 60, 700, 5000])               # (an empty quality line stops the reference: below)
        name = f"r{i}" if i % 97 else "dup"                      # duplicate ids: the first one wins
        tail = ["", " c=1", "\tx", " a\tb"][i % 4]               # comments after a blank, tabs inside the first token
        recs.append((name + tail, "".join(rnd.choice("ACGTNacgt") for _ in range(n)),
                     "".join(chr(rnd.randint(33, 73)) for _ in range(n))))
    files["a.fa"] = "".join(f">{h}\n{s}\n" for h, s, _ in recs)
    files["b.fq"] = "".join(f"@{h}\n{s}\n+\n{q}\n" for h, s, q in recs)
    files["c.fq"] = files["b.fq"][:-1]                           # no newline at the end of the last quality line
    files["d.fa"] = files["a.fa"].replace("\n", "\r\n")          # a '\r' stays part of its line
    files["e.fq"] = files["b.fq"] + "@cut\nACGT\n+\n"            # truncated last record: not indexed
    files["f.fa"] = files["a.fa"] + ">last"                      # header without a sequence line
    files["g.fq"] = ""                                           # empty file
    files["h.fa"] = files["a.fa"] + ">empty\n\n>x\nAC\n"        # an empty sequence line is a record of length 0
    for name, text in files.items():
        with open(os.path.join(w, name), "w", newline="") as f:
            f.write(text)
    return sorted(files)


def test_index_tool_threads_and_odd_inputs():
    """The mmap + threads index builder: any thread count gives the same file, and that file equals the
    reference's own goldpolish-index (oracle/_ref, build container only) on inputs that stress the line
    arithmetic."""
    ref = os.path.join(ROOT, "oracle", "_ref", "goldpolish-index")
    with _tmp() as w:
        for name in _odd_files(w):
            path = os.path.join(w, name)
            outs = []
            for threads in ("1", "3", "16"):
                out = path + f".idx{threads}"
                subprocess.check_call([os.path.join(BIN, "goldpolish-index"), path, out], env=dict(ENV, GP_INDEX_THREADS=threads))
                outs.append(open(out).read())
            assert outs[0] == outs[1] == outs[2], name
            if os.path.exists(ref) and os.path.getsize(path) > 0:
                subprocess.check_call([ref, path, path + ".ref"], env=ENV, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                assert sorted(outs[0].splitlines()) == sorted(open(path + ".ref").read().splitlines()), name
        # an empty quality line: btllib::calc_phred_avg refuses the range, the tool exits 1 (as the reference does)
        bad = os.path.join(w, "bad.fq")
        open(bad, "w").write("@a\nACGT\n+\nIIII\n@b\n\n+\n\n")
        assert subprocess.run([os.path.join(BIN, "goldpolish-index"), bad, bad + ".idx"], env=ENV, capture_output=True).returncode == 1
        if os.path.exists(ref):
            assert subprocess.run([ref, bad, bad + ".ref"], env=ENV, capture_output=True).returncode == 1


@pytest.mark.gpu
def test_fifo_server_two_devices_bounded_workers_concurrent_clients():
    """GP_DEVICES: one context + GPU thread per listed device, requests dealt by pending read bases; a bounded worker
    pool (3 workers for 9+ batches); clients that talk to the server concurrently, as the reference's driver does with
    its up-to-200 goldpolish-polish-batch processes (scripts/goldpolish:363-426).  Same payloads as the reference server."""
    import threading

    import sim
    import torch
    from oracle import ref_driver as rd
    g = _load("filters.json")
    case = g["cases"][0]
    devices = "0,1" if torch.cuda.device_count() >= 2 else "0,0"  # (two contexts on one GPU exercise the same code)
    env = dict(ENV, GP_DEVICES=devices, GP_SERVER_WORKERS="3")
    with _tmp() as w:
        d = sim.simulate(write_dir=w, **case["sim"])
        reads = os.path.join(w, "reads.fq" if d.fastq else "reads.fa")
        for f in (os.path.join(w, "draft.fa"), reads):
            subprocess.check_call([os.path.join(BIN, "goldpolish-index"), f, f + ".index"], env=ENV)
        bs = case["bsize"]
        bdir = os.path.join(w, "bfs")
        nb = len(case["batches"])
        results = {}
        with rd.BfServer(bdir, os.path.join(w, "draft.fa"), os.path.join(w, "draft.fa.index"), os.path.join(w, "mappings.paf"),
                         reads, reads + ".index", threads=2, binary=os.path.join(BIN, "goldpolish-targeted-bfs"), env=env) as srv:
            rounds = 3  # every batch three times under different names: 3 * nb requests in flight
            names = [f"{r}_{b}" for r in range(rounds) for b in range(nb)]
            for name in names:  # the handshake on the shared pipes is sequential (scripts/goldpolish:381-384)
                with open(os.path.join(bdir, "batch_name_input"), "w") as f:
                    f.write(name + "\n")
                with open(os.path.join(bdir, "batch_target_ids_input_ready")) as f:
                    f.read()

            def client(name):
                b = int(name.split("_")[1])
                with open(os.path.join(bdir, f"{name}-target_ids_input"), "w") as f:
                    for c in range(b * bs, min((b + 1) * bs, d.n_contigs)):
                        f.write(d.contig_name(c) + "\n")
                with open(os.path.join(bdir, f"{name}-bfs_ready")) as f:
                    f.read()
                results[name] = [sha(_parse_bf(os.path.join(bdir, f"{name}-k{k}.bf"))[1]) for k in KS]

            ths = [threading.Thread(target=client, args=(n,)) for n in names]
            for t in ths:
                t.start()
            for t in ths:
                t.join(timeout=300)
            assert all(not t.is_alive() for t in ths)
        for name in names:
            assert results[name] == case["batches"][int(name.split("_")[1])]["server_bf_sha256"], name


def _restated_ntedit_chain(records, bf_paths):
    """scripts/goldpolish-ntedit:20-40 by the C restatement (pinned to the reference by the golden vectors): the k chain
    over the batch's .bf files as ntedit-gr writes it (records < 100 bp dropped), then the 0.75 guard on the file
    sizes.  Returns the text of the file the flow keeps."""
    bfs = [np.frombuffer(_parse_bf(p)[1], dtype=np.uint8) for p in bf_paths]
    text_in, kept = "", []
    for name, seq in records:
        text_in += f">{name}\n{seq.decode()}\n"
        cur = seq
        for bf, k in zip(bfs, KS):
            cur, _ = ol.ntedit_contig(cur, bf, k)
            if cur is None:
                break
        if cur is not None:
            kept.append(f">{name}\n{cur.decode()}\n")
    text_out = "".join(kept)
    return text_in if ol.lib().gpo_guard_rejects(len(text_in), len(text_out)) else text_out


@pytest.mark.gpu
def test_polish_batch_dropin_fused_with_the_server():
    """goldpolish_b200's goldpolish-polish-batch (same command line as scripts/goldpolish-polish-batch:24-54) asks the
    server to polish the batch in the GPU pass that builds its filters; `batch.ntedited.fa` then equals what the
    reference's goldpolish-ntedit flow (its own ntedit-gr, k chain + guard; the C restatement of that flow where
    oracle/_ref is not built) makes of the same batch's .bf files, the .bf files are deleted afterwards and the
    done-pipe is signalled."""
    import shutil
    import threading

    import sim
    from oracle import ref_driver as rd
    g = _load("filters.json")
    case = g["cases"][1]
    with _tmp() as w:
        d = sim.simulate(write_dir=w, **case["sim"])
        reads = os.path.join(w, "reads.fq" if d.fastq else "reads.fa")
        for f in (os.path.join(w, "draft.fa"), reads):
            subprocess.check_call([os.path.join(BIN, "goldpolish-index"), f, f + ".index"], env=ENV)
        bs = case["bsize"]
        bdir = os.path.join(w, "bfs")
        with rd.BfServer(bdir, os.path.join(w, "draft.fa"), os.path.join(w, "draft.fa.index"), os.path.join(w, "mappings.paf"),
                         reads, reads + ".index", threads=2, binary=os.path.join(BIN, "goldpolish-targeted-bfs"), env=ENV) as srv:
            for b in range(len(case["batches"])):
                cs = list(range(b * bs, min((b + 1) * bs, d.n_contigs)))
                ids = [d.contig_name(c) for c in cs]
                # expected: plain protocol, then the reference's own ntedit-gr chain + guard on the .bf files
                plain = os.path.join(w, f"plain{b}")
                os.makedirs(plain)
                with open(os.path.join(plain, "batch.fa"), "w") as f:
                    for c in cs:
                        f.write(f">{d.contig_name(c)}\n{d.contig(c).decode()}\n")
                paths = srv.build(f"p{b}", ids)
                if rd.ref_available():
                    chosen, _ = rd.run_ntedit_chain(os.path.join(plain, "batch"), [paths[k] for k in KS])
                    expected = open(chosen).read()
                else:
                    expected = _restated_ntedit_chain([(d.contig_name(c), d.contig(c)) for c in cs], [paths[k] for k in KS])
                # drop-in: the reference driver's steps (scripts/goldpolish:363-426), then our polish-batch
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
                subprocess.check_call([os.path.join(BIN, "goldpolish-polish-batch"), "batch.fa", bdir, w, "pre", "4",
                                       "-k32", "-k28", "-k24", "-k20"] + [f"-b{name}-k{k}.bf" for k in KS] +
                                      ["--seq-ids", "seq_ids", "--bfs-ids-pipe", f"{name}-target_ids_input",
                                       "--bfs-ready-pipe", f"{name}-bfs_ready", "--batch-done-pipe", done_pipe, "-t", "1"],
                                      cwd=fused, env=dict(ENV, GP_POLISH_BATCH_STOP_AFTER="ntedit",
                                                          PATH=BIN + os.pathsep + os.environ.get("PATH", "")))
                t.join(timeout=60)
                assert got_done and got_done[0].strip() == "1"
                assert open(os.path.join(fused, "batch.ntedited.fa")).read() == expected, b
                # "@prep": what `goldpolish-mask -s -k32 batch.ntedited.fa` prints (scripts/goldpolish-make:65-66), by the
                # restatement that the reference script's own vectors pin (tests/test_mask.py) and by our mask tool
                from oracle import mask_oracle as mo
                lines = expected.split("\n")
                want = "".join(h + "\n" + mo.mask(q, 32) + "\n" for h, q in zip(lines[0::2], lines[1::2]) if h)
                prepd = os.path.join(fused, "batch.ntedited.prepd.fa")
                assert open(prepd).read() == want, b
                assert subprocess.check_output([os.path.join(BIN, "goldpolish-mask"), "-s", "-k32", "batch.ntedited.fa"],
                                               cwd=fused, env=ENV).decode() == want, b
                assert os.stat(prepd).st_mtime_ns >= os.stat(os.path.join(fused, "batch.ntedited.fa")).st_mtime_ns
                assert not any(os.path.exists(os.path.join(bdir, f"{name}-k{k}.bf")) for k in KS)
