"""CPU: the sharding bookkeeping bench.py uses for the strong-scaling run (no GPU, no collective): every batch lands on
exactly one rank, a rank's share is self-contained (entries re-indexed into its own read store, contigs with their
batches), and the guard rule applied per batch is the C ABI's."""
import numpy as np

from util import dataset, plan

import bench
import goldpolish_b200 as gp
from goldpolish_b200 import shard


def test_shares_partition_the_workload_and_are_self_contained():
    d = dataset(genome_len=200000)
    bs = 3
    pl = plan(d, bsize=bs)
    nb = len(pl.batch_entry_off) - 1
    rl = np.diff(d.read_off)
    off = pl.batch_entry_off.astype(np.int64)
    cs = np.concatenate([[0], np.cumsum(rl[pl.entries["read_id"]])])
    work = cs[off[1:]] - cs[off[:-1]] + 1
    world = 3
    assignment = shard.assign_batches(work.tolist(), world)
    assert sorted(b for a in assignment for b in a) == list(range(nb))
    loads = [int(sum(work[b] for b in a)) for a in assignment]
    assert max(loads) - min(loads) <= int(work.max())  # LPT: within one batch of each other
    seen_contigs = []
    for mine in assignment:
        sh = bench.LocalShare(d, pl, mine, bs)
        assert sh.batches.tolist() == sorted(mine)
        seen_contigs += sh.contigs.tolist()
        # entries name the same reads, through the local store
        k = 0
        for i, b in enumerate(mine):
            ents = pl.entries[off[b]:off[b + 1]]
            loc = sh.entries[int(sh.batch_entry_off[i]):int(sh.batch_entry_off[i + 1])]
            assert len(ents) == len(loc) and np.array_equal(ents["kmer_threshold"], loc["kmer_threshold"])
            for e, l in zip(ents[:3], loc[:3]):
                assert sh.read_seq[sh.read_off[l["read_id"]]:sh.read_off[l["read_id"] + 1]].tobytes() == d.read(int(e["read_id"]))
            k += len(ents)
        for i, c in enumerate(sh.contigs.tolist()):
            assert sh.contig_seq[sh.contig_off[i]:sh.contig_off[i + 1]].tobytes() == d.contig(c)
            assert sh.batches[sh.contig_batch[i]] == c // bs
    assert sorted(seen_contigs) == list(range(d.n_contigs))
    whole = bench.LocalShare(d, pl, list(range(nb)), bs)  # the identity share aliases the data set
    assert whole.read_seq is d.read_seq and whole.entries is pl.entries


def _fake_step(sh, shrink, drop_every):
    """Polished records of a share as a step could return them: each record `shrink` bases shorter, every
    `drop_every`-th one dropped; random filter payloads."""
    n = len(sh.contigs)
    dropped = (np.arange(n) % drop_every == 1).astype(np.uint8)
    lens = np.where(dropped == 0, np.diff(sh.contig_off) - shrink, 0)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    out = np.concatenate([sh.contig_seq[sh.contig_off[i]:sh.contig_off[i] + lens[i]] for i in range(n)])
    bfs = np.random.default_rng(shrink).integers(0, 256, size=(len(sh.batches), 4, 64), dtype=np.uint8)
    return out, off, dropped, bfs


def test_dump_outputs_writes_the_same_seeded_sample_every_time(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float arrays only, under 64 MB; the sample (a strict subset of the contigs and batches)
    depends on the inputs alone, not on what the step returned, so two builds dump the same positions; what is written
    is what the step returned, cut at DUMP_MAX_POLISHED bytes."""
    d = dataset(genome_len=200000)
    pl = plan(d, bsize=1)
    nb = len(pl.batch_entry_off) - 1
    sh = bench.LocalShare(d, pl, list(range(1, nb)), 1)  # a share: global contig / batch ids differ from local ones
    monkeypatch.setattr(bench, "DUMP_SAMPLE_BASES", sh.draft_bases // 3)
    out, off, dropped, bfs = _fake_step(sh, 0, 7)
    a = bench.dump_outputs(str(tmp_path / "a"), sh, out, off, dropped, bfs)
    # another build's outputs for the same inputs: other lengths, other drops, other filters -- same sample positions
    out2, off2, dropped2, bfs2 = _fake_step(sh, 5, 3)
    b = bench.dump_outputs(str(tmp_path / "b"), sh, out2, off2, dropped2, bfs2)
    assert np.array_equal(a["polished_sample_contigs"], b["polished_sample_contigs"])
    assert np.array_equal(a["filters_sample_batches"], b["filters_sample_batches"])
    assert 0 < len(a["polished_sample_contigs"]) < len(sh.contigs)
    assert len(a["filters_sample_batches"]) == bench.DUMP_FILTER_BATCHES < len(sh.batches)
    picked_bases = sum(int(d.contig_off[int(c) + 1] - d.contig_off[int(c)]) for c in a["polished_sample_contigs"])
    assert picked_bases <= bench.DUMP_SAMPLE_BASES or len(a["polished_sample_contigs"]) == 1
    total = 0
    for name in a:
        x = np.load(tmp_path / "a" / f"{name}.npy")
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, a[name]), name
        total += x.nbytes
    assert total <= 64 << 20
    lens = np.diff(off.astype(np.int64))
    assert np.array_equal(a["polished_len"], lens) and np.array_equal(a["dropped"], dropped)
    local = {int(c): i for i, c in enumerate(sh.contigs)}
    want = b"".join(out[int(off[local[int(c)]]):int(off[local[int(c)] + 1])].tobytes() for c in a["polished_sample_contigs"])
    assert len(want) > 0 and a["polished_sample"].astype(np.uint8).tobytes() == want
    lb = {int(g): i for i, g in enumerate(sh.batches)}
    assert np.array_equal(a["filters_sample"], bfs[[lb[int(g)] for g in a["filters_sample_batches"]]])
    # the byte cap cuts the concatenated sample
    monkeypatch.setattr(bench, "DUMP_MAX_POLISHED", len(want) // 2)
    c = bench.dump_outputs(str(tmp_path / "c"), sh, out, off, dropped, bfs)
    assert c["polished_sample"].astype(np.uint8).tobytes() == want[:len(want) // 2]


def test_guard_per_batch_is_the_c_abi_rule():
    d = dataset(genome_len=60000)
    bs = 2
    pl = plan(d, bsize=bs)
    sh = bench.LocalShare(d, pl, list(range(len(pl.batch_entry_off) - 1)), bs)
    n = len(sh.contigs)
    lens = np.diff(sh.contig_off)
    # "polished" records: batch 0 shrinks below 75 % (rejected: keeps its originals), batch 1 loses a record (dropped)
    out_len = lens.copy()
    out_len[0:2] = lens[0:2] // 2
    dropped = np.zeros(n, dtype=np.uint8)
    dropped[2] = 1
    out_len[2] = 0
    off = np.concatenate([[0], np.cumsum(out_len)]).astype(np.uint64)
    out = np.concatenate([sh.contig_seq[sh.contig_off[i]:sh.contig_off[i] + out_len[i]] for i in range(n)])
    new_out, new_off, new_dropped, n_rej = bench.apply_guard(sh, out, off, dropped, gp.guard_rejects)
    in0 = sum(sh.name_len[i] + 3 + lens[i] for i in (0, 1))
    out0 = sum(sh.name_len[i] + 3 + out_len[i] for i in (0, 1))
    assert gp.guard_rejects(int(in0), int(out0))
    rej1 = gp.guard_rejects(int(sum(sh.name_len[i] + 3 + lens[i] for i in (2, 3))), int(sh.name_len[3] + 3 + lens[3]))
    assert n_rej == 1 + int(rej1)
    for i in (0, 1):
        assert new_out[int(new_off[i]):int(new_off[i + 1])].tobytes() == d.contig(i) and not new_dropped[i]
    if not rej1:
        assert new_dropped[2] == 1 and new_off[3] == new_off[2]
    assert new_out[int(new_off[4]):int(new_off[5])].tobytes() == d.contig(4)
