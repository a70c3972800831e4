"""The limit paths of the level-synchronous build kernel against the C restatement, bit for bit: the epoch-tag clears
(forced on small inputs by narrowing the tags with GP_LEVEL_TIME_BITS), the tightest tag budget (8 k values,
kmer_threshold 24, 6-bit tags), both sides of every host limit that hands a batch to the in-order kernel (65 535
entries, 2^21 steps of 32 occurrences, kmer_threshold 24), and the overlapped pipeline with clears."""
import functools

import numpy as np
import pytest

from util import KS, dataset, ol, plan

pytestmark = pytest.mark.gpu

KS8 = (32, 30, 28, 26, 24, 22, 20, 18)
# thresholds of the entries of a batch copy, by pattern: all 24 (the largest the level kernel takes), 24 and 4
# alternating (the entries of one batch disagree), all 13
PATTERNS = 3


@pytest.fixture(scope="module")
def gp():
    import goldpolish_b200
    return goldpolish_b200


def pattern_thr(pattern, n):
    if pattern == 0:
        return np.full(n, 24, dtype=np.uint32)
    if pattern == 1:
        return np.where(np.arange(n) % 2 == 0, 24, 4).astype(np.uint32)
    return np.full(n, 13, dtype=np.uint32)


def stream_tags(read_lens, thr, ks, keep):
    """Tags one batch draws at least: every stream with k-mers draws one per list round and one for round 0, i.e.
    lread + 1, where lread = kmer_threshold - 2 + k index (the largest of the batch), less one without counters."""
    t = 0
    for ki, k in enumerate(ks):
        if len(read_lens) and (read_lens >= k).any():
            lmax = int(thr.max()) - 2 + ki
            t += (lmax if keep else lmax - 1) + 1
    return t


def min_clears(tags, time_bits):
    """Between two clears the epoch cannot pass 2^(32 - time_bits) - 2: fewer clears could not have held `tags`."""
    m = (1 << (32 - time_bits)) - 2
    return -(-tags // m) - 1


def level_width(floor, read_lens, batch_entry_off, entries, ks):
    """Time width of the level kernel: the smallest from `floor` (GP_LEVEL_TIME_BITS, else 16) up to 26 that holds 32
    occurrences per step of the longest stream, a read of length n >= k being ceil((n - k + 1) / 32) steps."""
    lens = read_lens[entries["read_id"]].astype(np.int64)
    longest = 0
    for k in ks:
        steps = np.where(lens >= k, (lens - k + 32) // 32, 0)
        for b in range(len(batch_entry_off) - 1):
            longest = max(longest, int(steps[int(batch_entry_off[b]):int(batch_entry_off[b + 1])].sum()))
    w = floor
    while w < 26 and (longest * 32) >> w:
        w += 1
    return w


def entries_of(ids, thr):
    e = np.zeros(len(ids), dtype=np.dtype([("read_id", np.uint32), ("kmer_threshold", np.uint32)]))
    e["read_id"], e["kmer_threshold"] = ids, thr
    return e


@functools.lru_cache(maxsize=None)
def _plan(bsize):
    d = dataset(genome_len=60000)
    return d, plan(d, bsize=bsize)


@functools.lru_cache(maxsize=None)
def _oracle(bsize, b, pattern):
    d, pl = _plan(bsize)
    ids = pl.entries["read_id"][int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]
    fs = ol.FilterSet(KS)
    for rid, t in zip(ids, pattern_thr(pattern, len(ids))):
        fs.add_read(d.read(int(rid)), int(t))
    return fs


def copies_plan(bsize, time_bits, keep):
    """Copies of the plan's batches, each under one threshold pattern, until at least 5 clears are certain at the width
    the kernel will use.  Returns (d, [(batch, pattern)], batch_entry_off, entries, width, least clears)."""
    d, pl = _plan(bsize)
    rlens = np.diff(d.read_off)
    nb = len(pl.batch_entry_off) - 1
    width = level_width(time_bits, rlens, pl.batch_entry_off, pl.entries, KS)  # (copies repeat the plan's batches)
    copies, tags = [], 0
    while min_clears(tags, width) < 5:
        for b in range(nb):
            ids = pl.entries["read_id"][int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]
            pat = (len(copies) + b) % PATTERNS
            copies.append((b, pat))
            tags += stream_tags(rlens[ids], pattern_thr(pat, len(ids)), KS, keep)
    ids, thr, off = [], [], [0]
    for b, pat in copies:
        i = pl.entries["read_id"][int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]
        ids.append(i)
        thr.append(pattern_thr(pat, len(i)))
        off.append(off[-1] + len(i))
    return (d, copies, np.array(off, dtype=np.uint64), entries_of(np.concatenate(ids), np.concatenate(thr)), width,
            min_clears(tags, width))


NARROW = [(bsize, tb, overlap, keep, 2) for bsize in (1, 8) for tb in (26, 24, 21) for overlap in ("0", "1") for keep in (0, 1)]
NARROW += [(bsize, 26, overlap, keep, 3) for bsize in (1, 8) for overlap in ("0", "1") for keep in (0, 1)]


@pytest.mark.parametrize("bsize,time_bits,overlap,keep,arrays", NARROW)
def test_narrow_tags_clear_and_match_the_oracle(gp, bsize, time_bits, overlap, keep, arrays, monkeypatch):
    """Narrow epoch tags: the planner clears the timestamp arrays again and again (at least 5 times by the tag count
    alone), with one and two streams in flight, with and without the counter round, with two and three arrays.  Every
    filter equals the restatement's; so do the counter bytes of one copy of each pattern.  The variable is a floor: the
    bsize-8 batch (1.8 Mbp of reads) needs 22 bits of time, so there 21 builds at 22."""
    monkeypatch.setenv("GP_LEVEL_TIME_BITS", str(time_bits))
    monkeypatch.setenv("GP_LEVEL_OVERLAP", overlap)
    monkeypatch.setenv("GP_LEVEL_ARRAYS", str(arrays))
    d, copies, off, entries, width, clears = copies_plan(bsize, time_bits, keep)
    assert clears >= 5 and width == (22 if (bsize, time_bits) == (8, 21) else time_bits)
    with gp.Context(keep_counters=keep) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        bfs = ctx.build_filters(off, entries)
        st = ctx.stats()
        assert st["build_kernel"] == 2 and st["level_time_bits"] == width
        assert ctx.build_round_times()["clear"][2] >= clears
        for c, (b, pat) in enumerate(copies):
            want = _oracle(bsize, b, pat)
            for ki in range(len(KS)):
                assert np.array_equal(bfs[c, ki], want.bfs[ki]), f"copy {c} (batch {b}, pattern {pat}) k={KS[ki]}"
        for pat in range(PATTERNS):
            assert any(bfs[c].any() for c, (_, p) in enumerate(copies) if p == pat), f"pattern {pat}: all filters empty"
        if keep:  # (all copies are one wave: every counting filter is still resident)
            for pat in range(PATTERNS):
                c = max(c for c, (_, p) in enumerate(copies) if p == pat)
                b = copies[c][0]
                for ki in range(len(KS)):
                    assert np.array_equal(ctx.fetch_cbf(c, ki), _oracle(bsize, b, pat).cbfs[ki]), f"counters: copy {c} k={KS[ki]}"


def test_tightest_tag_budget(gp, monkeypatch):
    """8 k values, kmer_threshold 24 everywhere (per-k thresholds 22..29), counter bytes kept, 6-bit tags: a stream
    needs up to 30 tags of 62, the planner clears before almost every stream.  Coverage is doubled (every read twice)
    so that counters climb to the top levels."""
    monkeypatch.setenv("GP_LEVEL_TIME_BITS", "26")
    d, pl = _plan(1)
    rlens = np.diff(d.read_off)
    ids, off, tags = [], [0], 0
    for b in range(3):
        i = pl.entries["read_id"][int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]
        i = np.concatenate([i, i])
        ids.append(i)
        off.append(off[-1] + len(i))
        tags += stream_tags(rlens[i], np.full(len(i), 24), KS8, True)
    assert min_clears(tags, 26) >= 5
    entries = entries_of(np.concatenate(ids), np.full(off[-1], 24, dtype=np.uint32))
    with gp.Context(ks=KS8, keep_counters=1) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        bfs = ctx.build_filters(np.array(off, dtype=np.uint64), entries)
        st = ctx.stats()
        assert st["build_kernel"] == 2 and st["level_time_bits"] == 26
        assert ctx.build_round_times()["clear"][2] >= min_clears(tags, 26)
        top = 0
        for b in range(3):
            fs = ol.FilterSet(KS8)
            for rid in ids[b]:
                fs.add_read(d.read(int(rid)), 24)
            for ki in range(len(KS8)):
                assert np.array_equal(bfs[b, ki], fs.bfs[ki]), f"batch {b} k={KS8[ki]}"
                cbf = ctx.fetch_cbf(b, ki)
                assert np.array_equal(cbf, fs.cbfs[ki]), f"counters: batch {b} k={KS8[ki]}"
                top = max(top, int(cbf.max()))
        assert bfs.any() and top >= 25


def _random_reads(rng, lens):
    return [bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=n)) for n in lens]


def _upload(ctx, reads):
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(r) for r in reads])
    ctx.upload_reads(np.frombuffer(b"".join(reads), dtype=np.uint8).copy(), off)


def _check(ctx, bfs, fs, ks, keep=True):
    assert bfs.any()
    for ki in range(len(ks)):
        assert np.array_equal(bfs[0, ki], fs.bfs[ki]), f"k={ks[ki]}"
        if keep:
            assert np.array_equal(ctx.fetch_cbf(0, ki), fs.cbfs[ki]), f"counters k={ks[ki]}"


def test_entry_anchor_limit(gp):
    """A batch of exactly 65 535 entries (the last one anchors steps at 65 534) is built by the level kernel; one entry
    more and the in-order kernel builds it.  Entries repeat 6 000 reads of 0..120 bases (some shorter than k) about 11
    times each, with thresholds 4..24, so that counters end on both sides of the thresholds."""
    rng = np.random.default_rng(65535)
    reads = _random_reads(rng, rng.integers(0, 121, size=6000))
    reads.append(_random_reads(rng, [100])[0])  # the last entries: k-mers for every k
    ids = rng.integers(0, len(reads), size=65535).astype(np.uint32)
    ids[-3:] = len(reads) - 1
    thr = rng.integers(4, 25, size=65535).astype(np.uint32)
    fs = ol.FilterSet(KS)
    for rid, t in zip(ids, thr):
        fs.add_read(reads[rid], int(t))
    with gp.Context(keep_counters=1) as ctx:
        _upload(ctx, reads)
        bfs = ctx.build_filters(np.array([0, 65535], dtype=np.uint64), entries_of(ids, thr))
        st = ctx.stats()
        assert st["build_kernel"] == 2 and st["level_time_bits"] >= 16
        _check(ctx, bfs, fs, KS)
        fs.add_read(reads[-1], 9)
        bfs = ctx.build_filters(np.array([0, 65536], dtype=np.uint64),
                                entries_of(np.append(ids, len(reads) - 1), np.append(thr, 9)))
        st = ctx.stats()
        assert st["build_kernel"] == 1 and st["level_time_bits"] == 0
        _check(ctx, bfs, fs, KS)


def test_occurrence_clock_limit(gp):
    """k = 32, one batch whose stream holds exactly 2^21 - 1 steps (occurrence times up to 2^26 - 1, next to the
    threshold in bits 26..31): the level kernel at 26-bit times.  One step more overflows the clock and the in-order
    kernel runs.  A 2 015-base read is 62 steps, a 2 047-base read 63, a 32-base read 1; 2 048 reads of 2 015 bases
    repeat about 16 times each, around the thresholds 4..24."""
    rng = np.random.default_rng(2 ** 21)
    reads = _random_reads(rng, [2015] * 2048 + [2047, 32])
    steps = lambda n: -(-(n - 32 + 1) // 32)
    n62 = (2 ** 21 - 1 - steps(2047)) // steps(2015)
    assert n62 * steps(2015) + steps(2047) == 2 ** 21 - 1 and n62 + 1 <= 65535
    ids = np.append(rng.integers(0, 2048, size=n62), 2048).astype(np.uint32)
    thr = rng.integers(4, 25, size=len(ids)).astype(np.uint32)
    fs = ol.FilterSet((32,))
    for rid, t in zip(ids, thr):
        fs.add_read(reads[rid], int(t))
    with gp.Context(ks=(32,), keep_counters=1) as ctx:
        _upload(ctx, reads)
        bfs = ctx.build_filters(np.array([0, len(ids)], dtype=np.uint64), entries_of(ids, thr))
        st = ctx.stats()
        assert st["build_kernel"] == 2 and st["level_time_bits"] == 26
        _check(ctx, bfs, fs, (32,))
        fs.add_read(reads[2049], 6)
        bfs = ctx.build_filters(np.array([0, len(ids) + 1], dtype=np.uint64), entries_of(np.append(ids, 2049), np.append(thr, 6)))
        assert ctx.stats()["build_kernel"] == 1
        _check(ctx, bfs, fs, (32,))


def test_threshold_limit(gp):
    """kmer_threshold 24 and 4 mixed in every batch: the level kernel; a single entry at 25 hands the call to the
    in-order kernel.  Both equal the restatement, counters included."""
    d, pl = _plan(1)
    off = pl.batch_entry_off
    nb = len(off) - 1
    thr = np.where(np.arange(len(pl.entries)) % 2 == 0, 24, 4).astype(np.uint32)

    def oracle(b, thr):
        fs = ol.FilterSet(KS)
        for e in range(int(off[b]), int(off[b + 1])):
            fs.add_read(d.read(int(pl.entries["read_id"][e])), int(thr[e]))
        return fs

    want = [oracle(b, thr) for b in range(nb)]
    with gp.Context(keep_counters=1) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        for algo in (2, 1):
            bfs = ctx.build_filters(off, entries_of(pl.entries["read_id"], thr))
            assert ctx.stats()["build_kernel"] == algo
            assert bfs.any()
            for b in range(nb):
                for ki in range(len(KS)):
                    assert np.array_equal(bfs[b, ki], want[b].bfs[ki]), f"kernel {algo} batch {b} k={KS[ki]}"
                    assert np.array_equal(ctx.fetch_cbf(b, ki), want[b].cbfs[ki]), f"counters: kernel {algo} batch {b} k={KS[ki]}"
            thr = thr.copy()
            thr[int(off[1])] = 25  # the first entry of batch 1
            want[1] = oracle(1, thr)


@pytest.mark.parametrize("resident", [0, 2])
def test_pipeline_with_clears(gp, resident, monkeypatch):
    """gp_pipeline_run with 6-bit tags, every filter resident and with a 2-batch pool (each wave's launch starts again
    from epoch 0): the payloads and polished records of the build and polish calls without narrow tags."""
    import torch
    d, pl = _plan(1)
    entries = entries_of(pl.entries["read_id"], np.full(len(pl.entries), 20, dtype=np.uint32))
    off = pl.batch_entry_off
    nb = len(off) - 1
    with gp.Context() as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        bfs = ctx.build_filters(off, entries)
        out, ooff, dropped = ctx.polish(d.contig_seq, d.contig_off, pl.contig_batch)
        out = out[:int(ooff[-1])].copy()
        assert ctx.stats()["level_time_bits"] < 26
    monkeypatch.setenv("GP_LEVEL_TIME_BITS", "26")
    with gp.Context(max_resident_filters=resident) as ctx:
        ctx.upload_reads(d.read_seq, d.read_off)
        pinned = torch.zeros((nb, len(KS), gp.BF_BYTES), dtype=torch.uint8).pin_memory()
        ctx.build_output(pinned)
        ctx.build_stage(off, entries)
        ctx.polish_stage(d.contig_seq, d.contig_off, pl.contig_batch)
        ctx.pipeline_run()
        got = ctx.build_fetch(out=pinned).numpy()
        out2, ooff2, dropped2 = ctx.polish_fetch()
        st = ctx.stats()
        assert st["build_kernel"] == 2 and st["level_time_bits"] == 26 and st["polish_reruns"] == 0
        assert ctx.build_round_times()["clear"][2] >= 1
        assert np.array_equal(got, bfs) and bfs.any()
        assert np.array_equal(ooff2, ooff) and np.array_equal(dropped2, dropped)
        assert np.array_equal(out2[:int(ooff2[-1])], out)
        ctx.build_output(None)
