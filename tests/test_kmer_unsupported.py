"""CPU: the unsupported-run rule of gp_polish_fetch_unsupported restated in numpy on top of the k-mer support
restatement (tests/test_kmer_support.py) -- the spans [p, p + k) of the valid k-mers the filter does not contain, merged
where they overlap or touch -- against the same merge over the C restatement's gpo_nthash_all plus filter lookups, on
the golden ntEdit cases, a simulated set and odd k; the word-level derivation the device runs (coverage from a bitmap
word and the one before it, run starts and lasts, prefix counts) restated on the same records; hand-built edges; the
kmers sum invariant and the BED layout the tools write."""
import json
import os

import numpy as np
import pytest

from test_kmer_support import BF_BITS, EMPTY, FULL, contains, kmer_hashes, support
from util import GOLDEN, KS, dataset, ol, oracle_build, oracle_polish_contig, plan


def merge_runs(pos, missing, k):
    """Runs (start, end, kmers) of the spans [p, p + k) of the k-mer starts pos[missing], bedtools-merge style."""
    m = np.asarray(pos, dtype=np.int64)[np.asarray(missing, dtype=bool)]
    if len(m) == 0:
        return []
    brk = np.flatnonzero(np.diff(m) > k) + 1  # a gap: the next span starts after this one's end
    first = np.concatenate([[0], brk])
    last = np.concatenate([brk - 1, [len(m) - 1]])
    return [(int(m[a]), int(m[b]) + k, int(b - a + 1)) for a, b in zip(first, last)]


def unsupported_runs(seq, bf, k):
    """The rule: runs of one record against one filter; None (a dropped record) has none."""
    if seq is None:
        return []
    pos, h = kmer_hashes(seq, k)
    return merge_runs(pos, ~contains(bf, h), k)


def unsupported_runs_by_oracle(seq, bf, k):
    pos, h = ol.nthash_all(seq, k)
    return merge_runs(pos, ~contains(bf, h), k)


# ---- the device's derivation, restated word by word ------------------------------------------------------------------
def miss_words(seq, bf, k):
    """The bitmap support_count_kernel stores: bit p % 32 of word p / 32 set for an unsupported start p."""
    pos, h = kmer_hashes(seq, k)
    bits = np.zeros((len(seq) + 31) // 32 * 32, dtype=np.uint8)
    bits[pos[~contains(bf, h)]] = 1
    return np.packbits(bits.reshape(-1, 32)[:, ::-1], axis=1).view(">u4").ravel().astype(np.uint64)


def _smear(x, k):
    span = 1
    while 2 * span <= k:
        x |= (x << np.uint64(span)) & np.uint64((1 << 64) - 1)
        span *= 2
    return x | ((x << np.uint64(k - span)) & np.uint64((1 << 64) - 1)) if span < k else x


def runs_from_words(w, k):
    """unsupported_count_kernel + the scans + unsupported_fill_kernel on one segment."""
    w = np.asarray(w, dtype=np.uint64)
    if len(w) == 0:
        return []
    prev = np.concatenate([[0], w[:-1]]).astype(np.uint64)
    nxt = np.concatenate([w[1:], [0]]).astype(np.uint64)
    c64 = _smear((w << np.uint64(32)) | prev, k)
    cov = c64 >> np.uint64(32)
    before = (c64 >> np.uint64(31)) & np.uint64(0xFFFFFFFF)
    next0 = (_smear((nxt << np.uint64(32)) | w, k) >> np.uint64(32)) & np.uint64(1)
    starts = cov & ~before & np.uint64(0xFFFFFFFF)
    lasts = cov & ~((cov >> np.uint64(1)) | (next0 << np.uint64(31))) & np.uint64(0xFFFFFFFF)
    popc = lambda a: np.array([bin(int(x)).count("1") for x in a], dtype=np.int64)
    run_scan, miss_scan = np.cumsum(popc(starts)), np.cumsum(popc(w))
    n = int(run_scan[-1])
    start, end, kmers = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int64)
    for f in range(len(w)):
        run0 = run_scan[f] - popc(starts[f:f + 1])[0]
        miss0 = miss_scan[f] - popc(w[f:f + 1])[0]
        s, l, m = int(starts[f]), int(lasts[f]), int(w[f])
        for b in range(32):
            below, upto = (1 << b) - 1, (2 << b) - 1
            if s >> b & 1:
                i = run0 + bin(s & below).count("1")
                start[i] = 32 * f + b
                kmers[i] -= miss0 + bin(m & below).count("1")
            if l >> b & 1:
                i = run0 + bin(s & upto).count("1") - 1
                end[i] = 32 * f + b + 1
                kmers[i] += miss0 + bin(m & upto).count("1")
    return list(zip(start.tolist(), end.tolist(), kmers.tolist()))


def derived(seq, bf, k):
    if seq is None or len(seq) < k:
        return []
    return runs_from_words(miss_words(seq, bf, k), k)


# ---- the restatement against the C restatement ----------------------------------------------------------------------
def _golden():
    g = json.load(open(os.path.join(GOLDEN, "ntedit_cases.json")))
    fs = ol.FilterSet(KS)
    for _ in range(5):
        fs.add_read(g["truth"].encode(), 4)
    return g, fs


def _check(rec, bf, k):
    runs = unsupported_runs(rec, bf, k)
    assert runs == unsupported_runs_by_oracle(rec, bf, k), k
    assert runs == derived(rec, bf, k), k
    kmers, present = support(rec, bf, k)
    assert sum(r[2] for r in runs) == kmers - present
    return runs


def test_golden_cases_agree_with_the_c_restatement():
    g, fs = _golden()
    n = 0
    for name, case in g["cases"].items():
        for rec in (case["draft"], case.get("chain")):
            if rec is None:
                continue
            for ki, k in enumerate(KS):
                n += len(_check(rec.encode(), fs.bfs[ki], k))
    assert n > 0


def test_simulated_set_agrees_with_the_c_restatement():
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    fsets = oracle_build(d, pl)
    n = 0
    for c in range(0, d.n_contigs, 3):
        fs = fsets[int(pl.contig_batch[c])]
        draft = d.contig(c)
        for rec in (draft, oracle_polish_contig(draft, fs.bfs)):
            if rec is None:
                continue
            for ki, k in enumerate(KS):
                n += len(_check(rec, fs.bfs[ki], k))
    assert n > 0


def test_odd_k_agrees_with_the_c_restatement():
    rng = np.random.default_rng(5)
    seq = np.array(list(b"ACGTacgt" * 5 + b"N"), dtype=np.uint8)[rng.integers(0, 41, 3000)].tobytes()
    fs = ol.FilterSet((31, 27, 23, 19))
    for _ in range(5):
        fs.add_read(seq[:2000], 4)
    for ki, k in enumerate(fs.ks):
        runs = _check(seq, fs.bfs[ki], k)
        assert len(runs) > 0 and runs[-1][1] > 2000, k


# ---- hand-built edges -------------------------------------------------------------------------------------------------
def filter_of(seq, k, present):
    """A filter holding exactly the k-mers of seq that start at the positions `present` (all four bits each)."""
    bf = np.zeros(BF_BITS // 8, dtype=np.uint8)
    pos, h = kmer_hashes(seq, k)
    keep = np.isin(pos, np.asarray(list(present), dtype=np.int64))
    n = (h[keep] & np.uint64(BF_BITS - 1)).astype(np.int64).ravel()
    np.bitwise_or.at(bf, n >> 3, (1 << (n & 7)).astype(np.uint8))
    return bf


def _acgt(n, seed=11):
    return np.array(list(b"ACGT"), dtype=np.uint8)[np.random.default_rng(seed).integers(0, 4, n)].tobytes()


def _distinct(n, k, seed=11):
    """n random bases whose k-mers are pairwise distinct, reverse complements included (so that a filter can hold all
    k-mers but chosen ones: at k = 4 there are only 136 such k-mers)."""
    rng = np.random.default_rng(seed)
    while True:
        seq, seen = bytearray(_acgt(k - 1, int(rng.integers(1 << 30)))), set()
        for _ in range(n - k + 1):
            for b in rng.permutation(list(b"ACGT")):
                h = int(kmer_hashes(bytes(seq[len(seq) - k + 1:]) + bytes([b]), k)[1][0, 0])
                if h not in seen:
                    seen.add(h)
                    seq.append(b)
                    break
            else:
                break
        if len(seq) == n:
            return bytes(seq)


def _length(k):
    return 120 if k == 4 else 500


@pytest.mark.parametrize("k", [4, 32])
def test_shorter_than_k_and_all_n(k):
    assert unsupported_runs(_acgt(k - 1), EMPTY, k) == [] == derived(_acgt(k - 1), EMPTY, k)
    assert unsupported_runs(b"N" * 200, EMPTY, k) == [] == derived(b"N" * 200, EMPTY, k)
    assert unsupported_runs(_acgt(k), EMPTY, k) == [(0, k, 1)] == derived(_acgt(k), EMPTY, k)
    assert unsupported_runs(b"", EMPTY, k) == []


@pytest.mark.parametrize("k", [4, 32])
def test_whole_record_and_both_ends(k):
    L = _length(k)
    seq = _distinct(L, k)
    n = L - k + 1
    assert _check(seq, EMPTY, k) == [(0, L, n)]
    assert _check(seq, FULL, k) == []
    # only the first and the last k-mer missing: runs at the record's first and last position
    bf = filter_of(seq, k, range(1, n - 1))
    assert _check(seq, bf, k) == [(0, k, 1), (L - k, L, 1)]


@pytest.mark.parametrize("k", [4, 32])
def test_touching_spans_merge_and_a_gap_splits(k):
    L = _length(k)
    seq = _distinct(L, k, seed=k)
    a = 30
    bf = filter_of(seq, k, set(range(L)) - {a, a + k})  # spans [a, a + k) and [a + k, a + 2k) touch
    assert _check(seq, bf, k) == [(a, a + 2 * k, 2)]
    bf = filter_of(seq, k, set(range(L)) - {a, a + k + 1})  # one position apart: two runs
    assert _check(seq, bf, k) == [(a, a + k, 1), (a + k + 1, a + 2 * k + 1, 1)]


def test_n_inside_a_run():
    k = 8
    seq = _distinct(60, k) + b"N" + _distinct(60, k, seed=3)
    # the windows around the N are no k-mers: the runs on either side end at the N and start after it
    assert _check(seq, EMPTY, k) == [(0, 60, 53), (61, 121, 53)]
    # a missing k-mer ending right before the N and one starting right after it: two runs around the gap
    bf = filter_of(seq, k, set(range(121)) - {52, 61})
    assert _check(seq, bf, k) == [(52, 60, 1), (61, 69, 1)]


@pytest.mark.parametrize("k", [4, 32])
def test_runs_crossing_words(k):
    L = _length(k)
    seq = _distinct(L, k, seed=7)
    n = L - k + 1
    for miss in ({31}, {28, 31 + k}, {30, 63, 95}, set(range(20, 80)), {0, 64 - k, 64, n - 1}, {n - 1}, {31, 32}):
        bf = filter_of(seq, k, set(range(n)) - miss)
        runs = _check(seq, bf, k)
        want = merge_runs(np.arange(n), np.isin(np.arange(n), list(miss)), k)
        assert runs == want, (k, sorted(miss))
    # a run over several words, starting and ending inside one
    bf = filter_of(seq, k, set(range(n)) - set(range(37, 100)))
    assert _check(seq, bf, k) == [(37, 99 + k, 63)]


def test_random_bitmaps_against_the_merge():
    rng = np.random.default_rng(1)
    for k in (4, 5, 17, 19, 31, 32):
        for density in (0.01, 0.05, 0.3):
            npos = int(rng.integers(k, 400))
            length = npos + k - 1
            miss = rng.random(npos) < density
            bits = np.zeros((length + 31) // 32 * 32, dtype=np.uint8)
            bits[np.flatnonzero(miss)] = 1
            w = np.packbits(bits.reshape(-1, 32)[:, ::-1], axis=1).view(">u4").ravel().astype(np.uint64)
            assert runs_from_words(w, k) == merge_runs(np.arange(npos), miss, k), (k, density)


# ---- the BED the tools write (gp_host.hpp::write_unsupported_bed, restated) -------------------------------------------
def unsupported_bed(names, ks, runs, emit=None) -> bytes:
    """runs[c][j]: the runs of record c for k index j (of the record the BED describes); emit[c]: the record is written."""
    out = []
    for c, name in enumerate(names):
        if emit is not None and not emit[c]:
            continue
        for j, k in enumerate(ks):
            out += [f"{name}\t{s}\t{e}\tk{k}\t{m}\n" for s, e, m in runs[c][j]]
    return "".join(out).encode()


def test_bed_layout():
    runs = [[[(0, 40, 3), (100, 132, 1)], []], [[], [(7, 31, 2)]], [[(5, 37, 1)], [(5, 33, 2)]]]
    t = unsupported_bed(["a", "b", "c"], (32, 24), runs, emit=[1, 1, 0]).decode()
    assert t == "a\t0\t40\tk32\t3\na\t100\t132\tk32\t1\nb\t7\t31\tk24\t2\n"
    assert unsupported_bed(["a"], (32,), [[[]]]) == b""
