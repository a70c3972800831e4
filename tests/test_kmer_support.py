"""CPU: the k-mer support rule of gp_polish_fetch_support restated in numpy -- ntHash by its definition, a k-mer counted at
every start whose k bases are ACGT of either case, "present" when all four bits h_i mod 2^22 are set in the filter the C
restatement's gpo_fill_bfs filled -- against the restatement's own gpo_nthash_all plus filter lookups, on the golden
ntEdit cases and a simulated set; hand-built records pin each edge; the QV rule and the TSV the tools write."""
import json
import math
import os

import numpy as np
import pytest

from util import GOLDEN, KS, dataset, ol, oracle_build, oracle_polish_contig, plan

M64 = (1 << 64) - 1
SEEDS = (0x3c8bfbb395c60474, 0x3193c18562a02b4c, 0x20323ed082572324, 0x295549f54be24456)  # A C G T
MULTI_SEED, MULTI_SHIFT = 0x90b45d39fb6da1fa, 27
BF_BITS = 1 << 22


def _srol(v, s):
    a, b = s % 31, s % 33
    hi, lo = v >> 33, v & ((1 << 33) - 1)
    hi = ((hi << a) | (hi >> (31 - a))) & ((1 << 31) - 1)
    lo = ((lo << b) | (lo >> (33 - b))) & ((1 << 33) - 1)
    return (hi << 33) | lo


# ROT[code, r] = srol(seed[code], r)
ROT = np.array([[_srol(s, r) for r in range(32)] for s in SEEDS], dtype=np.uint64)
_CODE = np.full(256, 4, dtype=np.int64)
for _i, _ch in enumerate(b"ACGT"):
    _CODE[_ch] = _i
    _CODE[_ch | 0x20] = _i


def kmer_hashes(seq: bytes, k: int):
    """(start positions, hashes[n, 4]) of every k-mer of only ACGTacgt, by the definition: fwd = XOR_i
    srol^{k-1-i}(seed[s_i]), rev = XOR_i srol^i(seed[comp s_i]), h0 = fwd + rev, h_j = h0 * (j ^ k * multiSeed),
    h_j ^= h_j >> 27."""
    code = _CODE[np.frombuffer(seq, dtype=np.uint8)]
    n = len(code) - k + 1
    if n <= 0:
        return np.zeros(0, dtype=np.int64), np.zeros((0, 4), dtype=np.uint64)
    bad = np.concatenate([[0], np.cumsum(code == 4)])
    pos = np.flatnonzero(bad[k:k + n] - bad[:n] == 0)
    fwd = np.zeros(len(pos), dtype=np.uint64)
    rev = np.zeros(len(pos), dtype=np.uint64)
    for i in range(k):
        c = code[pos + i]
        fwd ^= ROT[c, k - 1 - i]
        rev ^= ROT[3 - c, i]
    h = np.empty((len(pos), 4), dtype=np.uint64)
    h[:, 0] = fwd + rev
    for j in (1, 2, 3):
        t = h[:, 0] * np.uint64(j ^ ((k * MULTI_SEED) & M64))
        h[:, j] = t ^ (t >> np.uint64(MULTI_SHIFT))
    return pos, h


def contains(bf: np.ndarray, h: np.ndarray) -> np.ndarray:
    """KmerBloomFilter::contains for every row of hashes: bit n of the payload is bit n % 8 of byte n / 8."""
    n = (h & np.uint64(BF_BITS - 1)).astype(np.int64)
    bits = (np.asarray(bf, dtype=np.uint8)[n >> 3] >> (n & 7).astype(np.uint8)) & 1
    return bits.all(axis=1) if len(n) else np.zeros(0, dtype=bool)


def support(seq, bf, k):
    """(k-mers, present) of one record against one filter; None (a dropped record) counts nothing."""
    if seq is None:
        return 0, 0
    _, h = kmer_hashes(seq, k)
    return len(h), int(contains(bf, h).sum())


def support_by_oracle(seq: bytes, bf, k):
    pos, h = ol.nthash_all(seq, k)
    return len(pos), int(contains(bf, h).sum())


# ---- QV and the TSV (the host writer of gp_host.hpp, restated) ------------------------------------------------------
def qv(kmers: int, missing: int, k: int) -> str:
    if kmers == 0:
        return "NA"
    if missing == 0:
        return "inf"
    e = 1.0 - math.pow(1.0 - missing / kmers, 1.0 / k)
    return "%.4f" % (-10.0 * math.log10(e) + 0.0)  # (+ 0.0: QV 0 prints without a sign)


def kmer_qv_tsv(names, ks, counts, bits, polished_is_draft=False) -> bytes:
    """The TSV of ntedit-gr --kmer-qv / goldpolish-ntedit GP_KMER_QV=1 from counts[n, nk, 4] and bits[n_batches, nk]."""
    nk, nb = len(ks), len(bits)
    lines = ["#goldpolish_b200 k-mer support: k-mers per record position, missing = not contained in the filter of its batch",
             "#k\t" + "\t".join(str(k) for k in ks)]
    fill, fp = [], []
    for j in range(nk):
        if nb == 0:
            fill.append("NA")
            fp.append("NA")
            continue
        fill.append("%.6f" % (float(sum(int(bits[b][j]) for b in range(nb))) / (nb * 4194304.0)))
        s = 0.0
        for b in range(nb):
            s += math.pow(int(bits[b][j]) / 4194304.0, 4.0)
        fp.append("%.6g" % (s / nb))
    lines.append("#filter_fill\t" + "\t".join(fill))
    lines.append("#filter_fp_rate\t" + "\t".join(fp))
    lines.append("#name\tk\tdraft_kmers\tdraft_missing\tdraft_qv\tpolished_kmers\tpolished_missing\tpolished_qv")
    tot = [[0, 0, 0, 0] for _ in ks]
    for c, name in enumerate(names):
        for j, k in enumerate(ks):
            dk, dp, pk, pp = (int(x) for x in counts[c][j])
            dm = dk - dp
            pk, pm = (dk, dm) if polished_is_draft else (pk, pk - pp)
            lines.append(f"{name}\t{k}\t{dk}\t{dm}\t{qv(dk, dm, k)}\t{pk}\t{pm}\t{qv(pk, pm, k)}")
            for i, v in enumerate((dk, dm, pk, pm)):
                tot[j][i] += v
    for j, k in enumerate(ks):
        dk, dm, pk, pm = tot[j]
        lines.append(f"*\t{k}\t{dk}\t{dm}\t{qv(dk, dm, k)}\t{pk}\t{pm}\t{qv(pk, pm, k)}")
    return ("\n".join(lines) + "\n").encode()


# ---- the restatement against the C restatement ----------------------------------------------------------------------
def _golden():
    g = json.load(open(os.path.join(GOLDEN, "ntedit_cases.json")))
    fs = ol.FilterSet(KS)
    for _ in range(5):
        fs.add_read(g["truth"].encode(), 4)
    return g, fs


def test_golden_cases_agree_with_the_c_restatement():
    g, fs = _golden()
    checked = 0
    for name, case in g["cases"].items():
        for rec in (case["draft"], case.get("chain")):
            if rec is None:
                continue
            for ki, k in enumerate(KS):
                want = support_by_oracle(rec.encode(), fs.bfs[ki], k)
                assert support(rec.encode(), fs.bfs[ki], k) == want, (name, k)
                checked += want[0]
    assert checked > 0


def test_simulated_set_agrees_with_the_c_restatement():
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    fsets = oracle_build(d, pl)
    missing = 0
    for c in range(d.n_contigs):
        fs = fsets[int(pl.contig_batch[c])]
        draft = d.contig(c)
        polished = oracle_polish_contig(draft, fs.bfs)
        for rec in (draft, polished):
            if rec is None:
                continue
            for ki, k in enumerate(KS):
                got = support(rec, fs.bfs[ki], k)
                assert got == support_by_oracle(rec, fs.bfs[ki], k), (c, k)
                missing += got[0] - got[1]
    assert missing > 0  # the drafts carry errors the filters do not contain


def test_odd_k_agrees_with_the_c_restatement():
    rng = np.random.default_rng(5)
    seq = np.array(list(b"ACGTacgt" * 5 + b"N"), dtype=np.uint8)[rng.integers(0, 41, 3000)].tobytes()
    fs = ol.FilterSet((31, 27, 23, 19))
    for _ in range(5):  # the counting filter lets a k-mer in once it reaches the threshold
        fs.add_read(seq[:2000], 4)
    for ki, k in enumerate(fs.ks):
        want = support_by_oracle(seq, fs.bfs[ki], k)
        assert support(seq, fs.bfs[ki], k) == want and 0 < want[1] < want[0], k


# ---- hand-built edges -------------------------------------------------------------------------------------------------
FULL = np.full(BF_BITS // 8, 0xFF, dtype=np.uint8)  # every bit set: every k-mer is present
EMPTY = np.zeros(BF_BITS // 8, dtype=np.uint8)


@pytest.mark.parametrize("seq,k,kmers", [
    (b"ACGTACG", 8, 0),             # shorter than k
    (b"ACGTACGT", 8, 1),            # ends exactly at a k-mer
    (b"N" * 50, 8, 0),              # all N
    (b"ACGTACGTAC" + b"R" + b"ACGTACGTAC", 8, 6),  # IUPAC inside: only windows on either side, 3 + 3
    (b"ACGTNACGTACGT", 4, 1 + 5),   # N splits the record
    (b"", 4, 0),
])
def test_window_edges(seq, k, kmers):
    assert support(seq, FULL, k) == (kmers, kmers)
    assert support(seq, EMPTY, k) == (kmers, 0)
    assert support_by_oracle(seq, FULL, k) == (kmers, kmers)


def test_lower_case_hashes_like_upper_case():
    rng = np.random.default_rng(3)
    up = np.array(list(b"ACGT"), dtype=np.uint8)[rng.integers(0, 4, 500)].tobytes()
    mixed = bytes(ch | 0x20 if i % 3 == 0 else ch for i, ch in enumerate(up))
    fs = ol.FilterSet((24,))
    for _ in range(5):
        fs.add_read(up[:300], 4)
    assert np.array_equal(kmer_hashes(mixed, 24)[1], kmer_hashes(up, 24)[1])
    assert support(mixed, fs.bfs[0], 24) == support(up, fs.bfs[0], 24)
    assert support(mixed, fs.bfs[0], 24) == support_by_oracle(mixed, fs.bfs[0], 24)


def test_counted_per_position_not_per_distinct_kmer():
    seq = b"ACGTACGT" * 8  # 57 starts, 4 distinct 8-mers
    fs = ol.FilterSet((8,))
    for _ in range(5):
        fs.add_read(b"ACGTACGTACG", 4)
    assert support(seq, fs.bfs[0], 8) == (57, 57)


def test_qv_rule():
    assert qv(0, 0, 21) == "NA"
    assert qv(1000, 0, 21) == "inf"
    # Merqury: E = 1 - (1 - missing / total)^(1/k); QV = -10 log10 E
    e = -math.expm1(math.log1p(-10 / 1000) / 21)
    assert abs(float(qv(1000, 10, 21)) - (-10 * math.log10(e))) < 1e-4
    assert float(qv(1000, 10, 21)) < float(qv(1000, 1, 21))
    assert qv(5, 5, 21) == "0.0000"  # every k-mer missing: E = 1


def test_tsv_layout():
    counts = np.array([[[100, 90, 98, 98], [120, 100, 119, 110]], [[0, 0, 0, 0], [7, 7, 0, 0]]], dtype=np.uint64)
    bits = np.array([[1 << 20, 1 << 21]], dtype=np.uint64)
    t = kmer_qv_tsv(["a", "b"], (32, 24), counts, bits).decode().splitlines()
    assert t[1] == "#k\t32\t24"
    assert t[2] == "#filter_fill\t0.250000\t0.500000"
    assert t[3] == "#filter_fp_rate\t0.00390625\t0.0625"
    assert t[5] == f"a\t32\t100\t10\t{qv(100, 10, 32)}\t98\t0\tinf"
    assert t[7] == "b\t32\t0\t0\tNA\t0\t0\tNA"
    assert t[9] == f"*\t32\t100\t10\t{qv(100, 10, 32)}\t98\t0\tinf"
    assert t[10] == f"*\t24\t127\t20\t{qv(127, 20, 24)}\t119\t9\t{qv(119, 9, 24)}"
    kept = kmer_qv_tsv(["a", "b"], (32, 24), counts, bits, polished_is_draft=True).decode().splitlines()
    assert kept[5] == f"a\t32\t100\t10\t{qv(100, 10, 32)}\t100\t10\t{qv(100, 10, 32)}"
