"""k values that are not multiples of 4 (any k in 4..32), on the CPU: ntHash restated two ways, the padded-word algebra
the device uses for a partial last byte (gp_hashing.cuh::hash_kmer), and the k check of goldpolish-targeted-bfs."""
import os
import subprocess

import numpy as np
import pytest

from util import ROOT, ol

M64 = (1 << 64) - 1
SEED = {"A": 0x3c8bfbb395c60474, "C": 0x3193c18562a02b4c, "G": 0x20323ed082572324, "T": 0x295549f54be24456}
COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}
MULTI_SEED, MULTI_SHIFT = 0x90b45d39fb6da1fa, 27
CODE_SEED = [SEED["A"], SEED["C"], SEED["G"], SEED["T"]]  # 2-bit codes of the packed read store
ALL_K = range(4, 33)


def srol(v, s):
    """rotate the high 31 and the low 33 bits of v left by s, independently"""
    a, b = s % 31, s % 33
    hi, lo = v >> 33, v & ((1 << 33) - 1)
    hi = ((hi << a) | (hi >> (31 - a))) & ((1 << 31) - 1)
    lo = ((lo << b) | (lo >> (33 - b))) & ((1 << 33) - 1)
    return (hi << 33) | lo


def direct_nthash(seq: bytes, k: int):
    """Every k-mer of only A/C/G/T (either case) by the definition: fwd = XOR_i srol^{k-1-i}(seed[s_i]),
    rev = XOR_i srol^i(seed[comp s_i]), h0 = fwd + rev, h_j = h0 * (j ^ k * multiSeed), h_j ^= h_j >> 27."""
    s = seq.decode("latin-1").upper()
    pos, hs = [], []
    for p in range(len(s) - k + 1):
        kmer = s[p:p + k]
        if any(ch not in SEED for ch in kmer):
            continue
        fwd = rev = 0
        for i, ch in enumerate(kmer):
            fwd ^= srol(SEED[ch], k - 1 - i)
            rev ^= srol(SEED[COMP[ch]], i)
        h0 = (fwd + rev) & M64
        row = [h0]
        for j in (1, 2, 3):
            t = (h0 * (j ^ ((k * MULTI_SEED) & M64))) & M64
            row.append(t ^ (t >> MULTI_SHIFT))
        pos.append(p)
        hs.append(row)
    return pos, hs


def random_read(rng, n):
    """A read with upper- and lower-case bases, N runs and other non-ACGT bytes."""
    b = np.array(list(b"ACGTACGTACGTACGTacgtN"), dtype=np.uint8)[rng.integers(0, 21, n)]
    for _ in range(3):
        at = int(rng.integers(0, n))
        b[at:at + int(rng.integers(1, 6))] = ord(rng.choice(list("NnRYX-.")))
    return b.tobytes()


def test_two_nthash_statements_agree_for_every_k():
    rng = np.random.default_rng(2031)
    reads = [random_read(rng, int(rng.integers(40, 200))) for _ in range(6)]
    n = 0
    for k in ALL_K:
        for r in reads:
            pos, hs = ol.nthash_all(r, k)
            dpos, dhs = direct_nthash(r, k)
            assert pos.tolist() == dpos, k
            assert hs.tolist() == dhs, k
            n += len(dpos)
    assert n > 5000


def byte_tables():
    """tf[g][b] = XOR_j srol^{4g+3-j}(seed[code_j(b)]), tr[m][b] = XOR_j srol^{4m+j}(seed[3-code_j(b)])
    (gp_hashing.cuh::fill_hash_tables)"""
    tf = np.zeros((8, 256), dtype=np.uint64)
    tr = np.zeros((8, 256), dtype=np.uint64)
    for g in range(8):
        for b in range(256):
            f = r = 0
            for j in range(4):
                c = (b >> (2 * j)) & 3
                f ^= srol(CODE_SEED[c], 4 * g + 3 - j)
                r ^= srol(CODE_SEED[3 - c], 4 * g + j)
            tf[g, b], tr[g, b] = f, r
    return tf, tr


def sror_np(v, s):
    """inverse of srol on an array"""
    m31, m33 = np.uint64((1 << 31) - 1), np.uint64((1 << 33) - 1)
    hi, lo = v >> np.uint64(33), v & m33
    hi = ((hi >> np.uint64(s)) | (hi << np.uint64(31 - s))) & m31
    lo = ((lo >> np.uint64(s)) | (lo << np.uint64(33 - s))) & m33
    return (hi << np.uint64(33)) | lo


def test_padded_word_algebra_matches_nthash_for_every_k():
    """k = 4q - pad is hashed as the 4q-mer whose last pad bases read as A: fwd_k = sror^pad(fwd_ext ^ Cf) with
    Cf = XOR_{d<pad} srol^d(seedA), rev_k = rev_ext ^ Cr with Cr = XOR_{i=k}^{4q-1} srol^i(seedT)."""
    tf, tr = byte_tables()
    rng = np.random.default_rng(77)
    codes = rng.integers(0, 4, 3000).astype(np.uint64)
    seq = bytes(b"ACGT"[int(c)] for c in codes)
    for k in ALL_K:
        kq, pad = (k + 3) // 4, -k % 4
        npos = len(codes) - k + 1
        idx = np.arange(npos)[:, None] + np.arange(4 * kq)[None, :]
        win = np.where(np.arange(4 * kq)[None, :] < k, codes[np.minimum(idx, len(codes) - 1)], 0)  # bits beyond 2k zeroed
        fwd = np.zeros(npos, dtype=np.uint64)
        rev = np.zeros(npos, dtype=np.uint64)
        for m in range(kq):
            b = (win[:, 4 * m] | (win[:, 4 * m + 1] << np.uint64(2)) | (win[:, 4 * m + 2] << np.uint64(4)) |
                 (win[:, 4 * m + 3] << np.uint64(6))).astype(np.int64)
            fwd ^= tf[kq - 1 - m][b]
            rev ^= tr[m][b]
        cf = cr = 0
        for d in range(pad):
            cf ^= srol(SEED["A"], d)
        for i in range(k, 4 * kq):
            cr ^= srol(SEED["T"], i)
        if pad:
            fwd = sror_np(fwd ^ np.uint64(cf), pad)
            rev = rev ^ np.uint64(cr)
        with np.errstate(over="ignore"):
            h0 = fwd + rev
        pos, hs = ol.nthash_all(seq, k)
        assert pos.tolist() == list(range(npos)), k
        assert np.array_equal(h0, hs[:, 0]), k


BFS = os.path.join(ROOT, "goldpolish_b200", "bin", "goldpolish-targeted-bfs")


def _server_args(w, k):
    return [BFS] + [os.path.join(w, f) for f in ("t.fa", "t.fa.index", "m.paf", "r.fa", "r.fa.index")] + ["150", "40", "1", "32", str(k)]


@pytest.mark.parametrize("k", [25, 31, 3, 33, 0])
def test_targeted_bfs_k_range(k, tmp_path):
    """The server checks its k list before it loads anything or touches a device: any k in 4..32 passes (and the
    server goes on to the missing index), others are refused with the bound."""
    if not os.path.exists(BFS):
        pytest.skip("goldpolish-targeted-bfs not built")
    r = subprocess.run(_server_args(str(tmp_path), k), capture_output=True, text=True, timeout=60,
                       env=dict(os.environ, GP_QUIET="1"))
    assert r.returncode != 0
    if 4 <= k <= 32:
        assert "not supported" not in r.stderr and "cannot open" in r.stderr, r.stderr
    else:
        assert f"k = {k} is not supported: k must be within 4..32" in r.stderr, r.stderr
