"""CPU: the edit-record rules of gp_polish_fetch_edits restated in numpy, fed by ntEdit's C restatement with origins.
Replaying the records onto the draft must give the polished record (up to case) for the golden ntEdit cases and a
simulated set, and each normalisation rule is pinned on hand-built cases."""
import atexit
import ctypes as C
import json
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from util import GOLDEN, KS, ROOT, dataset, ol, oracle_build, oracle_polish_contig, plan

INS = 0xFFFFFFFF  # GP_EDIT_INSERTED
_origins_lib = None


def _lib():
    """tests/ntedit_origins.c (the C restatement's ntEdit with origins), compiled once per process into a temporary
    directory: the repository tree is not written to."""
    global _origins_lib
    if _origins_lib is None:
        d = tempfile.mkdtemp(prefix="gp_origins_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libntedit_origins.so")
        cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
        subprocess.check_call([cc, "-std=c11", "-O2", "-fPIC", "-shared", "-o", so,
                               os.path.join(ROOT, "tests", "ntedit_origins.c"), "-lm"])
        l = C.CDLL(so)
        l.ntedit_contig_origins.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(ol.NteditOpts),
                                            C.c_void_p, C.c_size_t, C.POINTER(ol.NteditStats), C.c_void_p]
        l.ntedit_contig_origins.restype = C.c_long
        _origins_lib = l
    return _origins_lib


def ntedit_contig_origins(seq: bytes, bf: np.ndarray, k: int, **kw):
    """ol.ntedit_contig plus the origin of every output byte: its position in `seq`, or INS.
    Returns (edited bytes or None if dropped, origins (uint32) or None, stats dict)."""
    o = ol.ntedit_opts(k, **kw)
    cap = 2 * len(seq) + 4096
    out = np.zeros(cap, dtype=np.uint8)
    org = np.zeros(cap, dtype=np.uint32)
    st = ol.NteditStats()
    bf = np.ascontiguousarray(bf, dtype=np.uint8)
    n = _lib().ntedit_contig_origins(seq, len(seq), bf.ctypes.data, bf.size, C.byref(o), out.ctypes.data, cap,
                                     C.byref(st), org.ctypes.data)
    if n == -1:
        return None, None, st.as_dict()
    if n < 0:
        raise RuntimeError("ntedit output buffer too small")
    return out[:n].tobytes(), org[:n].copy(), st.as_dict()
TYPES = ("SNV", "MNV", "INS", "DEL", "COMPLEX")


def _up(b: bytes) -> np.ndarray:
    a = np.frombuffer(b, dtype=np.uint8).copy()
    low = (a >= 97) & (a <= 122)
    a[low] -= 32
    return a


def derive_records(draft: bytes, out: bytes, origin) -> list:
    """(pos, REF, ALT, TYPE) of every gap between consecutive anchors, as include/goldpolish_b200.h states the rule:
    an anchor is a polished base whose origin is a draft base equal to it up to case; the contig ends are anchors."""
    D, O = _up(draft), _up(out)
    R = np.asarray(origin, dtype=np.uint32)
    assert len(R) == len(O)
    kept = R != INS
    org = R[kept].astype(np.int64)
    if np.any(org >= len(D)) or np.any(np.diff(org) <= 0):
        raise ValueError("origins of the non-inserted bases do not increase strictly")
    anchor = kept.copy()
    anchor[kept] = D[org] == O[kept]
    A = np.flatnonzero(anchor)
    a = np.concatenate([[-1], A])
    b = np.concatenate([A, [len(O)]])
    oa = np.concatenate([[-1], R[A].astype(np.int64)])
    ob = np.concatenate([R[A].astype(np.int64), [len(D)]])
    recs = []
    for t in np.flatnonzero((b - a > 1) | (ob - oa > 1)):
        ai, bi, oai, obi = int(a[t]), int(b[t]), int(oa[t]), int(ob[t])
        ref, alt = D[oai + 1:obi].tobytes(), O[ai + 1:bi].tobytes()
        if ref and alt:
            pos = oai + 1
            kind = "COMPLEX" if len(ref) != len(alt) else "SNV" if len(ref) == 1 else "MNV"
        else:
            kind = "DEL" if ref else "INS"
            if ai >= 0:  # the left anchor's base before both
                pos = oai
                ref, alt = D[oai:oai + 1].tobytes() + ref, D[oai:oai + 1].tobytes() + alt
            elif bi < len(O):  # at the contig start: the right anchor's base after both
                pos = 0
                ref, alt = ref + D[obi:obi + 1].tobytes(), alt + D[obi:obi + 1].tobytes()
            else:
                pos = 0
        recs.append((pos, ref.decode(), alt.decode(), kind))
    return recs


def replay(draft: bytes, recs) -> bytes:
    """The draft with every record applied (upper case): what the records claim the polished record is."""
    D = _up(draft).tobytes()
    out, prev = [], 0
    for pos, ref, alt, _ in recs:
        assert pos >= prev and D[pos:pos + len(ref)] == ref.encode(), (pos, ref)
        out.append(D[prev:pos])
        out.append(alt.encode())
        prev = pos + len(ref)
    out.append(D[prev:])
    return b"".join(out)


def compose(origin, local):
    """Origins after one more round: `local` maps the round's output to its input, `origin` that input to the draft."""
    origin = np.asarray(origin, dtype=np.uint32)
    local = np.asarray(local, dtype=np.uint32)
    ins = local == INS
    return np.where(ins, np.uint32(INS), origin[np.where(ins, 0, local)] if len(origin) else np.uint32(INS)).astype(np.uint32)


def chain_with_origins(seq: bytes, bfs, ks=KS, **opts):
    """The k chain of scripts/goldpolish-ntedit:20-29 by the C restatement, with the composed origin map."""
    cur, origin = seq, np.arange(len(seq), dtype=np.uint32)
    for bf, k in zip(bfs, ks):
        cur, local, _ = ntedit_contig_origins(cur, bf, k, **opts)
        if cur is None:
            return None, None
        origin = compose(origin, local)
    return cur, origin


def _check_contig(draft: bytes, bfs, ks=KS, **opts):
    """The chain with origins gives the same bytes as the pinned restatement, and its records replay to it."""
    out, origin = chain_with_origins(draft, bfs, ks, **opts)
    assert out == oracle_polish_contig(draft, bfs, ks, **opts)
    if out is None:
        return None
    recs = derive_records(draft, out, origin)
    assert replay(draft, recs) == _up(out).tobytes()
    return recs


def _golden():
    with open(os.path.join(GOLDEN, "ntedit_cases.json")) as f:
        g = json.load(f)
    fs = ol.FilterSet(KS)
    for _ in range(5):
        fs.add_read(g["truth"].encode(), 4)
    return g, fs


def test_golden_cases_replay_to_the_polished_records():
    g, fs = _golden()
    kinds = set()
    for name, rec in g["cases"].items():
        draft = rec["draft"].encode()
        recs = _check_contig(draft, fs.bfs)
        if rec["chain"] is None:
            assert recs is None, name
            continue
        kinds.update(r[3] for r in recs)
        if rec["chain"].upper() == rec["draft"].upper():
            assert recs == [], name
        if "mode0" in rec:  # one round at k 32 in the other modes / limits of the golden file
            for opts, key in (({"mode": 0}, "mode0"), ({"mode": 2, "max_insertions": 2, "max_deletions": 2}, "mode2"),
                              ({"mask": 0, "max_insertions": 3, "max_deletions": 10}, "nomask_i3_d10")):
                out, local, _ = ntedit_contig_origins(draft, fs.bfs[0], 32, **opts)
                assert out.decode() == rec[key]
                assert replay(draft, derive_records(draft, out, local)) == _up(out).tobytes()
    assert {"SNV", "INS", "DEL"} <= kinds


def test_simulated_set_replays():
    d = dataset(genome_len=60000)
    pl = plan(d, bsize=1)
    fsets = oracle_build(d, pl)
    edited = 0
    for c in range(d.n_contigs):
        edited += bool(_check_contig(d.contig(c), fsets[int(pl.contig_batch[c])].bfs))
    assert edited > 0


def test_origins_increase_strictly():
    g, fs = _golden()
    for rec in g["cases"].values():
        draft = rec["draft"].encode()
        out, local, _ = ntedit_contig_origins(draft, fs.bfs[0], 32)
        if out is None:
            continue
        kept = local != INS
        assert np.all(np.diff(local[kept].astype(np.int64)) > 0) and np.all(local[kept] < len(draft))


D8 = b"ACGTACGT"
ID = list(range(8))


@pytest.mark.parametrize("out,origin,want", [
    (b"ACCTACGT", ID, [(2, "G", "C", "SNV")]),
    (b"ACCAACGT", ID, [(2, "GT", "CA", "MNV")]),
    (b"ACGTTACGT", [0, 1, 2, 3, INS, 4, 5, 6, 7], [(3, "T", "TT", "INS")]),
    (b"ACGACGT", [0, 1, 2, 4, 5, 6, 7], [(2, "GT", "G", "DEL")]),
    (b"GACGTACGT", [INS] + ID, [(0, "A", "GA", "INS")]),
    (b"CGTACGT", ID[1:], [(0, "AC", "C", "DEL")]),
    (b"ACGTACGTA", ID + [INS], [(7, "T", "TA", "INS")]),
    (b"ACGTACG", ID[:7], [(6, "GT", "G", "DEL")]),
    (b"ACGCCGT", [0, 1, 2, INS, INS, 6, 7], [(3, "TAC", "CC", "COMPLEX")]),
    (b"acgTACGT", ID, []),                                   # soft-masking is not an edit
    (b"CATGTGCA", ID, [(0, "ACGTACGT", "CATGTGCA", "MNV")]),  # no anchor at all
    (b"GG", [INS, INS], [(0, "ACGTACGT", "GG", "COMPLEX")]),
    (b"ACGGGTACGT", [0, 1, 2, INS, INS, 3, 4, 5, 6, 7], [(2, "G", "GGG", "INS")]),
])
def test_normalisation_rules(out, origin, want):
    recs = derive_records(D8, out, origin)
    assert recs == want
    assert replay(D8, recs) == _up(out).tobytes()


def test_iupac_draft_bases_are_written_as_they_are():
    assert derive_records(b"ACGTNCGT", b"ACGTACGT", list(range(8))) == [(4, "N", "A", "SNV")]
    assert derive_records(b"ACGTrCGT", b"ACGTACGT", list(range(8))) == [(4, "R", "A", "SNV")]


def test_insertion_deleted_by_a_later_round_leaves_no_record():
    round1 = np.array([0, 1, 2, 3, INS, 4, 5, 6, 7], dtype=np.uint32)  # "ACGT" + "G" + "ACGT"
    round2 = np.array([0, 1, 2, 3, 5, 6, 7, 8], dtype=np.uint32)       # the inserted G deleted again
    origin = compose(compose(np.arange(8, dtype=np.uint32), round1), round2)
    assert origin.tolist() == ID
    assert derive_records(D8, D8, origin) == []
    # ... while a deletion that a later round fills with another base is one substitution
    round2b = np.array([0, 1, 2, 3, INS, 5, 6, 7, 8], dtype=np.uint32)
    origin = compose(compose(np.arange(8, dtype=np.uint32), round1), round2b)
    assert derive_records(D8, b"ACGTCACGT", origin) == [(3, "T", "TC", "INS")]


def test_decreasing_origins_are_refused():
    with pytest.raises(ValueError):
        derive_records(D8, b"ACGTACGT", [0, 1, 2, 4, 3, 5, 6, 7])
    with pytest.raises(ValueError):
        derive_records(D8, b"ACG", [0, 1, 8])


def test_track_edits_with_hard_masking_is_refused():
    import goldpolish_b200 as gp
    with pytest.raises(gp.GpError) as e:
        gp.Context(track_edits=True, prep_mode=2, prep_k=32)
    assert e.value.code == -1 and "prep_mode 2" in str(e.value)
