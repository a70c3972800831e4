"""CPU: the oracle restatement (oracle/gp_oracle.c) against the golden vectors minted from the
reference's own code (tests/golden/make_golden.py), and -- when oracle/_ref is present -- live."""
import json
import os
import random
import re

import numpy as np
import pytest

from util import GOLDEN, KS, dataset, ol, plan, sha


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def test_nthash_known_answers():
    for rec in _load("nthash_kat.json"):
        pos, hs = ol.nthash_all(rec["seq"].encode(), rec["k"])
        assert pos.tolist() == rec["pos"]
        assert [[str(x) for x in row] for row in hs.tolist()] == rec["hashes"]


def test_nthash_canonical_symmetry():
    """fwd(kmer) == rev(revcomp(kmer)): the canonical hash is strand independent."""
    rng = random.Random(5)
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    for _ in range(200):
        k = rng.choice(KS)
        s = "".join(rng.choice("ACGT") for _ in range(k))
        rc = "".join(comp[c] for c in reversed(s))
        l = ol.lib()
        assert l.gpo_ntf64(s.encode(), k) == l.gpo_ntr64(rc.encode(), k)
        assert l.gpo_ntf64(s.encode(), k) + l.gpo_ntr64(s.encode(), k) == \
            (l.gpo_ntf64(rc.encode(), k) + l.gpo_ntr64(rc.encode(), k))


def test_filters_golden():
    import sim
    import goldpolish_b200 as gp
    for case in _load("filters.json")["cases"]:
        d = sim.simulate(**case["sim"])
        for b, rec in enumerate(case["batches"]):
            fs = ol.FilterSet(KS)
            for rid, thr in rec["entries"]:
                fs.add_read(d.read(rid), thr)
            assert [sha(x) for x in fs.bfs] == rec["bf_sha256"], (case["name"], b)
            assert [sha(x) for x in fs.cbfs] == rec["cbf_sha256"], (case["name"], b)
            assert rec["server_bf_sha256"] == rec["bf_sha256"]
        # the host planner reproduces the entries the reference server selected
        pl = gp.plan_batches(np.diff(d.contig_off), [d.contig_name(i) for i in range(d.n_contigs)],
                             [d.read_name(i) for i in range(d.n_reads)], d.read_phred, np.diff(d.read_off),
                             d.map_read, d.map_contig, bsize=case["bsize"])
        for b, rec in enumerate(case["batches"]):
            ents = pl.entries[int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]
            assert [[int(e["read_id"]), int(e["kmer_threshold"])] for e in ents] == rec["entries"]


def test_order_dependence_is_real():
    """Reversing the read order of a loaded batch changes the filter bits (SURVEY Appendix C):
    an unordered counting-filter update cannot be bit exact."""
    import sim
    case = [c for c in _load("filters.json")["cases"] if c["name"] == "loaded_bsize8"][0]
    d = sim.simulate(**case["sim"])
    rec = max(case["batches"], key=lambda r: len(r["entries"]))
    fs = ol.FilterSet(KS)
    for rid, thr in reversed(rec["entries"]):
        fs.add_read(d.read(rid), thr)
    assert [sha(x) for x in fs.cbfs] != rec["cbf_sha256"]


def _golden_cases():
    g = _load("ntedit_cases.json")
    truth = g["truth"].encode()
    fs = ol.FilterSet(KS)
    for _ in range(5):
        fs.add_read(truth, 4)
    assert [sha(b) for b in fs.bfs] == g["bf_sha256"]
    return g, fs


def test_ntedit_golden_cases():
    g, fs = _golden_cases()
    kinds = {}
    for name, rec in g["cases"].items():
        draft = rec["draft"].encode()
        for i, k in enumerate(KS):
            got, st = ol.ntedit_contig(draft, fs.bfs[i], k)
            want = rec["per_k"][str(k)]
            assert (got is None and want is None) or got.decode() == want, (name, k)
            assert st["ref_ub"] == 0
            for key, v in st.items():
                kinds[key] = kinds.get(key, 0) + v
        cur = draft
        for i, k in enumerate(KS):
            cur, _ = ol.ntedit_contig(cur, fs.bfs[i], k)
            if cur is None:
                break
        assert (cur is None and rec["chain"] is None) or cur.decode() == rec["chain"], name
        if "mode0" in rec:
            assert ol.ntedit_contig(draft, fs.bfs[0], 32, mode=0)[0].decode() == rec["mode0"]
            assert ol.ntedit_contig(draft, fs.bfs[0], 32, mode=2, max_insertions=2, max_deletions=2)[0].decode() == rec["mode2"]
            assert ol.ntedit_contig(draft, fs.bfs[0], 32, mask=0, max_insertions=3, max_deletions=10)[0].decode() == rec["nomask_i3_d10"]
    # the cases really exercise every edit kind
    for key in ("subs", "inss", "dels", "masks"):
        assert kinds[key] > 0, key
    # planted errors are repaired: the clean draft comes back unchanged and fixed drafts equal the truth
    assert g["cases"]["clean"]["chain"] == g["truth"]
    assert g["cases"]["ins_1_to_5"]["chain"] == g["truth"]  # isolated 1..5 bp insertions are deleted again
    assert g["cases"]["short_80bp"]["chain"] is None           # ntedit.cpp:1850
    assert g["cases"]["exactly_100bp"]["chain"] is not None


def test_ntedit_cli_golden_records():
    """Header = name + ' ' + comment, multi-line input joined, <100 bp record dropped (ntedit.cpp:1831-1853)."""
    g = _load("ntedit_cli.json")
    recs = g["edited_fasta"].strip().split("\n")
    assert recs[0] == ">c1 first comment here" and recs[2] == ">c3" and len(recs) == 4
    _, fs = _golden_cases()
    ins = {}
    name = None
    for ln in g["input_fasta"].splitlines():
        if ln.startswith(">"):
            name = ln[1:]
            ins[name] = ""
        else:
            ins[name] += ln
    assert ol.ntedit_contig(ins["c1 first comment here"].encode(), fs.bfs[0], 32)[0].decode() == recs[1]
    assert ol.ntedit_contig(ins["c3"].encode(), fs.bfs[0], 32)[0].decode() == recs[3]
    assert ol.ntedit_contig(ins["tiny"].encode(), fs.bfs[0], 32)[0] is None


def _reference_checks():
    """tests/golden/reference_checks.json (tests/golden/make_golden_reference_checks.py), or None before it is minted."""
    path = os.path.join(GOLDEN, "reference_checks.json")
    return _load("reference_checks.json") if os.path.exists(path) else None


def test_insertion_strings_match_reference_table():
    """multi_possible_bases (ntedit.cpp:198-343) is regenerated arithmetically; check it against the table minted
    from the reference source, or against that source itself when it is mounted."""
    path = "/root/reference/subprojects/ntedit/ntedit.cpp"
    g = _reference_checks()
    if g is None and not os.path.exists(path):
        pytest.skip("reference source not mounted and tests/golden/reference_checks.json not minted")
    tables = {}
    if g is not None:
        tables.update(g["insertion_strings"])
    if os.path.exists(path):
        from golden.make_golden_reference_checks import insertion_strings
        live = insertion_strings(os.path.dirname(os.path.dirname(os.path.dirname(path))))
        assert g is None or live == tables
        tables = live
    for first in "ACGT":
        strings = tables[first]
        assert len(strings) >= 341
        for i in range(341):
            buf = (b"\0" * 8)
            import ctypes as C
            out = C.create_string_buffer(8)
            n = ol.lib().gpo_insertion_string(ord(first), i, out)
            assert out.value.decode() == strings[i] and n == len(strings[i])


def test_thresholds_and_guard():
    l = ol.lib()
    # goldpolish_targeted_bfs.cpp:45-53
    assert [l.gpo_kmer_threshold(b) for b in (0, 1_000_000, 10_000_000, 37_100_000, 10**9)] == [5, 5, 7, 13, 13]
    # :96-99 truncation
    assert l.gpo_mappings_cap(7000, 40.0) == 28 and l.gpo_mappings_cap(249, 40.0) == 0
    # scripts/goldpolish-ntedit:31-34
    assert l.gpo_guard_rejects(10000, 7499) == 1 and l.gpo_guard_rejects(10000, 7500) == 0
    assert l.gpo_guard_rejects(3, 2) == 1  # 0.6666 < 0.75


def test_oracle_matches_reference_live():
    """Differential check against the reference's own functions: what they produced for these inputs, minted into
    tests/golden/reference_checks.json, and -- when oracle/_ref has been built -- live."""
    from oracle import ref_driver as rd
    g = _reference_checks()
    if g is None and not rd.ref_available():
        pytest.skip("oracle/_ref not built and tests/golden/reference_checks.json not minted")
    d = dataset(genome_len=30000, seed=99)
    pl = plan(d, bsize=2)
    b = int(np.argmax(np.diff(pl.batch_entry_off)))
    ents = pl.entries[int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]
    if g is not None:
        want = g["live"]
        assert want["batch"] == b
        fs = ol.FilterSet(KS)
        for e in ents:
            fs.add_read(d.read(int(e["read_id"])), int(e["kmer_threshold"]))
        assert [sha(x) for x in fs.bfs] == want["bf_sha256"] and [sha(x) for x in fs.cbfs] == want["cbf_sha256"]
        for c, steps in want["contigs"].items():
            cur, got = d.contig(int(c)), []
            for i, k in enumerate(KS):
                cur, _ = ol.ntedit_contig(cur, fs.bfs[i], k)
                got.append(None if cur is None else sha(cur))
                if cur is None:
                    break
            assert got == steps, c
    if not rd.ref_available():
        return
    import ctypes as C
    h = rd.harness()
    fs = ol.FilterSet(KS)
    ks = (C.c_uint * 4)(*KS)
    hb = h.ref_build_open(ks, 4, ol.CBF_COUNTERS, ol.BF_BYTES, 4)
    for e in ents:
        s = d.read(int(e["read_id"]))
        fs.add_read(s, int(e["kmer_threshold"]))
        h.ref_build_add_read(hb, s, len(s), int(e["kmer_threshold"]))
    for i in range(4):
        rb = np.zeros(ol.BF_BYTES, np.uint8); h.ref_build_get_bf(hb, i, rb.ctypes.data)
        rc = np.zeros(ol.CBF_COUNTERS, np.uint8); h.ref_build_get_cbf(hb, i, rc.ctypes.data)
        assert np.array_equal(rb, fs.bfs[i]) and np.array_equal(rc, fs.cbfs[i])
    h.ref_build_close(hb)
    for c in range(2 * b, min(2 * b + 2, d.n_contigs)):
        cur = d.contig(c)
        for i, k in enumerate(KS):
            got, _ = ol.ntedit_contig(cur, fs.bfs[i], k)
            cap = 3 * len(cur) + 4096
            buf = np.zeros(cap, np.uint8)
            n = h.ref_ntedit_contig(cur, len(cur), fs.bfs[i].ctypes.data, ol.BF_BYTES, k, 4, 5, 5, 1, 1, 0.5, 0.5,
                                    b"/dev/shm/gp_test_scratch.fa", buf.ctypes.data, cap)
            if n == -1:
                assert got is None
                break
            assert got == buf[:n].tobytes()
            cur = got


def test_python_planner_ntlink_filter_matches_reference_server():
    """ntLink-style triples: the planner's minimizer filter (goldpolish_b200/host.py::filter_ntlink, a restatement of
    AllMappings::filter, src/mappings.cpp:230-320) selects the reads the reference's own server selected -- the
    filters built from its entries equal the payloads that server wrote (binary search on the minimizer threshold at
    mx_max = 12 per 10 kbp, so the filter really drops reads)."""
    import sim
    import goldpolish_b200 as gp
    case = _load("filters.json")["ntlink"]
    d = sim.simulate(**case["sim"])
    pl = gp.plan_batches(np.diff(d.contig_off), [d.contig_name(i) for i in range(d.n_contigs)],
                         [d.read_name(i) for i in range(d.n_reads)], d.read_phred, np.diff(d.read_off),
                         d.map_read, d.map_contig, bsize=case["bsize"], subsample_max_per_10kbp=case["subsample_max"],
                         map_mx=d.map_mx, mx_max_per_10kbp=case["mx_max"])
    unfiltered = gp.plan_batches(np.diff(d.contig_off), [d.contig_name(i) for i in range(d.n_contigs)],
                                 [d.read_name(i) for i in range(d.n_reads)], d.read_phred, np.diff(d.read_off),
                                 d.map_read, d.map_contig, bsize=case["bsize"], subsample_max_per_10kbp=case["subsample_max"])
    assert len(pl.entries) < len(unfiltered.entries)
    for b, rec in enumerate(case["batches"]):
        fs = ol.FilterSet(KS)
        for e in pl.entries[int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]:
            fs.add_read(d.read(int(e["read_id"])), int(e["kmer_threshold"]))
        assert [sha(x) for x in fs.bfs] == rec["server_bf_sha256"], b


def test_reference_fixture_batches_through_the_port():
    """configs[0] on the CPU: the reference's in-tree draft fixture (committed gzip) + reads simulated from its in-tree
    expected output; the C restatement reproduces the reference's own filters and polished record (k chain + guard) of
    a few batches -- read selection by (truncated phred, id), thresholds, FASTQ index semantics included."""
    import fixture_reads as fr
    g = _load("fixtures.json")
    for which, picks in (("config1", (0, 57, 151)), ("target", (0, 6))):
        draft, truth = fr.load_fixture(which)
        reads, maps = fr.simulate_reads(truth)
        gg = g[which]
        assert len(reads) == gg["n_reads"] and sum(len(s) for _, s, _ in reads) == gg["read_bases"]
        seq_of = {n: s for n, s, _ in reads}
        phred_of = {n: float(q - 33) for n, s, q in reads}  # constant quality: mean of all but the last char - 33
        by_contig = {}
        for r, c, *_ in maps:
            by_contig.setdefault(c, []).append(r)
        for b in picks:
            name, seq = draft[b]
            ids = by_contig[name]
            chosen, thr = ol.select_reads(ids, [phred_of[i] for i in ids], [len(seq_of[i]) for i in ids], len(seq), 40.0)
            fs = ol.FilterSet(KS)
            for j in chosen:
                fs.add_read(seq_of[ids[j]], thr)
            assert [sha(x) for x in fs.bfs] == gg["batches"][b]["bf_sha256"], (which, b)
            cur = seq
            for ki, k in enumerate(KS):
                cur, _ = ol.ntedit_contig(cur, fs.bfs[ki], k)
            rec_in = b">" + name.encode() + b"\n" + seq + b"\n"
            rec_out = b">" + name.encode() + b"\n" + cur + b"\n"
            if ol.lib().gpo_guard_rejects(len(rec_in), len(rec_out)):
                rec_out = rec_in
            assert sha(rec_out) == gg["batches"][b]["polished_sha256"], (which, b)
