"""Mint tests/golden/reference_checks.json from the reference's OWN code (oracle/_ref and its ntedit.cpp source).

Run where the reference sources are present and oracle/_ref is built:
    make -C oracle ref REF=<reference checkout> && python tests/golden/make_golden_reference_checks.py <reference checkout>
Written (every value an OUTPUT of the reference):
  * insertion_strings   multi_possible_bases of subprojects/ntedit/ntedit.cpp (341 strings per first base)
  * live                the inputs of test_oracle_matches_reference_live: SHA-256 of the reference's filters and of its
                        per-k ntEdit output for each contig of the most loaded batch
  * ref_sample          the inputs of test_port_and_reference_agree_on_batches: SHA-256 of the reference's filter
                        payloads and its polished records (serve_batch + ntEdit chain + guard) per batch
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref_driver as rd  # noqa: E402
from util import KS, dataset, plan, sha  # noqa: E402

OUT = os.path.join(HERE, "reference_checks.json")


def insertion_strings(ref_root):
    src = open(os.path.join(ref_root, "subprojects", "ntedit", "ntedit.cpp")).read()
    body = src[src.index("multi_possible_bases = {"):src.index("/* Checks that the filepath is readable")]
    table = {}
    for first in "ACGT":
        m = re.search(r"\{\s*'%s',\s*\{(.*?)\}\s*\}" % first, body, re.S)
        table[first] = re.findall(r'"([ACGT]+)"', m.group(1))
    return table


def live():
    h = rd.harness()
    d = dataset(genome_len=30000, seed=99)
    pl = plan(d, bsize=2)
    b = int(np.argmax(np.diff(pl.batch_entry_off)))
    ents = pl.entries[int(pl.batch_entry_off[b]):int(pl.batch_entry_off[b + 1])]
    hb = h.ref_build_open((C.c_uint * 4)(*KS), 4, 10485760, 524288, 4)
    for e in ents:
        s = d.read(int(e["read_id"]))
        h.ref_build_add_read(hb, s, len(s), int(e["kmer_threshold"]))
    bfs, rec = [], {"batch": b, "bf_sha256": [], "cbf_sha256": [], "contigs": {}}
    for i in range(4):
        rb = np.zeros(524288, np.uint8); h.ref_build_get_bf(hb, i, rb.ctypes.data)
        rc = np.zeros(10485760, np.uint8); h.ref_build_get_cbf(hb, i, rc.ctypes.data)
        bfs.append(rb); rec["bf_sha256"].append(sha(rb)); rec["cbf_sha256"].append(sha(rc))
    h.ref_build_close(hb)
    for c in range(2 * b, min(2 * b + 2, d.n_contigs)):
        cur, steps = d.contig(c), []
        for i, k in enumerate(KS):
            cap = 3 * len(cur) + 4096
            buf = np.zeros(cap, np.uint8)
            n = h.ref_ntedit_contig(cur, len(cur), bfs[i].ctypes.data, 524288, k, 4, 5, 5, 1, 1, 0.5, 0.5,
                                    b"/dev/shm/gp_golden_scratch.fa", buf.ctypes.data, cap)
            if n == -1:
                steps.append(None)
                break
            cur = buf[:n].tobytes()
            steps.append(sha(cur))
        rec["contigs"][str(c)] = steps
    return rec


def ref_sample():
    from oracle.ref_sample import ReferenceSample
    w = dict(bsize=3, subsample_max=40.0, mx_max=150.0, mappings="paf")
    d = dataset(genome_len=60000)
    nb = (d.n_contigs + w["bsize"] - 1) // w["bsize"]
    batches = [nb - 1, 0]
    rs = ReferenceSample(w, d, batches, threads=2)
    try:
        r = rs.run()
        assert r["kind"] == "reference"
        return {"batches": batches,
                "filters_sha256": [sha(rs.filters(i)) for i in range(len(batches))],
                "polished": [[[n, hashlib.sha256(s).hexdigest()] for n, s in rs.polished(i)] for i in range(len(batches))]}
    finally:
        rs.close()


def main():
    assert rd.ref_available(), "build oracle/_ref first (make -C oracle ref REF=<reference checkout>)"
    out = {"insertion_strings": insertion_strings(sys.argv[1]), "live": live(), "ref_sample": ref_sample()}
    json.dump(out, open(OUT, "w"))
    print("written", OUT)


if __name__ == "__main__":
    main()
