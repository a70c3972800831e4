"""CPU: oracle/ref_sample.py drives the reference's own serve_batch + ntEdit chain + guard on chosen batches; its
single-thread fallback (the C restatement) must give the same filters and the same records, batch for batch."""
import json
import os

import numpy as np
import pytest

from util import GOLDEN, dataset, sha

from oracle import ref_driver as rd
from oracle.ref_sample import ReferenceSample

W = dict(bsize=3, subsample_max=40.0, mx_max=150.0, mappings="paf")


def test_port_and_reference_agree_on_batches():
    """Against what the reference produced for these batches (tests/golden/reference_checks.json), and -- when
    oracle/_ref has been built -- live."""
    d = dataset(genome_len=60000)
    nb = (d.n_contigs + W["bsize"] - 1) // W["bsize"]
    batches = [nb - 1, 0]  # any order, any subset
    path = os.path.join(GOLDEN, "reference_checks.json")
    if not os.path.exists(path) and not rd.ref_available():
        pytest.skip("oracle/_ref not built and tests/golden/reference_checks.json not minted")
    if os.path.exists(path):
        want = json.load(open(path))["ref_sample"]
        assert want["batches"] == batches
        port = ReferenceSample(W, d, batches, threads=1)
        port.kind = "port"
        try:
            port.run()
            for i in range(len(batches)):
                assert sha(port.filters(i)) == want["filters_sha256"][i], f"filters of batch {batches[i]}"
                assert [[n, sha(s)] for n, s in port.polished(i)] == want["polished"][i], f"records of batch {batches[i]}"
        finally:
            port.close()
    if not rd.ref_available():
        return
    ref = ReferenceSample(W, d, batches, threads=2)
    port = ReferenceSample(W, d, batches, threads=1)
    port.kind = "port"
    try:
        r = ref.run()
        q = port.run()
        assert r["kind"] == "reference" and q["kind"] == "port" and r["bases"] == q["bases"]
        for i in range(len(batches)):
            assert np.array_equal(ref.filters(i), port.filters(i)), f"filters of batch {batches[i]}"
            assert ref.polished(i) == port.polished(i), f"records of batch {batches[i]}"
            assert len(ref.polished(i)) > 0
    finally:
        ref.close()
        port.close()
