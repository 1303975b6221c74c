"""The real call stream of plain ngmlr -- every IAlignment::SingleAlign / BatchScore / SingleScore call the
unmodified reference makes on a FASTQ, recorded by the decorators of oracle/record_aligners.cpp
(oracle/_ref/ngmlr_rec; SURVEY.md section 7 step 0) with what the reference returned, stored as a sample --
replayed call by call:
  * CPU: through the oracle (pins the C restatement on retries x5, realignments, full matrices,
    corridors several thousand columns wide -- inputs the seeded generators only approximate);
  * GPU (-m gpu): through the CUDA library (batched convex path with the device text stage, sub-read
    scorer), bit for bit against what the reference returned."""
import lzma
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))


@pytest.fixture(scope="module")
def stream(tmp_path_factory):
    """A sample of the call stream (tests/golden/recorded_calls.bin.xz, written by tests/golden/make_ref_golden.py
    from `scripts/record_workload.py --reads 28 --genome-mb 1 --contigs 2 --threads 8 --median 5000 --sv --seed 7`)."""
    path = str(tmp_path_factory.mktemp("rec") / "calls.bin")
    with lzma.open(os.path.join(ROOT, "tests", "golden", "recorded_calls.bin.xz")) as f, open(path, "wb") as out:
        out.write(f.read())
    from replay_workload import parse
    aligns, pairs = parse(path)
    assert len(aligns) >= 40 and len(pairs) >= 1000
    return aligns, pairs


def _same(a, r):
    if a["threw"] or a["ret"] < 0:
        return r["ret"] < 0
    return (r["ret"] == a["ret"] and r["score_bits"] == a["score_bits"] and r["cigar"] == a["cigar"]
            and r["md"] == a["md"] and r["nm"] == a["nm"] and r["position_offset"] == a["po"]
            and r["qstart"] == a["qstart"] and r["qend"] == a["qend"])


def test_oracle_equals_the_reference_on_its_real_call_stream(stream, oracle):
    aligns, pairs = stream
    bad = [i for i, a in enumerate(aligns)
           if not _same(a, oracle.single_align(a["ref"], a["qry"], a["off"], a["len"], a["qs"], a["qe"]))]
    assert not bad, bad[:5]
    W = np.array([int(a["len"][0]) for a in aligns])
    # the stream really contains what the seeded generators lack: wide corridors and repeated / failed calls
    assert W.max() >= 1500 and len(aligns) > 28
    for r, q, sb in pairs[:1500]:
        assert int(np.float32(oracle.ssw_score(r, q)).view(np.uint32)) == sb


@pytest.mark.gpu
def test_cuda_library_equals_the_reference_on_its_real_call_stream(stream):
    from ngmlr_b200 import B200Aligner, PackedBatch
    aligns, pairs = stream
    al = B200Aligner(0)
    try:
        for on_device in (True, False):
            al.set_text_stage(on_device, False)
            batch = PackedBatch([a["ref"] for a in aligns], [a["qry"] for a in aligns], [a["off"] for a in aligns],
                                [a["len"] for a in aligns], [a["qs"] for a in aligns], [a["qe"] for a in aligns])
            res = al.BatchAlign(batch)
            bad = [i for i, (a, g) in enumerate(zip(aligns, res)) if not _same(a, g.as_dict())]
            assert not bad, (on_device, bad[:5])
        got = al.BatchScore([p[0] for p in pairs], [p[1] for p in pairs])
        want = np.array([p[2] for p in pairs], dtype=np.uint32)
        assert np.array_equal(got.view(np.uint32), want)
    finally:
        al.close()
