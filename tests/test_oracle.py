"""CPU tests: the oracle restatement against the committed golden vectors produced by the unmodified
reference (tests/golden/make_golden.py, tests/golden/make_ref_golden.py)."""
import numpy as np
import pytest

import cases
import golden_util as gu
from oracle_lib import DEFAULT_SCORING

REF_GOLD = gu.load("compiled_ref_golden.json")   # tests/golden/make_ref_golden.py


@pytest.mark.parametrize("setname", ["default", "weird", "mild"])
def test_oracle_matches_golden_convex(oracle, setname):
    for name, sc, probs, recs in gu.golden_sets():
        if name != setname:
            continue
        for i, (p, rec) in enumerate(zip(probs, recs)):
            res = oracle.single_align(p.ref, p.qry, p.offsets, p.lengths, p.ext_qstart, p.ext_qend,
                                      scoring=sc, rule=0)
            gu.check_against_record(res, rec, f"{name}[{i}]")
            _, bs, bx, by = oracle.fill(p.ref, p.qry, p.offsets, p.lengths, sc, 0)
            assert [int(np.float32(bs).view(np.uint32)), bx, by] == rec["best"], f"{name}[{i}] best cell"


def test_oracle_directions_match_golden(oracle):
    name, sc, probs, recs = gu.golden_sets()[0]
    for i, (p, rec) in enumerate(zip(probs, recs)):
        if (np.asarray(p.lengths) < 0).any():
            continue  # reference's offsetInMatrix goes backwards on negative lengths: layout-only
        dirs, *_ = oracle.fill(p.ref, p.qry, p.offsets, p.lengths, sc, 0)
        assert gu.digest(dirs) == rec["dirs_sha"], f"direction matrix {i}"


def test_rule2_equals_as_coded_rule(oracle):
    """The single-pass 'raw-run' form the CUDA kernel implements == the as-coded SSE path."""
    for sc, seed in ((DEFAULT_SCORING, 5), (cases.WEIRD_SCORING, 6), (cases.MILD_SCORING, 7)):
        for p in cases.random_problems(12, seed, max_len=700):
            a = oracle.fill(p.ref, p.qry, p.offsets, p.lengths, sc, 0)
            b = oracle.fill(p.ref, p.qry, p.offsets, p.lengths, sc, 2)
            assert np.array_equal(a[0], b[0]) and a[1:] == b[1:]


def test_scalar_rule_equals_sse_rule_for_default_scoring(oracle):
    for p in cases.random_problems(12, 11, max_len=700) + cases.edge_problems():
        a = oracle.fill(p.ref, p.qry, p.offsets, p.lengths, DEFAULT_SCORING, 0)
        b = oracle.fill(p.ref, p.qry, p.offsets, p.lengths, DEFAULT_SCORING, 1)
        assert np.array_equal(a[0], b[0]) and a[1:] == b[1:]


def test_oracle_sw_matches_golden(oracle):
    g = gu.load("sw_golden.json")
    refs, qrys = cases.sw_pairs(256, 31)
    assert gu.digest(b"".join(refs), b"".join(qrys)) == g["input_sha"]
    for r, q, want in zip(refs, qrys, g["scores"]):
        assert oracle.ssw_score(r, q) == want
        assert oracle.ssw_score(r, q, striped=True) == want
    long_ref = b"ACGT" * 700
    extra = [(long_ref, long_ref[:2000]), (long_ref, long_ref[:1000] + b"G" + long_ref[1000:2000]),
             (b"A" * 100001, b"A" * 10), (b"", b""), (b"A", b"A"), (b"ACGT", b"")]
    for (r, q), want in zip(extra, g["extra"]):
        assert oracle.ssw_score(r, q) == want
        assert oracle.ssw_score(r, q, striped=True) == want


def test_oracle_cells_formula(oracle):
    p = cases.random_problems(1, 3)[0]
    lo = np.maximum(p.offsets, 0)
    hi = np.minimum(p.offsets + p.lengths, len(p.ref))
    assert oracle.cells(len(p.ref), p.offsets, p.lengths) == int(np.maximum(hi - lo, 0).sum()) == p.cells


@pytest.mark.parametrize("sc,seed", [(DEFAULT_SCORING, 21), (cases.WEIRD_SCORING, 22), (cases.MILD_SCORING, 23)])
def test_oracle_vs_compiled_reference(oracle, sc, seed):
    gold = REF_GOLD["convex"][str(seed)]
    for i, (p, rec) in enumerate(zip(cases.random_problems(10, seed, max_len=900), gold["records"])):
        assert gu.digest(p.ref, p.qry, p.offsets, p.lengths) == rec["input_sha"], "generator drifted"
        b = oracle.single_align(p.ref, p.qry, p.offsets, p.lengths, p.ext_qstart, p.ext_qend, scoring=sc, rule=0)
        gu.check_against_record(b, rec, f"{seed}[{i}]")
        assert b["score_bits"] == rec["score_bits"]
        db = oracle.fill(p.ref, p.qry, p.offsets, p.lengths, sc, 0)
        assert gu.digest(db[0]) == rec["dirs_sha"] and [int(np.float32(db[1]).view(np.uint32)), *db[2:]] == rec["best"]
    refs, qrys = cases.sw_pairs(64, seed)
    for r, q, want in zip(refs, qrys, gold["sw"]):
        assert want == oracle.ssw_score(r, q) == oracle.ssw_score(r, q, striped=True)


def test_oracle_score_select_matches_golden(oracle):
    """ScoreBuffer::topNSE / computeMQ restatement (incl. libstdc++'s std::sort order among equal scores)
    against vectors recorded from the unmodified reference."""
    from oracle_lib import score_select_cases
    gold = gu.load("score_select_golden.json")
    scs = score_select_cases(77, 400)
    assert len(gold) == len(scs)
    for sc, g in zip(scs, gold):
        assert gu.digest(sc) == g["input_sha"], "generator drifted"
        order, kept, mq = oracle.score_select(sc)
        assert (kept, mq) == (g["kept"], g["mq"])
        assert gu.digest(order) == g["order_sha"]
        if g["order"] is not None:
            assert list(order) == g["order"]


def test_oracle_score_select_vs_compiled_reference(oracle):
    from oracle_lib import score_select_cases
    gold = REF_GOLD["score_select"]
    scs = [sc for sc in score_select_cases(5, 1500) if sc.size]
    assert len(scs) == len(gold["kept"])
    orders = []
    for sc, k, m in zip(scs, gold["kept"], gold["mq"]):
        o = oracle.score_select(sc)
        assert o[1:] == (k, m)
        orders.append(o[0])
    assert gu.digest(np.concatenate(orders)) == gold["order_sha"]


def test_raw_tail_corner_fuzz_against_the_compiled_reference():
    """scripts/fuzz_raw_tail.py (DESIGN.md section 2): the compiled reference's fill vs the single-pass rule 2
    the CUDA RAW kernel implements, on inputs built to hit the tail-cell best-tracking corner (narrow
    corridors, scorings outside the default class). The full run (1.2e8 cells, 0 mismatches) is recorded in
    DESIGN.md; this is its quick version, against the reference's fills stored for it."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "fuzz_raw_tail.py"), "--cells", "4e6", "--seed", "3",
                        "--golden", os.path.join(root, "tests", "golden", "compiled_ref_golden.json")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
    assert "mismatches 0" in r.stdout and "not vacuous" in r.stdout
