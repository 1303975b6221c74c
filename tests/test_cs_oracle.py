"""CPU tests of the candidate-search row: the C restatement (oracle/cs_oracle.c) and the numpy
builder of the reference-format index (ngmlr_b200/refindex.py) against what the WHOLE unmodified
reference (oracle/_ref/libngmlr_full.so: SequenceProvider, CompactPrefixTable, CS) returned, and
against each other."""
import numpy as np
import pytest

import cs_cases
from oracle_lib import CsOracle


@pytest.fixture(scope="module")
def contigs():
    return cs_cases.genome_contigs()


@pytest.fixture(scope="module")
def cs_oracle(contigs):
    o = CsOracle([c.tobytes() for c in contigs])
    yield o
    o.close()


@pytest.fixture(scope="module")
def built(contigs):
    """(EncodedReference, KmerIndex) of the test genome from the numpy builder, built once."""
    from ngmlr_b200 import refindex
    ref = refindex.encode_reference(contigs)
    return ref, refindex.build_index(ref)


def test_numpy_index_builder_equals_oracle(contigs, cs_oracle, built):
    ref, idx = built
    assert ref.concat_len == cs_oracle.concat_len and ref.ref_start == cs_oracle.ref_starts()
    assert np.array_equal(ref.enc, cs_oracle.encoded())
    tab, rci, pos = cs_oracle.index()
    assert np.array_equal(tab, idx.tab) and np.array_equal(rci, idx.rci) and np.array_equal(pos, idx.pos)
    packed = idx.packed_index().reshape(-1, 5)
    assert packed.shape[0] == 4 ** 13 + 1
    assert np.array_equal(packed[:, :4].copy().view(np.uint32).reshape(-1), tab)


def test_oracle_search_basic_properties(contigs, cs_oracle):
    g1 = contigs[0]
    res, mx = cs_oracle.search(g1[20000:20256].tobytes())
    assert res[0][1] // 16 == (1000 + 20000) // 16 and res[0][2] == 0 and mx == res[0][0] and 80 <= mx <= 82
    from ngmlr_b200 import synth
    res, mx = cs_oracle.search(synth.revcomp(g1[30000:30256]).tobytes())
    assert res[0][2] == 1 and abs(res[0][1] - (1000 + 30000)) <= 16
    assert cs_oracle.search(b"")[0] == [] and cs_oracle.search(b"ACGTACGTACGT")[0] == []


@pytest.fixture(scope="module")
def whole_ref():
    """What the unmodified reference, initialised on the test genome, returned (tests/golden/compiled_ref_golden.json,
    written by tests/golden/make_ref_golden.py)."""
    import golden_util as gu
    return gu.load("compiled_ref_golden.json")


def test_oracle_equals_whole_reference(contigs, cs_oracle, whole_ref):
    import golden_util as gu
    ref = whole_ref["whole_reference"]
    assert ref["concat_len"] == cs_oracle.concat_len and ref["ref_starts"] == cs_oracle.ref_starts()
    assert gu.digest(*cs_oracle.index()) == ref["index_sha"]
    subs = [s for s in cs_cases.subreads(250, 17, contigs) if len(s)]
    assert len(subs) == len(ref["search"])
    for sub, (sha, mh) in zip(subs, ref["search"]):
        got, got_mh = cs_oracle.search(sub)
        assert gu.digest(np.array([x[0] for x in got], np.float32), np.array([x[1] for x in got], np.uint64),
                         np.array([x[2] for x in got], np.int32)) == sha and got_mh == mh
    for p, sha in ref["decode"]:
        d = cs_oracle.decode(p)
        assert (None if d is None else gu.digest(d)) == sha, p
    # DecodeRefSequenceExact (alignment windows, corridor 0 as in extractReferenceSequenceForAlignment): the
    # reference's windows are those of decode_exact_golden.json (test_oracle_decode_exact_matches_golden)
    assert cs_oracle.decode_exact(cs_oracle.concat_len, 10) is None
    for st, ln, c, sha in ref["decode_exact_corridor"]:   # non-zero corridor as well
        assert gu.digest(cs_oracle.decode_exact(st, ln, c)) == sha


def test_oracle_decode_exact_matches_golden(contigs, cs_oracle):
    import golden_util as gu
    from ngmlr_b200 import refindex
    g = gu.load("decode_exact_golden.json")
    enc = refindex.encode_reference(contigs)
    wins = cs_cases.exact_windows(enc.ref_start, enc.ref_len)
    assert len(wins) == g["n"] and gu.digest(np.array(wins, dtype=np.int64)) == g["windows_sha"], "generator drifted"
    for (st, ln), sha in zip(wins, g["text_sha"]):
        assert gu.digest(cs_oracle.decode_exact(st, ln)) == sha, (st, ln)
    for st, ln, text in g["samples"]:
        assert cs_oracle.decode_exact(st, ln) == text.encode()


def test_cache_files_round_trip(contigs, tmp_path, built):
    """ngmfiles: what is written is read back identically (always runnable)."""
    from ngmlr_b200 import ngmfiles
    ref, idx = built
    ngmfiles.write_encoded_reference(str(tmp_path / "r-enc.2.ngm"), ref, skipped_lens=[8])
    ngmfiles.write_index(str(tmp_path / "r-ht-13-2.2.ngm"), idx)
    ref2, names = ngmfiles.read_encoded_reference(str(tmp_path / "r-enc.2.ngm"))
    assert np.array_equal(ref2.enc, ref.enc) and ref2.concat_len == ref.concat_len
    assert ref2.ref_start == ref.ref_start and ref2.ref_len == ref.ref_len and names[0] == "c0"
    idx2, skip, off = ngmfiles.read_index(str(tmp_path / "r-ht-13-2.2.ngm"))
    assert (idx2.k, skip, off) == (13, 2, 0)
    assert np.array_equal(idx2.tab, idx.tab) and np.array_equal(idx2.rci, idx.rci) and np.array_equal(idx2.pos, idx.pos)
    with open(tmp_path / "bad.ngm", "wb") as f:
        f.write(b"\0" * 64)
    with pytest.raises(ValueError):
        ngmfiles.read_index(str(tmp_path / "bad.ngm"))
    # the library's C writers / readers (csrc/ngm_files.cpp): same bytes, same arrays
    ngmfiles.c_write_encoded_reference(str(tmp_path / "c-enc.2.ngm"), ref, skipped_lens=[8])
    ngmfiles.c_write_index(str(tmp_path / "c-ht-13-2.2.ngm"), idx)
    assert open(tmp_path / "c-enc.2.ngm", "rb").read() == open(tmp_path / "r-enc.2.ngm", "rb").read()
    assert open(tmp_path / "c-ht-13-2.2.ngm", "rb").read() == open(tmp_path / "r-ht-13-2.2.ngm", "rb").read()
    ref3, names3 = ngmfiles.c_read_encoded_reference(str(tmp_path / "r-enc.2.ngm"))
    assert np.array_equal(ref3.enc, ref.enc) and ref3.concat_len == ref.concat_len
    assert ref3.ref_start == ref.ref_start and ref3.ref_len == ref.ref_len and names3 == names
    idx3, skip3, off3 = ngmfiles.c_read_index(str(tmp_path / "r-ht-13-2.2.ngm"))
    assert (idx3.k, skip3, off3) == (13, 2, 0)
    assert np.array_equal(idx3.tab, idx.tab) and np.array_equal(idx3.rci, idx.rci) and np.array_equal(idx3.pos, idx.pos)
    with pytest.raises(ValueError):
        ngmfiles.c_read_index(str(tmp_path / "bad.ngm"))
    blob = bytearray(open(tmp_path / "r-ht-13-2.2.ngm", "rb").read())
    blob[-1] ^= 0x40                      # broken signature: the reference would rebuild the table
    open(tmp_path / "sig.ngm", "wb").write(bytes(blob))
    with pytest.raises(ValueError, match="-5"):
        ngmfiles.c_read_index(str(tmp_path / "sig.ngm"))


def test_cache_files_are_byte_compatible_with_the_reference(contigs, tmp_path, built, whole_ref):
    """The UNMODIFIED reference writes <fasta>-enc.2.ngm and <fasta>-ht-13-2.2.ngm for the test genome (contig names
    with a description); ngmfiles and the library's C writers write the same bytes (the index file entirely; the
    encoded reference up to the end of the used part of binRef -- the reference writes its uninitialised allocation
    tail): digests of the reference's files are stored."""
    import golden_util as gu
    from ngmlr_b200 import ngmfiles
    gold = whole_ref["cache_files"]
    ref, idx = built
    names = gold["names"]
    assert names == [f"contig{i}" for i in range(len(contigs)) if contigs[i].size > 10]
    # writers: same bytes
    ngmfiles.write_index(str(tmp_path / "mine-ht.ngm"), idx)
    assert gu.digest(open(tmp_path / "mine-ht.ngm", "rb").read()) == gold["index_sha"]
    skipped = [int(c.size) for c in contigs if not c.size > 10]
    ngmfiles.write_encoded_reference(str(tmp_path / "mine-enc.ngm"), ref, names, skipped_lens=skipped)
    mine = open(tmp_path / "mine-enc.ngm", "rb").read()
    defined = 24 + 128 * len(ref.ref_start) + int(ref.enc.size)
    assert len(mine) == gold["enc_len"] and gu.digest(mine[:defined]) == gold["enc_defined_sha"]
    # ... and the library's C writers
    ngmfiles.c_write_index(str(tmp_path / "c-ht.ngm"), idx)
    assert gu.digest(open(tmp_path / "c-ht.ngm", "rb").read()) == gold["index_sha"]
    ngmfiles.c_write_encoded_reference(str(tmp_path / "c-enc.ngm"), ref, names, skipped_lens=skipped)
    assert open(tmp_path / "c-enc.ngm", "rb").read() == mine
    c_ref, c_names = ngmfiles.c_read_encoded_reference(str(tmp_path / "mine-enc.ngm"))
    assert np.array_equal(c_ref.enc, ref.enc) and c_ref.ref_start == ref.ref_start and c_names == names


class _OracleBackend:
    """The two backend operations of ngmlr_b200.intervals on the CPU oracle."""

    def __init__(self, cs_oracle, oracle):
        self.cs, self.o = cs_oracle, oracle

    def decode(self, starts, seq_lens):
        return [self.cs.decode_exact(int(s), int(n)) for s, n in zip(starts, seq_lens)]

    def align(self, tasks, refs, offsets, lengths):
        return [self.o.single_align(r, t.read_seq, o, l, t.ext_qstart, t.ext_qend)
                for t, r, o, l in zip(tasks, refs, offsets, lengths)]


def _interval_tasks(contigs, enc):
    """Intervals as processLongReadLIS would hand them to computeAlignment: read part, reference span
    (with some slack or some shortfall), 256-bp anchors (some reverse-coded), corridor estimate; plus
    realign / short-read / full-matrix variants and corridors that are too narrow at first."""
    from ngmlr_b200 import corridor, synth
    from ngmlr_b200.intervals import IntervalTask
    rng = np.random.default_rng(77)
    tasks = []
    for k in range(36):
        c = int(rng.integers(0, 2))
        L = int(rng.integers(300, 3000))
        s0 = int(rng.integers(200, contigs[c].size - L - 200))
        big_del = k % 5 == 0          # a long deletion in the read: the first corridor may be too narrow
        src = contigs[c][s0:s0 + L]
        if big_del:
            cut = int(rng.integers(40, 120))
            mid = L // 2
            src = np.concatenate([src[:mid], src[mid + cut:]])
        read, _ = synth.mutate(src, rng, err=0.10)
        ext_qs, ext_qe = (int(rng.integers(0, 30)), int(rng.integers(0, 30))) if k % 3 == 0 else (0, 0)
        on_start = enc.ref_start[c] + s0 - int(rng.integers(0, 40))
        on_stop = enc.ref_start[c] + s0 + L + int(rng.integers(0, 40))
        full_len = len(read) + ext_qs + ext_qe
        anchors = []
        for y in range(0, len(read) - 256, 256):
            x = int(y * (on_stop - on_start) / max(len(read), 1)) + int(rng.integers(-20, 21))
            rev = int(rng.integers(0, 2))
            on_read = (full_len - (y + ext_qs) - 256) if rev else (y + ext_qs)
            anchors.append((on_read, on_start + max(x, 0), rev))
        kind = k % 6
        t = IntervalTask(on_ref_start=on_start, on_ref_stop=on_stop, read_seq=read.tobytes(),
                         corridor=corridor.estimate_corridor(len(read), on_stop - on_start),
                         ext_qstart=ext_qs, ext_qend=ext_qe, full_read_length=full_len,
                         anchors=anchors if kind != 1 else [], realign=kind == 2,
                         full_alignment=kind == 3 and L < 900, short_read=kind == 4)
        if kind == 5:
            t.corridor = 40       # far too narrow: forces retries with wider corridors
            t.anchors = []
        tasks.append(t)
    return tasks


def test_batched_compute_alignment_equals_the_reference(contigs, cs_oracle, whole_ref, oracle):
    """ngmlr_b200.intervals.compute_alignments (window extraction, corridor per attempt, retry policy)
    with the oracle as its backend == AlignmentBuffer::computeAlignment of the unmodified reference."""
    import golden_util as gu
    from ngmlr_b200 import refindex
    from ngmlr_b200.intervals import compute_alignments
    enc = refindex.encode_reference(contigs)
    tasks = _interval_tasks(contigs, enc)
    want = whole_ref["whole_reference"]["compute_alignment"]
    assert len(want) == len(tasks)
    got, calls = compute_alignments(_OracleBackend(cs_oracle, oracle), tasks)
    n_valid = n_retry = 0
    for t, g, nc, w in zip(tasks, got, calls, want):
        assert (w is not None) == (g is not None), (t.corridor, nc)
        if g is None:
            continue
        n_valid += 1
        n_retry += nc > 1
        assert w["cigar_sha"] == gu.digest(g["cigar"]) and w["md_sha"] == gu.digest(g["md"])
        for k in ("qstart", "qend", "nm", "alignment_length", "cigar_op_count", "position_offset", "score_bits",
                  "identity_bits"):
            assert w[k] == g[k], k
    assert n_valid >= 24 and n_retry >= 3, (n_valid, n_retry)
