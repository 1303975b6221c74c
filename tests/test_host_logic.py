"""CPU tests of host-side logic: corridor geometry mirrors and batch packing."""
import numpy as np

from ngmlr_b200 import PackedBatch, corridor, synth


def test_corridor_with_anchors_matches_c_float_semantics():
    # hand-computed with float32 arithmetic as in src/AlignmentBuffer.cpp:129-197
    offs, lens = corridor.corridor_endpoints_with_anchors(1000, 1100, [0, 300, 600], [0, 256, 512], 1)
    k = np.float32(1000) / np.float32(1100)
    diffs = [np.float32(y) / k - np.float32(x) for x, y in ((0, 0), (300, 256), (600, 512))]
    right = max([d for d in diffs if d > 0] + [np.float32(0)])
    left = max([-d for d in diffs if not d > 0] + [np.float32(0)])
    left = np.float32(left + 128)
    right = np.float32(right + 128)
    left = np.float32(left + np.float32(np.float32(left + right) * np.float32(0.1)))
    right = np.float32(right + np.float32(np.float32(left + right) * np.float32(0.1)))
    assert lens[0] == int(np.float32(left + right))
    assert offs[0] == int(np.float32(np.float32(0) / k) - right)
    assert offs[999] == int(np.float32(np.float32(999) / k) - right)
    assert (np.diff(offs) >= 0).all() and (lens == lens[0]).all()


def test_other_corridors():
    o, l = corridor.corridor_linear(10, 40)
    assert list(o[:3]) == [-20, -19, -18] and (l == 40).all()
    o, l = corridor.corridor_full(5, 1000)
    assert (o == -200).all() and (l == 1200).all()
    o, l = corridor.corridor_endpoints(100, 120, 400)
    assert (l == 100).all() and o[0] == int((np.float32(0) - np.float32(50)) / (np.float32(100) / np.float32(120)))
    assert corridor.estimate_corridor(8000, 8100) == max(int(np.float32(100) * np.float32(2.1)), 1600)


def test_packed_batch_layout():
    probs = synth.pacbio_problems(3, genome_len=100_000, seed=4, median=1500)
    b = PackedBatch.from_problems(probs)
    assert b.n == 3 and b.row_start[-1] == sum(len(p.qry) for p in probs)
    assert b.offsets.dtype == np.int32 and b.lengths.size == b.row_start[-1]
    assert b.read_bases == sum(len(p.qry) for p in probs)


def test_synthetic_reads_have_requested_error_profile():
    rng = np.random.default_rng(1)
    g = synth.random_genome(50_000, 1)
    read, starts = synth.mutate(g[:20000], rng, err=0.15, ratio=(9, 4, 2))
    # more insertions than deletions -> read longer than the reference window
    assert 20000 * 1.02 < read.size < 20000 * 1.12
    assert starts[-1] == read.size and (np.diff(starts) >= 0).all()


def test_select_candidates_matches_oracle_and_golden(oracle):
    """ngmlr_b200_select_candidates (host glue, no GPU) == ScoreBuffer::topNSE/computeMQ."""
    import golden_util as gu
    from ngmlr_b200 import select_candidates
    from oracle_lib import score_select_cases
    gold = gu.load("score_select_golden.json")
    scs = score_select_cases(77, 400)
    start = np.zeros(len(scs) + 1, dtype=np.int64)
    start[1:] = np.cumsum([s.size for s in scs])
    order, kept, mq = select_candidates(start, np.concatenate(scs))
    for i, (sc, g) in enumerate(zip(scs, gold)):
        local = order[start[i]:start[i + 1]] - start[i]
        assert (int(kept[i]), int(mq[i])) == (g["kept"], g["mq"])
        assert gu.digest(local.astype(np.int32)) == g["order_sha"]
        o = oracle.score_select(sc)
        assert np.array_equal(local, o[0]) and (int(kept[i]), int(mq[i])) == o[1:]
    # empty batch
    o2, k2, m2 = select_candidates(np.zeros(1, np.int64), np.zeros(0, np.float32))
    assert o2.size == 0 and k2.size == 0 and m2.size == 0


def _text_stage_simple(runs, ref, ref_position, ext_qs, ext_qe):
    """Column-by-column restatement of convertCigar's bookkeeping (src/ConvexAlignFast.cpp:112-333):
    CIGAR with EQ/X merged into M, MD, NM, and the nmPerPosition triples {ref-16, read-16, errors in
    the last 32 alignment events} recorded once both positions passed 16 (addPosition :76-99)."""
    lead, trail = runs[0] >> 4, runs[-1] >> 4
    cig, md, nm_pos = [], [], []
    qstart = lead + ext_qs
    if qstart > 0:
        cig.append(f"{qstart}S")
    pos_ref, pos_read, ri = 0, lead, ref_position
    bits, level = 0, 0
    pend, md_run, matches, cols = 0, 0, 0, 0

    def note():
        if pos_read > 16 and pos_ref > 16:
            nm_pos.extend((pos_ref - 16, pos_read - 16, level))

    for r in runs[1:-1]:
        op, n = r & 15, r >> 4
        cols += n
        if op in (7, 8):
            pend += n
            for _ in range(n):
                if op == 8:
                    md.append(f"{md_run}{chr(ref[ri])}")
                    md_run = 0
                    bits = ((bits << 1) | 1) & 0xFFFFFFFF
                else:
                    md_run += 1
                    matches += 1
                    bits = (bits << 1) & 0xFFFFFFFF
                level = bin(bits).count("1")
                ri += 1
                note()
                pos_ref += 1
                pos_read += 1
        else:
            if pend:
                cig.append(f"{pend}M")
                pend = 0
            cig.append(f"{n}{'D' if op == 2 else 'I'}")
            if op == 2:
                md.append(f"{md_run}^")
                md_run = 0
            for k in range(n):
                bits = (bits << 1) & 0xFFFFFFFF
                if k == 0:
                    bits |= 1
                    level = max(level + 1, 0)
                if op == 2:
                    md.append(chr(ref[ri]))
                    ri += 1
                    note()
                    pos_ref += 1
            if op == 1:
                pos_read += n
    md.append(str(md_run))
    if pend:
        cig.append(f"{pend}M")
    qend = trail + ext_qe
    if qend > 0:
        cig.append(f"{qend}S")
    return "".join(cig), "".join(md), cols - matches, nm_pos, pos_ref, pos_read


def test_text_stage_fast_paths_equal_column_by_column_version():
    """binary_cigar_to_text writes the nmPerPosition triples of long match runs in bulk once the
    32-event error window is empty; compare with the column-by-column bookkeeping on random CIGARs
    (short and very long match runs, indel runs, leading positions below the 16-base margin)."""
    import ctypes as C
    from ngmlr_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(8)
    for case in range(300):
        runs, ref_need = [int(rng.integers(0, 40)) << 4 | 4], 0
        last = None
        for _ in range(int(rng.integers(1, 60))):
            op = int(rng.choice([7, 7, 7, 8, 1, 2]))
            if op == last:
                continue
            n = int(rng.choice([1, 2, 3, 5, 17, 31, 32, 33, 40, 100, 700])) if op == 7 else int(rng.integers(1, 6))
            runs.append(n << 4 | op)
            if op != 1:
                ref_need += n
            last = op
        runs.append(int(rng.integers(0, 30)) << 4 | 4)
        ref_position = int(rng.integers(0, 5))
        ref = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, ref_position + ref_need + 8)].tobytes()
        ext_qs, ext_qe = int(rng.integers(0, 3)), int(rng.integers(0, 3))
        arr = np.array(runs, dtype=np.int32)
        ints = (C.c_int32 * 12)()
        ident = C.c_float()
        cig, md = C.create_string_buffer(1 << 16), C.create_string_buffer(1 << 16)
        nm = np.zeros(3 * (ref_need + 8), dtype=np.int32)
        ok = lib.ngmlr_b200_debug_cigar_text(arr.ctypes.data_as(C.c_void_p), len(runs), ref, len(ref), ref_position,
                                             ext_qs, ext_qe, ints, C.byref(ident), cig, 1 << 16, md, 1 << 16,
                                             nm.ctypes.data_as(C.c_void_p), int(nm.size))
        assert ok == 1
        w_cig, w_md, w_nm, w_pos, w_lr, w_lq = _text_stage_simple(runs, ref, ref_position, ext_qs, ext_qe)
        assert cig.value.decode() == w_cig and md.value.decode() == w_md, case
        assert ints[3] == w_nm and ints[9] == w_lr and ints[10] == w_lq
        assert ints[11] * 3 == len(w_pos) and list(nm[:len(w_pos)]) == w_pos, case


def test_corridor_builders_equal_the_compiled_reference():
    """corridor.py (float32 numpy) against the reference's own getCorridorLinear / getCorridorFull /
    getCorridorEndpoints / AlignmentBuffer::getCorridorEndpointsWithAnchors / estimateCorridor
    (src/AlignmentBuffer.cpp:68-197, 1454-1467): digests of what they returned through oracle/ref_cs_shim.cpp
    (tests/golden/compiled_ref_golden.json, written by tests/golden/make_ref_golden.py)."""
    import cases
    import golden_util as gu
    gold = gu.load("compiled_ref_golden.json")["corridor"]
    cs = cases.corridor_fuzz_cases()
    assert len(gold) == len(cs)
    for c, g in zip(cs, gold):
        q, r, cor = c["q"], c["r"], c["corridor"]
        assert gu.digest(*corridor.corridor_linear(q, cor)) == g["linear"]
        assert gu.digest(*corridor.corridor_full(q, r)) == g["full"]
        for realign in (0, 1):
            eo, el = corridor.corridor_endpoints(q, r, cor, realign=bool(realign))
            assert gu.digest(eo, el) == g["endpoints"][realign], (q, r, cor, realign)
        eo, el = corridor.corridor_endpoints_with_anchors(q, r, c["ax"], c["ay"], c["multiplier"])
        assert gu.digest(eo, el) == g["anchors"], (q, r, c["anchors"], c["multiplier"])
        assert corridor.estimate_corridor(c["b"], c["d"]) == g["estimate"]


def test_corridor_builders_match_golden():
    """Always runnable: corridor.py against digests recorded from the reference's own builders."""
    import cases
    import golden_util as gu
    gold = gu.load("corridor_golden.json")
    cs = cases.corridor_cases()
    assert len(gold) == len(cs)
    for c, g in zip(cs, gold):
        assert gu.digest(*corridor.corridor_linear(c["q"], c["corridor"])) == g["linear"]
        assert gu.digest(*corridor.corridor_full(c["q"], c["r"])) == g["full"]
        assert gu.digest(*corridor.corridor_endpoints(c["q"], c["r"], c["corridor"], realign=bool(c["realign"]))) == g["endpoints"]
        ax = [a[1] - c["on_ref_start"] for a in c["anchors"]]
        ay = [c["full_len"] - a[0] - 256 - c["ext_qstart"] if a[2] else a[0] - c["ext_qstart"] for a in c["anchors"]]
        assert gu.digest(*corridor.corridor_endpoints_with_anchors(c["q"], c["r"], ax, ay, c["multiplier"])) == g["anchors"]


def test_split_read_follows_splitRead():
    from ngmlr_b200 import split_read
    s = bytes(range(256)) * 3 + b"ACGT" * 10
    parts = split_read(s)
    assert len(parts) == 3 and all(len(p) == 256 for p in parts) and b"".join(parts) == s[:768]
    assert split_read(b"ACGT" * 10) == [b"ACGT" * 10]          # shorter than one part: one sub-read
    assert split_read(b"A" * 256) == [b"A" * 256] and len(split_read(b"A" * 511)) == 1


def _binary_runs_from_text(cigar, md, ext_qs, ext_qe):
    """Rebuild the reference's binary CIGAR (len << 4 | op; EQ 7, X 8, I 1, D 2, S 4; leading and
    trailing clip entries always present) from CIGAR + MD text."""
    import re
    ops = [(int(n), o) for n, o in re.findall(r"(\d+)([MIDS])", cigar)]
    lead = ops.pop(0)[0] - ext_qs if ops and ops[0][1] == "S" else -ext_qs
    trail = ops.pop()[0] - ext_qe if ops and ops[-1][1] == "S" else -ext_qe
    # MD: numbers = matches, letters = mismatches, ^letters = deletions
    md_items = re.findall(r"(\d+)|(\^[A-Za-z]+)|([A-Za-z])", md)
    seq = []          # per aligned reference base of M/D: 'E' match, 'X' mismatch, 'D' deleted
    for num, dele, mis in md_items:
        if num:
            seq.extend("E" * int(num))
        elif dele:
            seq.extend("D" * (len(dele) - 1))
        else:
            seq.append("X")
    runs, si = [max(lead, 0) << 4 | 4], 0
    for n, o in ops:
        if o == "M":
            k = 0
            while k < n:
                kind = seq[si + k]
                j = k
                while j < n and seq[si + j] == kind:
                    j += 1
                runs.append((j - k) << 4 | (7 if kind == "E" else 8))
                k = j
            si += n
        elif o == "D":
            assert all(c == "D" for c in seq[si:si + n])
            runs.append(n << 4 | 2)
            si += n
        else:
            runs.append(n << 4 | 1)
    runs.append(max(trail, 0) << 4 | 4)
    return runs


def test_text_stage_equals_oracle_on_real_alignments(oracle):
    """The product's CIGAR/MD/NM/nmPerPosition stage (binary_cigar_to_text, via its host-only debug
    hook) on the alignments the oracle finds: same text and same nmPerPosition triples as the oracle's
    convertCigar restatement (which is pinned against the reference)."""
    import ctypes as C
    import cases
    from ngmlr_b200 import _lib
    lib = _lib.load()
    n_checked = 0
    for p in cases.random_problems(40, 515, max_len=1500):
        w = oracle.single_align(p.ref, p.qry, p.offsets, p.lengths, p.ext_qstart, p.ext_qend)
        if w["ret"] < 0 or w["status"]:
            continue
        runs = _binary_runs_from_text(w["cigar"], w["md"], p.ext_qstart, p.ext_qend)
        arr = np.array(runs, dtype=np.int32)
        ints = (C.c_int32 * 12)()
        ident = C.c_float()
        cap = 8 * (len(p.qry) + len(p.ref)) + 64
        cig, md = C.create_string_buffer(cap), C.create_string_buffer(cap)
        nm = np.zeros(3 * (2 * (len(p.qry) + 1) + len(p.ref)), dtype=np.int32)
        ref = bytes(p.ref)
        ok = lib.ngmlr_b200_debug_cigar_text(arr.ctypes.data_as(C.c_void_p), len(runs), ref, len(ref),
                                             w["position_offset"], p.ext_qstart, p.ext_qend, ints, C.byref(ident),
                                             cig, cap, md, cap, nm.ctypes.data_as(C.c_void_p), int(nm.size))
        assert ok == 1
        assert cig.value.decode() == w["cigar"] and md.value.decode() == w["md"]
        assert (ints[0], ints[1], ints[2], ints[3], ints[4], ints[5]) == (
            w["ret"], w["qstart"], w["qend"], w["nm"], w["alignment_length"], w["cigar_op_count"])
        assert (ints[7], ints[8], ints[9], ints[10]) == (w["first_ref"], w["first_read"], w["last_ref"], w["last_read"])
        assert np.float32(ident.value).view(np.uint32) == np.uint32(w["identity_bits"])
        assert ints[11] == w["nm_count"]
        assert np.array_equal(nm[:3 * ints[11]].reshape(-1, 3), w["nm_positions"])
        n_checked += 1
    assert n_checked >= 15
