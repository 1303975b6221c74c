"""Writes what the tests compare with the compiled UNMODIFIED reference (oracle/_ref, built by `make -C oracle ref`
from the reference's sources) as data, so that those comparisons run everywhere:

  compiled_ref_golden.json     corridor builders, ConvexAlignFast / StrippedSW, ScoreBuffer::topNSE, the RAW-tail
                               fuzz, SequenceProvider / CompactPrefixTable / CS on the cs_cases genome, the .ngm
                               cache files, AlignmentBuffer::computeAlignment, the IAlignment.h record layout, and the
                               records the plain ngmlr binary writes for its own test fixtures
  recorded_calls.bin.xz        a sample of the real call stream of plain ngmlr (scripts/record_workload.py):
                               SingleAlign / BatchScore / SingleScore inputs with the reference's results
  ref_fixtures/<test>/plain_ngmlr.sam.gz   the SAM file of plain ngmlr on a fixture, reads with varied qualities

Inputs are regenerated from seeds by the tests; only outputs are stored.

    REF=<ngmlr source tree> python tests/golden/make_ref_golden.py
"""
import ctypes as C
import gzip
import json
import lzma
import os
import shutil
import struct
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path.insert(0, TESTS)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

import cases  # noqa: E402
import cs_cases  # noqa: E402
from golden_util import digest  # noqa: E402
from make_golden import record  # noqa: E402
from oracle_lib import DEFAULT_SCORING, CsReference, Reference, score_select_cases  # noqa: E402

PLAIN = os.path.join(ROOT, "oracle", "_ref", "ngmlr")
REC = os.path.join(ROOT, "oracle", "_ref", "ngmlr_rec")


def corridors():
    lib = C.CDLL(CsReference.PATH)
    lib.ref_estimate_corridor.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_longlong]

    def run(kind, c, arg, realign=0):
        an = c["anchors"] if kind == 3 else []
        n = len(an)
        a0 = (C.c_int * max(n, 1))(*[a[0] for a in an])
        a1 = (C.c_ulonglong * max(n, 1))(*[a[1] for a in an])
        a2 = (C.c_int * max(n, 1))(*[a[2] for a in an])
        off = np.zeros(c["q"], dtype=np.int32)
        ln = np.zeros(c["q"], dtype=np.int32)
        h = lib.ref_corridor(kind, c["q"], c["r"], arg, realign, n, a0, a1, a2, C.c_ulonglong(c["on_ref_start"]),
                             c["ext_qstart"], 256, c["full_len"], off.ctypes.data_as(C.c_void_p),
                             ln.ctypes.data_as(C.c_void_p))
        assert h == c["q"]
        return digest(off, ln)

    # getCorridorFull is called with the reference length
    return [{"linear": run(0, c, c["corridor"]), "full": run(1, c, c["r"]),
             "endpoints": [run(2, c, c["corridor"], 0), run(2, c, c["corridor"], 1)],
             "anchors": run(3, c, c["multiplier"]),
             "estimate": lib.ref_estimate_corridor(c["a"], c["a"] + c["b"], c["c"], c["c"] + c["d"])}
            for c in cases.corridor_fuzz_cases()]


def convex():
    out = {}
    for sc, seed in ((DEFAULT_SCORING, 21), (cases.WEIRD_SCORING, 22), (cases.MILD_SCORING, 23)):
        ref = Reference(sc)
        refs, qrys = cases.sw_pairs(64, seed)
        out[str(seed)] = {"records": [record(ref, p) for p in cases.random_problems(10, seed, max_len=900)],
                          "sw": [ref.ssw_score(r, q) for r, q in zip(refs, qrys)]}
        ref.close()
    return out


def score_select():
    kept, mq, order = [], [], []
    for sc in score_select_cases(5, 1500):
        if sc.size == 0:
            continue
        o, k, m = CsReference.score_select(sc)
        kept.append(k)
        mq.append(m)
        order.append(o)
    return {"kept": kept, "mq": mq, "order_sha": digest(np.concatenate(order))}


def raw_tail(cells=4e6, seed=3):
    from fuzz_raw_tail import fill_digest, problems
    engines = {}
    fills = []
    for sc, r, q, o, l, _c in problems(seed, cells):
        if sc not in engines:
            engines[sc] = Reference(scoring=sc)
        fills.append(fill_digest(engines[sc].fill(r, q, o, l, 0)))
    for e in engines.values():
        e.close()
    return {"cells": cells, "seed": seed, "fills": fills}


def whole_reference(td):
    """Everything that needs the reference's singletons initialised on the cs_cases genome (one process)."""
    from ngmlr_b200 import refindex
    from test_cs_oracle import _interval_tasks
    contigs = cs_cases.genome_contigs()
    path = os.path.join(td, "ref.fa")
    with open(path, "w") as f:
        for i, c in enumerate(contigs):
            f.write(f">c{i}\n{c.tobytes().decode()}\n")
    ref = CsReference(path)
    out = {"concat_len": ref.concat_len, "ref_starts": ref.ref_starts(), "index_sha": digest(*ref.index())}
    subs = [s for s in cs_cases.subreads(250, 17, contigs) if len(s)]
    # the table size must not matter (overflow -> retry with a larger table)
    searches = [ref.search(s, table_bits=16) for s in subs]
    assert all(ref.search(s, table_bits=8) == w for s, w in zip(subs, searches))
    out["search"] = [[digest(np.array([x[0] for x in w], np.float32), np.array([x[1] for x in w], np.uint64),
                             np.array([x[2] for x in w], np.int32)), mh] for w, mh in searches]
    out["decode"] = [[p, None if (d := ref.decode(p)) is None else digest(d)]
                     for p in (0, 1, 999, 1000, 1001, 5555, 61000, ref.concat_len - 100, ref.concat_len - 1,
                               ref.concat_len)]
    assert ref.decode_exact(ref.concat_len, 10) is None
    out["decode_exact_corridor"] = [[st, ln, c, digest(ref.decode_exact(st, ln, c))]
                                    for st, ln, c in ((5000, 100, 12), (5001, 101, 12), (61000, 64, 40))]
    # AlignmentBuffer::computeAlignment
    lib = ref.lib
    enc = refindex.encode_reference(contigs)
    comp = []
    for t in _interval_tasks(contigs, enc):
        n = len(t.anchors)
        a0 = (C.c_int * max(n, 1))(*[a[0] for a in t.anchors])
        a1 = (C.c_ulonglong * max(n, 1))(*[a[1] for a in t.anchors])
        a2 = (C.c_int * max(n, 1))(*[a[2] for a in t.anchors])
        ints = (C.c_int * 12)()
        fl = (C.c_float * 2)()
        cap = 8 * len(t.read_seq) + 64
        cig, md = C.create_string_buffer(cap), C.create_string_buffer(cap)
        ok = lib.ref_compute_alignment(C.c_ulonglong(t.on_ref_start), C.c_ulonglong(t.on_ref_stop), n, a0, a1, a2,
                                       t.corridor, t.read_seq, t.ext_qstart, t.ext_qend, t.full_read_length,
                                       int(t.realign), int(t.full_alignment), int(t.short_read), ints, fl,
                                       cig, cap, md, cap, None, 0)
        comp.append(None if not ok else {
            "cigar_sha": digest(cig.value), "md_sha": digest(md.value),
            "qstart": ints[1], "qend": ints[2], "nm": ints[3], "alignment_length": ints[4],
            "cigar_op_count": ints[5], "position_offset": ints[11],
            "score_bits": int(np.float32(fl[0]).view(np.uint32)), "identity_bits": int(np.float32(fl[1]).view(np.uint32))})
    out["compute_alignment"] = comp
    return out


def cache_files(td):
    """The .ngm files the reference writes for the cs_cases genome (contig names with a description)."""
    contigs = cs_cases.genome_contigs()
    fasta = os.path.join(td, "cache.fa")
    with open(fasta, "w") as f:
        for i, c in enumerate(contigs):
            f.write(f">contig{i} some description\n{c.tobytes().decode()}\n")
    code = ("import ctypes, sys; lib = ctypes.CDLL(sys.argv[1]); "
            "sys.exit(lib.ref_cs_init_save(sys.argv[2].encode()))")
    subprocess.run([sys.executable, "-c", code, CsReference.PATH, fasta], check=True, capture_output=True)
    from ngmlr_b200 import ngmfiles
    enc = open(fasta + "-enc.2.ngm", "rb").read()
    _ref, names = ngmfiles.read_encoded_reference(fasta + "-enc.2.ngm")
    defined = 24 + 128 * len(_ref.ref_start) + int(_ref.enc.size)
    return {"names": names, "enc_len": len(enc), "enc_defined_sha": digest(enc[:defined]),
            "index_sha": digest(open(fasta + "-ht-13-2.2.ngm", "rb").read())}


def abi_layout(td):
    from test_abi import PROBE
    path = os.path.join(td, "p.cpp")
    open(path, "w").write(PROBE.replace("HEADER", '"IAlignment.h"'))
    src = os.path.join(os.environ["REF"], "src")
    subprocess.run(["g++", "-std=c++11", "-w", "-I", src, "-o", os.path.join(td, "p"), path,
                    "-Wl,--unresolved-symbols=ignore-all"], check=True)
    return subprocess.run([os.path.join(td, "p")], capture_output=True, text=True, check=True).stdout


def run_plain(td, fixture, ref_name, reads_name, extra, to_fastq):
    """plain ngmlr on a fixture, started as `ngmlr` in a directory of its own: the @PG line names no path."""
    d = os.path.join(HERE, "ref_fixtures", fixture)
    wd = os.path.join(td, fixture + "_" + to_fastq.__name__)
    os.makedirs(wd)
    op = gzip.open if ref_name.endswith(".gz") else open
    with op(os.path.join(d, ref_name), "rt") as f, open(os.path.join(wd, "ref.fa"), "w") as out:
        out.write(f.read())
    to_fastq(os.path.join(d, reads_name), os.path.join(wd, "reads.fq"))
    subprocess.run(["ngmlr", "-r", "ref.fa", "-q", "reads.fq", "-o", "out.sam", "--skip-write", "--no-progress",
                    *extra], executable=PLAIN, cwd=wd, check=True, capture_output=True, timeout=900)
    return open(os.path.join(wd, "out.sam"), "rb").read()


def fixtures(td):
    """Columns 1-6 of every record of plain ngmlr on the reference's own fixtures (the checks of
    test_ref_fixtures), and the whole SAM file with varied qualities (test_sam_text)."""
    from test_ref_fixtures import FIXTURE_RUNS, _to_fastq
    from test_sam_text import SAM_FIXTURES, _fastq_with_varied_qualities
    recs = {}
    for fixture, ref_name, reads_name, extra in FIXTURE_RUNS:
        sam = run_plain(td, fixture, ref_name, reads_name, extra, _to_fastq)
        recs[fixture] = [ln.split("\t")[:6] for ln in sam.decode().splitlines() if not ln.startswith("@")]
    for fixture, ref_name, reads_name in SAM_FIXTURES:
        sam = run_plain(td, fixture, ref_name, reads_name, ("-t", "1"), _fastq_with_varied_qualities)
        with gzip.GzipFile(os.path.join(HERE, "ref_fixtures", fixture, "plain_ngmlr.sam.gz"), "wb", mtime=0) as f:
            f.write(sam)
    return recs


def recorded_calls(td, max_aligns=48, min_pairs=1000):
    """The call stream of plain ngmlr on a small SV workload, cut to its first `min_pairs` BatchScore / SingleScore
    pairs and `max_aligns` SingleAlign records: the widest corridor and the repeated calls
    first, then the shortest."""
    from replay_workload import parse
    subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "record_workload.py"), "--reads", "28",
                    "--genome-mb", "1", "--contigs", "2", "--threads", "8", "--median", "5000", "--sv", "--seed", "7",
                    "--out", td], check=True, capture_output=True, timeout=900)
    buf = open(os.path.join(td, "calls.bin"), "rb").read()
    spans, at = [], 0          # (kind, start, end) of every record
    while at + 4 <= len(buf):
        kind = struct.unpack_from("<i", buf, at)[0]
        start = at
        if kind == 1:
            h = struct.unpack_from("<15i", buf, at)
            at += 60 + h[1] + h[2] + 8 * h[3] + h[13] + h[14]
        elif kind == 2:
            cnt = struct.unpack_from("<i", buf, at + 4)[0]
            at += 8
            for _ in range(cnt):
                rl, ql, _sb = struct.unpack_from("<3i", buf, at)
                at += 12 + rl + ql
        else:
            _k, rl, ql, _rc, _sb = struct.unpack_from("<5i", buf, at)
            at += 20 + rl + ql
        spans.append((kind, start, at))
    aligns = [s for s in spans if s[0] == 1]
    parsed, _ = parse(os.path.join(td, "calls.bin"))
    width = [int(a["len"][0]) if a["h"] else 0 for a in parsed]
    seen, repeated = set(), set()
    for i, a in enumerate(parsed):
        key = (a["ref"], a["qry"])
        (repeated if key in seen else seen).add(key)
    first = sorted(range(len(parsed)), key=lambda i: (-(width[i] == max(width)),
                                                      -((parsed[i]["ref"], parsed[i]["qry"]) in repeated),
                                                      len(parsed[i]["ref"]) + len(parsed[i]["qry"])))
    keep = set(first[:max_aligns])
    out, n_pairs = [], 0
    for k, (kind, s, e) in enumerate(spans):
        if kind == 1:
            if aligns.index((kind, s, e)) in keep:
                out.append(buf[s:e])
        elif n_pairs < min_pairs and kind == 3:
            out.append(buf[s:e])
            n_pairs += 1
        elif n_pairs < min_pairs:           # a BatchScore record, cut to the pairs still wanted
            cnt = min(struct.unpack_from("<i", buf, s + 4)[0], min_pairs - n_pairs)
            at = s + 8
            for _ in range(cnt):
                rl, ql, _sb = struct.unpack_from("<3i", buf, at)
                at += 12 + rl + ql
            out.append(struct.pack("<2i", 2, cnt) + buf[s + 8:at])
            n_pairs += cnt
    with open(os.path.join(HERE, "recorded_calls.bin.xz"), "wb") as f:
        f.write(lzma.compress(b"".join(out), preset=9 | lzma.PRESET_EXTREME))


def main():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref", "REF=" + os.environ["REF"]], check=True)
    assert os.path.exists(PLAIN), "the compiled reference is needed (REF=<ngmlr source tree>)"
    td = tempfile.mkdtemp(prefix="ref_golden_")
    try:
        out = {"corridor": corridors(), "convex": convex(), "score_select": score_select(), "raw_tail": raw_tail(),
               "cache_files": cache_files(td), "abi_layout": abi_layout(td), "fixture_records": fixtures(td)}
        # the reference keeps singletons: the whole-reference section runs in a process of its own
        p = subprocess.run([sys.executable, __file__, "--whole", td], check=True, capture_output=True, text=True)
        out["whole_reference"] = json.loads(p.stdout)
        with open(os.path.join(HERE, "compiled_ref_golden.json"), "w") as f:
            json.dump(out, f, separators=(",", ":"))
        os.makedirs(os.path.join(td, "rec"))
        recorded_calls(os.path.join(td, "rec"))
    finally:
        shutil.rmtree(td, ignore_errors=True)


if __name__ == "__main__":
    if sys.argv[1:2] == ["--whole"]:
        print(json.dumps(whole_reference(sys.argv[2])))
    else:
        main()
