"""SURVEY 8(f)4: the SAM text entry points (csrc/sam_text.cpp) against the unmodified reference writer.
CPU tests: the library's record formatter needs no device."""
import hashlib
import os
import subprocess
import sys

import pytest

import golden_util as gu
import sam_cases
from ngmlr_b200 import samtext as st

HERE = os.path.dirname(os.path.abspath(__file__))
FULL = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libngmlr_full.so")
GOLD = gu.load("sam_golden.json")
NAMES = [n.encode() for n in GOLD["ref_names"]]


def _ours(name, **kw):
    opts = dict(sam_cases.CONFIGS)[name]
    return st.sam_format(sam_cases.config_reads(name), NAMES, write_unmapped=opts["write_unmapped"],
                         bam_cigar_fix=opts["bam_cigar_fix"], rg_id=opts["rg_id"], **kw)


@pytest.mark.parametrize("name", [c[0] for c in sam_cases.CONFIGS])
def test_records_equal_the_reference_writers_golden_output(name):
    g = GOLD["configs"][name]
    text = _ours(name)
    lines = text.split(b"\n")[:-1]
    assert len(lines) == len(g["lines"])
    for i, (l, d) in enumerate(zip(lines, g["lines"])):
        assert hashlib.sha256(l).hexdigest()[:16] == d, f"{name}: line {i} differs: {l[:200]!r}"
    assert len(text) == g["bytes"] and hashlib.sha256(text).hexdigest() == g["sha256"]


@pytest.mark.parametrize("name", [c[0] for c in sam_cases.CONFIGS])
def test_header_equals_the_reference_prolog(name):
    sys.path.insert(0, os.path.join(HERE, "golden"))
    from make_sam_golden import CMDLINE, RG_FIELDS
    opts = dict(sam_cases.CONFIGS)[name]
    got = st.sam_header(NAMES, GOLD["ref_lens"], b"0.2.8", CMDLINE, rg_id=opts["rg_id"],
                        rg_fields=RG_FIELDS if opts["rg_id"] else None)
    assert got.decode() == GOLD["configs"][name]["header"]


@pytest.mark.skipif(not os.path.exists(FULL), reason="oracle/_ref/libngmlr_full.so not built")
@pytest.mark.parametrize("name", [c[0] for c in sam_cases.CONFIGS])
def test_records_equal_the_live_reference_writer(name):
    # the reference keeps singletons (SequenceProvider, Config): its writer runs in a process of its own
    p = subprocess.run([sys.executable, os.path.join(HERE, "golden", "make_sam_golden.py"), "--dump", name],
                       capture_output=True, check=True)
    want = p.stdout
    got = _ours(name)
    assert got == want


def test_output_does_not_depend_on_the_thread_count():
    one = _ours("default", threads=1)
    for t in (2, 3, 7, 32):
        assert _ours("default", threads=t) == one
    many = sam_cases.make_reads(5, n_reads=1500)
    assert st.sam_format(many, NAMES, threads=1) == st.sam_format(many, NAMES, threads=16)


def test_small_buffer_reports_the_size_and_writes_nothing():
    reads = sam_cases.config_reads("default")
    full = st.sam_format(reads, NAMES)
    rc, need, text = st.sam_format(reads, NAMES, cap=len(full) - 1)
    assert (rc, need, text) == (-2, len(full), b"")
    rc, need, text = st.sam_format(reads, NAMES, cap=len(full))
    assert rc == 0 and text == full
    assert st.sam_format([], NAMES) == b""


def _aln(reverse, **kw):
    d = dict(ref_pos=9, ref_id=0, reverse=reverse, score=10.0, mq=60, nm=0, identity=1.0, qstart=0, qend=0,
             cigar=b"4M", md=b"4")
    d.update(kw)
    return st.Alignment(**d)


def _quals(text):
    return [l.split(b"\t")[10] for l in text.split(b"\n")[:-1]]


def test_quality_orientation_as_coded_and_fixed():
    # src/SAMWriter.cpp:104-108 reverses the read's quality string in place for every reverse-strand record
    r = st.Read(b"q", b"ACGT", b"1234", [_aln(True), _aln(True), _aln(False), _aln(True)])
    assert _quals(st.sam_format([r], NAMES)) == [b"4321", b"1234", b"1234", b"4321"]
    assert _quals(st.sam_format([r], NAMES, fix_quality_orientation=True)) == [b"4321", b"4321", b"1234", b"4321"]
    seqs = [l.split(b"\t")[9] for l in st.sam_format([r], NAMES).split(b"\n")[:-1]]
    assert seqs == [b"ACGT", b"ACGT", b"ACGT", b"ACGT"]     # its own reverse complement
    r2 = st.Read(b"q", b"AACGN", b"12345", [_aln(True, cigar=b"5M", md=b"5")])
    assert st.sam_format([r2], NAMES).split(b"\t")[9:11] == [b"NCGTT", b"54321"]


def test_fasta_quality_is_never_reversed():
    # the reference reverses `length` bytes of the 2-byte "*" buffer here (undefined behaviour); a "*" stays a "*"
    r = st.Read(b"fa", b"ACGTT", b"*", [_aln(True, cigar=b"5M", md=b"5"), _aln(False, cigar=b"5M", md=b"5")])
    assert _quals(st.sam_format([r], NAMES)) == [b"*", b"*"]


def test_positions_are_truncated_as_the_reference_prints_them():
    # `m_Location + 1` is 64 bit, printed with %u in the POS column and with %d in SA:Z
    a = _aln(False, ref_pos=2**32 + 5)
    b = _aln(False, ref_pos=2**31 + 7, primary=False)
    lines = st.sam_format([st.Read(b"p", b"ACGT", None, [a, b])], NAMES).split(b"\n")
    assert lines[0].split(b"\t")[3] == b"6" and lines[1].split(b"\t")[3] == b"%d" % (2**31 + 8)
    assert b"SA:Z:" + NAMES[0] + b",%d,+,4M,60,0;" % (2**31 + 8 - 2**32) in lines[0]
    assert lines[1].split(b"\t")[1] == b"2048"


# ---- real records: the SAM file the unmodified ngmlr writes for its own fixtures, re-created from its fields -----
PLAIN = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "ngmlr")
FIX = os.path.join(HERE, "golden", "ref_fixtures")


def _fastq_with_varied_qualities(fa, fq):
    import gzip
    op = gzip.open if fa.endswith(".gz") else open
    reads, name, seq = {}, None, []
    with op(fa, "rt") as f:
        for line in list(f) + [">"]:
            line = line.rstrip("\n")
            if line.startswith(">"):
                if name is not None:
                    # the parser's normalisation (src/IParser.h:66-76): upper case, everything but ACGT becomes N
                    s = "".join(c if c in "ACGT" else "N" for c in "".join(seq).upper())
                    reads[name.split()[0][:249]] = (s, "".join(chr(35 + (i * 7 + len(s)) % 38) for i in range(len(s))))
                name, seq = line[1:], []
            else:
                seq.append(line.strip())
    with open(fq, "w") as out:
        for n, (s, q) in reads.items():
            out.write(f"@{n}\n{s}\n+\n{q}\n")
    return reads


def _rc(s):
    return s[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA"))


# (fixture, reference, reads) of the stored SAM files: plain ngmlr, one thread, reads with the qualities of
# _fastq_with_varied_qualities (tests/golden/ref_fixtures/<fixture>/plain_ngmlr.sam.gz, written by
# tests/golden/make_ref_golden.py)
SAM_FIXTURES = [("test_2", "ref_chr21_20kb.fa", "reads_100_2200bp.fa"), ("test_6", "reference.fasta.gz", "read.fa.gz")]


@pytest.mark.parametrize("test,ref_name,reads_name", SAM_FIXTURES)
def test_sam_file_of_the_unmodified_ngmlr_is_recreated_from_its_fields(tmp_path, test, ref_name, reads_name):
    import gzip
    import re
    d = os.path.join(FIX, test)
    fastq = _fastq_with_varied_qualities(os.path.join(d, reads_name), str(tmp_path / "reads.fq"))
    with gzip.open(os.path.join(d, "plain_ngmlr.sam.gz"), "rb") as f:
        raw = f.read()
    header = b"".join(l + b"\n" for l in raw.split(b"\n") if l.startswith(b"@"))
    body = raw[len(header):]
    # header fields
    names, lens, version, cmdline = [], [], None, None
    for l in header.split(b"\n"):
        f = l.split(b"\t")
        if f[0] == b"@SQ":
            names.append(f[1][3:])
            lens.append(int(f[2][3:]))
        elif f[0] == b"@PG":
            version = f[3][3:]
            cmdline = l.split(b"\tCL:", 1)[1]
    assert st.sam_header(names, lens, version, cmdline) == header
    # records -> reads (the records of a read are consecutive, in alignment order)
    reads, by_name = [], {}
    for l in body.split(b"\n")[:-1]:
        f = l.split(b"\t")
        name = f[0].decode()
        seq, qual = fastq[name]
        if name not in by_name:
            by_name[name] = st.Read(f[0], seq.encode(), qual.encode(), [])
            reads.append(by_name[name])
        flag = int(f[1])
        if flag & 4:
            continue
        tags = {t[:2]: t[5:] for t in f[11:]}
        length = len(seq)
        qs = int(tags[b"QS"])
        qe = length - int(tags[b"QE"])
        assert length - qs - qe == int(tags[b"XR"])
        assert f[9] == (_rc(seq.encode()) if flag & 16 else seq.encode())
        by_name[name].alignments.append(st.Alignment(
            ref_pos=int(f[3]) - 1, ref_id=names.index(f[2]), reverse=bool(flag & 16), score=float(tags[b"AS"]),
            mq=int(f[4]), nm=int(tags[b"NM"]), identity=float(tags[b"XI"]), qstart=qs, qend=qe, cigar=f[5],
            md=tags[b"MD"], sv_type=int(tags.get(b"SV", b"-1")), primary=not (flag & 0x800),
            cigar_ops=len(re.findall(rb"\d+[A-Z=]", f[5]))))
    assert sum(len(r.alignments) for r in reads) > 0
    got = st.sam_format(reads, names)
    assert got == body


# ---- the whole unmodified ngmlr with its SAMWriter replaced by the library at link time (oracle/swap_samwriter.cpp) ---
SAM_SWAPPED = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "ngmlr_sam")
LIBRARY = os.path.join(os.path.dirname(HERE), "ngmlr_b200", "libngmlr_b200.so")


def _run_ngmlr(exe, ref, fq, sam, threads):
    env = dict(os.environ, NGMLR_B200_LIB=LIBRARY)
    r = subprocess.run([exe, "-r", ref, "-q", fq, "-o", sam, "--skip-write", "--no-progress", "-t", str(threads)],
                       capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    return open(sam, "rb").read()


@pytest.mark.skipif(not (os.path.exists(PLAIN) and os.path.exists(SAM_SWAPPED)),
                    reason="oracle/_ref/ngmlr and ngmlr_sam not built")
@pytest.mark.parametrize("test,ref_name,reads_name,threads", [
    ("test_2", "ref_chr21_20kb.fa", "reads_100_2200bp.fa", 1), ("test_4", "reference.fasta.gz", "read.fa.gz", 4)])
def test_ngmlr_linked_with_the_library_writer_writes_the_same_sam_file(tmp_path, test, ref_name, reads_name, threads):
    """Plain ngmlr (its own aligners, CPU) with SAMWriter's member functions replaced by forwarders to
    ngmlr_b200_sam_header / ngmlr_b200_sam_format: the same file (one thread), the same records (several)."""
    import gzip
    d = os.path.join(FIX, test)
    ref = str(tmp_path / "ref.fa")
    op = gzip.open if ref_name.endswith(".gz") else open
    with op(os.path.join(d, ref_name), "rt") as f, open(ref, "w") as out:
        out.write(f.read())
    fq = str(tmp_path / "reads.fq")
    _fastq_with_varied_qualities(os.path.join(d, reads_name), fq)
    want = _run_ngmlr(PLAIN, ref, fq, str(tmp_path / "plain.sam"), threads)
    got = _run_ngmlr(SAM_SWAPPED, ref, fq, str(tmp_path / "plain.sam"), threads)   # same -o: same @PG command line ...
    want = want.replace(PLAIN.encode(), b"EXE")
    got = got.replace(SAM_SWAPPED.encode(), b"EXE")                                    # ... up to the binary's name
    assert got.count(b"\n") > 5
    if threads == 1:
        assert got == want
    else:
        assert sorted(got.split(b"\n")) == sorted(want.split(b"\n"))
