"""The reference's own test fixtures (test/data/test_2, test_4, test_5, test_6 with their expected
files, copied as data to tests/golden/ref_fixtures/; the checks of test/test_*.sh restated without
samtools / bedtools): BASELINE.json configs[0] verbatim.
  * CPU: what the unmodified reference binary (oracle/_ref/ngmlr) wrote for them (stored) reproduces
    expected.bed / expected.txt -- which validates the restated checks themselves;
  * GPU (-m gpu): the same binary with its aligners swapped for the CUDA plugin (oracle/_ref/ngmlr_b200)
    passes the same checks and writes the same SAM records as the plain binary.
FASTA reads are converted to FASTQ (constant quality 'I'): the reference overflows a 2-byte quality buffer
on reverse-strand FASTA reads (src/SAMWriter.cpp:104-108, BASELINE.md)."""
import gzip
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "ref_fixtures")
PLAIN = os.path.join(ROOT, "oracle", "_ref", "ngmlr")
SWAPPED = os.path.join(ROOT, "oracle", "_ref", "ngmlr_b200")


def _open(path):
    return gzip.open(path, "rt") if path.endswith(".gz") else open(path)


def _to_fastq(fa, fq):
    name, seq = None, []
    with _open(fa) as f, open(fq, "w") as out:
        def flush():
            if name is not None:
                s = "".join(seq)
                out.write(f"@{name}\n{s}\n+\n{'I' * len(s)}\n")
        for line in f:
            line = line.rstrip("\n")
            if line.startswith(">"):
                flush()
                name, seq = line[1:], []
            else:
                seq.append(line.strip())
        flush()


def _plain_ref(src, dst):
    with _open(src) as f, open(dst, "w") as out:
        out.write(f.read())


def _run(exe, tmp, test, ref_name, reads_name, extra=(), fasta_reads=False):
    d = os.path.join(FIX, test)
    ref = os.path.join(tmp, f"{test}_ref.fa")
    fq = os.path.join(tmp, f"{test}_reads.fq")
    _plain_ref(os.path.join(d, ref_name), ref)
    if fasta_reads:   # test_1 checks the FASTA parser's handling of long read names
        fq = os.path.join(d, reads_name)
    else:
        _to_fastq(os.path.join(d, reads_name), fq)
    sam = os.path.join(tmp, f"{test}_{os.path.basename(exe)}.sam")
    env = dict(os.environ, NGMLR_B200_LIB=os.path.join(ROOT, "ngmlr_b200", "libngmlr_b200.so"))
    r = subprocess.run([exe, "-r", ref, "-q", fq, "-o", sam, "--skip-write", "--no-progress", *extra],
                       capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln.rstrip("\n").split("\t") for ln in open(sam) if not ln.startswith("@")]


def _bed(records):
    """samtools view -Sb | bedtools bamtobed: chrom, start, end (reference span of the CIGAR), name, MAPQ, strand."""
    out = []
    for f in records:
        flag = int(f[1])
        if flag & 4:
            continue
        span = sum(int(n) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", f[5]) if op in "MDN=X")
        out.append("\t".join([f[2], str(int(f[3]) - 1), str(int(f[3]) - 1 + span), f[0], f[4],
                              "-" if flag & 16 else "+"]))
    return out


# (fixture, reference, reads, options) of the checks of test/test_*.sh.
# (test_1 -- read names longer than the parser's limit -- is not reproduced by the reference's own HEAD,
# which cuts names at 250 characters where expected.txt still holds 277; it concerns the FASTA parser only)
FIXTURE_RUNS = [("test_2", "ref_chr21_20kb.fa", "reads_100_2200bp.fa", ()),
                ("test_4", "reference.fasta.gz", "read.fa.gz", ("-x", "pacbio", "-t", "4")),
                ("test_5", "reference.fasta.gz", "read.fa.gz", ("-x", "pacbio", "-t", "4")),
                ("test_6", "reference.fasta.gz", "read.fa.gz", ("-x", "pacbio", "-t", "4"))]


def _checks(records):
    """records: fixture -> SAM records (lists of columns) of one binary on it."""
    # test_2: simple read lengths -> expected.bed
    assert _bed(records["test_2"]) == open(os.path.join(FIX, "test_2", "expected.bed")).read().splitlines()
    # test_4: primary alignment, columns 1-5 sorted
    got = sorted("\t".join(r[:5]) for r in records["test_4"])
    assert got == open(os.path.join(FIX, "test_4", "expected.txt")).read().splitlines()
    # test_5: max query name length (<= 254 characters of names); test_6: five reads -> five records
    assert sum(len(r[0]) + 1 for r in records["test_5"]) <= 254
    assert len(records["test_6"]) == 5   # samtools view -Sc


def _run_all(exe, tmp):
    return {t: _run(exe, tmp, t, ref, reads, extra) for t, ref, reads, extra in FIXTURE_RUNS}


def test_plain_reference_passes_its_own_fixture_checks():
    """Columns 1-6 of what plain ngmlr wrote for the fixtures (tests/golden/compiled_ref_golden.json, written by
    tests/golden/make_ref_golden.py) pass the restated checks."""
    import golden_util as gu
    _checks(gu.load("compiled_ref_golden.json")["fixture_records"])


@pytest.mark.gpu
@pytest.mark.skipif(not (os.path.exists(PLAIN) and os.path.exists(SWAPPED)), reason="oracle/_ref binaries not built")
def test_plugin_linked_ngmlr_passes_the_reference_fixture_checks(tmp_path):
    a = _run_all(SWAPPED, str(tmp_path))
    b = _run_all(PLAIN, str(tmp_path))
    _checks(a)
    _checks(b)
    for k in a:
        assert sorted(map(tuple, a[k])) == sorted(map(tuple, b[k])), k   # every SAM column, every record
