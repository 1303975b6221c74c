#!/usr/bin/env python
"""bench.py -- aligned Gbp/s of the convex-gap banded alignment hot path on B200.

One "step" = one pass of the hot path over one batch of synthetic PacBio-shaped reads: stage 0/2
(k-mer candidate search of every 256-bp sub-read, device-side window decode and StrippedSW scoring
of every candidate) followed by stage 4 (convex fill -> traceback -> binary CIGAR -> CIGAR/MD text of
the read's interval alignment): BASELINE.json configs[1] (synthetic 50 Mb
reference, ~8 kb reads, 15 % errors ins:del:sub 9:4:2, anchored corridor) sharded by read across
ranks (weak scaling: every rank aligns its own `--reads` reads per step; no per-step collective;
one NCCL broadcast of the reference at start-up).

  value      whole-job Gbp/s with the batch already resident in HBM (K x kernels only, CUDA events);
             the batch is dealt read by read to `--contexts` aligner contexts that run concurrently
  e2e        same metric through the public calls (B200Aligner -> C ABI) from HOST buffers:
             pack + H2D + kernels + D2H + CIGAR/MD text every step, same contexts
  roofline   fill kernel: algorithmic bytes per launch / mean launch time vs measured HBM peak
  cpu_baseline  the reference's own CPU ConvexAlignFast (oracle/_ref) or the oracle port, timed on
             this box's host cores on a bounded sample of the same workload

`--impl reference` times the CPU implementation instead (all host threads) and prints the same
line with "impl": "reference".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on (default)
    "pacbio50": dict(genome_mb=50.0, contigs=5, median=8000, err=0.15, ratio=(9, 4, 2), sv=False, hi=40000,
                     what="configs[1]: synthetic 50 Mb i.i.d. reference (5 contigs), PacBio-shaped reads (log-normal, "
                          "median 8 kb, 15% errors ins:del:sub 9:4:2, strand 50/50), one interval per read, corridor "
                          "from 256-bp anchors"),
    # configs[3] shape (reads and error model; reference size as given by --genome-mb)
    "ont": dict(genome_mb=50.0, contigs=5, median=20000, err=0.12, ratio=(1, 1, 1), sv=False, hi=100000,
                what="configs[3] shape: ONT-shaped reads (log-normal, median 20 kb, 12% errors 1:1:1), "
                     "--subread-corridor 40, one interval per read"),
    # configs[4] shape
    "sv": dict(genome_mb=50.0, contigs=5, median=8000, err=0.15, ratio=(9, 4, 2), sv=True, hi=40000,
               what="configs[4] shape: every read carries one insertion / deletion / inversion of 1-50 kb; indels up "
                    "to 3 kb inside one interval (anchor-widened corridors), longer ones as two intervals, inversions "
                    "as three (+ a full-matrix alignment of inverted segments up to 2 kb); retries with wider corridors"),
    # configs[2] shape: human-sized reference
    "3gb": dict(genome_mb=3000.0, contigs=24, median=8000, err=0.15, ratio=(9, 4, 2), sv=False, hi=40000,
                what="configs[2] shape: synthetic 3 Gb i.i.d. reference (24 contigs), PacBio-shaped reads"),
}


class Workload:
    """Reads as sequenced + the computeAlignment calls ngmlr would issue for them (ngmlr_b200.synth)."""

    def __init__(self, genome, contig_len, enc_ref, n_reads, seed, cfg):
        from ngmlr_b200 import synth
        self.genome, self.contig_len, self.enc = genome, contig_len, enc_ref
        self.reads, self.ivs = synth.simulate_reads(n_reads, genome, contig_len, seed, median=cfg["median"],
                                                    err=cfg["err"], ratio=cfg["ratio"], sv=cfg["sv"], hi=cfg["hi"])
        self.bases = sum(len(r) for r in self.reads)

    def g2c(self, pos):
        c = pos // self.contig_len
        return self.enc.ref_start[c] + (pos - c * self.contig_len)

    def tasks(self, ivs, read_map=None):
        from ngmlr_b200 import synth
        t = synth.interval_tasks(ivs, self.reads, self.g2c)
        if read_map is not None:
            for x in t:
                x.read_index = read_map[x.read_index]
        return t

    def slice(self, j, S):
        """Context j of S: reads j, j+S, ... and their intervals, read indices renumbered."""
        idx = list(range(j, len(self.reads), S))
        rmap = {r: k for k, r in enumerate(idx)}
        ivs = [iv for iv in self.ivs if iv.read in rmap]
        return [self.reads[r] for r in idx], ivs, rmap


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        import datetime
        rows = []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, f, float(f[1]), float(f[2])))
            except ValueError:
                continue
        # nvidia-smi is started ahead of the warm-up (it takes a few hundred ms to come up); only the samples taken
        # between mark_begin() and mark_end() -- the timed region -- count
        if self.t0 is not None and self.t1 is not None:
            inside = [r for r in rows if self.t0 - 0.025 <= r[0] <= self.t1 + 0.025]
            rows = inside or rows[-1:]
        sm, mx, reasons = [], [], set()
        for _ts, f, a, b in rows:
            sm.append(a)
            mx.append(b)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class CpuStage02:
    """Stage 0/2 on the CPU with the reference's own code (oracle/_ref/libngmlr_full.so: CS vote,
    DecodeRefSequence, StrippedSW), or with the oracle port when that library is absent."""

    def __init__(self, genome, n_contigs=5, prefer=None):
        n_contigs = int(n_contigs)
        if prefer is None and genome.size > 500_000_000:
            prefer = "port"   # the reference takes tens of minutes to index a human-sized FASTA; the C port builds
                              # the same index (tests/test_cs_oracle.py) in about a minute
        import ctypes as C
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib
        self.C = C
        step_c = genome.size // n_contigs
        contigs = [genome[i * step_c:(i + 1) * step_c] for i in range(n_contigs)]
        self.kind = "port"
        if prefer != "port" and oracle_lib.CsReference.available():
            try:
                fasta = f"/tmp/ngmlr_b200_bench_{os.getpid()}.fa"
                with open(fasta, "w") as f:
                    for i, c in enumerate(contigs):
                        f.write(f">c{i}\n{c.tobytes().decode()}\n")
                lib = C.CDLL(oracle_lib.CsReference.PATH)
                lib.ref_cs_init(fasta.encode())
                lib.ref_cs_probe_create.restype = C.c_void_p
                lib.ref_full_ssw_create.restype = C.c_void_p
                lib.ref_full_ssw_score.restype = C.c_float
                lib.ref_full_ssw_score.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
                self.fast = hasattr(lib, "ref_stage02_read")   # the whole per-read loop in C (no GIL between calls)
                if self.fast:
                    lib.ref_stage02_read.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int]
                self.lib = lib
                self.kind = "reference"
                os.unlink(fasta)
            except OSError:
                self.kind = "port"
        if self.kind == "port":
            self.orc = oracle_lib.CsOracle([c.tobytes() for c in contigs])
            self.ssw = oracle_lib.Oracle()

    def worker_state(self):
        if self.kind == "reference":
            return (self.C.c_void_p(self.lib.ref_cs_probe_create()), self.C.c_void_p(self.lib.ref_full_ssw_create()))
        return None

    _CPL = bytes.maketrans(b"ACGT", b"TGCA")

    def candidates(self, st, sub):
        """One sub-read through the reference's CS vote, DecodeRefSequence and StrippedSW:
        [(location, reverse, vote score, sw score)] in the reference's emission order."""
        C = self.C
        if self.kind == "port":
            sub = bytes(sub)
            cands, _ = self.orc.search(sub)
            out = []
            for (s_, loc, rev) in cands:
                w = self.orc.decode((loc - 20) % (1 << 64), 308) or b"N" * 308
                out.append((int(loc), int(rev), float(s_),
                            float(self.ssw.ssw_score(w, sub.translate(self._CPL)[::-1] if rev else sub))))
            return out
        sc = (C.c_float * 512)()
        lo = (C.c_ulonglong * 512)()
        rv = (C.c_int * 512)()
        mh = C.c_float()
        n = self.lib.ref_cs_search_p(st[0], bytes(sub), len(sub), 16, sc, lo, rv, 512, C.byref(mh))
        assert n <= 512
        out = []
        buf = C.create_string_buffer(312)
        for j in range(max(0, n)):
            if not self.lib.ref_cs_decode(C.c_ulonglong(lo[j] - 20), C.c_ulonglong(308), buf):
                buf.value = b"N" * 308
            q = bytes(sub).translate(self._CPL)[::-1] if rv[j] else bytes(sub)
            out.append((int(lo[j]), int(rv[j]), float(sc[j]), float(self.lib.ref_full_ssw_score(st[1], buf.value, q))))
        return out

    def read(self, st, qry):
        """All sub-reads of one read: vote, then score every candidate. Returns #candidates."""
        C = self.C
        if self.kind == "reference" and self.fast:
            return self.lib.ref_stage02_read(st[0], st[1], bytes(qry), len(qry), 256, 20, 308)
        n_c = 0
        for k in range(len(qry) // 256):
            sub = qry[k * 256:(k + 1) * 256]
            if self.kind == "reference":
                sc = (C.c_float * 512)()
                lo = (C.c_ulonglong * 512)()
                rv = (C.c_int * 512)()
                mh = C.c_float()
                n = self.lib.ref_cs_search_p(st[0], sub, len(sub), 16, sc, lo, rv, 512, C.byref(mh))
                buf = C.create_string_buffer(312)
                for j in range(max(0, min(n, 512))):
                    if not self.lib.ref_cs_decode(C.c_ulonglong(lo[j] - 20), C.c_ulonglong(308), buf):
                        buf.value = b"N" * 308
                    q = sub.translate(self._CPL)[::-1] if rv[j] else sub
                    self.lib.ref_full_ssw_score(st[1], buf.value, q)
                    n_c += 1
            else:
                cands, _ = self.orc.search(sub)
                for (_s, loc, rev) in cands:
                    w = self.orc.decode((loc - 20) % (1 << 64), 308) or b"N" * 308
                    self.ssw.ssw_score(w, sub.translate(self._CPL)[::-1] if rev else sub)
                    n_c += 1
        return n_c


def effective_cpus():
    """Host CPUs this process can really use: logical CPUs, limited by the affinity mask and by the
    container's CFS quota (cgroup v2 cpu.max / v1 cfs_quota_us) -- the GPU boxes expose 128 logical
    CPUs under a 16-CPU quota, and 128 busy threads there run slower than 32."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except (OSError, ValueError):
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    if quota:
        n = max(1, min(n, int(quota * 2)))   # 2 threads per quota CPU measured best for the CPU arm
    return n


def tune_malloc_for_threads():
    """The reference allocates its multi-megabyte direction matrix per SingleAlign call; with glibc's
    defaults every such allocation is an mmap/munmap pair and the threads of one process serialise on
    the kernel's address-space lock (measured here: 4 threads = 1.0x one thread). Keeping large blocks
    in per-thread arenas lets the CPU arm scale with the host threads -- the faster, fairer baseline."""
    import ctypes as C
    try:
        libc = C.CDLL("libc.so.6")
        libc.mallopt(C.c_int(-3), C.c_int(1 << 30))    # M_MMAP_THRESHOLD
        libc.mallopt(C.c_int(-1), C.c_int(1 << 30))    # M_TRIM_THRESHOLD
        libc.mallopt(C.c_int(-8), C.c_int(256))        # M_ARENA_MAX
    except OSError:
        pass


def cpu_reference_run(work_items, threads, impl, stage02=None, keep=None):
    """work_items: [(read bytes as sequenced, [AlignProblem of each interval of the read])]; every read goes
    through stage 0/2 (when stage02 is given) and every problem through SingleAlign, on `threads` host
    threads (ctypes releases the GIL). impl: 'reference' = oracle/_ref (unmodified ConvexAlignFast),
    'port' = oracle C port. keep: dict that receives {(read, k): result dict} (parity check)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    tune_malloc_for_threads()
    work = list(range(len(work_items)))
    lock = threading.Lock()
    engines = [(oracle_lib.Reference() if impl == "reference" else oracle_lib.Oracle(),
                stage02.worker_state() if stage02 else None) for _ in range(threads)]

    def worker(t):
        eng, st = engines[t]
        while True:
            with lock:
                if not work:
                    break
                i = work.pop()
            read, probs = work_items[i]
            if stage02:
                stage02.read(st, read)
            for k, p in enumerate(probs):
                r = eng.single_align(p.ref, p.qry, p.offsets, p.lengths, p.ext_qstart, p.ext_qend)
                if keep is not None:
                    keep[(i, k)] = r

    ts = [threading.Thread(target=worker, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    if impl == "reference":
        for eng, _ in engines:
            eng.close()
    return dt


def cpu_impl_kind():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    if oracle_lib.Reference.available():
        try:
            oracle_lib.Reference().close()
            return "reference"
        except OSError:
            pass
    oracle_lib.Oracle()
    return "port"


def cpu_work_items(wl, n_reads):
    """The first n_reads reads of the workload with the first-attempt SingleAlign problems of their intervals."""
    by_read = {}
    for iv in wl.ivs:
        if iv.read < n_reads:
            by_read.setdefault(iv.read, []).append(iv)
    return [(wl.reads[r], [iv.problem(wl.genome, wl.reads) for iv in by_read.get(r, [])]) for r in range(n_reads)]


def build_reference(args, cfg, rank, world, dev):
    """The synthetic genome is generated and 4-bit encoded on rank 0, then ONE NCCL broadcast of the packed
    reference (ngmlr_b200.parallel.broadcast_reference); every rank decodes the flat genome it simulates its
    reads from. The k-mer index is built on each rank's own GPU (main()). No collective per step."""
    from ngmlr_b200 import parallel, refindex, synth
    n_contigs = cfg["contigs"]
    contig_len = int(args.genome_mb * 1e6) // n_contigs
    genome = enc_ref = None
    t0 = time.perf_counter()
    if rank == 0:
        genome = synth.random_genome(contig_len * n_contigs, 1)
        enc_ref = refindex.encode_reference([genome[i * contig_len:(i + 1) * contig_len] for i in range(n_contigs)])
    if world > 1:
        enc_ref = parallel.broadcast_reference(enc_ref, src=0, device=dev)
        if rank != 0:
            genome = np.concatenate(refindex.decode_contigs(enc_ref))
    return genome, contig_len, enc_ref, time.perf_counter() - t0


def ialignment_batch_align(wl, ivs, gpu_results, steps, gpu_id):
    """The same problems pushed through the reference's plugin surface itself: CreateAlignment(gpu_id) ->
    IAlignment::BatchAlign through the vtable with host strings, CorridorLine arrays and caller-allocated
    `Align` records (ngmlr_b200_plugin_time_batch_align builds them from flat arrays and times only the
    BatchAlign calls). Full fidelity of the drop-in object: CIGAR / MD text AND the nmPerPosition array (12
    bytes per alignment column) are written into the caller's buffers by host threads. Results are verified
    against what the resident pipeline produced for the same intervals."""
    import ctypes as C
    from ngmlr_b200 import PackedBatch, _lib
    lib = _lib.load()
    lib.CreateAlignment.restype = C.c_void_p
    lib.CreateAlignment.argtypes = [C.c_int]
    lib.DeleteAlignment.argtypes = [C.c_void_p]
    i32p, i64p = C.POINTER(C.c_int32), C.POINTER(C.c_int64)
    lib.ngmlr_b200_plugin_time_batch_align.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                                       i32p, i32p, i64p, i32p, i32p, C.c_int, C.POINTER(C.c_double),
                                                       i32p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    probs = [iv.problem(wl.genome, wl.reads) for iv in ivs]
    pb = PackedBatch.from_problems(probs)
    a = lib.CreateAlignment(gpu_id)
    assert a, "CreateAlignment failed"
    n = pb.n
    rets = np.zeros(n, np.int32)
    bits = np.zeros(n, np.uint32)
    crc = np.zeros(n, np.uint32)
    sec = C.c_double(0)
    args = pb.c_args()
    lib.ngmlr_b200_plugin_time_batch_align(a, n, args[1], args[3], args[5], args[6], args[7], args[8], args[9], 1,
                                           C.byref(sec), rets.ctypes.data_as(i32p), bits.ctypes.data_as(C.POINTER(C.c_uint32)),
                                           crc.ctypes.data_as(C.POINTER(C.c_uint32)))   # warm-up (arenas, pinned buffers)
    rc = lib.ngmlr_b200_plugin_time_batch_align(a, n, args[1], args[3], args[5], args[6], args[7], args[8], args[9], steps,
                                                C.byref(sec), rets.ctypes.data_as(i32p),
                                                bits.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                crc.ctypes.data_as(C.POINTER(C.c_uint32)))
    lib.DeleteAlignment(a)
    assert rc == 0, "IAlignment::BatchAlign threw"

    def fnv(s):
        c = 2166136261
        for ch in s.encode():
            c = ((c ^ ch) * 16777619) & 0xffffffff
        return c

    checked = 0
    for i, g in enumerate(gpu_results):
        d = g.as_dict()
        if d["ret"] < 0:
            assert rets[i] < 0
            continue
        assert int(bits[i]) == d["score_bits"] and int(crc[i]) == fnv(d["cigar"] + d["md"]), \
            f"IAlignment::BatchAlign differs from the resident pipeline on interval {i}"
        checked += 1
    bases = sum(len(p.qry) for p in probs)
    return {"value": bases * steps / sec.value / 1e9, "unit": "Gbp/s", "ms_per_batch": 1e3 * sec.value / steps,
            "problems": n, "read_bases": bases, "verified_against_resident_pipeline": checked,
            "note": "CreateAlignment -> IAlignment::BatchAlign (vtable), host strings + CorridorLine[] in, caller-owned "
                    "Align buffers out incl. nmPerPosition; one aligner object, one batch in flight"}


def sam_text_run(wl, ivs, gpu_results, st02, threads, ref_sample=256):
    """SURVEY 8(f)4 beside the alignment numbers: the SAM records of the first context's slice (its reads with the
    CIGAR / MD / NM / identity the device text stage produced for them) formatted by the library's host threads
    (ngmlr_b200_sam_format), MB of SAM text per second; the unmodified SAMWriter (one thread, as one ngmlr worker
    runs it) on the first `ref_sample` reads of the same records beside it, and the two texts compared."""
    from ngmlr_b200 import samtext as st
    by_read = {}
    for iv, g in zip(ivs, gpu_results):
        if g.ret < 0:
            continue
        pos = iv.ref_start + g.PositionOffset
        by_read.setdefault(iv.read, []).append(st.Alignment(
            ref_pos=int(pos % wl.contig_len), ref_id=int(pos // wl.contig_len), reverse=bool(iv.reverse),
            score=float(g.Score), mq=60, nm=int(g.NM), identity=float(g.Identity), qstart=int(g.QStart),
            qend=int(g.QEnd), cigar=g.pBuffer1.encode() if isinstance(g.pBuffer1, str) else bytes(g.pBuffer1),
            md=g.pBuffer2.encode() if isinstance(g.pBuffer2, str) else bytes(g.pBuffer2), sv_type=int(g.svType),
            primary=len(by_read.get(iv.read, [])) == 0, cigar_ops=int(g.cigarOpCount)))
    reads = []
    for r in sorted(by_read):
        seq = bytes(wl.reads[r])
        qual = bytes((33 + (i * 7) % 41) for i in range(64)) * (len(seq) // 64 + 1)
        reads.append(st.Read(b"read_%d" % r, seq, qual[:len(seq)], by_read[r]))
    n_contigs = int(wl.genome.size // wl.contig_len)
    names = [b"c%d" % i for i in range(n_contigs)]
    packed = st.PackedReads(reads)
    text = st.sam_format(packed, names, threads=threads)
    out = {"unit": "MB/s of SAM text", "reads": len(reads), "records": sum(len(r.alignments) for r in reads),
           "bytes": len(text)}
    for label, t_ in (("value", threads), ("one_thread", 1)):
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            rc, need, _txt = st.sam_format(packed, names, threads=t_, cap=len(text))
            dt = time.perf_counter() - t0
            assert rc == 0 and need == len(text)
            best = dt if best is None else min(best, dt)
        out[label] = len(text) / best / 1e6
    out["threads"] = threads
    if st02 is not None and getattr(st02, "kind", "") == "reference":
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib
        ref = oracle_lib.SamReference(st02.lib)
        sample = reads[:ref_sample]
        pk = ref.pack(sample)
        want = ref.write(1, pk)
        t0 = time.perf_counter()
        ref.write(1, pk, cap=len(want))
        dt = time.perf_counter() - t0
        got = st.sam_format(sample, ref.names, threads=threads)
        assert got == want, "SAM text differs from the unmodified SAMWriter's"
        out["reference_writer"] = {"value": len(want) / dt / 1e6, "threads": 1, "reads": len(sample),
                                   "verified_bytes": len(want)}
    return out


def integrated_run(wl_cfg, genome, contig_len, n_contigs, enc_ref, index, n_reads, cpu_threads, gpu_threads=16):
    """The UNMODIFIED ngmlr end to end, twice on the same FASTQ: the plain binary (oracle/_ref/ngmlr, its own
    ConvexAlignFast / StrippedSW on `cpu_threads` threads) and the same objects linked with the CUDA plugin
    behind IAlignment (oracle/_ref/ngmlr_b200; every blocking SingleAlign of its `gpu_threads` worker threads
    parked in the plugin's cross-thread batcher). Both start from the SAME on-disk caches -- written here from
    the encoded reference and the k-mer index that was built on the GPU (ngmlr_b200.ngmfiles, byte-compatible
    with ngmlr's own -enc.2.ngm / -ht-13-2.2.ngm), so neither run builds an index. SAM records must be
    identical. Everything outside IAlignment (FASTQ parsing, CS vote, chaining, SV logic, SAM writing) is
    the reference's own CPU code in both runs -- the integrated ratio is bounded by it (Amdahl)."""
    import shutil
    import tempfile
    from ngmlr_b200 import ngmfiles, synth
    plain = os.path.join(ROOT, "oracle", "_ref", "ngmlr")
    swapped = os.path.join(ROOT, "oracle", "_ref", "ngmlr_b200")
    if not (os.path.exists(plain) and os.path.exists(swapped)):
        return {"unavailable": "oracle/_ref/ngmlr{,_b200} not built"}
    d = tempfile.mkdtemp(prefix="ngmlr_b200_integrated_")
    try:
        ref = os.path.join(d, "ref.fa")
        with open(ref, "w") as f:
            for c in range(n_contigs):
                s = genome[c * contig_len:(c + 1) * contig_len].tobytes().decode()
                f.write(f">c{c}\n" + "\n".join(s[k:k + 80] for k in range(0, len(s), 80)) + "\n")
        ngmfiles.c_write_encoded_reference(ref + "-enc.2.ngm", enc_ref, [f"c{c}" for c in range(n_contigs)])
        ngmfiles.c_write_index(ref + "-ht-13-2.2.ngm", index, skip=2)
        reads, _ = synth.simulate_reads(n_reads, genome, contig_len, 77, median=wl_cfg["median"], err=wl_cfg["err"],
                                        ratio=wl_cfg["ratio"], sv=wl_cfg["sv"], hi=wl_cfg["hi"])
        fq = os.path.join(d, "reads.fq")
        bases = 0
        with open(fq, "w") as f:
            for i, r in enumerate(reads):
                s = r.decode()
                bases += len(s)
                f.write(f"@r{i}\n{s}\n+\n{'I' * len(s)}\n")
        out = {"reads": n_reads, "read_bases": bases}
        sams = {}
        for name, exe, t, extra in (("cpu", plain, cpu_threads, {}),
                                    ("b200", swapped, gpu_threads, {"NGMLR_B200_BATCH_WINDOW_US": "200",
                                                                     "NGMLR_B200_BATCH_MAX": "512",
                                                                     "NGMLR_B200_BATCH_SERVERS": "2",
                                                                     "NGMLR_B200_HOST_THREADS": "4",
                                                                     "NGMLR_B200_STATS": "1"})):
            sam = os.path.join(d, name + ".sam")
            env = dict(os.environ, NGMLR_B200_LIB=os.path.join(ROOT, "ngmlr_b200", "libngmlr_b200.so"), **extra)
            import resource
            ru0 = resource.getrusage(resource.RUSAGE_CHILDREN)
            t0 = time.perf_counter()
            r = subprocess.run([exe, "-r", ref, "-q", fq, "-o", sam, "-t", str(t), "--no-progress"],
                               capture_output=True, text=True, env=env, timeout=1800)
            wall = time.perf_counter() - t0
            ru1 = resource.getrusage(resource.RUSAGE_CHILDREN)
            cpu_s = (ru1.ru_utime - ru0.ru_utime) + (ru1.ru_stime - ru0.ru_stime)
            if r.returncode != 0:
                return {"unavailable": f"{name} run failed: {r.stderr[-300:]}"}
            built = "Building reference index" in r.stderr or "Building reference index" in r.stdout
            sams[name] = sorted(ln for ln in open(sam) if not ln.startswith("@"))
            stats = [ln for ln in r.stderr.splitlines() if ln.startswith("[ngmlr_b200]")]
            out[name] = {"threads": t, "wall_s": wall, "cpu_s": cpu_s, "gbp_per_s": bases / wall / 1e9,
                         "built_its_own_index": built,
                         "env": extra, "plugin_stats": stats or None}
        out["sam_identical"] = sams["cpu"] == sams["b200"]
        out["sam_records"] = len(sams["cpu"])
        out["speedup"] = out["cpu"]["wall_s"] / out["b200"]["wall_s"]
        out["note"] = ("whole unmodified ngmlr processes incl. start-up and cache loading; caches written from the "
                       "GPU-built index (ngmfiles), identical for both")
        return out
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="pacbio50", choices=sorted(CONFIGS))
    ap.add_argument("--reads", type=int, default=8192, help="reads per step per GPU")
    ap.add_argument("--genome-mb", type=float, default=0.0, help="reference size (0 = the config's)")
    ap.add_argument("--dp-only", action="store_true", help="time stage 4 (convex alignment) alone")
    ap.add_argument("--stagger-ms", type=float, default=0.0,
                    help="device-resident leg: context j starts j x this many ms after context 0 (inside the timed region)")
    ap.add_argument("--contexts", type=int, default=4, help="aligner contexts (host threads/streams) per GPU")
    ap.add_argument("--fill-ctas", type=int, default=0,
                    help="0 (default): fill launches of short-lived CTAs on a low-priority stream; n > 0: a persistent "
                         "fill grid of n CTAs per SM per launch in the concurrent phases")
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads in the CPU baseline sample (0 = auto)")
    ap.add_argument("--parity-reads", type=int, default=0, help="reads compared CPU vs GPU (0 = the CPU sample)")
    ap.add_argument("--profile-only", action="store_true",
                    help="stop after the solo phase (one context, whole batch resident): what ncu captures")
    ap.add_argument("--integrated-only", action="store_true", help="run only the whole-ngmlr comparison")
    ap.add_argument("--integrated-threads", type=int, default=16,
                    help="worker threads of the plugin-linked ngmlr (16 = the GPU boxes' CPU quota measured best: "
                         "every thread blocks ~10 ms per SingleAlign batch, more threads only oversubscribe the CPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed device-resident path computed in its last step (the alignment of every "
                         "interval, stage 0/2 candidates and scores) to DIR/<name>.npy, at most 64 MB in all")
    ap.add_argument("--integrated-reads", type=int, default=-1,
                    help="reads of the whole-ngmlr comparison (plain binary vs plugin-linked binary); "
                         "-1 = 2000 at N=1 on configs up to 100 Mb, else 0 (skipped)")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    cfg = CONFIGS[args.config]
    if args.genome_mb <= 0:
        args.genome_mb = cfg["genome_mb"]
    workload_name = cfg["what"] + f"; reference {args.genome_mb:g} Mb"

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = effective_cpus()
    os.environ.setdefault("NGMLR_B200_HOST_THREADS",
                          str(max(2, min(16, (os.cpu_count() or 1) // max(1, world * max(1, args.contexts))))))

    from ngmlr_b200 import synth

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        from ngmlr_b200 import refindex
        kind = cpu_impl_kind()
        n_genome = int(args.genome_mb * 1e6)
        contig_len = n_genome // cfg["contigs"]
        genome = synth.random_genome(contig_len * cfg["contigs"], 1)
        threads = cores
        # bounded sample: ~8 reads per thread per step (dynamic scheduling evens out the read lengths)
        n = args.cpu_sample or max(threads, min(args.reads, 8 * threads))
        wl = Workload(genome, contig_len, None, n, 2, cfg)
        items = cpu_work_items(wl, n)
        bases = wl.bases
        cells = sum(p.cells for _r, ps in items for p in ps)
        st02 = None if args.dp_only else CpuStage02(genome, cfg["contigs"])
        for _ in range(max(1, min(args.warmup, 1))):   # grows the per-thread malloc arenas, warms the caches
            cpu_reference_run(items, threads, kind, st02)
        times = [cpu_reference_run(items, threads, kind, st02) for _ in range(args.steps)]
        t = float(np.sum(times))
        val = bases * args.steps / t / 1e9
        line = {"metric": "aligned_gbp_per_s", "value": val, "unit": "Gbp/s", "impl": "reference",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": val / 5.56e-4, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_name, "reads_per_step": n, "read_bases_per_step": bases,
                           "dp_cells_per_step": cells},
                "cpu_baseline": {"value": val, "unit": "Gbp/s", "cores": threads, "kind": kind,
                                 "sample": f"{n} reads ({bases} bases, {cells} DP cells) per step, {threads} threads "
                                           f"(= usable CPUs: {os.cpu_count()} logical, container quota applied), "
                                           + ("ConvexAlignFast::SingleAlign only" if args.dp_only else
                                              f"CS vote + DecodeRefSequence + StrippedSW ({st02.kind}) then ConvexAlignFast::SingleAlign"),
                                 "mcells_per_s_per_core": cells * args.steps / t / threads / 1e6},
                "e2e": {"value": val, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py --impl b200 needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    genome, contig_len, enc_ref, t_ref = build_reference(args, cfg, rank, world, dev)

    from ngmlr_b200 import B200Aligner, IntervalBatch, PackedReads
    if args.integrated_only:
        a0 = B200Aligner(local_rank)
        a0.set_reference(enc_ref)
        a0.build_index(enc_ref)
        print(json.dumps(integrated_run(cfg, genome, contig_len, cfg["contigs"], enc_ref, a0.get_index(),
                                        max(args.integrated_reads, 500), cores, args.integrated_threads)))
        a0.close()
        return
    wl = Workload(genome, contig_len, enc_ref, args.reads, 2 + rank, cfg)   # reads sharded by rank: own reads per rank
    bases = wl.bases
    all_reads = PackedReads(wl.reads)
    all_ivs = IntervalBatch(wl.tasks(wl.ivs))
    # S independent aligner contexts (own stream, own device arenas), driven by S host threads --
    # the reference's model of one aligner object per worker thread. The step's batch is dealt to the
    # contexts read by read (context j takes reads j, j+S, ...); their work overlaps on the GPU, which
    # hides the tail of each fill launch and the traceback behind another context's fill, and (end to
    # end) the host side of one slice behind the kernels of the others.
    S = max(1, args.contexts)
    streams = [torch.cuda.Stream(device=dev, priority=-1) for _ in range(S)]  # outrank the fill launches
    als = [B200Aligner(local_rank, stream=st_.cuda_stream) for st_ in streams]
    al = als[0]
    # one copy of the encoded reference per GPU; the k-mer index is built from it ON the device
    # (CompactPrefixTable::CreateTable as kernels) and shared by the GPU's contexts
    al.set_reference(enc_ref)
    t_idx0 = time.perf_counter()
    n_positions = al.build_index(enc_ref)
    t_index = time.perf_counter() - t_idx0
    for a_ in als[1:]:
        a_.share_reference(al)
    sl_reads, sl_ivs, sl_bases = [], [], []
    for j in range(S):
        r_, iv_, rmap = wl.slice(j, S)
        sl_reads.append(PackedReads(r_))
        sl_ivs.append(IntervalBatch(wl.tasks(iv_, rmap)))
        sl_bases.append(sum(len(x) for x in r_))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def run_threads(fn):
        ts = [threading.Thread(target=fn, args=(j,)) for j in range(S)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()

    # ---- (a) one context alone on the whole batch: per-kernel durations for the roofline (the fill
    # kernel timed in isolation, inputs resident) ----
    n_sub = al.reads_upload(all_reads)
    al.intervals_upload(all_ivs)
    for _ in range(args.warmup):
        if not args.dp_only:
            al.cs_run()
        al.run()
    barrier()
    fill_ms, tb_ms, tx_ms, cs_ms = [], [], [], []
    n_cand = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(streams[0])
    for _ in range(args.steps):
        n_cand, ms_ = (0, 0.0) if args.dp_only else al.cs_run()
        cs_ms.append(ms_)
        al.run()
        st = al.stats()
        fill_ms.append(st["fill_ms"])
        tb_ms.append(st["traceback_ms"])
        tx_ms.append(st["text_ms"])
    e1.record(streams[0])
    torch.cuda.synchronize(dev)
    solo_ms = e0.elapsed_time(e1)
    if args.profile_only:
        print(json.dumps({"profile_only": True, "fill_ms": float(np.mean(fill_ms)), "traceback_ms": float(np.mean(tb_ms)),
                          "text_ms": float(np.mean(tx_ms)), "stage02_ms": float(np.mean(cs_ms)), "solo_ms_per_step":
                          solo_ms / args.steps}))
        return
    gpu_first = al.fetch()                 # first-attempt alignments of every interval (parity check below)
    st = al.stats()
    cells = st["cells"]
    gpu_first = [gpu_first[i] for i in range(len(gpu_first))]
    gpu_cs = None if args.dp_only else al.cs_fetch()
    n_first_valid = sum(1 for r, iv in zip(gpu_first, wl.ivs) if r.ret == len(wl.reads[iv.read]))

    # ---- (b) device-resident timed region: every context keeps its slice in HBM, exactly K steps ----
    # By default the fill launches are short-lived CTAs on a low-priority stream, so the latency-bound kernels of
    # the S contexts (candidate search, traceback, text) and the copies' bookkeeping kernels slip in between;
    # --fill-ctas n selects a persistent fill grid of n CTAs per SM per launch instead.
    for a_ in als:
        a_.set_fill_ctas_per_sm(args.fill_ctas if S > 1 else 0)

    def resident_warm(j):
        als[j].reads_upload(sl_reads[j])
        als[j].intervals_upload(sl_ivs[j])
        for _ in range(args.warmup):
            if not args.dp_only:
                als[j].cs_run()
            als[j].run()

    sampler = ClockSampler(local_rank)
    sampler.start()
    run_threads(resident_warm)
    barrier()
    sampler.mark_begin()
    cur = torch.cuda.current_stream(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    for st_ in streams:
        st_.wait_event(e0)
    ends = [torch.cuda.Event() for _ in range(S)]

    def dev_worker(j):
        if args.stagger_ms > 0:
            time.sleep(j * args.stagger_ms * 1e-3)
        for _ in range(args.steps):
            if not args.dp_only:
                als[j].cs_run()
            als[j].run()
        ends[j].record(streams[j])

    run_threads(dev_worker)
    for j in range(S):
        cur.wait_event(ends[j])
    e1.record(cur)
    barrier()
    sampler.mark_end()
    clocks = sampler.stop()
    dev_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, als, args.dp_only)

    # ---- (c) end to end from host buffers through the public calls: per step every context uploads its
    # reads ONCE (reads_upload), runs stage 0/2 on their sub-reads and brings candidates + scores back
    # (cs_run, cs_fetch), then computeAlignment for its intervals (compute_alignments: windows by position,
    # corridors in closed form, read parts by index; retries inside the call) -> CIGAR / MD / NM / regions on
    # the host. ----
    io = [dict(h2d=0, d2h=0, attempts=0, invalid=0) for _ in range(S)]

    def e2e_steps(j, k):
        a_ = als[j]
        for _ in range(k):
            a_.reads_upload(sl_reads[j])
            h2d = a_.reads_h2d_bytes()
            d2h = 0
            if not args.dp_only:
                m_, _ms = a_.cs_run()
                cstart, _sc, _lo, _rv, sw_, _mx = a_.cs_fetch()   # candidates + scores -> host
                assert m_ == cstart[-1] and sw_.size == m_
                d2h += 17 * int(m_) + 12 * (len(cstart) - 1)
            out, att = a_.compute_alignments(sl_ivs[j])
            cst = a_.compute_alignments_stats()
            h2d += cst["h2d_bytes"]
            d2h += cst["d2h_bytes"]
            bad = sum(1 for i in range(len(out)) if out.ret(i) < 0)
            io[j].update(h2d=h2d, d2h=d2h, attempts=int(att.sum()), invalid=bad, n=len(out),
                         host_ms={k_: cst[k_] for k_ in ("host_pack_ms", "host_h2d_ms", "host_run_ms", "host_d2h_ms",
                                                         "host_text_ms")})
            del out

    run_threads(lambda j: e2e_steps(j, 1))
    barrier()
    t0 = time.perf_counter()
    run_threads(lambda j: e2e_steps(j, args.steps))
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    e2e_h2d = sum(x["h2d"] for x in io)
    e2e_d2h = sum(x["d2h"] for x in io)
    n_invalid = sum(x["invalid"] for x in io)
    assert n_invalid <= max(2, len(wl.ivs) // 200), f"bench: {n_invalid} of {len(wl.ivs)} intervals without an alignment"

    t_dev = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(bases), float(cells)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    dev_ms, e2e_ms = (float(x) for x in t_dev.cpu())
    tot_bases, tot_cells = (float(x) for x in tot.cpu())

    if rank == 0:
        value = tot_bases * args.steps / (dev_ms * 1e-3) / 1e9
        e2e_val = tot_bases * args.steps / (e2e_ms * 1e-3) / 1e9
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst)" if peaks else "fallback 6650 GB/s"
        # algorithmic bytes of ONE fill launch (DESIGN.md section 4): 0.25 B per DP cell (2-bit direction) +
        # sequences read once; corridor rows are generated on the device from 28-byte closed forms
        seq_b = sum(iv.ref_len + iv.read_len for iv in wl.ivs)
        algo_bytes = cells * 0.25 + seq_b + 112 * len(wl.ivs)
        fill_s = float(np.mean(fill_ms)) * 1e-3
        achieved = algo_bytes / fill_s / 1e9
        sm_mhz = float(clocks.get("sm_mhz") or 1965.0)
        # SURVEY section 8(d): 148 SMs x 128 lanes x clock / >= 25 instructions per cell
        issue_bound = 148 * 128 * sm_mhz * 1e6 / 25.0
        traffic = None
        alu_ops = lane_instr = None
        try:  # DRAM bytes of one fill launch from the committed ncu capture (same workload only)
            tr = json.load(open(os.path.join(ROOT, "profiles", "fill_traffic.json")))
            if tr.get("reads_per_step") == args.reads and tr.get("config", "pacbio50") == args.config:
                traffic = tr["dram_bytes_per_launch"]
            alu_ops = tr.get("alu_pipe_lane_ops_per_cell")   # a property of the kernel's code, not of the batch
            lane_instr = tr.get("lane_instructions_per_cell")
        except Exception:
            pass
        # the pipe that binds (DESIGN.md 4.1): compares / selects / min-max run on the ALU pipe only, 16 lanes per
        # clock and SM sub-partition; ops per cell from the same ncu capture
        alu_bound = 148 * 4 * 16 * sm_mhz * 1e6 / alu_ops if alu_ops else None
        # what the kernel's own instruction count allows at one warp-instruction per clock and sub-partition (the
        # final build issues 67.4 lane-instructions per useful cell incl. block ramp and chunk hand-off)
        own_issue_bound = 148 * 128 * sm_mhz * 1e6 / lane_instr if lane_instr else None
        line = {
            "metric": "aligned_gbp_per_s", "value": value, "unit": "Gbp/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": e2e_val / 5.56e-4,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name, "config": args.config, "reads_per_step_per_gpu": args.reads,
                       "intervals_per_step_per_gpu": len(wl.ivs),
                       "read_bases_per_step": tot_bases, "dp_cells_per_step": tot_cells,
                       "parallelism": f"read-sharded x{world}, no per-step collective; {S} aligner contexts/GPU, "
                                      + (f"persistent fill grid {args.fill_ctas} CTAs/SM per launch" if args.fill_ctas
                                         else "fill = short-lived CTAs on a low-priority stream"),
                       "l2": "inputs+direction arena per step exceed L2 (direction writes alone "
                             f"{st['dir_bytes'] / 1e6:.0f} MB/step/GPU)",
                       "vs_baseline_note": "e2e (host buffers in, CIGAR/MD text out) / README.md:25 whole-pipeline "
                                           "5.56e-4 Gbp/s on 10 Opteron cores; the same-box CPU arm is cpu_baseline / "
                                           "--impl reference"},
            "reads_per_s": args.reads * world * args.steps / (dev_ms * 1e-3),
            "gcells_per_s": tot_cells * args.steps / (dev_ms * 1e-3) / 1e9,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel": "convex_fill_kernel", "launch_ms": fill_s * 1e3,
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "gcells_per_s_kernel": cells / fill_s / 1e9,
                         "issue_bound_gcells_per_s": issue_bound / 1e9,
                         "frac_of_issue_bound": cells / fill_s / issue_bound,
                         "alu_pipe_bound_gcells_per_s": alu_bound / 1e9 if alu_bound else None,
                         "frac_of_alu_pipe_bound": cells / fill_s / alu_bound if alu_bound else None,
                         "own_instruction_count_bound_gcells_per_s": own_issue_bound / 1e9 if own_issue_bound else None,
                         "frac_of_own_instruction_count_bound": cells / fill_s / own_issue_bound if own_issue_bound else None,
                         "note": "integer/float DP: instruction-issue bound (SURVEY 8(d): 148 SMs x 128 lanes x clock / "
                                 "25 instructions per cell), not HBM bound; the HBM fraction is structurally ~0.02. The "
                                 "kernel issues 67.4 lane-instructions per useful cell (ncu, profiles/fill_traffic.json): "
                                 "issue slots 85 % busy, ALU pipe 67 %"},
            "kernel_ms_per_step": {"fill": float(np.mean(fill_ms)), "traceback": float(np.mean(tb_ms)),
                                   "text": float(np.mean(tx_ms)),
                                   "stage02_cs_vote_decode_score": float(np.mean(cs_ms))},
            "stage02": {"subreads_per_step_per_gpu": n_sub, "candidates_per_step_per_gpu": int(n_cand),
                        "sw_cell_updates_per_step_per_gpu": int(n_cand) * 257 * 307,
                        "reference_setup_s": t_ref, "index_build_on_device_s": t_index,
                        "index_build_kernels_ms": al.index_build_ms, "index_positions": int(n_positions)},
            "e2e": {"value": e2e_val, "unit": "Gbp/s", "h2d_bytes_per_step": e2e_h2d,
                    "d2h_bytes_per_step": e2e_d2h, "ms_per_step": e2e_ms / args.steps,
                    "host_ms_per_slice_first_attempt": {k: float(np.mean([x["host_ms"][k] for x in io]))
                                                        for k in io[0].get("host_ms", {})},
                    "singlealign_calls_per_step": sum(x["attempts"] for x in io),
                    "intervals_without_alignment": n_invalid,
                    "note": f"reads_upload -> cs_run -> cs_fetch -> compute_alignments per context and step; each of the "
                            f"{S} contexts takes every {S}-th read"},
            "solo": {"gbp_per_s": bases * args.steps / (solo_ms * 1e-3) / 1e9, "ms_per_step": solo_ms / args.steps,
                     "first_attempt_valid": n_first_valid, "intervals": len(wl.ivs),
                     "note": "one context alone on the whole batch, same K steps (kernels not overlapped)"},
            # per context and step: cs count, sizes, 4 x (scan init + scan), vote, count widening, compaction,
            # window decode + score (14) + fill, traceback, text (3)
            "gpu_launches": (3 if args.dp_only else 17) * S * args.steps,
            "clocks": clocks,
        }
        # CPU baseline on this box's host cores, bounded sample of the same workload -- and the parity check:
        # the CPU arm's alignments, candidates and scores against what the GPU produced for the same reads
        try:
            kind = cpu_impl_kind()
            threads = cores
            n = args.cpu_sample or max(threads, min(len(wl.reads), 8 * threads))
            items = cpu_work_items(wl, n)
            st02 = None if args.dp_only else CpuStage02(genome, cfg["contigs"])
            cpu_reference_run(items, threads, kind, st02)   # warm-up: per-thread malloc arenas, caches
            keep = {}
            t = cpu_reference_run(items, threads, kind, st02, keep=keep)
            sb = sum(len(r) for r, _ in items)
            sc = sum(p.cells for _r, ps in items for p in ps)
            line["cpu_baseline"] = {"value": sb / t / 1e9, "unit": "Gbp/s", "cores": threads, "kind": kind,
                                    "sample": f"first {n} reads of the batch ({sb} bases, {sc} DP cells), "
                                              f"{threads} threads, {t:.1f} s, stages: "
                                              + ("4 only" if st02 is None else f"0/2 ({st02.kind}) + 4"),
                                    "mcells_per_s_per_core": sc / t / threads / 1e6}
            line["parity_checked"] = parity_check(wl, keep, gpu_first, gpu_cs, st02,
                                                  args.parity_reads or min(n, 64))
        except AssertionError:
            raise
        except Exception as ex:  # the baseline is reported, never required for the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "Gbp/s", "cores": 0, "kind": "unavailable",
                                    "sample": repr(ex)}
        try:   # the plugin surface itself, on the first context's slice of the batch
            k_ = len(wl.ivs) if len(wl.ivs) <= 2048 else 2048
            line["e2e_ialignment"] = ialignment_batch_align(wl, wl.ivs[:k_], gpu_first[:k_], max(2, args.steps // 2),
                                                            local_rank)
        except AssertionError:
            raise
        except Exception as ex:
            line["e2e_ialignment"] = {"value": None, "note": repr(ex)}
        if world == 1:   # SURVEY 8(f)4: the SAM text of the batch's records
            try:
                line["sam_text"] = sam_text_run(wl, wl.ivs, gpu_first, locals().get("st02"), cores)
            except AssertionError:
                raise
            except Exception as ex:
                line["sam_text"] = {"value": None, "note": repr(ex)}
        n_int = args.integrated_reads
        if n_int < 0:
            n_int = 2000 if (world == 1 and args.genome_mb <= 100 and not args.dp_only) else 0
        if n_int > 0:
            try:
                line["integrated"] = integrated_run(cfg, genome, contig_len, cfg["contigs"], enc_ref, al.get_index(),
                                                    n_int, cores, args.integrated_threads)
            except Exception as ex:
                line["integrated"] = {"unavailable": repr(ex)}
        print(json.dumps(line))
    for a_ in als:
        a_.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = (64 << 20) - (1 << 16)   # 64 MB less room for the .npy headers
ALIGN_FIELDS = ("ret", "Score", "Identity", "PositionOffset", "QStart", "QEnd", "NM", "alignmentLength", "cigarOpCount",
                "svType")


def dump_outputs(out_dir, als, dp_only):
    """What a caller of the timed path receives after its last step, as float32 / float64 .npy files: every context's
    alignments (fetch; one row per interval, contexts in order, CIGAR and MD text as CRC-32 and length) and stage 0/2
    results (cs_fetch: per sub-read candidate ranges and best score, per candidate vote score, location, strand and
    StrippedSW score). Per-candidate arrays that would exceed 64 MB in all are cut to a fixed, seeded sample of
    candidates, whose indices are written as cs_sample.npy."""
    import zlib
    os.makedirs(out_dir, exist_ok=True)
    al = {k: [] for k in ALIGN_FIELDS + ("first_position", "last_position", "cigar_crc32", "cigar_len", "md_crc32",
                                         "md_len")}
    cs = {k: [] for k in ("cs_start", "cs_max_score", "cs_vote_score", "cs_location", "cs_reverse", "cs_sw_score")}
    base = 0
    for a_ in als:
        for r in a_.fetch():
            for k in ALIGN_FIELDS:
                al[k].append(getattr(r, k))
            al["first_position"].append(r.firstPosition)
            al["last_position"].append(r.lastPosition)
            for k, t in (("cigar", r.pBuffer1), ("md", r.pBuffer2)):
                b = t.encode() if isinstance(t, str) else bytes(t)
                al[k + "_crc32"].append(zlib.crc32(b))
                al[k + "_len"].append(len(b))
        if not dp_only:
            start, sc, lo, rv, sw, mx = a_.cs_fetch()
            cs["cs_start"].append(start[:-1] + base)
            base += int(start[-1])
            for k, v in (("cs_max_score", mx), ("cs_vote_score", sc), ("cs_location", lo), ("cs_reverse", rv),
                         ("cs_sw_score", sw)):
                cs[k].append(v)
    arrays = {"align_" + k: np.asarray(v, dtype=np.float32 if k in ("Score", "Identity") else np.float64)
              for k, v in al.items()}
    if not dp_only:
        cs = {k: np.concatenate(v) for k, v in cs.items()}
        cs["cs_start"] = np.append(cs["cs_start"], base)
        for k in ("cs_start", "cs_location"):
            arrays[k] = cs[k].astype(np.float64)
        for k in ("cs_max_score", "cs_vote_score", "cs_reverse", "cs_sw_score"):
            arrays[k] = cs[k].astype(np.float32)
        per_cand = ("cs_vote_score", "cs_location", "cs_reverse", "cs_sw_score")
        fixed = sum(v.nbytes for k, v in arrays.items() if k not in per_cand)
        row = sum(arrays[k].itemsize for k in per_cand)
        keep = max(0, (DUMP_BYTES - fixed) // (row + 8))
        if base > keep:
            idx = np.sort(np.random.default_rng(0).choice(base, size=keep, replace=False))
            for k in per_cand:
                arrays[k] = arrays[k][idx]
            arrays["cs_sample"] = idx.astype(np.float64)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def parity_check(wl, cpu_aligned, gpu_first, gpu_cs, st02, n_stage02_reads):
    """The CPU arm's outputs (the reference's own code where oracle/_ref exists) against the GPU's for the
    same reads, outside every timed region. Stage 4: every interval of the CPU sample -- score bits, CIGAR,
    MD, NM, positions. Stage 0/2: the candidate lists (order, location, strand, vote score) and StrippedSW
    scores of every sub-read of the first reads. A mismatch fails the run."""
    by_read = {}
    for gi, iv in enumerate(wl.ivs):
        by_read.setdefault(iv.read, []).append(gi)
    n_al = 0
    for (r, k), want in cpu_aligned.items():
        g = gpu_first[by_read[r][k]].as_dict()
        if want["ret"] < 0 or g["ret"] < 0:   # no alignment: the reference leaves the other fields undefined
            assert want["ret"] < 0 and g["ret"] < 0, f"parity: read {r} interval {k}: ret cpu {want['ret']} gpu {g['ret']}"
            n_al += 1
            continue
        for key in ("ret", "score_bits", "cigar", "md", "nm", "position_offset", "qstart", "qend", "alignment_length"):
            assert want[key] == g[key], f"parity: read {r} interval {k}: {key} differs (cpu {want[key]!r:.80} gpu {g[key]!r:.80})"
        n_al += 1
    out = {"alignments": n_al, "fields": "ret, score bits, CIGAR, MD, NM, PositionOffset, QStart, QEnd, alignmentLength"}
    if gpu_cs is not None and st02 is not None:
        cstart, cs_sc, cs_lo, cs_rv, cs_sw, _mx = gpu_cs
        s = 0   # global sub-read index
        n_sub = n_c = 0
        wstate = st02.worker_state()
        for r in range(len(wl.reads)):
            read = wl.reads[r]
            parts = max(1, len(read) // 256)
            if r < n_stage02_reads and len(read) >= 256:
                for k in range(parts):
                    want = st02.candidates(wstate, read[k * 256:(k + 1) * 256])
                    a, b = int(cstart[s + k]), int(cstart[s + k + 1])
                    got = [(int(cs_lo[j]), int(cs_rv[j]), float(cs_sc[j]), float(cs_sw[j])) for j in range(a, b)]
                    assert want == got, f"parity: read {r} sub-read {k}: candidates differ (cpu {want[:3]} gpu {got[:3]})"
                    n_sub += 1
                    n_c += len(want)
            s += parts
        out.update(subreads=n_sub, candidates=n_c,
                   stage02_fields="candidate order, location, strand, vote score, StrippedSW score")
    return out


if __name__ == "__main__":
    main()
