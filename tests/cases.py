"""Seeded alignment-problem generators shared by the CPU and GPU tests."""
import numpy as np

from ngmlr_b200 import corridor, synth

WEIRD_SCORING = (1.0, -20.0, -1.0, -1.0, -1.0, 0.15)   # SURVEY section 7: SSE path != scalar rule
MILD_SCORING = (2.0, -5.0, -3.0, -2.0, -0.5, 0.05)


def random_problems(n, seed, min_len=40, max_len=1500, modes=(0, 1, 2, 3)):
    """Mixed bag: anchored corridors, narrow corridors (forces invalid paths), full matrices,
    N runs in the reference window."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        L = int(rng.integers(min_len, max_len))
        g = synth.random_genome(max_len + 4000, int(rng.integers(1 << 30)))
        if rng.random() < 0.2:
            g[rng.integers(0, g.size, size=60)] = ord("N")
        p = synth.make_problem(g, int(rng.integers(0, 3000)), L, rng,
                               err=float(rng.choice([0.02, 0.15, 0.3])),
                               multiplier=int(rng.integers(1, 3)), reverse=bool(rng.integers(0, 2)))
        mode = int(rng.choice(modes))
        if mode == 1:
            w = int(rng.integers(5, 60))
            p.offsets = (p.offsets + (p.lengths[0] - w) // 2).astype(np.int32)
            p.lengths = np.full_like(p.lengths, w)
        elif mode == 2:
            p.offsets, p.lengths = corridor.corridor_full(len(p.qry), len(p.ref))
        elif mode == 3:
            p.offsets, p.lengths = corridor.corridor_linear(len(p.qry), int(rng.integers(20, 200)))
        p.ext_qstart = int(rng.integers(0, 50))
        p.ext_qend = int(rng.integers(0, 50))
        out.append(p)
    return out


def edge_problems():
    """Hand-built edge cases: tiny inputs, ragged per-row corridors, corridors hanging off both ends
    of the reference, rows with no cells, non-monotone offsets, single-row reads."""
    rng = np.random.default_rng(99)
    g = synth.random_genome(3000, 5)
    out = []
    base = synth.make_problem(g, 100, 400, rng, err=0.1)
    H = len(base.qry)
    # ragged lengths and jittered offsets
    p = synth.AlignProblem(base.ref, base.qry, (base.offsets + rng.integers(-3, 4, H)).astype(np.int32),
                           (base.lengths + rng.integers(-20, 20, H)).astype(np.int32))
    out.append(p)
    # corridor far left of the reference (mostly x < 0) and far right (x >= refLen)
    out.append(synth.AlignProblem(base.ref, base.qry, (base.offsets - 300).astype(np.int32), base.lengths.copy()))
    out.append(synth.AlignProblem(base.ref, base.qry, (base.offsets + 350).astype(np.int32), base.lengths.copy()))
    # some rows empty (length 0 / negative)
    ln = base.lengths.copy()
    ln[50:60] = 0
    ln[200] = -5
    out.append(synth.AlignProblem(base.ref, base.qry, base.offsets.copy(), ln))
    # non-monotone offsets (zig-zag)
    zig = (base.offsets + ((np.arange(H) % 7) * 5 - 15)).astype(np.int32)
    out.append(synth.AlignProblem(base.ref, base.qry, zig, base.lengths.copy()))
    # tiny reads: 1, 2, 31, 32, 33 rows
    for h in (1, 2, 31, 32, 33, 64, 65):
        q = base.qry[:h]
        o, l = corridor.corridor_linear(h, 40)
        out.append(synth.AlignProblem(base.ref[:80], q, o, l))
    # identical sequences (long diagonal) and completely different ones (all STOP / zero)
    o, l = corridor.corridor_linear(300, 64)
    out.append(synth.AlignProblem(base.ref[:300], base.ref[:300], o, l))
    out.append(synth.AlignProblem(b"A" * 300, b"C" * 300, o, l))
    # homopolymers: massive ties between D / I / diagonal
    out.append(synth.AlignProblem(b"A" * 300, b"A" * 280, o[:280], l[:280]))
    # width-1 and width-2 corridors
    o1 = np.arange(200, dtype=np.int32)
    out.append(synth.AlignProblem(base.ref[:220], base.ref[:200], o1, np.ones(200, np.int32)))
    out.append(synth.AlignProblem(base.ref[:220], base.ref[:200], o1, np.full(200, 2, np.int32)))
    # reference window shorter than the corridor reach, N-only read
    out.append(synth.AlignProblem(base.ref[:50], base.qry[:300], base.offsets[:300].copy(), base.lengths[:300].copy()))
    out.append(synth.AlignProblem(base.ref[:300], b"N" * 200, o[:200], l[:200]))
    # lower-case / mixed bytes compare as raw bytes
    out.append(synth.AlignProblem(base.ref[:300].lower(), base.ref[:300], o, l))
    return out


def sw_pairs(n, seed):
    """(ref window, sub-read) pairs shaped like ScoreBuffer's: 306-char window, 256-char sub-read
    (src/ScoreBuffer.cpp:110, ScoreBuffer.h:71-72), plus ragged/odd ones."""
    rng = np.random.default_rng(seed)
    g = synth.random_genome(200000, seed + 7)
    refs, qrys = [], []
    for i in range(n):
        start = int(rng.integers(100, g.size - 2000))
        kind = i % 8
        if kind < 5:
            win = g[start - 20:start - 20 + 306]
            sub, _ = synth.mutate(g[start:start + 300], rng, err=float(rng.choice([0.0, 0.1, 0.2])))
            sub = sub[:256]
        elif kind == 5:   # unrelated
            win = g[start:start + 306]
            sub = synth.random_genome(256, int(rng.integers(1 << 30)))
        elif kind == 6:   # with N and lower case
            win = g[start:start + 306].copy()
            win[rng.integers(0, 306, 10)] = ord("N")
            sub = np.frombuffer(g[start + 10:start + 266].tobytes().lower(), dtype=np.uint8)
        else:             # ragged lengths
            win = g[start:start + int(rng.integers(1, 700))]
            sub = g[start:start + int(rng.integers(1, 600))]
        refs.append(bytes(win.tobytes()))
        qrys.append(bytes(np.asarray(sub, dtype=np.uint8).tobytes()))
    return refs, qrys


def corridor_cases(seed=33, n=48):
    """Seeded parameter sets for the corridor builders (row 7): dicts with q, r, corridor, realign,
    multiplier, anchors [(onRead, onRef, isReverse)], on_ref_start, ext_qstart, full_len."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        q = int(rng.integers(1, 5000))
        r = int(max(1, q + rng.integers(-q // 3 - 1, q // 3 + 2)))
        on_ref_start = int(rng.integers(1000, 10**9))
        ext_qs = int(rng.integers(0, 50))
        full_len = q + ext_qs + int(rng.integers(0, 300))
        anchors = [(int(rng.integers(0, q + 1)) + ext_qs, on_ref_start + int(rng.integers(0, r + 1)),
                    int(rng.integers(0, 2))) for _a in range(int(rng.integers(0, 12)))]
        out.append(dict(q=q, r=r, corridor=int(rng.choice([40, 400, 1600, 3333, 8192])),
                        realign=int(rng.integers(0, 2)), multiplier=int(rng.choice([1, 1, 2, 4])),
                        anchors=anchors, on_ref_start=on_ref_start, ext_qstart=ext_qs, full_len=full_len))
    return out


def corridor_fuzz_cases(seed=21, n=60):
    """Seeded inputs of the corridor builders compared with the compiled reference (test_host_logic): dicts with
    q, r, corridor, on_ref_start, ext_qstart, full_len, anchors [(onRead, onRef, isReverse)], their (x, y) form
    ax / ay, multiplier, and the four arguments a, b, c, d of estimateCorridor(a, a + b, c, c + d)."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        q = int(rng.integers(1, 6000))
        r = int(max(1, q + rng.integers(-q // 3 - 1, q // 3 + 2)))
        cor = int(rng.choice([40, 400, 1600, 3333, 8192]))
        # anchored corridor: forward and reverse anchors (mapping to (x, y) as at src/AlignmentBuffer.cpp:149-158)
        on_ref_start = int(rng.integers(1000, 10**9))
        ext_qs = int(rng.integers(0, 50))
        full_len = q + ext_qs + int(rng.integers(0, 300))
        anchors, ax, ay = [], [], []
        for _a in range(int(rng.integers(0, 12))):
            on_read = int(rng.integers(0, q + 1)) + ext_qs
            on_ref = on_ref_start + int(rng.integers(0, r + 1))
            rev = int(rng.integers(0, 2))
            anchors.append((on_read, on_ref, rev))
            ax.append(on_ref - on_ref_start)
            ay.append(full_len - on_read - 256 - ext_qs if rev else on_read - ext_qs)
        mult = int(rng.choice([1, 1, 2, 4]))
        a, b = int(rng.integers(0, 50000)), int(rng.integers(0, 50000))
        c, d = int(rng.integers(0, 10**9)), int(rng.integers(0, 60000))
        out.append(dict(q=q, r=r, corridor=cor, on_ref_start=on_ref_start, ext_qstart=ext_qs, full_len=full_len,
                        anchors=anchors, ax=ax, ay=ay, multiplier=mult, a=a, b=b, c=c, d=d))
    return out
