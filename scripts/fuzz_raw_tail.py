#!/usr/bin/env python
"""Targeted fuzz of the one corner the CUDA RAW fill does not replay literally (DESIGN.md section 2): the
reference's SSE blocks first compute EVERY cell of a row -- including its last <= 12 columns -- and feed those
values to the best-cell tracking (src/ConvexAlignFast.cpp:1165-1170); the scalar tail then recomputes the last
<= 12 columns with the scalar rule and tracks again (:1179, :1270-1275). The oracle's rule 2 / the RAW kernel
track only the final value of every cell. A difference needs a scoring outside the default class (where SSE and
scalar values of a cell can differ at all) AND a tail cell whose SSE value beats every cell seen so far while
its final value does not.

Compares the COMPILED REFERENCE's fill (oracle/_ref/libngmlr_ref.so: directions, best score bits, best cell)
with the oracle's rule 2 on inputs built to hit the corner: corridors 13-48 columns wide (a third to all of every
row is "tail"), scorings with cheap gap opens / expensive mismatches, short periodic sequences that tie a lot.
Prints the number of cells and mismatches; exits non-zero on any mismatch."""
import argparse
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SCORINGS = [(1.0, -20.0, -1.0, -1.0, -1.0, 0.15), (2.0, -8.0, -1.0, -2.0, -0.5, 0.3), (1.0, -3.0, -0.5, -0.5, -0.25, 0.05),
            (3.0, -30.0, -2.0, -1.0, -1.0, 0.0), (1.0, -1.0, -1.0, -1.0, -1.0, 0.15), (2.0, -5.0, -5.0, -5.0, -1.0, 0.15)]


def problems(seed, max_cells):
    """The seeded fuzz inputs: (scoring, ref, qry, offsets, lengths, cells), 200 per scoring in turn, until
    `max_cells` cells are reached."""
    from ngmlr_b200 import corridor, synth
    rng = np.random.default_rng(seed)
    cells = 0
    n = 0
    while cells < max_cells:
        sc = SCORINGS[n % len(SCORINGS)]
        for _ in range(200):
            H = int(rng.integers(20, 400))
            W = int(rng.integers(13, 49))
            kind = int(rng.integers(0, 3))
            if kind == 0:      # periodic: many equal-score paths
                unit = synth.random_genome(int(rng.integers(1, 5)), int(rng.integers(1 << 30)))
                r = np.tile(unit, H + 80)[:H + 60]
            else:
                r = synth.random_genome(H + 60, int(rng.integers(1 << 30)))
            q, _ = synth.mutate(r[10:10 + H], rng, err=float(rng.choice([0.05, 0.2, 0.4])))
            q = q[:H] if q.size >= H else np.concatenate([q, r[:H - q.size]])
            shift = int(rng.integers(-5, 15))
            o, l = corridor.corridor_linear(len(q), W)
            o = (o + 10 + shift).astype(np.int32)
            c = int(np.maximum(np.minimum(o + l, len(r)) - np.maximum(o, 0), 0).sum())
            cells += c
            yield sc, r.tobytes(), q.tobytes(), o, l, c
        n += 1


def fill_digest(res):
    """Directions, best score bits and best cell of one fill, as stored by --golden files."""
    dirs, bs, bx, by = res
    h = hashlib.sha256(np.ascontiguousarray(dirs).tobytes())
    h.update(np.array([np.float32(bs).view(np.uint32), bx, by], dtype=np.int64).tobytes())
    return h.hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=float, default=1.2e8)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--golden", default=None,
                    help="JSON file with the reference's fill digests for --cells / --seed (tests/golden/"
                         "compiled_ref_golden.json, section raw_tail): compare with those instead of the compiled "
                         "reference")
    args = ap.parse_args()
    from oracle_lib import Oracle, Reference
    orc = Oracle()
    golden = None
    if args.golden:
        import json
        golden = json.load(open(args.golden))["raw_tail"]
        assert golden["cells"] == args.cells and golden["seed"] == args.seed, "golden file is for another run"
        golden = golden["fills"]
    engines = {}
    cells = 0
    bad = 0
    n = 0
    per_scoring = {}
    n_scalar_probe = n_scalar_differs = 0
    for sc, r, q, o, l, c in problems(args.seed, args.cells):
        if golden is not None:
            want = golden[n]
        else:
            if sc not in engines:
                engines[sc] = Reference(scoring=sc)
            want = fill_digest(engines[sc].fill(r, q, o, l, 0))
        b = orc.fill(r, q, o, l, sc, 2)
        if n_scalar_probe < 3000:   # how often does this input separate the SSE semantics from the scalar rule at all?
            n_scalar_probe += 1
            n_scalar_differs += fill_digest(orc.fill(r, q, o, l, sc, 1)) != want
        cells += c
        per_scoring[sc] = per_scoring.get(sc, 0) + c
        if fill_digest(b) != want:
            bad += 1
            print("MISMATCH", sc, len(q), int(l[0]), b[1:], file=sys.stderr)
        n += 1
    for e in engines.values():
        e.close()
    if golden is not None:
        assert n == len(golden), "golden file is for another run"
    print(f"{n_scalar_differs} of the first {n_scalar_probe} problems separate the as-coded SSE semantics from the pure "
          f"scalar rule (the fuzz is not vacuous)")
    print(f"cells {cells} problems {n} mismatches {bad}; cells per scoring: "
          + ", ".join(f"{k}: {v}" for k, v in per_scoring.items()))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
