#!/usr/bin/env python3
"""Checks what `bench.py --dump-outputs DIR` wrote against the CPU reference.

    python tools/check_bench_dumps.py DIR [--batch-log2 20]

bench.py times verify, sign, x25519, genpub and x25519_base on fixed synthetic inputs and dumps a fixed sample of the rows
each pass returned (DIR/rows.npy holds the row indices, DIR/<pass>.npy the rows as float32).  This script regenerates the
same inputs (bench.synth_inputs with rank 0's seed), recomputes genpub, sign, x25519 and x25519_base of the sampled rows with
the CPU reference (the compiled reference when present, else the oracle port) and compares byte for byte.  The verify
passes must accept every row (verify, e2e, e2e_pageable); the 1 KB end-to-end pass must reject exactly the rows bench.py
corrupted (every tenth).  Exit code 0 when everything matches, 1 with a list of the differences otherwise.
"""
import argparse
import os
import sys

sys.dont_write_bytecode = True              # reads the tree, writes nothing into it
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

import bench  # noqa: E402

SEED = 0x5EED0001                           # bench.run_ours: synth_inputs(n, 0x5EED0001 + rank), rank 0 dumps


def load(d, name, width):
    path = os.path.join(d, name + ".npy")
    if not os.path.exists(path):
        raise SystemExit(f"{path} is missing")
    a = np.load(path)
    if not np.array_equal(a, np.round(a)) or a.min() < 0 or a.max() > 255:
        raise SystemExit(f"{name}.npy does not hold byte values")
    a = a.astype(np.uint8)
    return a.reshape(len(a), width) if width > 1 else a.reshape(-1)


def check(d, batch_log2, cpu=None):
    """Returns a list of human-readable differences (empty when the dumps are right)."""
    if cpu is None:
        from cpu_ref import best_cpu_impl
        cpu = best_cpu_impl()
    n = 1 << batch_log2
    rows = np.load(os.path.join(d, "rows.npy"))
    if not np.array_equal(rows, np.round(rows)) or rows.min() < 0 or rows.max() >= n:
        return [f"rows.npy does not hold row indices of a batch of 2^{batch_log2}"]
    rows = rows.astype(np.int64)
    if not np.array_equal(rows, bench.dump_rows(n)):
        return [f"rows.npy is not bench.py's sample for a batch of 2^{batch_log2}"]
    sec, msgs, pts = bench.synth_inputs(n, SEED)
    sec, msgs, pts = sec[rows], msgs[rows], pts[rows]
    pub = cpu.genpub(sec)
    want = {"genpub": pub, "sign": cpu.sign(sec, pub, msgs, fixed_len=64), "x25519": cpu.x25519(sec, pts), "x25519_base": cpu.x25519_base(sec)}
    errors = []
    for name, w in want.items():
        got = load(d, name, w.shape[1])
        if got.shape != w.shape:
            errors.append(f"{name}: shape {got.shape}, expected {w.shape}")
            continue
        bad = np.nonzero((got != w).any(axis=1))[0]
        if len(bad):
            errors.append(f"{name}: {len(bad)} of {len(w)} rows differ from the CPU reference, first rows {rows[bad[:5]].tolist()}")
    for name in ("verify", "e2e", "e2e_pageable"):
        got = load(d, name, 1)
        if got.shape != rows.shape or not (got == 1).all():
            errors.append(f"{name}: {int((got != 1).sum())} of {len(got)} valid signatures not accepted")
    got = load(d, "e2e_1kb", 1)
    want_ok = (rows % 10 != 0).astype(np.uint8)                 # bench.py corrupts rows 0, 10, 20, ... of the 1 KB leg
    if got.shape != rows.shape or not (got == want_ok).all():
        errors.append(f"e2e_1kb: {int((got != want_ok).sum())} of {len(got)} decisions differ from 'reject exactly the rows = 0 (mod 10)'")
    return errors


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("dir")
    ap.add_argument("--batch-log2", type=int, default=20)
    args = ap.parse_args()
    errors = check(args.dir, args.batch_log2)
    for e in errors:
        print("MISMATCH", e)
    rows = len(np.load(os.path.join(args.dir, "rows.npy")))
    print(("FAIL" if errors else "OK") + f": {rows} rows of 2^{args.batch_log2}, genpub / sign / x25519 / x25519_base against the CPU reference, "
          "verify / e2e / e2e_pageable / e2e_1kb decisions")
    return 1 if errors else 0


if __name__ == "__main__":
    sys.exit(main())
