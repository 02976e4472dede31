"""tools/check_bench_dumps.py without a GPU: on dumps made up from the CPU reference in bench.py's layout it passes, and it
reports a single changed byte, a wrong decision and a dump of the wrong batch size."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import check_bench_dumps  # noqa: E402


def write_dumps(d, cpu, log2):
    import bench
    n = 1 << log2
    rows = bench.dump_rows(n)
    sec, msgs, pts = bench.synth_inputs(n, check_bench_dumps.SEED)
    sec, msgs, pts = sec[rows], msgs[rows], pts[rows]
    pub = cpu.genpub(sec)
    outs = {"genpub": pub, "sign": cpu.sign(sec, pub, msgs, fixed_len=64), "x25519": cpu.x25519(sec, pts), "x25519_base": cpu.x25519_base(sec),
            "verify": np.ones(len(rows), np.uint8), "e2e": np.ones(len(rows), np.uint8), "e2e_pageable": np.ones(len(rows), np.uint8),
            "e2e_1kb": (rows % 10 != 0).astype(np.uint8)}
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "rows.npy"), rows.astype(np.float64))
    for name, a in outs.items():
        np.save(os.path.join(d, name + ".npy"), a.astype(np.float32))


def test_checker_accepts_right_dumps_and_reports_wrong_ones(tmp_path, cpu):
    d = str(tmp_path / "dumps")
    write_dumps(d, cpu, 10)
    assert check_bench_dumps.check(d, 10, cpu) == []
    assert check_bench_dumps.check(d, 11, cpu)                      # another batch size: other inputs
    sign = np.load(os.path.join(d, "sign.npy"))
    sign[7, 33] = (sign[7, 33] + 1) % 256
    np.save(os.path.join(d, "sign.npy"), sign)
    errs = check_bench_dumps.check(d, 10, cpu)
    assert len(errs) == 1 and errs[0].startswith("sign: 1 of 1024 rows differ") and "[7]" in errs[0], errs
    write_dumps(d, cpu, 10)
    kb = np.load(os.path.join(d, "e2e_1kb.npy"))
    kb[20] = 1                                                       # a corrupted signature accepted
    np.save(os.path.join(d, "e2e_1kb.npy"), kb)
    errs = check_bench_dumps.check(d, 10, cpu)
    assert len(errs) == 1 and errs[0].startswith("e2e_1kb: 1 of 1024"), errs
