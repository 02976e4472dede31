"""Throughput of batched ZIP215 verification against per-signature ZIP215 on one GPU, through the device API.

    python tools/bench_verify_batched.py [--n 1048576] [--rounds 5] [--out FILE]

2^20 signatures over 64-byte messages (signed on the GPU), in three workloads:
  honest       every row valid
  invalid_0.1% 0.1 % of the rows at random positions have a corrupted message (their batch equations fail and the
               rows of those groups are re-checked one by one)
  adversarial  one invalid row in every group of VERIFY_BATCH_ROWS rows, so every row is re-checked
For each workload, ed25519_verify_zip215_batched_dev (fixed seed) and ed25519_verify_policy_batch_dev(VERIFY_ZIP215)
alternate for --rounds rounds after a warm-up, so that clock and neighbour drift hit them alike.  A sample is --reps
back-to-back calls timed with CUDA events; every batched output must equal the per-signature output.  The working set
(2^20 records of 2.4 KB) is far larger than L2.  Prints one JSON line with M verify/s (median and every round) and the
card, its power limit and SM clocks read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_verify_policy import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5, help="calls per timed sample")
    ap.add_argument("--workloads", default="honest,invalid_0.1%,adversarial")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import libeddsa_b200 as ed
    assert torch.cuda.is_available(), "needs a CUDA device"
    n, K = args.n, ed.VERIFY_BATCH_ROWS
    rng = np.random.default_rng(2026)
    sec = torch.from_numpy(rng.integers(0, 256, (n, 32), dtype=np.uint8)).cuda()
    msgs = torch.from_numpy(rng.integers(0, 256, (n, 64), dtype=np.uint8)).cuda()
    pub = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    sig = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    ed.ed25519_genpub_batch_dev(pub, sec)
    ed.ed25519_sign_batch_dev(sig, sec, pub, msgs, None, 64)
    seed = bytes(range(32))
    rows = np.arange(n)
    bad = {"honest": np.zeros(0, np.int64),
           "invalid_0.1%": rng.choice(n, n // 1000, replace=False),
           # within a pass, lane l of warp w holds rows 32 K w + l + 32 r: rows with r = 0 put one invalid row in every group
           "adversarial": rows[(rows % (32 * K)) < 32]}
    ok_b = torch.zeros(n, dtype=torch.uint8, device="cuda")
    ok_z = torch.zeros(n, dtype=torch.uint8, device="cuda")

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            fn()
        b.record()
        b.synchronize()
        return args.reps * n / (a.elapsed_time(b) * 1e-3) / 1e6

    res = {"n": n, "batch_rows": K, "rounds": args.rounds, "workloads": {}}
    before = card()
    for wl in args.workloads.split(","):
        m = msgs.clone()
        if len(bad[wl]):
            idx = torch.from_numpy(bad[wl]).cuda()
            m[idx, 0] ^= 1
        batched = lambda: ed.ed25519_verify_zip215_batched_dev(ok_b, sig, pub, m, None, 64, seed)          # noqa: E731
        single = lambda: ed.ed25519_verify_policy_batch_dev(ok_z, sig, pub, m, None, 64, ed.VERIFY_ZIP215)  # noqa: E731
        for f in (batched, single, batched, single):     # warm-up: module load, pool growth, tables
            f()
        torch.cuda.synchronize()
        assert torch.equal(ok_b, ok_z), f"{wl}: batched output differs from per-signature ZIP215"
        assert int(ok_z.sum()) == n - len(bad[wl]), f"{wl}: unexpected accept count"
        rb, rz = [], []
        for _ in range(args.rounds):
            rb.append(timed(batched))
            rz.append(timed(single))
        assert torch.equal(ok_b, ok_z)
        mb, mz = statistics.median(rb), statistics.median(rz)
        res["workloads"][wl] = {"invalid_rows": int(len(bad[wl])), "m_verify_per_s": {"batched": round(mb, 3), "zip215": round(mz, 3)},
                                "batched_over_zip215": round(mb / mz, 4),
                                "all_rounds": {"batched": [round(x, 3) for x in rb], "zip215": [round(x, 3) for x in rz]}}
    res["card_before"], res["card_after"] = before, card()
    res["library"] = ed.LIB_PATH if os.environ.get("LIBEDDSA_B200_SO") else "default"
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
