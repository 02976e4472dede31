"""Throughput of the three verify acceptance rules (REFERENCE, STRICT, ZIP215) on one GPU, through the device API.

    python tools/bench_verify_policy.py [--n 1048576] [--rounds 5] [--out FILE]

2^20 honest signatures over 64-byte messages (signed on the GPU) are verified by ed25519_verify_policy_batch_dev; after a
warm-up of every rule, the rules alternate in one process for --rounds rounds, so that clock and neighbour drift hit them
alike.  A sample is --reps back-to-back calls timed with CUDA events; every call must accept every signature.
Prints one JSON line: M verify/s per rule (median and every round), the card, its power limit and SM clocks read in the same
run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, limit, sm, sm_max = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit_w": float(limit), "sm_mhz": float(sm), "sm_max_mhz": float(sm_max)}
    except Exception as e:                            # the numbers are still measured; the card's details are then missing
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5, help="calls per timed sample")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import libeddsa_b200 as ed
    assert torch.cuda.is_available(), "needs a CUDA device"
    n = args.n
    rng = np.random.default_rng(2026)
    sec = torch.from_numpy(rng.integers(0, 256, (n, 32), dtype=np.uint8)).cuda()
    msgs = torch.from_numpy(rng.integers(0, 256, (n, 64), dtype=np.uint8)).cuda()
    pub = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    sig = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    ed.ed25519_genpub_batch_dev(pub, sec)
    ed.ed25519_sign_batch_dev(sig, sec, pub, msgs, None, 64)
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    rules = {"reference": ed.VERIFY_REFERENCE, "strict": ed.VERIFY_STRICT, "zip215": ed.VERIFY_ZIP215}

    def run(policy):
        ok.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            ed.ed25519_verify_policy_batch_dev(ok, sig, pub, msgs, None, 64, policy)
        b.record()
        b.synchronize()
        assert int(ok.sum()) == n, "a rule rejected an honest signature"
        return args.reps * n / (a.elapsed_time(b) * 1e-3) / 1e6

    for p in rules.values():                          # warm-up: module load, pool growth, tables
        run(p)
        run(p)
    before = card()
    rates = {k: [] for k in rules}
    for _ in range(args.rounds):
        for k, p in rules.items():
            rates[k].append(run(p))
    res = {"n": n, "rounds": args.rounds, "m_verify_per_s": {k: round(statistics.median(v), 3) for k, v in rates.items()},
           "all_rounds": {k: [round(x, 3) for x in v] for k, v in rates.items()},
           "vs_reference": {k: round(statistics.median(v) / statistics.median(rates["reference"]) - 1, 4) for k, v in rates.items()},
           "card_before": before, "card_after": card()}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
