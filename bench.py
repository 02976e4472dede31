#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200-native Ed25519 / X25519 batch engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch-log2 20] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): Ed25519 verify/s, sign/s & X25519 ops/s, batch 2^20 per GPU.
A "step" is one pass of the hot path over one synthetic batch: 2^20 independent Ed25519
verifications of (pubkey, 64-byte message, signature) triples — BASELINE config 1's workload —
resident in HBM.  The same protocol is then repeated for sign, x25519, genpub and x25519_base and
reported under "also" (each with its own integer-multiply roofline fraction).

  value     device-timed (CUDA events on the launching stream) whole-job ops/s, inputs resident in HBM
  e2e       same metric through the public host-buffer C-ABI (ed25519_verify_batch) from pinned host
            memory: H2D of sig/pub/msg and D2H of the accept flags inside the timed region
  roofline  compute-bound on the 32x32->64 integer multiplier (IMAD.WIDE, fmaheavy pipe); peak measured
            on this pool's B200s (profiles/r01_pipe_microbench.md): 32 wide multiplies/clk/SM.  "frac" counts the
            field work the engine EXECUTES (half-size scalars: ~133 k wide multiplies per signature),
            "frac_reference_fm" the field work the reference's algorithm would need (232 k) at our rate —
            that one can exceed 1 because the algorithm, not the pipe, got faster
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, kind "reference"; oracle port otherwise) on the
            box's host cores, one instance per core, bounded sample of the same workload
One process per GPU; batches are sharded by rank (no collective on the data path); the timed region
is bracketed by barrier + synchronize and the max over ranks is reported.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "Ed25519 verify/s (batch 2^20 per GPU, 64 B messages); sign/s and X25519 ops/s under 'also'"
UNIT = "ops/s"

# ---- integer-multiply roofline model (DESIGN.md §4) -------------------------------------------------
# measured on this pool's B200 (tools/pipe_bench.cu, profiles/r01_pipe_microbench.md):
IMAD_WIDE_PER_CLK_PER_SM = 32.0      # IMAD.WIDE.U32 thread-instructions / clk / SM (IMAD lo: 64)
SM_COUNT = 148
SM_MAX_MHZ = 1965.0
PEAK_TMULS = IMAD_WIDE_PER_CLK_PER_SM * SM_COUNT * SM_MAX_MHZ * 1e6 / 1e12   # 9.31 T wide multiplies / s
PROD_M, PROD_S = 72, 44              # wide multiplies per field multiplication / squaring as emitted (8 x 32-bit limbs: 64 + 8 fold, 36 + 8 fold)
# field operations per op: reference counts (SURVEY.md §8d, instrumented reference) and the counts
# this engine executes (tests/test_host_sim.py::test_field_op_counts pins them)
REF_FM = {"verify": (2291, 1514), "sign": (506, 254), "genpub": (506, 254), "x25519_base": (505, 254), "x25519": (1292, 1278)}
OURS_FM_SINGLE = {"sign": (313, 254), "genpub": (313, 254), "x25519_base": (312, 254), "x25519": (1283, 1272)}   # 43-row signed radix-64 comb
# the kernels share one inversion (254 S + 11 M) among up to EDG_BATCH = 32 operations of a thread, +3 M per operation;
# a thread of the persistent grid gets n / (resident threads) operations, so at 2^20 per GPU the share is 14..28
EDG_BATCH = 32
RESIDENT_THREADS = {"sign": 148 * 512, "genpub": 148 * 512, "x25519_base": 148 * 512, "x25519": 4 * 148 * 128}   # k_comb: one block of 512 threads per SM


def ours_fm(op, n=1 << 20):
    m, s_ = OURS_FM_SINGLE[op]
    share = max(1.0, min(float(EDG_BATCH), n / RESIDENT_THREADS[op]))
    return (m - 11 + 11 / share + 3, s_ - 254 + 254 / share)


OURS_FM = {op: ours_fm(op) for op in RESIDENT_THREADS}


def verify_fm(nwin):
    """Field operations of one verification with half-size scalars (csrc/hgcd.cuh) over nwin 4-bit windows: two
    decompressions and two 8-entry tables (168 M + 510 S), per window 4 doublings + 2 additions (28 M + 16 S; the
    first window has no doublings), 16 base-table additions; no inversion (the result is compared projectively)."""
    return (267 + 28 * nwin, 494 + 16 * nwin)


# nwin = 33 for 85 % of random challenges (32: 10 %, 34: 4.4 %, 35: 0.3 %; measured over 300 000 random t,
# tests/test_host_sim.py::test_half_gcd).  A warp of the loop kernel runs the maximum over its 32 lanes; the front
# kernel hands out records sorted by window count (<= 33 from the front of the array, the rest from the back), so
# 95.3 % of the warps run 33 windows and the others ~34.9: 33.1 on average (unsorted it would be 33.9).
VERIFY_NWIN_WARP_MEAN = 33.1
OURS_FM["verify"] = verify_fm(VERIFY_NWIN_WARP_MEAN)
OURS_FM_SINGLE["verify"] = verify_fm(33)
IO_BYTES = {"verify": 64 + 32 + 64 + 1, "sign": 32 + 32 + 64 + 64, "genpub": 64, "x25519_base": 64, "x25519": 96}


def products(fm):
    return fm[0] * PROD_M + fm[1] * PROD_S


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [s for s, p in zip(sm, pw) if p >= 0.6 * max(pw)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "reasons": sorted(reasons)}


def synth_inputs(n, seed):
    """Synthetic random keys / messages for one rank (counter-based generator, reproducible on host and device side)."""
    rng = np.random.Generator(np.random.Philox(key=seed))
    sec = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    msgs = rng.integers(0, 256, (n, 64), dtype=np.uint8)
    pts = rng.integers(0, 256, (n, 32), dtype=np.uint8)      # bit 255 left random, as in the reference's KAT table
    return sec, msgs, pts


DUMP_ROWS = 1 << 16          # rows of every output written by --dump-outputs: 16 MiB of signatures, 41.5 MiB in all


def dump_rows(n):
    """The rows --dump-outputs writes: all of them for small batches, else a fixed seeded sample (the same in every run)."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0x5EED00D0).choice(n, DUMP_ROWS, replace=False))


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_rates(n_sample, seconds, threads, ops=("verify",)):
    from cpu_ref import best_cpu_impl, OP_GENPUB, OP_SIGN, OP_VERIFY, OP_X25519, OP_X25519_BASE
    cpu = best_cpu_impl()
    sec, msgs, pts = synth_inputs(n_sample, 0x5EED0001)
    pub = cpu.genpub(sec)
    sig = cpu.sign(sec, pub, msgs, fixed_len=64)
    out = {}
    for op in ops:
        if op == "verify":
            out[op] = cpu.time_op(OP_VERIFY, seconds, threads, n_sample, sig, pub, msgs, 64)
        elif op == "sign":
            out[op] = cpu.time_op(OP_SIGN, seconds, threads, n_sample, sec, pub, msgs, 64)
        elif op == "genpub":
            out[op] = cpu.time_op(OP_GENPUB, seconds, threads, n_sample, sec)
        elif op == "x25519":
            out[op] = cpu.time_op(OP_X25519, seconds, threads, n_sample, sec, pts)
        elif op == "x25519_base":
            out[op] = cpu.time_op(OP_X25519_BASE, seconds, threads, n_sample, sec)
    return cpu.kind, out


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    from cpu_ref import best_cpu_impl, OP_VERIFY
    cores = os.cpu_count() or 1
    cpu = best_cpu_impl()
    n_sample = min(1 << args.batch_log2, 4096 * cores)
    sec, msgs, _ = synth_inputs(n_sample, 0x5EED0001)
    pub = cpu.genpub(sec)
    sig = cpu.sign(sec, pub, msgs, fixed_len=64)
    for _ in range(args.warmup):
        cpu.verify(sig, pub, msgs, fixed_len=64)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ok = cpu.verify(sig, pub, msgs, fixed_len=64)
    dt = time.perf_counter() - t0
    assert ok.all()
    value = n_sample * args.steps / dt
    sample = f"{n_sample} of the 2^{args.batch_log2} (pubkey, 64 B msg, sig) triples per step, one reference instance per core ({cores} threads)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic", "config": {"workload": f"ed25519_verify, 64 B messages, CPU sample of {n_sample} ops per step", "batch_per_step": n_sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": cpu.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this engine has no CPU path (use --impl reference for the CPU arm)")
    os.environ["EDDSA_B200_DEVICES"] = f"{local}," if world > 1 else os.environ.get("EDDSA_B200_DEVICES", "0,")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout at the first collective; keep stdout for the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            gloo = dist.new_group(backend="gloo")
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    import libeddsa_b200 as ed
    ed.init()

    n = 1 << args.batch_log2
    K, W = args.steps, max(args.warmup, 3)
    sec, msgs, pts = synth_inputs(n, 0x5EED0001 + rank)

    def pinned(a):
        return torch.from_numpy(a).pin_memory()

    h_sec, h_msg, h_pts = pinned(sec), pinned(msgs), pinned(pts)
    d_sec, d_msg, d_pts = h_sec.to(dev), h_msg.to(dev), h_pts.to(dev)
    d_pub = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    d_sig = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    d_ok = torch.empty((n,), dtype=torch.uint8, device=dev)
    d_out = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # valid triples, produced by the (parity-tested) GPU sign path
    ed.ed25519_genpub_batch_dev(d_pub, d_sec)
    ed.ed25519_sign_batch_dev(d_sig, d_sec, d_pub, d_msg, fixed_len=64)
    torch.cuda.synchronize()

    passes = {
        "verify": lambda: ed.ed25519_verify_batch_dev(d_ok, d_sig, d_pub, d_msg, fixed_len=64),
        "sign": lambda: ed.ed25519_sign_batch_dev(d_sig, d_sec, d_pub, d_msg, fixed_len=64),
        "x25519": lambda: ed.x25519_batch_dev(d_out, d_sec, d_pts),
        "genpub": lambda: ed.ed25519_genpub_batch_dev(d_pub, d_sec),
        "x25519_base": lambda: ed.x25519_base_batch_dev(d_out, d_sec),
    }

    rows = dump_rows(n) if args.dump_outputs and rank == 0 else None
    outputs = {}

    def keep(name, a):
        """For --dump-outputs: the sampled rows of what the last timed step of a pass returned, as float32."""
        if rows is not None:
            a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
            outputs[name] = a[rows].astype(np.float32)

    from libeddsa_b200 import sharding

    def barrier():
        sharding.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return sharding.max_over_ranks(x, dev)

    def timed(fn, steps, warmup):
        """W untimed + K timed steps; every step bracketed by CUDA events on the launching stream; L2 is
        flushed (256 MB write) between steps, outside the events.  Returns (total ms, per-launch ms list)."""
        for _ in range(warmup):
            fn()
        barrier()
        evs = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        barrier()
        per = [a.elapsed_time(b) for a, b in evs]
        return max_over_ranks(sum(per)), per

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ed.launch_count()
    total_ms, per = timed(passes["verify"], K, W)
    keep("verify", d_ok)
    launches = (ed.launch_count() - launches0) * K // (K + W)       # kernels launched by the K timed passes
    assert bool(d_ok.all().item()), "verify rejected a valid signature"
    value = world * n * K / (total_ms * 1e-3)
    kernel_ms = statistics.mean(per)

    also = {}
    results = {"sign": d_sig, "x25519": d_out, "genpub": d_pub, "x25519_base": d_out}
    for name in ("sign", "x25519", "genpub", "x25519_base"):
        ms, p = timed(passes[name], K, W)
        keep(name, results[name])
        rate = world * n * K / (ms * 1e-3)
        per_gpu = rate / world
        also[name] = {"value": rate, "unit": UNIT, "ms_per_step": ms / K,
                      "roofline_frac_executed": per_gpu * products(OURS_FM[name]) / 1e12 / PEAK_TMULS,
                      "roofline_frac_reference_fm": per_gpu * products(REF_FM[name]) / 1e12 / PEAK_TMULS}
    # restore valid signatures for the e2e leg (sign overwrote d_sig with identical bytes; keep it explicit)
    torch.cuda.synchronize()

    # ---- end to end through the public host-buffer C-ABI, pinned host memory --------------------------
    h_sig, h_pub = pinned(d_sig.cpu().numpy()), pinned(d_pub.cpu().numpy())
    h_ok = torch.empty(n, dtype=torch.uint8).pin_memory()
    L = ed.lib()
    import ctypes
    vp = lambda t: ctypes.c_void_p(t.data_ptr())

    def e2e_step():
        rc = L.ed25519_verify_batch(n, vp(h_ok), vp(h_sig), vp(h_pub), vp(h_msg), None, 64)
        if rc:
            raise RuntimeError(f"ed25519_verify_batch failed: {rc} {L.eddsa_b200_last_error()}")

    for _ in range(W):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_step()
    own_s = time.perf_counter() - t0                             # this rank's own K steps (before waiting for the others)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    per_rank = [own_s]
    if world > 1:
        t_all = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(t_all, torch.tensor([own_s], dtype=torch.float64, device=dev))
        per_rank = [float(t.item()) for t in t_all]
    assert bool(h_ok.all().item())
    keep("e2e", h_ok)
    e2e_value = world * n * K / e2e_s
    # ---- the same from ordinary (pageable) memory: the library stages through its pinned slots ------------------
    p_sig, p_pub, p_msg, p_ok = np.array(h_sig.numpy()), np.array(h_pub.numpy()), np.array(h_msg.numpy()), np.empty(n, np.uint8)
    ap = lambda a: ctypes.c_void_p(a.ctypes.data)

    def e2e_pageable_step():
        rc = L.ed25519_verify_batch(n, ap(p_ok), ap(p_sig), ap(p_pub), ap(p_msg), None, 64)
        if rc:
            raise RuntimeError(f"ed25519_verify_batch failed: {rc} {L.eddsa_b200_last_error()}")

    def wall(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        barrier()
        return max_over_ranks(time.perf_counter() - t0)

    pg_s = wall(e2e_pageable_step, K, 1)
    assert p_ok.all()
    keep("e2e_pageable", p_ok)
    also["e2e_pageable"] = {"value": world * n * K / pg_s, "unit": UNIT, "api": "ed25519_verify_batch, ordinary (malloc) host buffers: staged through the "
                            "library's pinned slots with memcpy", "ms_per_step": pg_s / K * 1e3}
    del p_sig, p_pub, p_msg

    # ---- BASELINE config 5's shape end to end: 1 KB messages, 10 % corrupted, pinned host buffers ----------------
    mlen = 1024
    g1 = torch.Generator(device=dev)
    g1.manual_seed(0x5EED0005 + rank)
    d_msg1k = torch.randint(0, 256, (n, mlen), dtype=torch.uint8, device=dev, generator=g1)
    ed.ed25519_sign_batch_dev(d_sig, d_sec, d_pub, d_msg1k, fixed_len=mlen)
    bad = torch.arange(0, n, 10, device=dev)
    d_sig[bad, 3 + (bad % 40)] ^= 1
    h_msg1k = torch.empty((n, mlen), dtype=torch.uint8, pin_memory=True)
    h_msg1k.copy_(d_msg1k)
    h_sig1k = torch.empty((n, 64), dtype=torch.uint8, pin_memory=True)
    h_sig1k.copy_(d_sig)
    torch.cuda.synchronize()
    del d_msg1k

    def e2e_1kb_step():
        rc = L.ed25519_verify_batch(n, vp(h_ok), vp(h_sig1k), vp(h_pub), vp(h_msg1k), None, mlen)
        if rc:
            raise RuntimeError(f"ed25519_verify_batch failed: {rc} {L.eddsa_b200_last_error()}")

    kb_s = wall(e2e_1kb_step, K, 1)
    assert int(h_ok.sum().item()) == n - len(bad)
    keep("e2e_1kb", h_ok)
    kb_bytes = n * (64 + 32 + mlen)
    also["e2e_1kb"] = {"value": world * n * K / kb_s, "unit": UNIT, "api": "ed25519_verify_batch (host buffers, pinned), 1024-byte messages, 10 % of the signatures corrupted",
                       "ms_per_step": kb_s / K * 1e3, "h2d_bytes_per_step": kb_bytes, "h2d_gbs_per_gpu": kb_bytes * K / kb_s / 1e9,
                       "note": "copy-bound: every signature brings 1 120 bytes over PCIe; compare h2d_gbs_per_gpu with also.inproc.copy_bandwidth"}
    del h_msg1k, h_sig1k
    clocks = sampler.stop() if rank == 0 else None

    # ---- single operations of eddsa.h (batch of one on the GPU) next to the reference's CPU time ------------------
    if rank == 0:
        also["single_op_latency_us"] = single_op_latency(ed, h_sec.numpy(), h_pub.numpy(), h_sig.numpy(), h_msg.numpy(), h_pts.numpy())

    # ---- the library's own multi-device path on BASELINE configs 4 and 5 (one process, all N devices) ------------
    # rank 0 runs tools/inproc_bench.py as a subprocess; the other ranks wait on a CPU (gloo) barrier so that their
    # GPUs are idle (an NCCL barrier would spin a kernel on them)
    torch.cuda.synchronize()
    del flush
    torch.cuda.empty_cache()
    ed.shutdown()
    if world > 1:
        dist.barrier()
    if rank == 0 and not args.no_inproc:
        also["inproc"] = run_inproc(world, K)
    if world > 1:
        dist.barrier(group=gloo)

    if rank == 0:
        # ---- roofline of the dominant kernel (k_verify) ---------------------------------------------
        per_gpu = n / (kernel_ms * 1e-3)
        achieved = per_gpu * products(OURS_FM["verify"]) / 1e12
        roofline = {
            "bound": "int32-multiply (IMAD.WIDE on the fmaheavy pipe; compute-bound, see DESIGN.md §4)",
            "kernel": "k_verify_scalars + k_verify_points + k_verify (one step = %d launches: three stages per pass of up to 1 212 416 signatures)" % max(int(launches) // K, 1),
            "achieved": achieved, "peak": PEAK_TMULS, "unit": "T wide-multiplies/s (32x32->64)", "frac": achieved / PEAK_TMULS,
            "frac_reference_fm": per_gpu * products(REF_FM["verify"]) / 1e12 / PEAK_TMULS,
            "peak_source": "measured: tools/pipe_bench.cu on this pool's B200 = 32 IMAD.WIDE/clk/SM x 148 SM x 1965 MHz (profiles/r01_pipe_microbench.md)",
            "wide_multiplies_per_op_executed": products(OURS_FM["verify"]),
            "wide_multiplies_per_op_reference_fm": products(REF_FM["verify"]),
            "kernel_ms_per_launch": kernel_ms,
            "stages": ncu_stages(),
            "traffic": ncu_traffic(n),
            "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of the three stages from the ncu --set full capture on 2^18 signatures "
                            "(profiles/r02_ncu_summary.json), scaled to this batch; the 2.4 KB record the front stages hand to the window "
                            "loop (two 8-entry point tables) is written once and read back ~2x: ~5 % of HBM bandwidth",
            "hbm": {"algorithmic_bytes_per_launch": n * IO_BYTES["verify"],
                    "achieved_gbs": n * IO_BYTES["verify"] / (kernel_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak(),
                    "note": "HBM is not the bound: <0.1 % of measured copy bandwidth"},
        }
        cores = os.cpu_count() or 1
        cpu_b = None
        if world == 1:
            kind, rates = cpu_rates(4096 * min(cores, 16), 2.0, cores, ops=("verify", "sign", "x25519", "genpub", "x25519_base"))
            _, single = cpu_rates(2048, 1.5, 1, ops=("verify",))
            cpu_b = {"value": rates["verify"], "unit": UNIT, "cores": cores, "kind": kind,
                     "sample": f"{4096 * min(cores, 16)} of the same synthetic triples, every thread looping its slice for 2.0 s (one instance per core)",
                     "single_thread": single["verify"], "also": {k: v for k, v in rates.items() if k != "verify"}}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (8 saturated 32-bit limbs, IMAD.WIDE carry chains)",
            "data": "synthetic",
            "config": {"workload": "ed25519_verify of 2^%d random valid (pubkey, 64 B msg, sig) triples per GPU (BASELINE config 1)" % args.batch_log2,
                       "batch_per_gpu": n, "global_batch": n * world, "msg_len": 64, "sharding": "by rank, no collective",
                       "l2": "inputs 168 MB > 126 MB L2 and a 256 MB flush write between timed steps"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * (64 + 32 + 64), "d2h_bytes_per_step": n,
                    "api": "ed25519_verify_batch (host buffers, pinned)", "ms_per_step": e2e_s / K * 1e3,
                    "ms_per_step_by_rank": [round(t / K * 1e3, 3) for t in per_rank],
                    "note": "value = all ranks' signatures / the slowest rank's time; the ranks share one host (pinned buffers and PCIe "
                            "paths on whichever NUMA node each process landed), so their own times differ — see ms_per_step_by_rank"},
            "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu_b, "also": also, "clocks": clocks,
        }
        if rows is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "rows.npy"), rows.astype(np.float64))
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def single_op_latency(ed, sec, pub, sig, msg, pts, calls=300):
    """Median wall time of one call of each eddsa.h function (a batch of one on the GPU: H2D, kernels, D2H, synchronise)
    and of the same call into the reference's CPU library."""
    import ctypes
    from cpu_ref import have_reference, reference_path
    ours = ed.lib()
    ref = ctypes.CDLL(reference_path()) if have_reference() else None
    out = ctypes.create_string_buffer(64)
    rows = [(sec[i].tobytes(), pub[i].tobytes(), sig[i].tobytes(), msg[i].tobytes(), pts[i].tobytes()) for i in range(64)]

    def med(fn):
        for i in range(30):
            fn(rows[i % 64])
        ts = []
        for i in range(calls):
            r = rows[i % 64]
            t0 = time.perf_counter()
            fn(r)
            ts.append(time.perf_counter() - t0)
        return round(statistics.median(ts) * 1e6, 1)

    res = {}
    for name, lib in (("gpu", ours), ("reference_cpu", ref)):
        if lib is None:
            continue
        lib.ed25519_verify.restype = ctypes.c_bool
        res[name] = {
            "ed25519_genpub": med(lambda r: lib.ed25519_genpub(out, r[0])),
            "ed25519_sign_64B": med(lambda r: lib.ed25519_sign(out, r[0], r[1], r[3], ctypes.c_size_t(64))),
            "ed25519_verify_64B": med(lambda r: lib.ed25519_verify(r[2], r[1], r[3], ctypes.c_size_t(64))),
            "x25519": med(lambda r: lib.x25519(out, r[0], r[4])),
            "x25519_base": med(lambda r: lib.x25519_base(out, r[0])),
        }
    res["note"] = "median of %d calls; the GPU figure is one thread of one kernel chain plus two copies and a synchronise — latency-bound callers should batch" % calls
    return res


def run_inproc(world, reps):
    cmd = [sys.executable, os.path.join(ROOT, "tools", "inproc_bench.py"), "--devices", str(world), "--reps", str(reps)]
    drop = ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "GROUP_RANK", "MASTER_ADDR", "MASTER_PORT", "EDDSA_B200_DEVICES", "OMP_NUM_THREADS")
    env = {k: v for k, v in os.environ.items() if k not in drop and not k.startswith("TORCHELASTIC")}
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    try:
        res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
        for line in reversed(res.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"error": (res.stderr or res.stdout)[-600:]}
    except Exception as e:                                       # noqa: BLE001 — the headline line must still be printed
        return {"error": repr(e)}


VERIFY_STAGES = ("verify_scalars", "verify_points", "verify_loop")


def ncu_traffic(n):
    """DRAM bytes per pass over n signatures, from the committed ncu capture (None if it is not there)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_summary.json")))
        per_op = sum(d[k]["dram_read_bytes"] + d[k]["dram_write_bytes"] for k in VERIFY_STAGES) / d["ops_per_launch"]
        return int(per_op * n)
    except Exception:
        return None


def ncu_stages():
    """The three kernels of a verify pass as captured by ncu on 2^18 signatures (profiles/r02_ncu_summary.json): share of the
    pass and multiplier-pipe utilisation of each — context for the pass-level roofline above, not measured live."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_summary.json")))
        tot = sum(d[k]["duration_ms"] for k in VERIFY_STAGES)
        return {d[k]["kernel"]: {"share_of_pass": round(d[k]["duration_ms"] / tot, 3), "fmaheavy_pipe_busy_pct": d[k]["fmaheavy_pipe_busy_pct"],
                                 "registers": d[k]["registers_per_thread"]} for k in VERIFY_STAGES}
    except Exception:
        return None


def hbm_peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        return 6650.0


def main():
    sys.dont_write_bytecode = True       # the tree may be read-only: importing the package and the CPU checker writes nothing there
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-log2", type=int, default=20)
    ap.add_argument("--no-inproc", action="store_true", help="skip the in-library multi-device leg (configs 4 and 5 at 2^24)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step of each pass returned "
                    "(rank 0, a fixed sample of rows) to DIR/<name>.npy as float32, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this project's GPU path (--impl ours)")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
