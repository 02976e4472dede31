"""GPU tests with structured inputs (run on the B200 box: `pytest -m gpu`): the device code paths that SHA-512 challenges and
random keys almost never drive into their rare branches, checked on the hardware against Python integers, the host builds of
the same headers and the CPU reference.

A  half_gcd (hgcd.cuh) and the verify loop's 16-bit recoding on the device (k_sc_selftest ops 3..5), on challenges that reach
   every branch class (tests/structured_inputs.py), bit-exact with both host builds of the header and with a plain Euclid.
B  the fixed-base comb (signed radix-64 recoding + tensor-core lookup) on scalars with structured digits, reached through
   x25519_base, whose kernel computes clamp(s) mod L itself.
C  the key conversions on non-canonical, off-curve and small y, host and device-pointer API.
D  device-pointer calls larger than one pass of the persistent grid (slow), and guard bytes around every output.
E  the outputs bench.py dumps, checked against the CPU reference (slow).
The same generators run on the SIMT emulator without a GPU (tests/host_sim/sim_scenarios.py: real_kernels_structured).
"""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import structured_inputs as si
from edmodel import L

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def to_rows(vals, width=32):
    return np.frombuffer(b"".join(v.to_bytes(width, "little") for v in vals), np.uint8).reshape(-1, width)


def from_rows(a):
    return [int.from_bytes(a[i].tobytes(), "little") for i in range(len(a))]


# ------------------------------------------------------------------------------------------------ A: half_gcd, recoding
def test_device_half_gcd_on_structured_challenges(ed):
    """k_sc_selftest ops 3 / 4 on every input of structured_inputs.half_gcd_inputs(): (rho, tau) bit for bit equal to the host
    build of hgcd.cuh in both flavours (portable C++ and the device paths under the PTX interpreter) and to the plain Euclid;
    rho odd, tau = rho t (mod 8L), tau < 2^128 and |rho| < 2^160 unless the result is the fallback (1, t)."""
    import ctypes
    import test_host_sim as ths
    ts = si.half_gcd_inputs()
    counts = si.class_counts(ts)
    print("half_gcd inputs by branch class:", counts)
    assert all(counts[k] >= m for k, m in si.MIN_CLASS_COUNT.items()), counts
    a = to_rows(ts)
    z = np.zeros_like(a)
    tau_d, rho_d = ed.sc_selftest(a, z, z, 3), ed.sc_selftest(a, z, z, 4)
    rho_w = rho_d.view(np.uint32)
    hosts = [ths._build("ops_host", flavour) for flavour in ("host", "device")]
    rho = (ctypes.c_uint32 * 8)(); tau = (ctypes.c_uint32 * 8)(); neg = ctypes.c_uint32()
    N = 8 * L
    for i, t in enumerate(ts):
        tw = (ctypes.c_uint32 * 8)(*[(t >> (32 * k)) & 0xFFFFFFFF for k in range(8)])
        for h in hosts:
            h.hs_half_gcd(rho, ctypes.byref(neg), tau, tw)
            assert bytes(tau) == tau_d[i].tobytes(), (t, h.device_paths, "tau")
            assert list(rho)[:6] == rho_w[i, :6].tolist() and rho_w[i, 6] == 0 and rho_w[i, 7] == neg.value, (t, h.device_paths, "rho")
        r = int.from_bytes(rho_d[i, :24].tobytes(), "little")
        r = -r if rho_w[i, 7] else r
        ta = int.from_bytes(tau_d[i].tobytes(), "little")
        assert r % 2 == 1 and (r * t - ta) % N == 0, t
        want_r, want_ta, info = si.half_gcd_model(t)
        assert (r, ta) == (want_r, want_ta), (t, info)
        if info["fallback"]:
            assert (r, ta) == (1, t)
        else:
            assert ta < 2**128 and abs(r) < 2**160, t


def test_device_window_recoding(ed):
    """k_sc_selftest op 5 (sc_recode_window): the 16 signed 16-bit digits d_k in [-2^15, 2^15) with sum d_k 2^(16 k) = x, for 0,
    1, L - 1, values made of 0x7fff / 0x8000 / 0xffff digit runs and random x < L."""
    xs = si.recode_window_values()
    z = np.zeros((len(xs), 32), np.uint8)
    es = from_rows(ed.sc_selftest(to_rows(xs), z, z, 5))
    for x, e in zip(xs, es):
        ds = si.window_digits(e)
        assert all(-2**15 <= d < 2**15 for d in ds) and sum(d << (16 * k) for k, d in enumerate(ds)) == x, (x, e)


# ------------------------------------------------------------------------------------------------ B: comb scalars
def test_x25519_base_with_structured_comb_digits(ed, cpu):
    """Raw x25519_base scalars s = v + jL in [2^254, 2^255), s = 0 (mod 8), with random bit 255 and bits 0..2: the kernel's
    clamp(s) mod L is the target v, whose 43 signed radix-64 digits are structured (structured_inputs.comb_targets).  Rows
    shuffled among random scalars; the host API and x25519_base_batch_dev against the CPU reference, a subset against the
    big-integer model u = (1 + y) / (1 - y) of v B."""
    import torch
    scal, targets, unreachable = si.comb_batch(n_random=3000)
    reach = [v for v in targets if v is not None]
    digits = [si.comb_digits(v) for v in reach]

    def run_of(ds, value):
        best = cur = 0
        for d in ds:
            cur = cur + 1 if d == value else 0
            best = max(best, cur)
        return best
    kinds = {"top digit 1": sum(ds[-1] == 1 for ds in digits), "10+ zero digits in a row": sum(run_of(ds, 0) >= 10 for ds in digits),
             "10+ digits 31 in a row": sum(run_of(ds, 31) >= 10 for ds in digits), "10+ digits -32 in a row": sum(run_of(ds, -32) >= 10 for ds in digits),
             "one non-zero digit above digit 0": sum(sum(d != 0 for d in ds[1:]) == 1 for ds in digits)}
    print(f"comb targets: {len(reach)} reachable through x25519_base, {unreachable} dropped; {kinds}")
    assert len(reach) >= 800 and all(c >= 20 for c in kinds.values()), kinds
    sa = np.frombuffer(b"".join(scal), np.uint8).reshape(-1, 32).copy()
    want = cpu.x25519_base(sa)
    got = ed.x25519_base_batch(sa)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert not len(bad), [(int(i), targets[i]) for i in bad[:5]]
    dev = torch.device("cuda:0")
    out = torch.empty((len(sa), 32), dtype=torch.uint8, device=dev)
    ed.x25519_base_batch_dev(out, torch.from_numpy(sa).to(dev))
    assert (out.cpu().numpy() == want).all()
    rng = random.Random(3)
    for i in rng.sample([i for i, v in enumerate(targets) if v is not None], 60):
        assert got[i].tobytes() == si.x25519_base_model(targets[i]), targets[i]


# ------------------------------------------------------------------------------------------------ C: conversions
def test_key_conversions_with_structured_keys(ed, cpu):
    """pk_ed25519_to_x25519 on every non-canonical y in [p, 2^255) with both sign bits, y in {0, 1, p - 1} and "-0", off-curve
    y and random keys; sk_ed25519_to_x25519 on random and constant keys — host API, device-pointer API and CPU reference agree."""
    import torch
    dev = torch.device("cuda:0")
    pks = np.frombuffer(b"".join(si.pk_structured()), np.uint8).reshape(-1, 32).copy()
    want = np.frombuffer(b"".join(cpu.pk_to_x25519(pks[i].tobytes()) for i in range(len(pks))), np.uint8).reshape(-1, 32)
    assert (ed.pk_ed25519_to_x25519_batch(pks) == want).all()
    out = torch.empty((len(pks), 32), dtype=torch.uint8, device=dev)
    ed.pk_ed25519_to_x25519_batch_dev(out, torch.from_numpy(pks).to(dev))
    assert (out.cpu().numpy() == want).all()
    rng = np.random.default_rng(31)
    sks = rng.integers(0, 256, (1000, 32), dtype=np.uint8)
    sks[0], sks[1], sks[2] = 0, 0xFF, 0x80
    want = np.frombuffer(b"".join(cpu.sk_to_x25519(sks[i].tobytes()) for i in range(len(sks))), np.uint8).reshape(-1, 32)
    assert (ed.sk_ed25519_to_x25519_batch(sks) == want).all()
    out = torch.empty((len(sks), 32), dtype=torch.uint8, device=dev)
    ed.sk_ed25519_to_x25519_batch_dev(out, torch.from_numpy(sks).to(dev))
    assert (out.cpu().numpy() == want).all()


# ------------------------------------------------------------------------------------------------ D: device-API shapes
GUARD = 64                                     # bytes of pattern before and after every output (a multiple of the 16-byte alignment)


def guarded(n, width, dev, lead=GUARD):
    """(whole buffer, output view of n x width bytes starting `lead` bytes in, copy of the initial pattern)."""
    import torch
    total = lead + n * width + GUARD
    buf = (torch.arange(total, dtype=torch.int64, device=dev) * 37 + 11).remainder(251).to(torch.uint8)
    view = buf[lead:lead + n * width].view(n, width) if width > 1 else buf[lead:lead + n]
    return buf, view, buf.clone()


def assert_guards(buf, pattern, lead, nbytes, what):
    b, p = buf.cpu().numpy(), pattern.cpu().numpy()
    assert (b[:lead] == p[:lead]).all(), f"{what}: bytes before the output were written"
    assert (b[lead + nbytes:] == p[lead + nbytes:]).all(), f"{what}: bytes after the output were written"


def ragged_subset(blob, off, idx):
    """The messages of rows idx as their own ragged batch (blob, offsets)."""
    parts = [blob[int(off[i]):int(off[i + 1])] for i in idx]
    sub_off = np.zeros(len(idx) + 1, np.uint64)
    sub_off[1:] = np.cumsum([len(p) for p in parts])
    return (np.concatenate(parts) if parts else np.zeros(0, np.uint8)), sub_off


def test_every_device_entry_point_leaves_its_neighbours_alone(ed, cpu):
    """Each of the seven device-pointer entry points writes into a view inside a larger tensor on a non-default stream, with n
    not a multiple of 32 (the comb's tail warp recomputes the last operation and must drop it): the results equal the CPU
    reference and the guard bytes before and after every output (the verify flags at an odd offset) are unchanged."""
    import torch
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(41)
    n = 32 * 37 + 13
    sec, pts = rng.integers(0, 256, (n, 32), dtype=np.uint8), rng.integers(0, 256, (n, 32), dtype=np.uint8)
    lens = rng.integers(0, 150, n)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    blob = rng.integers(0, 256, int(off[-1]) + 16, dtype=np.uint8)
    pub = cpu.genpub(sec)
    sig = cpu.sign(sec, pub, blob, off=off)
    bad = sig.copy()
    bad[::7, 40] ^= 1
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_sec, d_pts, d_pub, d_blob, d_off, d_bad = t(sec), t(pts), t(pub), t(blob), t(off.astype(np.int64)), t(bad)
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    outs = {}
    with torch.cuda.stream(stream):
        for name, width, lead, call in (
                ("genpub", 32, GUARD, lambda o: ed.ed25519_genpub_batch_dev(o, d_sec)),
                ("sign", 64, GUARD, lambda o: ed.ed25519_sign_batch_dev(o, d_sec, d_pub, d_blob, off=d_off)),
                ("verify", 1, GUARD + 3, lambda o: ed.ed25519_verify_batch_dev(o, d_bad, d_pub, d_blob, off=d_off)),
                ("x25519", 32, GUARD, lambda o: ed.x25519_batch_dev(o, d_sec, d_pts)),
                ("x25519_base", 32, GUARD, lambda o: ed.x25519_base_batch_dev(o, d_sec)),
                ("pk", 32, GUARD, lambda o: ed.pk_ed25519_to_x25519_batch_dev(o, d_pub)),
                ("sk", 32, GUARD, lambda o: ed.sk_ed25519_to_x25519_batch_dev(o, d_sec))):
            buf, view, pattern = guarded(n, width, dev, lead)
            call(view)
            outs[name] = (buf, view, pattern, lead, n * width)
    stream.synchronize()
    for name, (buf, view, pattern, lead, nbytes) in outs.items():
        assert_guards(buf, pattern, lead, nbytes, name)
    got = {k: v[1].cpu().numpy() for k, v in outs.items()}
    assert (got["genpub"] == pub).all() and (got["sign"] == sig).all()
    assert (got["verify"] == cpu.verify(bad, pub, blob, off=off)).all() and got["verify"].sum() == n - len(range(0, n, 7))
    assert (got["x25519"] == cpu.x25519(sec, pts)).all() and (got["x25519_base"] == cpu.x25519_base(sec)).all()
    assert (got["pk"] == ed.pk_ed25519_to_x25519_batch(pub)).all() and (got["sk"] == ed.sk_ed25519_to_x25519_batch(sec)).all()


@pytest.mark.slow
def test_x25519_calls_beyond_one_grid_pass(ed, cpu):
    """x25519_batch_dev and x25519_base_batch_dev at n = 40 x 512 x SMs + 77: more than EDG_BATCH = 32 operations per resident
    thread, so the kernels' outer grid-stride loop runs a second, ragged time.  Assumes 512 resident threads per SM for both
    kernels (DESIGN.md §3, bench.py: RESIDENT_THREADS — one 512-thread comb block, four 128-thread ladder blocks per SM).  Every
    row from the second pass's start minus 2048 to the end and a random sample of the rest against the CPU reference; guard
    bytes around both outputs."""
    import torch
    dev = torch.device("cuda:0")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    n = 40 * 512 * sms + 77
    g = torch.Generator(device=dev)
    g.manual_seed(0x5EED0D01)
    sec = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=g)
    pts = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=g)
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(stream):
        xbuf, xout, xpat = guarded(n, 32, dev)
        ed.x25519_batch_dev(xout, sec, pts)
        bbuf, bout, bpat = guarded(n, 32, dev)
        ed.x25519_base_batch_dev(bout, sec)
    stream.synchronize()
    assert_guards(xbuf, xpat, GUARD, 32 * n, "x25519")
    assert_guards(bbuf, bpat, GUARD, 32 * n, "x25519_base")
    first = 32 * 512 * sms - 2048
    rows = np.concatenate([np.arange(first, n), np.random.default_rng(5).choice(first, 20000, replace=False)])
    idx = torch.from_numpy(rows).to(dev)
    s, p = sec[idx].cpu().numpy(), pts[idx].cpu().numpy()
    for name, out, want in (("x25519", xout, cpu.x25519(s, p)), ("x25519_base", bout, cpu.x25519_base(s))):
        got = out[idx].cpu().numpy()
        bad = np.nonzero((got != want).any(axis=1))[0]
        assert not len(bad), (name, rows[bad[:5]].tolist())


@pytest.mark.slow
def test_genpub_and_ragged_sign_beyond_one_fixed_base_pass(ed, cpu):
    """ed25519_genpub_batch_dev and a ragged ed25519_sign_batch_dev (messages of 0..200 bytes) at n = 2^21 + 5013, longer than one
    fixed-base pass of 2^21 operations (the second pass indexes off + first).  Every row round-trips through
    ed25519_verify_batch_dev; the rows around the pass boundary and at both ends equal the CPU reference."""
    import torch
    dev = torch.device("cuda:0")
    n = (1 << 21) + 5013
    rng = np.random.default_rng(61)
    sec = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    lens = rng.integers(0, 201, n)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    blob = rng.integers(0, 256, int(off[-1]) + 16, dtype=np.uint8)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_sec, d_blob, d_off = t(sec), t(blob), t(off.astype(np.int64))
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(stream):
        pbuf, pub, ppat = guarded(n, 32, dev)
        ed.ed25519_genpub_batch_dev(pub, d_sec)
        sbuf, sig, spat = guarded(n, 64, dev)
        ed.ed25519_sign_batch_dev(sig, d_sec, pub, d_blob, off=d_off)
        obuf, ok, opat = guarded(n, 1, dev, GUARD + 1)
        ed.ed25519_verify_batch_dev(ok, sig, pub, d_blob, off=d_off)
    stream.synchronize()
    assert_guards(pbuf, ppat, GUARD, 32 * n, "genpub")
    assert_guards(sbuf, spat, GUARD, 64 * n, "sign")
    assert_guards(obuf, opat, GUARD + 1, n, "verify")
    assert bool(ok.all().item()), np.nonzero(ok.cpu().numpy() == 0)[0][:10]
    rows = np.concatenate([np.arange(0, 2048), np.arange((1 << 21) - 2048, (1 << 21) + 2048), np.arange(n - 2048, n)])
    got_pub, got_sig = pub.cpu().numpy()[rows], sig.cpu().numpy()[rows]
    want_pub = cpu.genpub(sec[rows])
    assert (got_pub == want_pub).all(), rows[np.nonzero((got_pub != want_pub).any(axis=1))[0][:5]].tolist()
    sub_blob, sub_off = ragged_subset(blob, off, rows)
    want_sig = cpu.sign(sec[rows], want_pub, sub_blob, off=sub_off)
    assert (got_sig == want_sig).all(), rows[np.nonzero((got_sig != want_sig).any(axis=1))[0][:5]].tolist()


# ------------------------------------------------------------------------------------------------ E: bench.py's outputs
@pytest.mark.slow
def test_bench_dumps_match_the_cpu_reference(tmp_path):
    """bench.py --dump-outputs at 2^16, then tools/check_bench_dumps.py: sign, genpub, x25519 and x25519_base of the timed steps
    equal the CPU reference, the verify legs accept every valid signature and reject exactly the corrupted ones.  Control: one
    changed byte of sign.npy is reported."""
    out = tmp_path / "dumps"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch-log2", "16", "--steps", "1", "--warmup", "0", "--no-inproc",
                          "--dump-outputs", str(out)], capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stderr[-3000:]
    chk = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "check_bench_dumps.py"), str(out), "--batch-log2", "16"],
                         capture_output=True, text=True, timeout=1200)
    assert chk.returncode == 0 and "OK" in chk.stdout, chk.stdout[-3000:] + chk.stderr[-3000:]
    sign = np.load(out / "sign.npy")
    sign[123, 45] = (sign[123, 45] + 1) % 256
    np.save(out / "sign.npy", sign)
    chk = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "check_bench_dumps.py"), str(out), "--batch-log2", "16"],
                         capture_output=True, text=True, timeout=1200)
    assert chk.returncode == 1 and "sign: 1 of" in chk.stdout, chk.stdout[-3000:]
