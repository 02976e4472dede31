"""Unit tests of the DEVICE code's arithmetic without a GPU: the .cuh headers under
libeddsa_b200/csrc are plain C++ inline functions, so tests/host_sim compiles them for the host
(g++) and this file checks them against Python big integers, hashlib and the golden fixtures.
This is test infrastructure only — the shipped library contains no host build of these functions.
"""
import ctypes
import hashlib
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import golden_util as gu
from edmodel import L, P

HS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_sim")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
A8 = ctypes.c_uint32 * 8


def _build(name, flavour="host"):
    """flavour "host": the portable host paths of the headers.  flavour "device": the DEVICE paths (everything under
    `#if defined(__CUDA_ARCH__)` — PTX carry chains, funnel shifts, byte permutes, 128-bit loads, cp.async staging), with
    the inline PTX rewritten into calls of a PTX interpreter (host_sim/ptx_rewrite.py, ptx_emul.h), one lane per call."""
    src = os.path.join(HS, name + ".cpp")
    if flavour == "host":
        so = os.path.join(HS, "lib" + name + ".so")
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", so, src], check=True)
    else:
        gen = os.path.join(HS, "_ptx")
        os.makedirs(os.path.join(gen, "tests", "host_sim"), exist_ok=True)
        subprocess.run([sys.executable, os.path.join(HS, "ptx_rewrite.py"), os.path.join(ROOT, "libeddsa_b200", "csrc"),
                        os.path.join(gen, "libeddsa_b200", "csrc")], check=True, stdout=subprocess.DEVNULL)
        gsrc = os.path.join(gen, "tests", "host_sim", name + ".cpp")
        with open(gsrc, "w") as f:
            f.write(open(src).read())
        so = os.path.join(HS, "lib" + name + "_ptx.so")
        # -fno-gnu-unique: the interpreter's per-statement programs are static locals of inline functions; as GNU_UNIQUE
        # symbols they would be shared by every library of the process that contains the same function
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-D__CUDA_ARCH__=1000",
                        "-D__CUDACC__", "-include", os.path.join(HS, "ptx_emul.h"), "-o", so, gsrc], check=True)
    lib = ctypes.CDLL(so)
    lib.device_paths = flavour == "device"
    return lib


@pytest.fixture(scope="module", params=["host", "device"])
def fe(request):
    return _build("fe_host", request.param)


@pytest.fixture(scope="module", params=["host", "device"])
def ops(request):
    return _build("ops_host", request.param)


def val(words):
    return sum(int(x) << (32 * i) for i, x in enumerate(words))


def W8(x):
    return [(x >> (32 * i)) & 0xFFFFFFFF for i in range(8)]


def call(f, *args):
    r = A8()
    f(r, *[A8(*a) for a in args])
    return list(r)


EDGE = [0, 1, 2, 19, 37, 38, 39, P - 1, P, P + 1, P + 18, 2 * P, 2 * P + 1, 2 * P + 37, 2**255 - 20, 2**255 - 1, 2**255, 2**255 + 18,
        2**256 - 39, 2**256 - 38, 2**256 - 1, 2**256 - 2**32, 2**224, 2**32 - 1]


def test_fe_arithmetic_on_all_256_bit_inputs(fe):
    """Operands are any values < 2^256 (weakly reduced); results are exact modulo p and again < 2^256,
    including the all-ones / near-2p / near-2^256 corner cases where the folding carries twice."""
    rng = random.Random(1)
    cases = [(a, b) for a in EDGE for b in EDGE] + [(rng.getrandbits(256), rng.getrandbits(256)) for _ in range(3000)]
    for a, b in cases:
        A, B = W8(a), W8(b)
        assert val(call(fe.h_fe_mul, A, B)) % P == a * b % P
        assert val(call(fe.h_fe_sq, A)) % P == a * a % P
        assert val(call(fe.h_fe_mul121665, A)) % P == a * 121665 % P
        assert val(call(fe.h_fe_sub, A, B)) % P == (a - b) % P
        assert val(call(fe.h_fe_add, A, B)) % P == (a + b) % P
        assert val(call(fe.h_fe_neg, A)) % P == (-a) % P


def test_fe_canonical_bytes(fe):
    """fld_import semantics (all 256 bits, bit 255 -> +19, i.e. the integer mod p) and canonical export."""
    rng = random.Random(2)
    for e in EDGE + [rng.getrandbits(256) for _ in range(3000)]:
        r = A8()
        fe.h_fe_from_bytes(r, e.to_bytes(32, "little"))
        assert val(r) % P == e % P
        out = ctypes.create_string_buffer(32)
        fe.h_fe_to_bytes(out, r)
        assert int.from_bytes(out.raw, "little") == e % P
        assert fe.h_fe_is_zero(r) == (1 if e % P == 0 else 0)
        assert val(call(fe.h_fe_canon, W8(e))) == e % P


def test_fe_inverse_and_pow2523(fe):
    rng = random.Random(3)
    for t in [1, 2, P - 1, P + 5, 2**256 - 1] + [rng.getrandbits(256) for _ in range(100)]:
        assert val(call(fe.h_fe_inv, W8(t))) % P == pow(t % P, P - 2, P)
        assert val(call(fe.h_fe_pow2523, W8(t))) % P == pow(t % P, (P - 5) // 8, P)
    for z in (0, P, 2 * P):                                   # inv(0) = 0 for every representative of 0 (SURVEY Q7)
        assert val(call(fe.h_fe_inv, W8(z))) % P == 0


def test_sc_reduce_muladd_recode(fe):
    rng = random.Random(4)

    def W(x, n):
        return (ctypes.c_uint32 * n)(*[(x >> (32 * i)) & 0xFFFFFFFF for i in range(n)])

    def V(a):
        return sum(int(x) << (32 * i) for i, x in enumerate(a))

    cases = [0, 1, L - 1, L, L + 1, 2 * L, 3 * L - 1, 2**252, 2**256 - 1, 2**512 - 1, (2**512 // L) * L, (2**512 // L) * L - 1, L * L]
    cases += [rng.getrandbits(512) for _ in range(3000)] + [rng.getrandbits(rng.randrange(1, 512)) for _ in range(1000)]
    for x in cases:
        r = (ctypes.c_uint32 * 8)()
        fe.h_sc_reduce512(r, W(x, 16))
        assert V(r) == x % L
    for k in range(0, 17):                                     # S + kL is reduced, never rejected (Q1)
        x = 12345 + k * L
        if x < 2**256:
            r = (ctypes.c_uint32 * 8)()
            fe.h_sc_reduce256(r, W(x, 8))
            assert V(r) == 12345
    for _ in range(1000):
        a, b, c = rng.getrandbits(256), rng.getrandbits(253), rng.getrandbits(256)
        r = (ctypes.c_uint32 * 8)()
        fe.h_sc_muladd(r, W(a, 8), W(b, 8), W(c, 8))
        assert V(r) == (a * b + c) % L
    for x in [0, 1, L - 1] + [rng.randrange(L) for _ in range(500)]:
        e = (ctypes.c_uint32 * 9)()
        fe.h_sc_recode(e, W(x, 8))
        w = fe.h_comb_w()                                      # signed radix-2^w digits of the fixed-base comb
        rows, half = (255 + w - 1) // w, 1 << (w - 1)
        ds = [((V(e) >> (w * j)) & (2 * half - 1)) - half for j in range(rows)]
        assert V(e) >> (w * rows) == 0
        assert all(-half <= d < half for d in ds) and sum(d * (2 * half)**j for j, d in enumerate(ds)) == x


def test_sha512_prefixed_streams(fe):
    """The register-prefix + global-message formulation equals SHA-512 of the concatenation for every
    length around the block boundaries and for unaligned message pointers."""
    rng = random.Random(5)

    def H(pre, msg, off):
        buf = ctypes.create_string_buffer(len(msg) + off + 32)
        base = ctypes.addressof(buf)
        pad = (-base) % 16 + off
        ctypes.memmove(base + pad, msg, len(msg))
        out = ctypes.create_string_buffer(64)
        fe.h_sha512(out, pre, len(pre), ctypes.c_void_p(base + pad), ctypes.c_uint64(len(msg)))
        return out.raw

    for npre in (0, 32, 64):
        for n in list(range(0, 270)) + [1023, 1024, 1025, 4096]:
            off = rng.choice((0, 0, 1, 4, 8))
            pre, msg = rng.randbytes(npre), rng.randbytes(n)
            assert H(pre, msg, off) == hashlib.sha512(pre + msg).digest(), (npre, n, off)


def test_ops_against_golden(ops):
    """The per-thread operation bodies (ops.cuh) reproduce the reference on the fixtures."""
    out = ctypes.create_string_buffer(32)
    sig = ctypes.create_string_buffer(64)
    point, scalar, result = gu.x25519_kat()
    for i in list(range(0, 1024, 16)):
        ops.hs_x25519(out, scalar[i].tobytes(), point[i].tobytes())
        assert out.raw == result[i].tobytes()
    point, scalar, result = gu.x25519_edge()
    for i in range(len(point)):
        ops.hs_x25519(out, scalar[i].tobytes(), point[i].tobytes())
        assert out.raw == result[i].tobytes()
    sec, pub, sg, msgs = gu.ed25519_kat()
    for i in list(range(0, 1024, 37)) + [111, 112, 127, 128, 239, 240, 1023]:
        ops.hs_genpub(out, sec[i].tobytes())
        assert out.raw == pub[i].tobytes()
        ops.hs_sign(sig, sec[i].tobytes(), pub[i].tobytes(), msgs[i], ctypes.c_uint64(len(msgs[i])))
        assert sig.raw == sg[i].tobytes()
        assert ops.hs_verify(sg[i].tobytes(), pub[i].tobytes(), msgs[i], ctypes.c_uint64(len(msgs[i]))) == 1
    bs, bo = gu.x25519_base_kat()
    for i in range(0, len(bs), 8):
        ops.hs_x25519_base(out, bs[i].tobytes())
        assert out.raw == bo[i].tobytes()
    edsk, edpk, xsk, xpk = gu.convert_kat()
    for i in range(0, len(edsk), 4):
        ops.hs_sk_conv(out, edsk[i].tobytes())
        assert out.raw == xsk[i].tobytes()
        ops.hs_pk_conv(out, edpk[i].tobytes())
        assert out.raw == xpk[i].tobytes()


def test_ops_adversarial_verify(ops):
    sig, pub, msgs, cls, expect = gu.verify_adv()
    bad = []
    for i in list(range(0, len(sig), 3)) + [i for i in range(len(sig)) if cls[i] >= 16]:
        got = ops.hs_verify(sig[i].tobytes(), pub[i].tobytes(), msgs[i], ctypes.c_uint64(len(msgs[i])))
        if got != expect[i]:
            bad.append((i, int(cls[i])))
    assert not bad, bad[:10]
    # the full-length fallback (rho, tau) = (1, t): 64 windows, every signature — it must decide identically
    for i in list(range(0, len(sig), 11)) + [i for i in range(len(sig)) if cls[i] >= 16][::3]:
        got = ops.hs_verify_full(sig[i].tobytes(), pub[i].tobytes(), msgs[i], ctypes.c_uint64(len(msgs[i])))
        assert got == expect[i], (i, int(cls[i]))
        assert ops.device_paths or 56 <= ops.hs_last_nwin() <= 64
    if ops.device_paths:       # the loop with its cp.async staging through shared memory, as k_verify runs it
        for i in list(range(0, len(sig), 7)) + [i for i in range(len(sig)) if cls[i] >= 16][::2]:
            got = ops.hs_verify_staged(sig[i].tobytes(), pub[i].tobytes(), msgs[i], ctypes.c_uint64(len(msgs[i])))
            assert got == expect[i], (i, int(cls[i]))


def wtab_expected(m, e):
    """Entry e of window table m as 96 bytes: (y+x, y-x, 2dxy) of e * 2^(128 m) * B, canonical, from the big-integer model."""
    import edmodel as em
    x, y = em.mul(e << (128 * m), em.B) if e else (0, 1)
    return b"".join(v.to_bytes(32, "little") for v in ((y + x) % em.P, (y - x) % em.P, 2 * em.D * x * y % em.P))


WTAB_SAMPLE = [0, 1, 2, 3, 7, 8, 9, 255, 256, 4095, 4096, 12345, 16384, 32767, 32768]


def test_window_tables_host_build(ops):
    """wtab_base / wtab_build8 (the code k_wtab_base / k_wtab_build run on the device) against the big-integer model."""
    n = ctypes.c_uint32()
    ops.hs_wtab.restype = ctypes.POINTER(ctypes.c_uint32)
    tab = ops.hs_wtab(ctypes.byref(n))
    assert n.value == 32769
    raw = np.ctypeslib.as_array(tab, shape=(2, 32769, 24)).view(np.uint8).reshape(2, 32769, 96)
    rng = random.Random(5)
    for m in range(2):
        for e in WTAB_SAMPLE + [rng.randrange(32769) for _ in range(40)]:
            assert raw[m, e].tobytes() == wtab_expected(m, e), (m, e)


def test_comb_table_host_build(ops):
    """The fixed-base comb table (k_comb_base / k_comb_rows run this code on the device): entry [j][k] =
    (k + 1) * 2^(W j) * B in affine precomputed form, every entry against the big-integer model."""
    import edmodel as em
    rows, entries = ctypes.c_int(), ctypes.c_int()
    ops.hs_comb.restype = ctypes.POINTER(ctypes.c_uint32)
    tab = ops.hs_comb(ctypes.byref(rows), ctypes.byref(entries))
    rows, entries = rows.value, entries.value
    w = entries.bit_length()                                   # entries = 2^(w-1)
    assert rows == (255 + w - 1) // w
    raw = np.ctypeslib.as_array(tab, shape=(rows, entries, 24)).view(np.uint8).reshape(rows, entries, 96)
    em.check_comb_table(raw, w)


def test_tensor_core_lookup_layout(ops):
    """The fragment-order comb table (comb_mma_word, the code k_comb_layout runs) together with the lookup's indexing —
    which thread's product lands in which word of which lane's exchange area — emulated with the PTX fragment layouts
    of mma.sync.m16n8k32.u8: every lane must receive exactly entry |digit| of the row, for every |digit| 0 .. ENTRIES."""
    rows, entries = ctypes.c_int(), ctypes.c_int()
    ops.hs_comb.restype = ctypes.POINTER(ctypes.c_uint32)
    tab = ops.hs_comb(ctypes.byref(rows), ctypes.byref(entries))
    rows, entries = rows.value, entries.value
    if entries < 16:
        pytest.skip("the tensor-core lookup needs rows of 16 or 32 entries")
    std = np.ctypeslib.as_array(tab, shape=(rows, entries, 24))
    rng = random.Random(9)
    out = (ctypes.c_uint32 * (32 * 24))()
    for row in (0, 1, rows // 2, rows - 1):
        for trial in range(3):
            absd = [rng.randrange(entries + 1) for _ in range(32)]
            if trial == 0:
                absd = [(l * 5 + row) % (entries + 1) for l in range(32)]      # every value 0 .. ENTRIES occurs
            ops.hs_mma_select(out, row, (ctypes.c_uint32 * 32)(*absd))
            got = np.ctypeslib.as_array(out).reshape(32, 24)
            for lane, d in enumerate(absd):
                want = std[row, d - 1] if d else np.zeros(24, np.uint32)
                assert (got[lane] == want).all(), (row, lane, d)


def test_half_gcd(ops):
    """hgcd.cuh: (rho, tau) is a lattice vector (tau = rho t mod 8L), rho is odd, and both are short — for random t,
    for structured t (tiny, huge partial quotients, even-rho traps) and for the documented fallback.  Beyond these
    invariants the result is deterministic: it must be exactly the vector a plain extended Euclid on (8L, t) stops at
    (tests/structured_inputs.py: half_gcd_model).  The structured challenges place partial quotients of 2^16 - 1 .. 2^64 at
    chosen continued-fraction depths, so that every rare branch (no Lehmer step, the word-shift loop, the large quotient
    across 2^128, even rho, the rv < 2^96 fallback) is taken a minimum number of times."""
    import structured_inputs as si
    N = 8 * L
    legacy = si.half_gcd_legacy_ts()
    ts = si.half_gcd_inputs()
    counts = si.class_counts(ts)
    print("half_gcd inputs by branch class:", counts)
    assert all(counts[k] >= m for k, m in si.MIN_CLASS_COUNT.items()), counts
    rho = (ctypes.c_uint32 * 8)(); tau = (ctypes.c_uint32 * 8)(); neg = ctypes.c_uint32()
    worst = 0; falls = 0
    legacy_set = set(legacy)
    for t in ts:
        tw = (ctypes.c_uint32 * 8)(*[(t >> (32 * i)) & 0xffffffff for i in range(8)])
        ops.hs_half_gcd(rho, ctypes.byref(neg), tau, tw)
        r = sum(int(rho[i]) << (32 * i) for i in range(8)); ta = sum(int(tau[i]) << (32 * i) for i in range(8))
        assert rho[6] == 0 and rho[7] == 0 and neg.value in (0, 1), t
        r = -r if neg.value else r
        assert r % 2 == 1, (t, r)
        assert (r * t - ta) % N == 0, (t, r, ta)
        want_r, want_ta, info = si.half_gcd_model(t)
        assert (r, ta) == (want_r, want_ta), (t, r, ta, want_r, want_ta, info)
        if info["fallback"]:
            assert (r, ta) == (1, t)
            falls += t in legacy_set                     # fallback (rho, tau) = (1, t): allowed, must be rare
        else:
            assert ta < 2**128 and abs(r) < 2**160, (t, r, ta)
            if t in legacy_set:
                worst = max(worst, abs(r).bit_length(), ta.bit_length())
    assert falls <= 10, falls                      # only structured t (short even vectors such as t = L - 1) may fall back
    assert worst <= 150, worst


def test_batch_inversion(ops):
    """Montgomery's trick shares one exponentiation among up to EDG_BATCH = 32 values (the shipped batch size); zeros
    (any representative) stay zero and do not poison their neighbours (inv(0) = 0, SURVEY Q7) — including the first
    and the last element, runs of zeros, and an all-zero batch."""
    rng = random.Random(6)
    for cnt in range(1, 33):
        for trial in range(12):
            vals = [rng.getrandbits(256) for _ in range(cnt)]
            for j in range(cnt):
                if rng.random() < 0.25:
                    vals[j] = rng.choice([0, P, 2 * P])
            if trial == 0:
                vals[0] = 0
            elif trial == 1:
                vals[-1] = P
            elif trial == 2:
                vals = [rng.choice([0, P, 2 * P]) for _ in range(cnt)]
            elif trial == 3 and cnt > 9:
                vals[9:] = [0] * (cnt - 9)
            buf = ctypes.create_string_buffer(b"".join(v.to_bytes(32, "little") for v in vals))
            ops.hs_batch_inv(buf, cnt)
            for j, v in enumerate(vals):
                got = int.from_bytes(buf.raw[32 * j:32 * j + 32], "little")
                assert got == pow(v % P, P - 2, P), (cnt, j)
    if ops.device_paths:
        return                  # the operation counters are host-path instrumentation
    m, s = ctypes.c_ulong(), ctypes.c_ulong()
    ops.hs_counts(ctypes.byref(m), ctypes.byref(s), 1)
    buf = ctypes.create_string_buffer(b"".join(rng.getrandbits(255).to_bytes(32, "little") for _ in range(8)))
    ops.hs_batch_inv(buf, 8)
    ops.hs_counts(ctypes.byref(m), ctypes.byref(s), 1)
    assert (m.value, s.value) == (11 + 3 * 8, 254)           # one inversion + 3 multiplications per element


def test_field_op_counts(ops):
    """Field multiplications / squarings executed per operation — the figures the integer-multiply
    roofline in bench.py and DESIGN.md §4 is computed from (reference counts: SURVEY.md §8d)."""
    import bench
    if ops.device_paths:
        pytest.skip("the operation counters are host-path instrumentation")

    def counts():
        m, s = ctypes.c_ulong(), ctypes.c_ulong()
        ops.hs_counts(ctypes.byref(m), ctypes.byref(s), 1)
        return m.value, s.value

    sec, pub, sig, msgs = gu.ed25519_kat()
    out = ctypes.create_string_buffer(64)
    i = 100
    counts()
    ops.hs_genpub(out, sec[i].tobytes())
    assert counts() == bench.OURS_FM_SINGLE["genpub"]
    ops.hs_sign(out, sec[i].tobytes(), pub[i].tobytes(), msgs[i], ctypes.c_uint64(len(msgs[i])))
    assert counts() == bench.OURS_FM_SINGLE["sign"]
    assert ops.hs_verify(sig[i].tobytes(), pub[i].tobytes(), msgs[i], ctypes.c_uint64(len(msgs[i]))) == 1
    assert counts() == bench.verify_fm(ops.hs_last_nwin()) and 32 <= ops.hs_last_nwin() <= 34
    ops.hs_x25519_base(out, sec[i].tobytes())
    assert counts() == bench.OURS_FM_SINGLE["x25519_base"]
    ops.hs_x25519(out, sec[i].tobytes(), pub[i].tobytes())
    assert counts() == bench.OURS_FM_SINGLE["x25519"]
    for op, (m, s) in bench.OURS_FM_SINGLE.items():    # never more field operations than the reference spends
        assert m + s <= bench.REF_FM[op][0] + bench.REF_FM[op][1]


def test_device_path_emulation_detects_a_wrong_carry_chain(tmp_path):
    """Negative control of the "device" flavour: one operand number changed in one carry chain of the rewritten fe.cuh (the
    second product of a multiplication row accumulates into the wrong word) and the multiplication check fails — the PTX
    interpreter really executes the device code's chains."""
    gen = tmp_path / "gen"
    (gen / "tests" / "host_sim").mkdir(parents=True)
    subprocess.run([sys.executable, os.path.join(HS, "ptx_rewrite.py"), os.path.join(ROOT, "libeddsa_b200", "csrc"),
                    str(gen / "libeddsa_b200" / "csrc")], check=True, stdout=subprocess.DEVNULL)
    f = gen / "libeddsa_b200" / "csrc" / "fe.cuh"
    text = f.read_text()
    good = "madc.lo.cc.u32 %2, %10, %13, %2; madc.hi.cc.u32 %3, %10, %13, %3;"
    assert text.count(good) == 1                                 # cmad<4>: the row of four products with a carry-out word
    f.write_text(text.replace(good, "madc.lo.cc.u32 %2, %10, %13, %2; madc.hi.cc.u32 %3, %10, %13, %2;"))
    (gen / "tests" / "host_sim" / "fe_host.cpp").write_text(open(os.path.join(HS, "fe_host.cpp")).read())
    so = tmp_path / "libfe_bad.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-D__CUDA_ARCH__=1000", "-D__CUDACC__",
                    "-include", os.path.join(HS, "ptx_emul.h"), "-o", str(so), str(gen / "tests" / "host_sim" / "fe_host.cpp")], check=True)
    bad = ctypes.CDLL(str(so))
    rng = random.Random(12)
    wrong = 0
    for _ in range(50):
        a, b = rng.getrandbits(256), rng.getrandbits(256)
        wrong += val(call(bad.h_fe_mul, W8(a), W8(b))) % P != a * b % P
    assert wrong > 40


def test_ragged_tile_ordering():
    """kernel_common.cuh: the message kernels visit a tile of consecutive operations of a ragged batch in order of message length
    (ragged_key + the shared-memory bitonic sort block_sort_u32).  The device code, compiled for the host as a block of one
    thread: every operation of the tile is visited exactly once, in non-decreasing (capped) length order; operations past the
    end of the batch sort last; huge lengths saturate instead of overflowing into the index bits."""
    gen = os.path.join(HS, "_ptx")
    os.makedirs(os.path.join(gen, "tests", "host_sim"), exist_ok=True)
    subprocess.run([sys.executable, os.path.join(HS, "ptx_rewrite.py"), os.path.join(ROOT, "libeddsa_b200", "csrc"),
                    os.path.join(gen, "libeddsa_b200", "csrc")], check=True, stdout=subprocess.DEVNULL)
    gsrc = os.path.join(gen, "tests", "host_sim", "kernel_common_host.cpp")
    with open(gsrc, "w") as f:
        f.write(open(os.path.join(HS, "kernel_common_host.cpp")).read())
    so = os.path.join(HS, "libkernel_common_host_ptx.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-D__CUDA_ARCH__=1000", "-D__CUDACC__",
                    "-I" + os.path.join(HS, "fake_cuda"), "-include", os.path.join(HS, "ptx_emul.h"), "-o", so, gsrc], check=True)
    lib = ctypes.CDLL(so)
    lib.hs_tile_order.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int]
    rng = np.random.default_rng(13)
    for bits in (9, 10, 11):
        tile = 1 << bits
        cap = (1 << (32 - bits)) - 2
        for n, base, maxlen in ((tile, 0, 300), (3 * tile + 17, 3 * tile, 5000), (tile + 5, 0, 1), (2 * tile, tile, 0), (tile // 2, 0, 70)):
            lens = rng.integers(0, maxlen + 1, size=n).astype(np.uint64)
            if maxlen == 5000:
                lens[base + 3] = cap + 12345                      # longer than the key can say
                lens[base + 4] = 1 << 40
            off = np.zeros(n + 1, np.uint64)
            off[1:] = np.cumsum(lens)
            keys = np.zeros(tile, np.uint32)
            lib.hs_tile_order(keys.ctypes.data, off.ctypes.data, base, n, bits)
            live = min(tile, n - base)
            assert (np.diff(keys.astype(np.int64)) >= 0).all()
            idx = (keys[:live] & (tile - 1)).astype(np.int64)
            assert sorted(idx.tolist()) == list(range(live))         # every operation of the tile exactly once
            assert (keys[live:] == 0xFFFFFFFF).all()                 # slots past the end of the batch sort last
            want = np.minimum(lens[base + idx], cap).astype(np.int64)
            assert ((keys[:live] >> bits).astype(np.int64) == want).all() and (np.diff(want) >= 0).all()
