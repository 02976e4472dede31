"""The public-data flavour of the field arithmetic (fe.cuh: pub_mul, pub_sq, pub_add, pub_sub, pub_neg, pub_dbl with
pub_settle_add / pub_settle_sub, and pub_pow2523) against the constant-time forms, bit for bit, on the host build of the
headers: the portable host paths and the DEVICE paths (inline PTX run by the interpreter of host_sim/ptx_emul.h).

The rare path (a carry or borrow out of word 0 that still has to travel through words 1..7) runs with probability below
4e-7 per operation on random data, so the operands are crafted to take it, and each test asserts how many did.
"""
import ctypes
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from edmodel import P

HS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_sim")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = 0xFFFFFFFF

# op: 0 mul, 1 sq, 2 add, 3 sub, 4 neg, 5 dbl, 6 pow2523.  Per item: both flavours, the public one settled, and its flag.
SHIM = r"""
#include "libeddsa_b200/csrc/fe.cuh"
#include <string.h>
using namespace edg;
extern "C" {
void h_pub_check(int op, long n, const uint32_t *a, const uint32_t *b, uint32_t *r_ct, uint32_t *r_pub, uint8_t *pend) {
    for (long i = 0; i < n; i++) {
        fe x, y, r0, r1;
        memcpy(x.v, a + 8 * i, 32); memcpy(y.v, b + 8 * i, 32);
        bool p = false;
        switch (op) {
        case 0: fe_mul(r0, x, y); p = pub_mul(r1, x, y); pub_settle_add(r1, p); break;
        case 1: fe_sq(r0, x); p = pub_sq(r1, x); pub_settle_add(r1, p); break;
        case 2: fe_add(r0, x, y); p = pub_add(r1, x, y); pub_settle_add(r1, p); break;
        case 3: fe_sub(r0, x, y); p = pub_sub(r1, x, y); pub_settle_sub(r1, p); break;
        case 4: fe_neg(r0, x); p = pub_neg(r1, x); pub_settle_sub(r1, p); break;
        case 5: fe_dbl(r0, x); p = pub_dbl(r1, x); pub_settle_add(r1, p); break;
        default: fe_pow2523(r0, x); pub_pow2523(r1, x); break;
        }
        memcpy(r_ct + 8 * i, r0.v, 32); memcpy(r_pub + 8 * i, r1.v, 32);
        pend[i] = p;
    }
}
// first operand x = base + k (k = 0, 1, ..) in word 0 .. of the seed for which pub_mul(x, y) (op 0) or pub_sq(x) (op 1)
// leaves a pending carry: the multiplication inputs whose rare path is too unlikely to hit by sampling
long h_pub_find(int op, const uint32_t *base, const uint32_t *y_in, long tries, uint32_t *found) {
    fe x, y, r;
    memcpy(x.v, base, 32); memcpy(y.v, y_in, 32);
    for (long k = 0; k < tries; k++) {
        x.v[0] = base[0] + (uint32_t)k;
        x.v[1] = base[1] + (uint32_t)(k >> 20);
        if (op == 0 ? pub_mul(r, x, y) : pub_sq(r, x)) { memcpy(found, x.v, 32); return k; }
    }
    return -1;
}
}
"""


def build_shim(tmp, flavour):
    """The shim above against the headers: flavour "host" (portable paths) or "device" (PTX carry chains, interpreted)."""
    os.makedirs(tmp, exist_ok=True)
    so = os.path.join(tmp, f"libfe_pub_{flavour}.so")
    if flavour == "host":
        src = os.path.join(tmp, "fe_pub_shim.cpp")
        with open(src, "w") as f:
            f.write(SHIM)
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", ROOT, "-o", so, src], check=True)
    else:
        gen = os.path.join(tmp, "gen")
        subprocess.run([sys.executable, os.path.join(HS, "ptx_rewrite.py"), os.path.join(ROOT, "libeddsa_b200", "csrc"),
                        os.path.join(gen, "libeddsa_b200", "csrc")], check=True, stdout=subprocess.DEVNULL)
        src = os.path.join(gen, "fe_pub_shim.cpp")
        with open(src, "w") as f:
            f.write(SHIM)
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-D__CUDA_ARCH__=1000",
                        "-D__CUDACC__", "-include", os.path.join(HS, "ptx_emul.h"), "-I", gen, "-o", so, src], check=True)
    return ctypes.CDLL(so)


def run(lib, op, a, b):
    """(constant-time result, public result, pending flags) of op over the rows of a, b (n x 8 uint32)."""
    a = np.ascontiguousarray(a, dtype=np.uint32)
    b = np.ascontiguousarray(b, dtype=np.uint32)
    n = len(a)
    r_ct = np.zeros((n, 8), np.uint32)
    r_pub = np.zeros((n, 8), np.uint32)
    pend = np.zeros(n, np.uint8)
    vp = ctypes.c_void_p
    lib.h_pub_check(ctypes.c_int(op), ctypes.c_long(n), vp(a.ctypes.data), vp(b.ctypes.data), vp(r_ct.ctypes.data), vp(r_pub.ctypes.data),
                    vp(pend.ctypes.data))
    return r_ct, r_pub, pend


def words(x):
    return [(x >> (32 * i)) & M32 for i in range(8)]


def value(w):
    return sum(int(v) << (32 * i) for i, v in enumerate(w))


def crafted_pairs(seed=1):
    """Operand pairs (a, b) for the add / sub family: word 0 within 38 of 2^32, runs of 0xffffffff words, values in
    [2^256 - 38, 2^256), a - b borrowing into a zero low word, plus random pairs."""
    rng = random.Random(seed)
    top = (1 << 256)
    rows = []
    for d in range(40):
        rows.append((top - 1 - d, top - 1 - rng.randrange(40)))                     # both near 2^256: add wraps twice
        rows.append((top - 1 - d, rng.randrange(1, 80)))                            # a + small crosses 2^256
        rows.append(((M32 - d) | (rng.getrandbits(224) << 32), top - 1 - rng.randrange(38)))
        rows.append((rng.randrange(40), rng.randrange(40, 200)))                    # a - b < 0, zero words above
        rows.append((0, top - 1 - rng.randrange(38)))                               # 0 - b, b in [2^256 - 38, 2^256)
        rows.append((d, top - 1 - d))
        rows.append((rng.randrange(38) << 0, (top - 1) ^ rng.randrange(1 << 5)))
        rows.append(((M32 - rng.randrange(38)) + (((1 << 224) - 1) << 32), 1 + rng.randrange(38)))   # a in [2^256 - 38, 2^256)
    for _ in range(400):
        rows.append((rng.getrandbits(256), rng.getrandbits(256)))
    a = np.array([words(x) for x, _ in rows], np.uint32)
    b = np.array([words(y) for _, y in rows], np.uint32)
    return a, b


def mul_operands(lib, op, count, seed=2):
    """count operands (a, b) for which pub_mul (op 0) / pub_sq (op 1) takes its rare path, found by a scan of word 0."""
    rng = random.Random(seed)
    a_rows, b_rows = [], []
    while len(a_rows) < count:
        base = np.array(words(rng.getrandbits(256) | (1 << 255)), np.uint32)
        y = np.array(words(rng.getrandbits(256) | (1 << 255)), np.uint32)
        found = np.zeros(8, np.uint32)
        k = lib.h_pub_find(ctypes.c_int(op), ctypes.c_void_p(base.ctypes.data), ctypes.c_void_p(y.ctypes.data), ctypes.c_long(1 << 26),
                           ctypes.c_void_p(found.ctypes.data))
        if k >= 0:
            a_rows.append(found.copy())
            b_rows.append(y)
    return np.array(a_rows, np.uint32), np.array(b_rows, np.uint32)


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    return build_shim(str(tmp_path_factory.mktemp("fe_pub_host")), "host")


@pytest.fixture(scope="module")
def mul_rare(host_lib):
    """Operands that take the rare path of pub_mul and of pub_sq (searched once with the fast host build)."""
    return {op: mul_operands(host_lib, op, 6, seed=2 + op) for op in (0, 1)}


@pytest.fixture(scope="module", params=["host", "device"])
def lib(request, tmp_path_factory, host_lib):
    if request.param == "host":
        return host_lib
    return build_shim(str(tmp_path_factory.mktemp("fe_pub_device")), "device")


@pytest.mark.parametrize("op", [2, 3, 4, 5])
def test_add_family_bit_identical(lib, op):
    a, b = crafted_pairs()
    r_ct, r_pub, pend = run(lib, op, a, b)
    assert np.array_equal(r_ct, r_pub)
    # the crafted rows take the rare path; the 400 random rows essentially never do
    assert int(pend[:-400].sum()) >= 20, f"op {op}: only {int(pend.sum())} rare paths taken"
    assert int(pend[-400:].sum()) <= 2
    for i in range(0, len(a), 7):                        # and the results are right modulo p
        x, y, r = value(a[i]), value(b[i]), value(r_pub[i])
        want = {2: x + y, 3: x - y, 4: -x, 5: 2 * x}[op] % P
        assert r % P == want and r < (1 << 256)


@pytest.mark.parametrize("op", [0, 1])
def test_mul_sq_bit_identical(lib, mul_rare, op):
    a_rare, b_rare = mul_rare[op]
    rng = np.random.default_rng(5)
    a = np.concatenate([a_rare, rng.integers(0, 1 << 32, (300, 8), dtype=np.uint32)])
    b = np.concatenate([b_rare, rng.integers(0, 1 << 32, (300, 8), dtype=np.uint32)])
    r_ct, r_pub, pend = run(lib, op, a, b)
    assert np.array_equal(r_ct, r_pub)
    assert int(pend[:len(a_rare)].sum()) == len(a_rare), "every searched operand takes the rare path"
    for i in range(0, len(a), 11):
        x, y, r = value(a[i]), value(b[i]), value(r_pub[i])
        assert r % P == (x * y if op == 0 else x * x) % P


def test_pow2523_bit_identical(lib):
    rng = np.random.default_rng(9)
    a = rng.integers(0, 1 << 32, (6, 8), dtype=np.uint32)
    a[0] = words((1 << 256) - 1)
    a[1] = words(P - 1)
    r_ct, r_pub, _ = run(lib, 6, a, a)
    assert np.array_equal(r_ct, r_pub)
