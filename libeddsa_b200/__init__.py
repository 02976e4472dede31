"""libeddsa_b200 — Python binding (ctypes) of the B200-native Ed25519 / X25519 batch engine.

This module is a thin mirror of the C interface (include/eddsa.h, include/eddsa_batch.h): the same
function names, argument order and meaning as the reference's eddsa.h
(/root/reference/lib/eddsa.h:44-81), plus the batch variants.  All arithmetic happens in the CUDA
kernels inside ``libeddsa_b200.so``; there is no Python or CPU implementation behind these calls —
if the shared library is missing, or no CUDA device is usable, they raise.

    import libeddsa_b200 as ed
    pub = ed.ed25519_genpub(sec)                       # bytes in / bytes out, batch of one on the GPU
    ok  = ed.ed25519_verify_batch(sig, pub, msgs, fixed_len=64)     # numpy uint8 arrays, host buffers
    ed.ed25519_verify_batch_dev(ok_t, sig_t, pub_t, msgs_t, fixed_len=64)   # torch CUDA tensors, async
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIBEDDSA_B200_SO") or os.path.join(_HERE, "libeddsa_b200.so")   # override: tuning variants only
_lib = None

ED25519_KEY_LEN = 32
ED25519_SIG_LEN = 64
X25519_KEY_LEN = 32

# acceptance rules of ed25519_verify_policy_batch / _dev (include/eddsa_batch.h: EDDSA_B200_VERIFY_*)
VERIFY_REFERENCE = 0   # libeddsa v0.8, what ed25519_verify_batch decides: S mod L, any A encoding, cofactorless
VERIFY_STRICT = 1      # RFC 8032 with canonical encodings (libsodium): S < L, canonical A and R, no small-order A or R
VERIFY_ZIP215 = 2      # ZIP 215: S < L, any encoding of A and R, cofactored
# signatures per batch equation of ed25519_verify_zip215_batched / _dev (include/eddsa_batch.h: EDDSA_B200_VERIFY_BATCH_ROWS)
VERIFY_BATCH_ROWS = 8


class EddsaB200Error(RuntimeError):
    pass


def build(verbose=False):
    """Compile libeddsa_b200.so in-tree (nvcc, sm_100a).  Works without a GPU."""
    jobs = str(min(8, os.cpu_count() or 1))
    res = subprocess.run(["make", "-C", _HERE, "-j", jobs], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
    if res.returncode != 0:
        raise EddsaB200Error("building libeddsa_b200.so failed")
    return LIB_PATH


def lib():
    """The loaded C library (raises if it has not been built — there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EddsaB200Error(f"{LIB_PATH} not found: run `make -C libeddsa_b200` (or __graft_entry__.build()) first")
        L = ctypes.CDLL(LIB_PATH)
        vp, sz, ip = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
        for name, args in {
            "ed25519_genpub_batch": [sz, vp, vp],
            "ed25519_sign_batch": [sz, vp, vp, vp, vp, vp, sz],
            "ed25519_verify_batch": [sz, vp, vp, vp, vp, vp, sz],
            "ed25519_verify_policy_batch": [sz, vp, vp, vp, vp, vp, sz, ip],
            "ed25519_verify_zip215_batched": [sz, vp, vp, vp, vp, vp, sz, vp],
            "x25519_batch": [sz, vp, vp, vp],
            "x25519_base_batch": [sz, vp, vp],
            "pk_ed25519_to_x25519_batch": [sz, vp, vp],
            "sk_ed25519_to_x25519_batch": [sz, vp, vp],
            "ed25519_genpub_batch_dev": [sz, vp, vp, vp],
            "ed25519_sign_batch_dev": [sz, vp, vp, vp, vp, vp, sz, vp],
            "ed25519_verify_batch_dev": [sz, vp, vp, vp, vp, vp, sz, vp],
            "ed25519_verify_policy_batch_dev": [sz, vp, vp, vp, vp, vp, sz, ip, vp],
            "ed25519_verify_zip215_batched_dev": [sz, vp, vp, vp, vp, vp, sz, vp, vp],
            "x25519_batch_dev": [sz, vp, vp, vp, vp],
            "x25519_base_batch_dev": [sz, vp, vp, vp],
            "pk_ed25519_to_x25519_batch_dev": [sz, vp, vp, vp],
            "sk_ed25519_to_x25519_batch_dev": [sz, vp, vp, vp],
            "eddsa_b200_fe_selftest": [sz, vp, vp, vp, ip],
            "eddsa_b200_sc_selftest": [sz, vp, vp, vp, vp, ip],
            "eddsa_b200_verify_tables": [vp, sz],
            "eddsa_b200_comb_table": [vp, sz],
            "eddsa_b200_debug_peek_staging": [ip, ip, vp, sz],
            "eddsa_b200_init": [],
            "eddsa_b200_device_count": [],
            "eddsa_b200_set_device_count": [ip],
        }.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = ctypes.c_int
        L.eddsa_b200_shutdown.restype = None
        L.eddsa_b200_launch_count.restype = ctypes.c_ulonglong
        L.eddsa_b200_verify_tables.restype = ctypes.c_size_t
        L.eddsa_b200_comb_table.restype = ctypes.c_size_t
        L.eddsa_b200_debug_peek_staging.restype = ctypes.c_size_t
        L.eddsa_b200_last_error.restype = ctypes.c_char_p
        L.ed25519_verify.restype = ctypes.c_bool
        L.ed25519_verify.argtypes = [vp, vp, vp, sz]
        L.ed25519_sign.argtypes = [vp, vp, vp, vp, sz]
        _lib = L
    return _lib


def _check(rc, what):
    if rc != 0:
        msg = lib().eddsa_b200_last_error().decode(errors="replace")
        raise EddsaB200Error(f"{what} failed with code {rc}: {msg}")


def init():
    _check(lib().eddsa_b200_init(), "eddsa_b200_init")


def shutdown():
    lib().eddsa_b200_shutdown()


def device_count():
    return lib().eddsa_b200_device_count()


def set_device_count(count):
    _check(lib().eddsa_b200_set_device_count(count), "eddsa_b200_set_device_count")


def launch_count():
    return int(lib().eddsa_b200_launch_count())


# ------------------------------------------------------------------------------------------------
# host-buffer batch API (numpy)
# ------------------------------------------------------------------------------------------------
def _arr(a, width, name):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.size % width:
        raise ValueError(f"{name}: size {a.size} is not a multiple of {width}")
    return a.reshape(-1, width)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def _msgs(msgs, off, fixed_len, n):
    msgs = np.ascontiguousarray(msgs, dtype=np.uint8).reshape(-1) if msgs is not None else np.zeros(0, np.uint8)
    if off is not None:
        off = np.ascontiguousarray(off, dtype=np.uint64)
        if off.shape != (n + 1,):
            raise ValueError("off must hold n + 1 offsets")
        if n and int(off[-1]) > msgs.size:
            raise ValueError("offsets run past the message blob")
    elif n * fixed_len > msgs.size:
        raise ValueError("message blob shorter than n * fixed_len")
    if msgs.size == 0:
        msgs = np.zeros(16, np.uint8)
    return msgs, off


def ed25519_genpub_batch(sec):
    sec = _arr(sec, 32, "sec")
    pub = np.empty_like(sec)
    _check(lib().ed25519_genpub_batch(len(sec), _p(pub), _p(sec)), "ed25519_genpub_batch")
    return pub


def ed25519_sign_batch(sec, pub, msgs, off=None, fixed_len=0):
    sec, pub = _arr(sec, 32, "sec"), _arr(pub, 32, "pub")
    if len(sec) != len(pub):
        raise ValueError("sec / pub length mismatch")
    msgs, off = _msgs(msgs, off, fixed_len, len(sec))
    sig = np.empty((len(sec), 64), np.uint8)
    _check(lib().ed25519_sign_batch(len(sec), _p(sig), _p(sec), _p(pub), _p(msgs), _p(off), fixed_len), "ed25519_sign_batch")
    return sig


def ed25519_verify_batch(sig, pub, msgs, off=None, fixed_len=0):
    sig, pub = _arr(sig, 64, "sig"), _arr(pub, 32, "pub")
    if len(sig) != len(pub):
        raise ValueError("sig / pub length mismatch")
    msgs, off = _msgs(msgs, off, fixed_len, len(sig))
    ok = np.empty(len(sig), np.uint8)
    _check(lib().ed25519_verify_batch(len(sig), _p(ok), _p(sig), _p(pub), _p(msgs), _p(off), fixed_len), "ed25519_verify_batch")
    return ok


def ed25519_verify_policy_batch(sig, pub, msgs, off=None, fixed_len=0, policy=VERIFY_STRICT):
    """ed25519_verify_batch under the acceptance rule `policy` (VERIFY_REFERENCE, VERIFY_STRICT or VERIFY_ZIP215)."""
    sig, pub = _arr(sig, 64, "sig"), _arr(pub, 32, "pub")
    if len(sig) != len(pub):
        raise ValueError("sig / pub length mismatch")
    msgs, off = _msgs(msgs, off, fixed_len, len(sig))
    ok = np.empty(len(sig), np.uint8)
    _check(lib().ed25519_verify_policy_batch(len(sig), _p(ok), _p(sig), _p(pub), _p(msgs), _p(off), fixed_len, policy),
           "ed25519_verify_policy_batch")
    return ok


def _seed(seed):
    if seed is None:
        return None
    seed = bytes(seed)
    if len(seed) != 32:
        raise ValueError("seed must be 32 bytes")
    return ctypes.create_string_buffer(seed, 32)


def ed25519_verify_zip215_batched(sig, pub, msgs, off=None, fixed_len=0, seed=None):
    """ZIP 215 decisions (equal to ed25519_verify_policy_batch(..., VERIFY_ZIP215)) by randomised batch equations over
    groups of VERIFY_BATCH_ROWS rows.  seed: 32 bytes, or None for fresh random bytes; never a value signers know."""
    sig, pub = _arr(sig, 64, "sig"), _arr(pub, 32, "pub")
    if len(sig) != len(pub):
        raise ValueError("sig / pub length mismatch")
    msgs, off = _msgs(msgs, off, fixed_len, len(sig))
    ok = np.empty(len(sig), np.uint8)
    _check(lib().ed25519_verify_zip215_batched(len(sig), _p(ok), _p(sig), _p(pub), _p(msgs), _p(off), fixed_len, _seed(seed)),
           "ed25519_verify_zip215_batched")
    return ok


def x25519_batch(scalar, point):
    scalar, point = _arr(scalar, 32, "scalar"), _arr(point, 32, "point")
    if len(scalar) != len(point):
        raise ValueError("scalar / point length mismatch")
    out = np.empty_like(scalar)
    _check(lib().x25519_batch(len(scalar), _p(out), _p(scalar), _p(point)), "x25519_batch")
    return out


def x25519_base_batch(scalar):
    scalar = _arr(scalar, 32, "scalar")
    out = np.empty_like(scalar)
    _check(lib().x25519_base_batch(len(scalar), _p(out), _p(scalar)), "x25519_base_batch")
    return out


def pk_ed25519_to_x25519_batch(pk):
    pk = _arr(pk, 32, "pk")
    out = np.empty_like(pk)
    _check(lib().pk_ed25519_to_x25519_batch(len(pk), _p(out), _p(pk)), "pk_ed25519_to_x25519_batch")
    return out


def sk_ed25519_to_x25519_batch(sk):
    sk = _arr(sk, 32, "sk")
    out = np.empty_like(sk)
    _check(lib().sk_ed25519_to_x25519_batch(len(sk), _p(out), _p(sk)), "sk_ed25519_to_x25519_batch")
    return out


def verify_tables():
    """Diagnostic: the device-built window tables of B and 2^128 B as a (2, 32769, 3, 32) uint8 array."""
    out = np.empty((2, 32769, 3, 32), np.uint8)
    got = lib().eddsa_b200_verify_tables(_p(out), out.nbytes)
    if got != out.nbytes:
        raise EddsaB200Error(f"eddsa_b200_verify_tables returned {got}: " + lib().eddsa_b200_last_error().decode(errors="replace"))
    return out


def comb_table():
    """Diagnostic: the device-built fixed-base comb table as a (rows, entries, 96) uint8 array."""
    buf = np.empty(1 << 21, np.uint8)
    got = lib().eddsa_b200_comb_table(_p(buf), buf.nbytes)
    if got == 0 or got % 96:
        raise EddsaB200Error(f"eddsa_b200_comb_table returned {got}: " + lib().eddsa_b200_last_error().decode(errors="replace"))
    shape = {43 * 32: (43, 32), 51 * 16: (51, 16), 64 * 8: (64, 8)}[got // 96]   # comb window W = 6 / 5 / 4 (sc.cuh: EDG_COMB_W)
    return buf[:got].reshape(shape + (96,)).copy()


def peek_staging(which, slot, length):
    """Diagnostic: the first `length` bytes of a staging buffer of the current device (see eddsa_batch.h)."""
    buf = np.zeros(length, np.uint8)
    got = lib().eddsa_b200_debug_peek_staging(which, slot, _p(buf), length)
    return buf[:got]


def sc_selftest(a, b, c, op):
    """Diagnostic: scalar operation `op` on n x 32-byte operands on the device: 0 (a + 2^256 b) mod L, 1 a mod L,
    2 a b + c mod L, 3 tau and 4 |rho| (words 0..5; word 7 = 1 if rho < 0) of the half-size verification scalars of
    t = a < L, 5 a < 2^253 recoded to the verify loop's signed 16-bit digits (a + 2^15 sum_k 2^(16 k))."""
    a, b, c = _arr(a, 32, "a"), _arr(b, 32, "b"), _arr(c, 32, "c")
    out = np.empty_like(a)
    _check(lib().eddsa_b200_sc_selftest(len(a), _p(out), _p(a), _p(b), _p(c), op), "eddsa_b200_sc_selftest")
    return out


def fe_selftest(a, b, op):
    """Diagnostic: field operation `op` on n x 32-byte operands, executed by the device field library."""
    a, b = _arr(a, 32, "a"), _arr(b, 32, "b")
    out = np.empty_like(a)
    _check(lib().eddsa_b200_fe_selftest(len(a), _p(out), _p(a), _p(b), op), "eddsa_b200_fe_selftest")
    return out


# ------------------------------------------------------------------------------------------------
# eddsa.h single-operation API (bytes) — calls the exported C symbols of the same name
# ------------------------------------------------------------------------------------------------
def _buf(b, n, name):
    b = bytes(b)
    if len(b) != n:
        raise ValueError(f"{name} must be {n} bytes")
    return b


def ed25519_genpub(sec):
    out = ctypes.create_string_buffer(32)
    lib().ed25519_genpub(out, _buf(sec, 32, "sec"))
    return out.raw


def ed25519_sign(sec, pub, data):
    out = ctypes.create_string_buffer(64)
    data = bytes(data)
    lib().ed25519_sign(out, _buf(sec, 32, "sec"), _buf(pub, 32, "pub"), data, len(data))
    return out.raw


def ed25519_verify(sig, pub, data):
    data = bytes(data)
    return bool(lib().ed25519_verify(_buf(sig, 64, "sig"), _buf(pub, 32, "pub"), data, len(data)))


def x25519_base(scalar):
    out = ctypes.create_string_buffer(32)
    lib().x25519_base(out, _buf(scalar, 32, "scalar"))
    return out.raw


def x25519(scalar, point):
    out = ctypes.create_string_buffer(32)
    lib().x25519(out, _buf(scalar, 32, "scalar"), _buf(point, 32, "point"))
    return out.raw


def pk_ed25519_to_x25519(pk):
    out = ctypes.create_string_buffer(32)
    lib().pk_ed25519_to_x25519(out, _buf(pk, 32, "pk"))
    return out.raw


def sk_ed25519_to_x25519(sk):
    out = ctypes.create_string_buffer(32)
    lib().sk_ed25519_to_x25519(out, _buf(sk, 32, "sk"))
    return out.raw


# ------------------------------------------------------------------------------------------------
# device-buffer batch API (torch CUDA uint8 tensors; enqueued on torch's current stream)
# ------------------------------------------------------------------------------------------------
def _stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dp(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def ed25519_genpub_batch_dev(pub, sec):
    n = sec.numel() // 32
    _check(lib().ed25519_genpub_batch_dev(n, _dp(pub), _dp(sec), _stream()), "ed25519_genpub_batch_dev")


def ed25519_sign_batch_dev(sig, sec, pub, msgs, off=None, fixed_len=0):
    n = sec.numel() // 32
    _check(lib().ed25519_sign_batch_dev(n, _dp(sig), _dp(sec), _dp(pub), _dp(msgs), _dp(off), fixed_len, _stream()), "ed25519_sign_batch_dev")


def ed25519_verify_batch_dev(ok, sig, pub, msgs, off=None, fixed_len=0):
    n = sig.numel() // 64
    _check(lib().ed25519_verify_batch_dev(n, _dp(ok), _dp(sig), _dp(pub), _dp(msgs), _dp(off), fixed_len, _stream()), "ed25519_verify_batch_dev")


def ed25519_verify_policy_batch_dev(ok, sig, pub, msgs, off=None, fixed_len=0, policy=VERIFY_STRICT):
    n = sig.numel() // 64
    _check(lib().ed25519_verify_policy_batch_dev(n, _dp(ok), _dp(sig), _dp(pub), _dp(msgs), _dp(off), fixed_len, policy, _stream()),
           "ed25519_verify_policy_batch_dev")


def ed25519_verify_zip215_batched_dev(ok, sig, pub, msgs, off=None, fixed_len=0, seed=None):
    n = sig.numel() // 64
    _check(lib().ed25519_verify_zip215_batched_dev(n, _dp(ok), _dp(sig), _dp(pub), _dp(msgs), _dp(off), fixed_len, _seed(seed), _stream()),
           "ed25519_verify_zip215_batched_dev")


def x25519_batch_dev(out, scalar, point):
    n = scalar.numel() // 32
    _check(lib().x25519_batch_dev(n, _dp(out), _dp(scalar), _dp(point), _stream()), "x25519_batch_dev")


def x25519_base_batch_dev(out, scalar):
    n = scalar.numel() // 32
    _check(lib().x25519_base_batch_dev(n, _dp(out), _dp(scalar), _stream()), "x25519_base_batch_dev")


def pk_ed25519_to_x25519_batch_dev(out, pk):
    n = pk.numel() // 32
    _check(lib().pk_ed25519_to_x25519_batch_dev(n, _dp(out), _dp(pk), _stream()), "pk_ed25519_to_x25519_batch_dev")


def sk_ed25519_to_x25519_batch_dev(out, sk):
    n = sk.numel() // 32
    _check(lib().sk_ed25519_to_x25519_batch_dev(n, _dp(out), _dp(sk), _stream()), "sk_ed25519_to_x25519_batch_dev")
