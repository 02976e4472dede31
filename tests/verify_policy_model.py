"""TEST INFRASTRUCTURE: big-integer decision model of the three acceptance rules of ed25519_verify_policy_batch
(include/eddsa_batch.h: REFERENCE = libeddsa's rule, STRICT = RFC 8032 with canonical encodings as libsodium decides,
ZIP215 = Zcash's ZIP 215) and a deterministic generator of the rows the committed verify fixtures lack.

The model decides from the rule table alone, on edmodel.py's curve (constants, point decoding, encodings, torsion points),
with the group law in extended coordinates so that a few thousand rows take seconds:

                 S            A encoding     R encoding       small-order A, R   equation
    REFERENCE    mod L        any            canonical        allowed            S B - t A - R == O
    STRICT       S < L        canonical      canonical        rejected           S B - t A - R == O
    ZIP215       S < L        any            any              allowed            8 (S B - t A - R) == O

t = SHA-512(R || A || M) mod L over the bytes as given; off-curve A or R are rejected by every rule.
"""
import functools
import hashlib

import numpy as np

import edmodel as em
from edmodel import D, L, P

REFERENCE, STRICT, ZIP215 = 0, 1, 2
POLICIES = (REFERENCE, STRICT, ZIP215)
NAMES = {REFERENCE: "reference", STRICT: "strict", ZIP215: "zip215"}

O = (0, 1, 1, 0)


def ext(pt):
    x, y = pt
    return (x, y, 1, x * y % P)


def padd(p, q):
    """Complete addition on -x^2 + y^2 = 1 + d x^2 y^2, extended coordinates (the law ge.cuh implements)."""
    x1, y1, z1, t1 = p
    x2, y2, z2, t2 = q
    a = (y1 - x1) * (y2 - x2) % P
    b = (y1 + x1) * (y2 + x2) % P
    c = 2 * D * t1 * t2 % P
    d = 2 * z1 * z2 % P
    e, f, g, h = b - a, d - c, d + c, b + a
    return (e * f % P, g * h % P, f * g % P, e * h % P)


def pmul(k, p):
    r = O
    while k > 0:
        if k & 1:
            r = padd(r, p)
        p = padd(p, p)
        k >>= 1
    return r


def is_identity(p):
    return p[0] % P == 0 and (p[1] - p[2]) % P == 0


def affine(p):
    zi = pow(p[2], P - 2, P)
    return (p[0] * zi % P, p[1] * zi % P)


def small_order(pt):
    return is_identity(pmul(8, ext(pt)))


def decode(b):
    """32 bytes -> (affine point or None when y is not on the curve, canonical).  Like the reference's decoder: y >= p is
    reduced and x = 0 with the sign bit set stays 0; canonical = the bytes are what encoding the point gives back."""
    v = int.from_bytes(bytes(b), "little")
    y, sign = v & ((1 << 255) - 1), v >> 255
    canon = y < P
    y %= P
    x = em.recover_x(y, sign)
    if x is None:
        return None, False
    if x == 0 and sign:
        canon = False
    return (x, y), canon


def decisions(sig, pub, msg):
    """(REFERENCE, STRICT, ZIP215) decisions for one row."""
    return _decisions(bytes(sig), bytes(pub), bytes(msg))


@functools.lru_cache(maxsize=None)
def _decisions(sig, pub, msg):
    A, a_canon = decode(pub)
    R, r_canon = decode(sig[:32])
    if A is None or R is None:
        return (0, 0, 0)
    s = int.from_bytes(sig[32:], "little")
    t = em.h_mod_l(sig[:32], pub, msg)
    d = padd(padd(pmul(s % L, ext(em.B)), pmul(t, ext(em.neg(A)))), ext(em.neg(R)))
    holds, holds8 = is_identity(d), is_identity(pmul(8, d))
    reference = r_canon and holds
    strict = s < L and a_canon and r_canon and not small_order(A) and not small_order(R) and holds
    zip215 = s < L and holds8
    return (int(reference), int(strict), int(zip215))


def decide_rows(rows):
    """rows: iterable of (sig, pub, msg, cls) -> uint8 array (n, 3) of decisions, columns in POLICIES order."""
    return np.array([decisions(s, p, m) for s, p, m, _ in rows], np.uint8).reshape(-1, 3)


# ------------------------------------------------------------------------------------------------------------------------------
# rows: (sig 64 bytes, pub 32 bytes, msg bytes, class)
# ------------------------------------------------------------------------------------------------------------------------------
def fixture_rows():
    """The committed adversarial fixtures (verify_adv.bin + verify_torsion.bin) and the reference's decisions."""
    import golden_util as gu
    sig, pub, msgs, cls, expect = gu.verify_adv()
    return [(sig[i].tobytes(), pub[i].tobytes(), msgs[i], int(cls[i])) for i in range(len(sig))], expect.astype(np.uint8)


# classes of the generated rows
G_TORSION_R = 101        # honest key, R = r B + T (T one of the 7 nonzero torsion points), signed over those R bytes
G_SMALL_R_ENCODING = 102  # honest key, R a non-canonical or "-0" encoding of a small-order point, S = t a
G_ZIP_ONLY_S_PLUS_L = 103  # each ZIP215-only row with S + L
G_S_BOUNDARY = 104       # S at the boundary of the range check: L - 1, L, L + 1, 2^253, 2^256 - 1 and s + k L
G_MIXED_ORDER_KEY = 105  # canonical mixed-order key a B + T, honest signature

MIN_ROWS = {G_TORSION_R: 56, G_SMALL_R_ENCODING: 48, G_ZIP_ONLY_S_PLUS_L: 150, G_S_BOUNDARY: 40, G_MIXED_ORDER_KEY: 56}


def _key(seed):
    sk = hashlib.sha256(b"verify-policy key %d" % seed).digest()
    a, prefix = em.clamp_scalar(sk)
    return a % L, prefix


def _msg(tag, i):
    return hashlib.sha512(b"verify-policy msg %s %d" % (tag, i)).digest()[: (i * 7) % 70]


def _enc(pt):
    return em.enc(pt)


def _smul_b(k):
    return affine(pmul(k, ext(em.B)))


def small_order_encodings():
    """Every encoding of a small-order point that is not its canonical one and still decodes to it: y + p for y < 19 (both
    sign bits where x = 0, the sign of x otherwise) and "-0" (x = 0 with the sign bit set)."""
    out = []
    for pt in em.small_order_points():
        x, y = pt
        if y < 19:
            out.append(em.enc(pt, noncanonical=True))
            if x == 0:
                out.append(em.enc(pt, noncanonical=True, flip_sign=True))
        if x == 0:
            out.append(em.enc(pt, flip_sign=True))
    return sorted(set(out))


@functools.lru_cache(maxsize=None)
def generated_rows():
    """The deterministic extra rows, as a list of (sig, pub, msg, class); asserts the minimum count of every class."""
    torsion = em.small_order_points()               # k T8, k = 0..7
    rows = []
    # honest key, R = r B + T for each nonzero torsion point T, signed over the bytes of R: S B - t A - R = -T
    for i in range(8):
        a, prefix = _key(i)
        A = _enc(_smul_b(a))
        for k in range(1, 8):
            msg = _msg(b"torsion-r", 8 * i + k)
            r = em.h_mod_l(prefix, msg, bytes([k]))
            R = _enc(affine(padd(pmul(r, ext(em.B)), ext(torsion[k]))))
            s = (r + em.h_mod_l(R, A, msg) * a) % L
            rows.append((R + s.to_bytes(32, "little"), A, msg, G_TORSION_R))
    # honest key, R an alternative encoding of a small-order point, S = t a: S B - t A - R = -R
    encs = small_order_encodings()
    for i in range(8):
        a, _ = _key(100 + i)
        A = _enc(_smul_b(a))
        for j, R in enumerate(encs):
            msg = _msg(b"small-r", 16 * i + j)
            s = em.h_mod_l(R, A, msg) * a % L
            rows.append((R + s.to_bytes(32, "little"), A, msg, G_SMALL_R_ENCODING))
    # canonical mixed-order keys a B + T with honest signatures: S B - t A - R = -t T
    for i in range(8):
        a, prefix = _key(200 + i)
        for k in range(1, 8):
            A = _enc(affine(padd(pmul(a, ext(em.B)), ext(torsion[k]))))
            msg = _msg(b"mixed", 8 * i + k)
            r = em.h_mod_l(prefix, msg)
            R = _enc(_smul_b(r))
            s = (r + em.h_mod_l(R, A, msg) * a) % L
            rows.append((R + s.to_bytes(32, "little"), A, msg, G_MIXED_ORDER_KEY))
    # S at the range check.  The identity key makes the equation hold for every S whatever t is (R = (S mod L) B), so there the
    # range check alone decides; on honest rows S = s + k L keeps the equation and only the range check rejects it
    ident = _enc((0, 1))
    for j, s in enumerate((L - 1, L, L + 1, 2**253, 2**256 - 1, 0, 1, L - 2)):
        for m in range(3):
            R = _enc(_smul_b(s % L))
            rows.append((R + s.to_bytes(32, "little"), ident, _msg(b"bound-ident", 3 * j + m), G_S_BOUNDARY))
    for i in range(8):
        a, prefix = _key(300 + i)
        A = _enc(_smul_b(a))
        msg = _msg(b"bound", i)
        r = em.h_mod_l(prefix, msg)
        R = _enc(_smul_b(r))
        s = (r + em.h_mod_l(R, A, msg) * a) % L
        top = (2**256 - 1 - s) // L
        for S in (s, s + L, s + top * L, L - 1, L, L + 1, 2**253, 2**256 - 1):
            rows.append((R + S.to_bytes(32, "little"), A, msg, G_S_BOUNDARY))
    # every row only ZIP215 accepts (fixtures and the rows above) again with S + L: every rule rejects it
    fx, _ = fixture_rows()
    base = fx + rows
    dec = decide_rows(base)
    for (sig, pub, msg, _), d in zip(base, dec):
        if tuple(d) == (0, 0, 1):
            S = int.from_bytes(sig[32:], "little") + L
            if S < 2**256:
                rows.append((sig[:32] + S.to_bytes(32, "little"), pub, msg, G_ZIP_ONLY_S_PLUS_L))
    counts = {c: sum(1 for r in rows if r[3] == c) for c in MIN_ROWS}
    assert all(counts[c] >= m for c, m in MIN_ROWS.items()), counts
    return rows


@functools.lru_cache(maxsize=None)
def all_rows():
    """Fixture rows followed by generated rows, with the model's decisions (n, 3) and the classes."""
    fx, _ = fixture_rows()
    rows = fx + generated_rows()
    return rows, decide_rows(rows), np.array([r[3] for r in rows], np.int64)


def as_arrays(rows):
    """rows -> (sig (n, 64) uint8, pub (n, 32) uint8, blob uint8, off uint64 (n + 1)) for the batch API (ragged form)."""
    import golden_util as gu
    sig = np.frombuffer(b"".join(r[0] for r in rows), np.uint8).reshape(-1, 64).copy()
    pub = np.frombuffer(b"".join(r[1] for r in rows), np.uint8).reshape(-1, 32).copy()
    blob, off = gu.ragged([r[2] for r in rows])
    if blob.size == 0:
        blob = np.zeros(16, np.uint8)
    return sig, pub, blob, off


def libsodium_decision(sig, pub, msg):
    """crypto_sign_open of PyNaCl (libsodium): 1 if it accepts the signed message."""
    import nacl.bindings as nb
    try:
        nb.crypto_sign_open(bytes(sig) + bytes(msg), bytes(pub))
        return 1
    except Exception:
        return 0
