"""TEST INFRASTRUCTURE: structured inputs for the scalar code whose rare branches random data almost never reaches.

* challenges t for the half-size verification scalars (libeddsa_b200/csrc/hgcd.cuh: half_gcd), with a plain Euclid on
  (8L, t) that classifies each of them by the branch it drives the device code into;
* values for the verify loop's signed 16-bit recoding (ops.cuh: sc_recode_window);
* targets for the fixed-base comb's signed radix-64 recoding (sc.cuh: sc_recode_comb), reached from outside through
  x25519_base, whose scalar is clamped and reduced mod L by the kernel itself;
* Ed25519 public keys for the key conversion with non-canonical, off-curve and small y.

Used by tests/test_host_sim.py (host builds of the headers), tests/test_gpu_structured.py (the B200) and the emulator scenario
of tests/host_sim/sim_scenarios.py (the real kernels without a GPU).  Everything is deterministic for a given seed.
"""
import random

from edmodel import L, P

N8L = 8 * L
R128, R96 = 1 << 128, 1 << 96
# partial quotients the word-shift and Lehmer limits of half_gcd care about: 16-bit Lehmer cofactor limit, the 32-bit
# leading-word window (V == 0 needs a quotient of about 2^32 or more), and a quotient that spans two whole words
BIG_QUOTIENTS = [2**16 - 1, 2**16, 2**32 - 1, 2**32, 2**33, 2**64]


# ------------------------------------------------------------------------------------------------ half_gcd
def half_gcd_model(t):
    """What half_gcd computes, by the plain extended Euclid on (8L, t): remainders r_j = b_j t (mod 8L), r_0 = 8L, r_1 = t,
    stopped at the first remainder below 2^128.  Odd cofactor: that vector; even cofactor: the next one (then odd), unless
    the remainder is below 2^96, where the next cofactor could exceed 160 bits and the result is (1, t).
    Returns (rho, tau, info) with rho signed and info the branch class of the input (see classify)."""
    r0, r1, b0, b1 = N8L, t, 0, 1
    qs = []
    while r1 >= R128:
        q = r0 // r1
        r0, r1, b0, b1 = r1, r0 - q * r1, b1, b0 - q * b1
        qs.append(q)
    info = {"maxq": max(qs, default=0), "cross_q": qs[-1] if qs else 0, "even": b1 % 2 == 0, "fallback": False, "steps": len(qs)}
    if b1 % 2:
        return b1, r1, info
    if r1 < R96:
        info["fallback"] = True
        return 1, t, info
    q = r0 // r1
    info["maxq"] = max(info["maxq"], q)
    return b0 - q * b1, r0 - q * r1, info


def classify(t):
    """The branch classes of half_gcd an input reaches (a set of names)."""
    _, _, info = half_gcd_model(t)
    c = set()
    if info["maxq"] >= 2**16:
        c.add("quotient >= 2^16")               # no Lehmer step possible: single steps with an under-estimated quotient
    if info["maxq"] >= 2**33:
        c.add("quotient >= 2^33")               # V == 0: the word-shift loop runs
    if info["maxq"] >= 2**64:
        c.add("quotient >= 2^64")               # ... by two words or more
    if info["cross_q"] >= 2**32:
        c.add("large quotient across 2^128")
    if info["even"]:
        c.add("even rho")
    if info["fallback"]:
        c.add("fallback (1, t)")
    return c


# minimum number of inputs of each class in half_gcd_inputs(): the generator provably reaches every branch
MIN_CLASS_COUNT = {"quotient >= 2^16": 100, "quotient >= 2^33": 60, "quotient >= 2^64": 20, "large quotient across 2^128": 40,
                   "even rho": 300, "fallback (1, t)": 20}


def half_gcd_legacy_ts(seed=11):
    """The inputs test_half_gcd has always used: tiny values, neighbours of L and of powers of two, inverses of small numbers
    mod 8L, random values of every size and 3000 uniform challenges."""
    rng = random.Random(seed)
    N = N8L
    ts = [0, 1, 2, 3, 5, 2**127, 2**128 - 1, 2**128, 2**128 + 1, L - 1, L - 2, (N + 1) // 2 % L, (L + 1) // 2, L // 3, L // 5,
          2**200, 2**252, 2**251 + 7, (1 << 129) + 1, N // (2**64 + 13) % L, pow(3, -1, N) % L, pow(5, -1, N) % L,
          pow(2**64 + 1, -1, N) % L, pow(2**126 + 1, -1, N) % L, pow(2**130 + 3, -1, N) % L]
    ts += [rng.getrandbits(k) % L for k in (16, 64, 100, 128, 129, 160, 200, 252) for _ in range(40)]
    ts += [rng.randrange(L) for _ in range(3000)]
    return ts


def _small_quotient(rng):
    return rng.choice((1, 1, 1, 1, 2, 2, 3, 4, 5, 7, 11, 20))


def cf_challenge(qs, rem):
    """The t < L whose Euclid on (8L, t) starts with the partial quotients qs = q_1 .. q_m exactly and whose remainder after
    them is close to rem (below it, if any admissible value is).  None if no such t exists.
    (8L, t) = P (r_m, r_{m+1}) with P = prod [[q, 1], [1, 0]]; 8L = a r_m + b r_{m+1} fixes r_{m+1} modulo a."""
    a, b, c, d = 1, 0, 0, 1
    for q in qs:
        a, b, c, d = a * q + b, a, c * q + d, c
    y0 = N8L * pow(b, -1, a) % a if a > 1 else 0
    ymax = (N8L - 1) // (a + b)                              # r_{m+1} < r_m
    if y0 > ymax:
        return None
    y = y0 + max(0, min(rem, ymax) - y0) // a * a
    x = (N8L - b * y) // a
    t = c * x + d * y
    return t if 0 < t < L else None


def _prefix_to(rng, target_a, first=None):
    """Random small partial quotients (the first one >= 8, so that t < L) while the leading convergent denominator stays
    below target_a."""
    qs = [first if first is not None else rng.randrange(8, 40)]
    a, b = qs[0], 1
    while True:
        q = _small_quotient(rng)
        if a * q + b > target_a:
            return qs
        qs.append(q)
        a, b = a * q + b, a


def half_gcd_structured(seed=12):
    """Challenges with a chosen large partial quotient Q (BIG_QUOTIENTS) placed by its continued-fraction depth: as the first
    quotient, deep above 2^128, at the step that crosses 2^128 (with the next remainder anywhere below 2^128, below 2^96 —
    the fallback when the cofactor is even — or tiny), and right after the crossing."""
    rng = random.Random(seed)
    ts = []
    for Q in BIG_QUOTIENTS:
        for rep in range(24):
            # Q as q_1: t ~ 8L / Q
            t = cf_challenge([Q] + [_small_quotient(rng) for _ in range(rng.randrange(0, 4))], rng.randrange(1, N8L // Q // 2 + 2))
            ts.append(t)
            # Q deep above 2^128: r_m ~ 2^(128 + e) after it
            e = rng.randrange(1, 100)
            qs = _prefix_to(rng, N8L >> (128 + e + Q.bit_length()))
            ts.append(cf_challenge(qs + [Q], rng.getrandbits(128 + e)))
            # Q across 2^128: r_{m-1} ~ Q 2^128, r_m in [2^128, 2^130), r_{m+1} < 2^128 of several sizes
            qs = _prefix_to(rng, N8L >> (129 + Q.bit_length()))
            for rem in (rng.getrandbits(128), rng.getrandbits(120), R96 - 1 - rng.getrandbits(40), rng.getrandbits(90), rng.getrandbits(20)):
                ts.append(cf_challenge(qs + [Q], rem))
                ts.append(cf_challenge(qs + [Q + 1], rem))     # the other parity of the cofactor
            # Q right after the crossing: r_m < 2^128 <= r_{m-1}
            qs = _prefix_to(rng, N8L >> 127)
            ts.append(cf_challenge(qs + [Q], rng.getrandbits(127 - min(Q.bit_length(), 100))))
    return [t for t in ts if t is not None]


def half_gcd_inputs(seed=11, n_random=3000):
    """The full set: the legacy list, the structured challenges, and n_random further uniform t < L (deduplicated)."""
    rng = random.Random(seed + 1000)
    ts = half_gcd_legacy_ts(seed) + half_gcd_structured(seed + 1) + [rng.randrange(L) for _ in range(n_random)]
    seen, out = set(), []
    for t in ts:
        if t not in seen:
            seen.add(t)
            out.append(t)
    return out


def class_counts(ts):
    counts = {k: 0 for k in MIN_CLASS_COUNT}
    for t in ts:
        for c in classify(t):
            counts[c] += 1
    return counts


# ------------------------------------------------------------------------------------------------ verify-loop recoding
def recode_window_values(seed=13, n_random=2000):
    """x < 2^253 for sc_recode_window: 0, 1, L - 1 and values made of runs of the 16-bit digits 0x7fff, 0x8000 and 0xffff
    (where the offset 0x8000 per digit carries or does not), plus random x < L."""
    rng = random.Random(seed)
    xs = [0, 1, 2, L - 1, L - 2, 2**252, 2**252 - 1, 2**253 - 1]
    for d in (0x7FFF, 0x8000, 0xFFFF, 0x0000):
        for lo in range(0, 16, 3):
            for hi in range(lo + 1, 17, 4):
                x = sum(d << (16 * k) for k in range(lo, hi))
                xs.append(x)
                xs.append(x + rng.randrange(1 << (16 * lo)) if lo else x + 1)
    for _ in range(200):
        x = sum(rng.choice((0x7FFF, 0x8000, 0xFFFF, 0, rng.getrandbits(16))) << (16 * k) for k in range(16))
        xs.append(x)
    xs = [x % (1 << 253) for x in xs]
    return xs + [rng.randrange(L) for _ in range(n_random)]


def window_digits(e, nwin=16, w=16):
    """The signed digits a recoded value e holds: ((e >> w k) mod 2^w) - 2^(w-1)."""
    return [((e >> (w * k)) & ((1 << w) - 1)) - (1 << (w - 1)) for k in range(nwin)]


# ------------------------------------------------------------------------------------------------ fixed-base comb
COMB_W, COMB_ROWS = 6, 43


def comb_value(digits):
    return sum(d << (COMB_W * j) for j, d in enumerate(digits))


def comb_targets(seed=14):
    """Residues v in [0, L) whose signed radix-64 recoding (43 digits in [-32, 32)) is structured: small values, 64^k, 64^k - 1
    and 32 * 64^k, single non-zero digits, runs of zero digits, all-31 and all-(-32) low digits under a positive top digit,
    alternating signs, L - 1, L - 2, L - 64^k, and values x = 2^b - 1 (x + 32 sum 64^j carries through every word)."""
    rng = random.Random(seed)
    vs = list(range(0, 65))
    for k in range(43):
        vs += [64**k, 64**k - 1, 32 * 64**k, L - 64**k, 64**k + 1]
        for d in (1, 2, 17, 31, -1, -32):
            if k:
                vs.append((1 << (COMB_W * (k + 1))) + d * 64**k)          # a single non-zero digit under a top digit
            vs.append(d * 64**k if d > 0 else None)
    for lo in range(0, 43, 3):                                             # runs of zero digits inside random digits
        for ln in (1, 5, 12, 30):
            ds = [rng.randrange(-32, 32) for _ in range(42)] + [rng.randrange(0, 2)]
            ds[lo:lo + ln] = [0] * len(ds[lo:lo + ln])
            vs.append(comb_value(ds))
    for k in range(1, 43):
        for top in (1, 2, 31):
            vs.append(comb_value([31] * k + [top]))
            vs.append(comb_value([-32] * k + [top]))
            vs.append(comb_value([31 if j % 2 else -32 for j in range(k)] + [top]))
            vs.append(comb_value([(-1) ** j * rng.randrange(1, 33) for j in range(k)] + [top]))
    vs += [L - 1, L - 2, L - 3, (L - 1) // 2, 2**252, 2**252 - 1]
    vs += [(1 << b) - 1 for b in range(1, 253)]
    # x25519_base reaches v only for v = 2, 4, 5, 7 (mod 8) (see x25519_base_scalar): every target also comes with its lowest
    # digit nudged into one of these classes, which keeps the structure of all the digits above it
    vs += [v + next(c for c in range(8) if (v + c) % 8 in (2, 4, 5, 7)) for v in vs if v is not None]
    out, seen = [], set()
    for v in vs:
        if v is not None and 0 <= v < L and v not in seen:
            seen.add(v)
            out.append(v)
    return out


def comb_digits(v):
    """The recoding the comb computes: e = v + 32 sum_j 64^j, digit_j = ((e >> 6 j) mod 64) - 32."""
    e = v + sum(32 << (COMB_W * j) for j in range(COMB_ROWS))
    assert e >> (COMB_W * COMB_ROWS) == 0
    return [((e >> (COMB_W * j)) & 63) - 32 for j in range(COMB_ROWS)]


def x25519_base_scalar(v, rng):
    """A raw x25519_base scalar whose clamped value s = v + j L lies in [2^254, 2^255) with s = 0 (mod 8): the kernel's
    clamp(s) mod L is then v.  Bit 255 and bits 0..2, which the clamp overwrites, are random.  None if no such j exists
    (half of all v: [2^254, 2^255) holds the four multiples j = 4 .. 7 of L, and s = 0 (mod 8) needs j = 3 v (mod 8), so
    that all but the top ~2^-125 of [0, L) are reachable exactly when v = 2, 4, 5 or 7 (mod 8))."""
    jmin = -(-(2**254 - v) // L)
    cands = [j for j in range(jmin, jmin + 5) if (v + j * L) % 8 == 0 and 2**254 <= v + j * L < 2**255]
    if not cands:
        return None
    s = v + rng.choice(cands) * L
    s |= rng.getrandbits(3) | (rng.getrandbits(1) << 255)
    return s.to_bytes(32, "little")


def clamp_mod_l(raw):
    s = int.from_bytes(raw, "little")
    s &= ~7
    s &= (1 << 255) - 1
    s |= 1 << 254
    return s % L


def comb_batch(seed=16, n_random=1000, limit=None):
    """x25519_base scalars for every reachable comb target (at most `limit` of them) mixed with n_random random scalars, rows
    shuffled so that structured scalars share warps (and so the tensor-core lookup) with random ones.
    Returns (rows: list of 32-byte scalars, targets: v per row or None for the random rows, unreachable: targets dropped)."""
    rng = random.Random(seed)
    rows, targets, unreachable = [], [], 0
    for v in comb_targets(seed):
        s = x25519_base_scalar(v, rng)
        if s is None:
            unreachable += 1
            continue
        rows.append(s)
        targets.append(v)
    if limit is not None:
        rows, targets = rows[:limit], targets[:limit]
    rows += [rng.getrandbits(256).to_bytes(32, "little") for _ in range(n_random)]
    targets += [None] * n_random
    perm = list(range(len(rows)))
    rng.shuffle(perm)
    return [rows[i] for i in perm], [targets[i] for i in perm], unreachable


def x25519_base_model(v):
    """u = (1 + y) / (1 - y) of v * B from the big-integer model, 32 bytes (u = 0 for the identity: inv(0) = 0)."""
    import edmodel as em
    _, y = em.mul(v, em.B) if v else (0, 1)
    return ((1 + y) * em.inv((1 - y) % P) % P).to_bytes(32, "little")


# ------------------------------------------------------------------------------------------------ key conversion
def pk_structured(seed=15, n_random=200):
    """32-byte Ed25519 public keys for the conversion u = (1 + y) / (1 - y): every non-canonical y in [p, 2^255) with both
    sign bits, y in {0, 1, p - 1} and their "-0" encodings (sign bit set with x = 0), y = 2 and other off-curve y, random
    keys (mostly off-curve) and keys of real points."""
    import edmodel as em
    rng = random.Random(seed)
    ys = [(y, s) for y in range(P, 2**255) for s in (0, 1)]
    ys += [(y, s) for y in (0, 1, 2, 3, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2) for s in (0, 1)]
    off = [y for y in range(2, 400) if not em.on_curve_y(y.to_bytes(32, "little"))][:20]
    ys += [(y, rng.getrandbits(1)) for y in off]
    keys = [(y | (s << 255)).to_bytes(32, "little") for y, s in ys]
    keys += [rng.getrandbits(256).to_bytes(32, "little") for _ in range(n_random)]
    keys += [em.enc(em.mul(rng.randrange(1, L), em.B)) for _ in range(20)]
    return keys
