"""Generates verify_settle.bin: valid signatures that take every pending-carry settle site of the verify window loops.

EDG_VERIFY_STEP (libeddsa_b200/csrc/ops.cuh) settles the pending carries of its public-data field operations in one
rarely taken branch per group of operations (28 settle sites in 8 groups).  On random data a site of an addition or
subtraction runs with probability about 38 / 2^33 per execution, so honest signatures almost never reach it.  This script
searches numbered candidates with the site probe of tests/host_sim/settle_probe.py (a host build of the headers that counts
each site) and keeps, for every site, the first candidate in index order that takes it with no other flag of its group set
(so that a flag missing from the group's OR changes the result as well as a settle that does not run):

  key    the settle of nt = -t2d (cached addition) depends on the table entry alone: it runs only for a key whose table
         of -A holds an entry with word 0 of t2d in {0} or within 37 of 2^32 (about 1 key in 7 M).  Candidate i is the
         secret key KEY_TAG || i (little-endian u64); the first such key signs the rows and the first pool rows.
  rows   per-signature: that key and one nonce point; candidate i signs the 32-byte message TAG || i.  Only rows whose
         own window count is 33 are kept (a warp runs the maximum of its lanes, and a longer run rescales every later
         value).  Searched with ed25519_verify_loop (cofactorless), until every site is found.
  lanes  batched ZIP215: candidate i is the 8-subset of a pool of POOL honest rows drawn by splitmix64 from i
         (settle_probe.cpp: candidate_lane), all included, under the committed SEED.  Searched with
         ed25519_verify_batched_loop<8> until every site is found.  A lane is kept for a site only when both mutants of
         the site also make its equation fail (a lane can take a site without depending on it: T3 enters the next
         addition only through C = T t2d, and t2d = 0 for an identity entry).  The sites of the base-table step run 16
         times per lane, so this phase needs a few 10^7 lanes: most of the run time.

Candidates are searched in chunks of CHUNK; all workers of a round take consecutive chunks, and a round's hits are merged
in index order, so the output does not depend on the number of workers.  Byte for byte reproducible:
    python tests/golden/make_verify_settle.py [--check]      # --check: compare with the committed file instead of writing

Format (little-endian): b"VSETTLE1", u32 rows, u32 pool, u32 lanes, u32 K, seed[32];
  rows  x (sig[64], pub[32], msg[32], u64 index, u32 taken, u32 alone)      taken / alone: bitmaps of sites
  pool  x (sig[64], pub[32], msg[32])
  lanes x (u64 index, u32 taken, u32 alone, u8 rows[K])                        rows: indices into the pool
"""
import concurrent.futures as cf
import ctypes
import hashlib
import os
import struct
import sys
import tempfile
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "host_sim"))
import edmodel as em  # noqa: E402
import settle_probe  # noqa: E402

OUT = os.path.join(HERE, "verify_settle.bin")
MAGIC = b"VSETTLE1"
TAG = b"verify-settle row message"[:24].ljust(24, b".")
SEED = hashlib.sha256(b"verify-settle batch seed").digest()
KEY_TAG = b"verify-settle secret key"[:24].ljust(24, b".")
POOL = 64
CHUNK = 4096
SITES = settle_probe.SITES


def key(sk):
    """An honest key: a = clamp(SHA-512(sk)), A = a B (prime order); and its nonce r (R = r B)."""
    a, prefix = em.clamp_scalar(sk)
    r = em.h_mod_l(prefix, b"verify-settle nonce")
    return a, prefix, em.enc(em.mul(a, em.B)), r, em.enc(em.mul(r, em.B))


def pool_rows(sk0):
    """POOL honest rows over 8 keys (the first: sk0), each signed as RFC 8032 signs (deterministic nonces)."""
    rows = []
    for k in range(8):
        a, prefix, A, _, _ = key(sk0 if k == 0 else hashlib.sha256(b"verify-settle pool key %d" % k).digest())
        for i in range(POOL // 8):
            msg = hashlib.sha256(b"verify-settle pool %d %d" % (k, i)).digest()
            rows.append((em.sign_with(a, prefix, A, msg), A, msg))
    return rows


def search(call, want_all):
    """First candidate (in index order) per site of want_all: {site: (index, taken, alone)}, searched until every site is
    found.  call(start, count, want) returns the hits of one chunk as (index, taken, alone)."""
    found, start = {}, 0
    workers = os.cpu_count() or 1
    with cf.ThreadPoolExecutor(workers) as ex:
        while len(found) < len(want_all):
            want = sum(1 << s for s in want_all if s not in found)
            chunks = list(ex.map(lambda c: call(start + c * CHUNK, CHUNK, want), range(workers)))
            for hits in chunks:
                for idx, taken, alone in hits:
                    for s in want_all:
                        if s not in found and alone >> s & 1:
                            found[s] = (idx, taken, alone)
            start += workers * CHUNK
    return found, start


def _hits(fn, *args):
    def call(start, count, want):
        idx, tk, al = (np.zeros(count, t) for t in (np.uint64, np.uint32, np.uint32))
        vp = ctypes.c_void_p
        n = fn(*args, ctypes.c_uint64(start), ctypes.c_uint64(count), ctypes.c_uint32(want), vp(idx.ctypes.data), vp(tk.ctypes.data),
               vp(al.ctypes.data), ctypes.c_long(count))
        if n < 0:
            raise SystemExit("a candidate failed to verify")
        return [(int(idx[k]), int(tk[k]), int(al[k])) for k in range(n)]
    return call


def lane_bitmaps(lib, rows):
    """(taken, alone) site bitmaps of the lane of rows [(sig, pub, 32-byte msg)] under SEED."""
    off = np.arange(len(rows) + 1, dtype=np.uint64) * 32
    taken, alone = ctypes.c_uint32(), ctypes.c_uint32()
    ok = lib.sp_batched(b"".join(r[0] for r in rows), b"".join(r[1] for r in rows), b"".join(r[2] for r in rows),
                        ctypes.c_void_p(off.ctypes.data), SEED, ctypes.byref(taken), ctypes.byref(alone))
    assert ok == 1
    return taken.value, alone.value


def generate(log=print):
    with tempfile.TemporaryDirectory() as tmp:
        lib = ctypes.CDLL(settle_probe.build(tmp, "host", opt=["-O3", "-march=native"]))
    lib.sp_init()
    assert lib.sp_sites() == SITES
    K = lib.sp_lane_rows()
    b32 = lambda x: (x % em.L).to_bytes(32, "little")
    t0 = time.time()
    keys = _hits(lib.sp_search_keys, KEY_TAG)
    found, n = search(lambda *c: [(i, 1, 1) for i, _, _ in keys(*c)], [0])
    sk = KEY_TAG + struct.pack("<Q", found[0][0])
    log(f"key: {n} candidates in {time.time() - t0:.0f} s")
    a, _, A, r, R = key(sk)

    t0 = time.time()
    found, n = search(_hits(lib.sp_search_rows, b32(a), b32(r), A, R, TAG), range(SITES))
    log(f"rows: {n} candidates in {time.time() - t0:.0f} s")
    rows = []
    for idx in sorted({v[0] for v in found.values()}):
        msg = TAG + struct.pack("<Q", idx)
        t = em.h_mod_l(R, A, msg)
        sig = R + ((r + t * a) % em.L).to_bytes(32, "little")
        taken, alone = next((v[1], v[2]) for v in found.values() if v[0] == idx)
        rows.append((sig, A, msg, idx, taken, alone))

    pool = pool_rows(sk)
    psig, ppub, pmsg = (b"".join(p[k] for p in pool) for k in range(3))
    t0 = time.time()
    found, n = search(_hits(lib.sp_search_lanes, psig, ppub, pmsg, POOL, SEED), range(SITES))
    log(f"lanes: {n} candidates in {time.time() - t0:.0f} s")
    lanes = []
    for idx in sorted({v[0] for v in found.values()}):
        sel = (ctypes.c_int * K)()
        lib.sp_lane_rows_of(sel, ctypes.c_uint64(idx), POOL)
        taken, alone = lane_bitmaps(lib, [pool[k] for k in sel])
        lanes.append((idx, taken, alone, bytes(list(sel))))

    out = [MAGIC, struct.pack("<4I", len(rows), POOL, len(lanes), K), SEED]
    out += [s + p + m + struct.pack("<QII", i, tk, al) for s, p, m, i, tk, al in rows]
    out += [s + p + m for s, p, m in pool]
    out += [struct.pack("<QII", i, tk, al) + sel for i, tk, al, sel in lanes]
    return b"".join(out)


def load(path=None):
    """(rows, pool, lanes, seed): rows [(sig, pub, msg, index, taken, alone)], pool [(sig, pub, msg)],
    lanes [(index, taken, alone, [pool indices])]."""
    data = open(path or OUT, "rb").read()
    assert data[:8] == MAGIC
    nrows, npool, nlanes, K = struct.unpack_from("<4I", data, 8)
    seed, pos = data[24:56], 56
    rows, pool, lanes = [], [], []
    for _ in range(nrows):
        rows.append((data[pos:pos + 64], data[pos + 64:pos + 96], data[pos + 96:pos + 128]) + struct.unpack_from("<QII", data, pos + 128))
        pos += 144
    for _ in range(npool):
        pool.append((data[pos:pos + 64], data[pos + 64:pos + 96], data[pos + 96:pos + 128]))
        pos += 128
    for _ in range(nlanes):
        i, tk, al = struct.unpack_from("<QII", data, pos)
        lanes.append((i, tk, al, list(data[pos + 16:pos + 16 + K])))
        pos += 16 + K
    assert pos == len(data)
    return rows, pool, lanes, seed


if __name__ == "__main__":
    t0 = time.time()
    blob = generate()
    print(f"{len(blob)} bytes in {time.time() - t0:.0f} s on {os.cpu_count()} threads")
    if "--check" in sys.argv:
        same = open(OUT, "rb").read() == blob
        print("identical to", OUT if same else "DIFFERENT from " + OUT)
        sys.exit(0 if same else 1)
    with open(OUT, "wb") as f:
        f.write(blob)
