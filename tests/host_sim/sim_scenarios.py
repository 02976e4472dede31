"""TEST INFRASTRUCTURE: scenarios for the host layer (libeddsa_b200/csrc/host.c) on the CUDA runtime simulator
(tests/host_sim/cudasim.cpp).  tests/test_host_pipeline.py runs each scenario in a fresh interpreter

    python tests/host_sim/sim_scenarios.py <scenario>

because host.c reads its environment once per process.  The product binding (libeddsa_b200/__init__.py) is used as it
is; only its library path is pointed at tests/host_sim/libeddsa_sim.so = host.c + the simulator.  Results are checked
against the CPU reference / oracle (tests/cpu_ref.py).
"""
import ctypes
import os
import sys
import threading

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS):
    if p not in sys.path:
        sys.path.insert(0, p)

SIM_SO = os.environ.get("CUDASIM_SO") or os.path.join(HERE, "libeddsa_sim.so")      # override: the mutants of test_host_pipeline.py
EINVAL = -1
(API_MALLOC, API_MALLOC_HOST, API_MEMCPY_ASYNC, API_MEMSET_ASYNC, API_EVENT_RECORD, API_EVENT_SYNC, API_STREAM_WAIT, API_POOL_ALLOC,
 API_FREE_ASYNC, API_STREAM_CREATE, API_EVENT_CREATE, API_LAUNCH, API_SET_DEVICE, API_POOL_CREATE, API_KERNEL_FAULT, API_STREAM_SYNC) = range(16)
API_NAMES = ["cudaMalloc", "cudaMallocHost", "cudaMemcpyAsync", "cudaMemsetAsync", "cudaEventRecord", "cudaEventSynchronize", "cudaStreamWaitEvent",
             "cudaMallocFromPoolAsync", "cudaFreeAsync", "cudaStreamCreate", "cudaEventCreate", "kernel launch", "cudaSetDevice", "cudaMemPoolCreate",
             "kernel fault", "cudaStreamSynchronize"]
L_X25519, L_X25519_BASE, L_GENPUB, L_SIGN, L_VERIFY, L_PK_CONV, L_SK_CONV, L_FE_TEST, L_SC_TEST, L_TABLES = range(10)
K_DEVICE, K_PINNED = 0, 1
STAT_NAMES = ["h2d_bytes", "d2h_bytes", "h2d_copies", "d2h_copies", "kernels", "pageable_async", "memsets", "dev_allocs", "host_allocs", "pool_allocs",
              "max_chunk_items", "event_syncs"]
P = 2**255 - 19


class Sim:
    """The simulator's control surface + the product binding loaded on top of it."""

    def __init__(self):
        import libeddsa_b200 as ed
        ed.LIB_PATH = SIM_SO
        self.ed = ed
        self.L = L = ed.lib()
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        L.cudasim_error_count.restype = ctypes.c_uint64
        L.cudasim_first_error.restype = ctypes.c_char_p
        L.cudasim_fail.argtypes = [ctypes.c_int, ctypes.c_long]
        L.cudasim_stats.argtypes = [vp]
        L.cudasim_launch_log.argtypes = [vp, sz]
        L.cudasim_launch_log.restype = sz
        L.cudasim_pending_ops.restype = sz
        L.cudasim_live_allocs.argtypes = [ctypes.c_int, vp]
        L.cudasim_live_allocs.restype = sz
        L.cudasim_find.argtypes = [vp, sz, sz]
        L.cudasim_find.restype = sz
        L.cudasim_user_alloc.argtypes = [sz, ctypes.c_int, ctypes.c_int]
        L.cudasim_user_alloc.restype = vp
        L.cudasim_user_free.argtypes = [vp]
        L.cudasim_stream_create.argtypes = [ctypes.c_int]
        L.cudasim_stream_create.restype = vp
        L.cudasim_set_device.argtypes = [ctypes.c_int]
        L.cudasim_config.argtypes = [ctypes.c_int] * 3

    def errors(self):
        return int(self.L.cudasim_error_count())

    def first_error(self):
        return self.L.cudasim_first_error().decode()

    def stats(self):
        buf = (ctypes.c_uint64 * 12)()
        self.L.cudasim_stats(buf)
        return dict(zip(STAT_NAMES, [int(x) for x in buf]))

    def reset(self):
        self.L.cudasim_reset_stats()

    def launches(self, op=None):
        buf = (ctypes.c_uint64 * (3 * 4096))()
        k = self.L.cudasim_launch_log(buf, 4096)
        rows = [(int(buf[3 * i]), int(buf[3 * i + 1]), int(buf[3 * i + 2])) for i in range(min(k, 4096))]
        return [r for r in rows if r[1] != L_TABLES and (op is None or r[1] == op)]

    def pending(self):
        return int(self.L.cudasim_pending_ops())

    def live(self, kind=-1):
        b = ctypes.c_uint64(0)
        k = self.L.cudasim_live_allocs(kind, ctypes.byref(b))
        return int(k), int(b.value)

    def find(self, rows, width=16):
        """How often the first `width` bytes of any of the rows occur in memory the library owns."""
        blob = b"".join(bytes(r[:width]) for r in rows)
        return int(self.L.cudasim_find(blob, len(blob) // width, width))

    def user_array(self, nbytes, kind, dev=0):
        """A caller-owned buffer the simulator knows as page-locked host memory (kind 1) or device memory (kind 0)."""
        p = self.L.cudasim_user_alloc(max(nbytes, 1), kind, dev)
        arr = np.ctypeslib.as_array((ctypes.c_uint8 * max(nbytes, 1)).from_address(p))[:nbytes]
        return arr, p

    def clean(self, pageable_ok=False):
        """After a successful call: no simulator complaints, nothing left queued, no async copy touched pageable memory."""
        assert self.errors() == 0, self.first_error()
        assert self.pending() == 0, f"{self.pending()} operations still queued after the call returned"
        if not pageable_ok:
            assert self.stats()["pageable_async"] == 0, "cudaMemcpyAsync on pageable memory (serialises on real hardware)"


def rng(seed):
    return np.random.default_rng(seed)


def rand_rows(r, n, width=32):
    return r.integers(0, 256, size=(n, width), dtype=np.uint8)


def make_signed(cpu, r, n, fixed_len=None, max_len=0):
    """n key pairs, messages (fixed length or ragged 0..max_len) and their signatures from the CPU checker."""
    sec = rand_rows(r, n)
    pub = cpu.genpub(sec)
    if fixed_len is not None:
        msgs = r.integers(0, 256, size=n * fixed_len, dtype=np.uint8)
        off = None
        sig = cpu.sign(sec, pub, msgs, None, fixed_len)
    else:
        lens = r.integers(0, max_len + 1, size=n)
        off = np.zeros(n + 1, np.uint64)
        off[1:] = np.cumsum(lens)
        msgs = r.integers(0, 256, size=int(off[-1]) + 1, dtype=np.uint8)
        sig = cpu.sign(sec, pub, msgs, off, 0)
    return sec, pub, msgs, off, sig


def mutate(r, sig, pub, frac=0.1):
    """Corrupt a fraction of the rows (signature or key bits); returns the copies."""
    sig, pub = sig.copy(), pub.copy()
    n = len(sig)
    for i in r.choice(n, size=max(1, int(n * frac)), replace=False) if n else []:
        if r.integers(0, 2):
            sig[i, r.integers(0, 64)] ^= 1 << r.integers(0, 8)
        else:
            pub[i, r.integers(0, 32)] ^= 1 << r.integers(0, 8)
    return sig, pub


def eq(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and (a == b).all(), f"{what}: {int((a != b).sum())} bytes differ"


def fe_add_expected(a, b):
    """(a + b) mod p for n x 32-byte little-endian rows, as canonical bytes, compared modulo p by the caller."""
    return [(int.from_bytes(bytes(x), "little") + int.from_bytes(bytes(y), "little")) % P for x, y in zip(a, b)]


def check_fe_add(out, a, b, sample=None):
    idx = range(len(a)) if sample is None else sample
    for i in idx:
        got = int.from_bytes(bytes(out[i]), "little") % P
        want = (int.from_bytes(bytes(a[i]), "little") + int.from_bytes(bytes(b[i]), "little")) % P
        assert got == want, f"fe add row {i}"


# ======================================================================================================================
def scenario_all_ops():
    """Every batch entry point, small and awkward sizes, against the CPU checker; the simulator sees a clean run."""
    from cpu_ref import best_cpu_impl, Oracle
    sim, cpu, orc = Sim(), best_cpu_impl(), Oracle()
    ed = sim.ed
    r = rng(1)
    for n in (0, 1, 2, 31, 32, 33, 257):
        sec, pub, msgs, off, sig = make_signed(cpu, r, n, fixed_len=37)
        eq(ed.ed25519_genpub_batch(sec), pub, f"genpub n={n}")
        sim.clean()
        eq(ed.ed25519_sign_batch(sec, pub, msgs, None, 37), sig, f"sign n={n}")
        sim.clean()
        bad_sig, bad_pub = mutate(r, sig, pub, 0.3) if n else (sig, pub)
        eq(ed.ed25519_verify_batch(bad_sig, bad_pub, msgs, None, 37), cpu.verify(bad_sig, bad_pub, msgs, None, 37), f"verify n={n}")
        sim.clean()
        if n:
            assert ed.ed25519_verify_batch(sig, pub, msgs, None, 37).all()
        pts = rand_rows(r, n)
        eq(ed.x25519_batch(sec, pts), cpu.x25519(sec, pts), f"x25519 n={n}")
        eq(ed.x25519_base_batch(sec), cpu.x25519_base(sec), f"x25519_base n={n}")
        sim.clean()
        pk, sk = ed.pk_ed25519_to_x25519_batch(pub), ed.sk_ed25519_to_x25519_batch(sec)
        for i in range(0, n, 17):
            assert bytes(pk[i]) == orc.pk_to_x25519(bytes(pub[i])) and bytes(sk[i]) == orc.sk_to_x25519(bytes(sec[i]))
        sim.clean()
    # zero-length messages and a NULL blob are legal when nothing is hashed
    sec, pub, msgs, off, sig = make_signed(cpu, r, 5, fixed_len=0)
    eq(ed.ed25519_sign_batch(sec, pub, None, None, 0), sig, "sign of empty messages")
    assert ed.ed25519_verify_batch(sig, pub, None, None, 0).all()
    # offsets that do not start at zero, and a ragged batch whose messages are all empty
    sec, pub, msgs, off, sig = make_signed(cpu, r, 50, max_len=33)
    shifted = np.concatenate([rand_rows(r, 1, 13).reshape(-1), msgs])
    off13 = off + np.uint64(13)
    eq(ed.ed25519_sign_batch(sec, pub, shifted, off13, 0), sig, "sign with offsets starting at 13")
    assert ed.ed25519_verify_batch(sig, pub, shifted, off13, 0).all()
    zero_off = np.full(51, 7, np.uint64)
    empty_sig = cpu.sign(sec, pub, shifted, zero_off, 0)
    eq(ed.ed25519_sign_batch(sec, pub, shifted, zero_off, 0), empty_sig, "ragged sign of empty messages")
    assert ed.ed25519_verify_batch(empty_sig, pub, shifted, zero_off, 0).all()
    sim.clean()
    # argument errors: EINVAL, a message, nothing launched
    L = sim.L
    before = ed.launch_count()
    assert L.ed25519_genpub_batch(3, None, sec.ctypes.data) == EINVAL and b"NULL" in L.eddsa_b200_last_error()
    assert L.ed25519_verify_batch(3, sig.ctypes.data, sig.ctypes.data, pub.ctypes.data, None, None, 5) == EINVAL
    dec = np.array([0, 5, 3, 9], np.uint64)
    assert L.ed25519_verify_batch(3, sig.ctypes.data, sig.ctypes.data, pub.ctypes.data, sig.ctypes.data, dec.ctypes.data, 0) == EINVAL
    assert b"non-decreasing" in L.eddsa_b200_last_error()
    assert ed.launch_count() == before
    sim.clean()


def scenario_chunks():
    """The chunk schedule of run_shard (one simulated SM: a verify wave is 512 signatures, a pass 8192)."""
    from cpu_ref import best_cpu_impl
    assert os.environ.get("CUDASIM_SMS") == "1" and os.environ.get("CUDASIM_DEVICES") == "1"
    sim, cpu = Sim(), best_cpu_impl()
    ed, L = sim.ed, sim.L
    r = rng(2)
    n = 20037
    sec, pub, msgs, off, sig = make_signed(cpu, r, n, fixed_len=64)
    bad_sig, bad_pub = mutate(r, sig, pub, 0.1)
    want = cpu.verify(bad_sig, bad_pub, msgs, None, 64)
    assert 0 < want.sum() < n
    # ordinary memory: chunks of 1, 1, 2, 4, 8 waves, then whole passes
    sim.reset()
    eq(ed.ed25519_verify_batch(bad_sig, bad_pub, msgs, None, 64), want, "verify from pageable memory")
    sim.clean()
    assert [x[2] for x in sim.launches(L_VERIFY)] == [512, 512, 1024, 2048, 4096, 8192, 3653], sim.launches(L_VERIFY)
    st = sim.stats()
    assert st["h2d_bytes"] == n * (64 + 32 + 64) and st["d2h_bytes"] == n and st["d2h_copies"] == 7
    # page-locked caller memory: used directly, chunks of 1, 2, 4, 8 waves, then whole passes
    bufs = {}
    for name, arr in (("sig", bad_sig), ("pub", bad_pub), ("msgs", msgs), ("ok", np.zeros(n, np.uint8))):
        a, p = sim.user_array(arr.nbytes, K_PINNED)
        a[:] = arr.reshape(-1)
        bufs[name] = (a, p)
    sim.reset()
    rc = L.ed25519_verify_batch(n, bufs["ok"][1], bufs["sig"][1], bufs["pub"][1], bufs["msgs"][1], None, 64)
    assert rc == 0, L.eddsa_b200_last_error()
    eq(bufs["ok"][0], want, "verify from page-locked memory")
    sim.clean()
    assert [x[2] for x in sim.launches(L_VERIFY)] == [512, 1024, 2048, 4096, 8192, 4165], sim.launches(L_VERIFY)
    # mixed: only the output is page-locked
    sim.reset()
    bufs["ok"][0][:] = 7
    rc = L.ed25519_verify_batch(n, bufs["ok"][1], bad_sig.ctypes.data, bad_pub.ctypes.data, msgs.ctypes.data, None, 64)
    assert rc == 0
    eq(bufs["ok"][0], want, "verify into a page-locked result array")
    sim.clean()
    # ~1 KB items: copies take as long as the kernels, the chunk size stays constant (a sixteenth of the shard in whole waves)
    n2 = 10000
    sec2, pub2, msgs2, off2, sig2 = make_signed(cpu, r, n2, fixed_len=1024)
    sig2[::7, 3] ^= 4
    sim.reset()
    eq(ed.ed25519_verify_batch(sig2, pub2, msgs2, None, 1024), cpu.verify(sig2, pub2, msgs2, None, 1024), "verify of 1 KB messages")
    sim.clean()
    sizes = [x[2] for x in sim.launches(L_VERIFY)]
    assert sizes == [512] * 19 + [n2 - 19 * 512], sizes
    # the other operations: 65536 items and four times more each chunk when staged; quarters of the shard when page-locked
    n3 = 300000
    a, b = rand_rows(r, n3), rand_rows(r, n3)
    sim.reset()
    out = ed.fe_selftest(a, b, 2)
    check_fe_add(out, a, b, range(0, n3, 997))
    check_fe_add(out, a, b, [65535, 65536, 140535, 140536, n3 - 1])
    sim.clean()
    assert [x[2] for x in sim.launches(L_FE_TEST)] == [65536, 75000, 75000, 75000, 9464], sim.launches(L_FE_TEST)
    pa, pb, po = sim.user_array(a.nbytes, K_PINNED), sim.user_array(b.nbytes, K_PINNED), sim.user_array(a.nbytes, K_PINNED)
    pa[0][:] = a.reshape(-1)
    pb[0][:] = b.reshape(-1)
    sim.reset()
    assert L.eddsa_b200_fe_selftest(n3, po[1], pa[1], pb[1], 2) == 0
    check_fe_add(po[0].reshape(-1, 32), a, b, range(0, n3, 997))
    sim.clean()
    assert [x[2] for x in sim.launches(L_FE_TEST)] == [75000] * 4


def scenario_budget():
    """EDDSA_B200_CHUNK_MB=1: chunks shrink to the staging budget; one item larger than the budget grows the buffers."""
    from cpu_ref import best_cpu_impl
    assert os.environ.get("EDDSA_B200_CHUNK_MB") == "1"
    sim, cpu = Sim(), best_cpu_impl()
    ed = sim.ed
    r = rng(3)
    n = 100000
    a, b = rand_rows(r, n), rand_rows(r, n)
    sim.reset()
    out = ed.fe_selftest(a, b, 2)
    check_fe_add(out, a, b, range(0, n, 499))
    sim.clean()
    sizes = [x[2] for x in sim.launches(L_FE_TEST)]
    assert max(sizes) == 32768 and sum(sizes) == n, sizes      # 2 x 32 bytes per item, 2 MB budget
    # ragged messages, lengths 0..300, one of 3 MB in the middle (over budget: the pipeline drains and re-allocates)
    n = 3000
    sec = rand_rows(r, n)
    pub = cpu.genpub(sec)
    lens = r.integers(0, 301, size=n)
    lens[1234] = 3 << 20
    lens[5] = 0
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum(lens)
    msgs = r.integers(0, 256, size=int(off[-1]), dtype=np.uint8)
    want_sig = cpu.sign(sec, pub, msgs, off, 0)
    sim.reset()
    sig = ed.ed25519_sign_batch(sec, pub, msgs, off, 0)
    eq(sig, want_sig, "ragged sign with a 3 MB message")
    sim.clean()
    assert len(sim.launches(L_SIGN)) >= 3
    bad_sig, bad_pub = mutate(r, sig, pub, 0.2)
    bad_sig[1234, 40] ^= 1
    sim.reset()
    eq(ed.ed25519_verify_batch(bad_sig, bad_pub, msgs, off, 0), cpu.verify(bad_sig, bad_pub, msgs, off, 0), "ragged verify with a 3 MB message")
    sim.clean()
    lg = sim.launches(L_VERIFY)
    assert sum(x[2] for x in lg) == n and any(x[2] == 1 for x in lg), lg       # the big message travels alone


def scenario_multi():
    """Sharding over four simulated devices: contiguous index ranges, fewer devices for small batches, the caller's device kept."""
    from cpu_ref import best_cpu_impl
    assert os.environ.get("CUDASIM_DEVICES") == "4"
    sim, cpu = Sim(), best_cpu_impl()
    ed, L = sim.ed, sim.L
    r = rng(4)
    assert ed.device_count() == 4
    L.cudasim_set_device(3)                                     # the caller works on device 3
    n = 100001
    a, b = rand_rows(r, n), rand_rows(r, n)
    sim.reset()
    out = ed.fe_selftest(a, b, 2)
    check_fe_add(out, a, b, list(range(0, n, 499)) + [24999, 25000, 25001, 50000, 75000, 75001, n - 1])
    sim.clean()
    lg = sorted(sim.launches(L_FE_TEST))
    assert [(d, m) for d, _, m in lg] == [(0, 25000), (1, 25000), (2, 25000), (3, 25001)], lg
    assert L.cudasim_current_device() == 3
    for n_small, want_devs in ((16384, 1), (16385, 2), (40000, 3), (65536, 4)):
        sim.reset()
        out = ed.fe_selftest(a[:n_small], b[:n_small], 3)
        sim.clean()
        assert len({d for d, _, _ in sim.launches(L_FE_TEST)}) == want_devs, (n_small, sim.launches(L_FE_TEST))
    ed.set_device_count(2)
    assert ed.device_count() == 2
    sim.reset()
    sec = rand_rows(r, 40000)
    eq(ed.ed25519_genpub_batch(sec), cpu.genpub(sec), "genpub over two devices")
    sim.clean()
    assert sorted((d, m) for d, _, m in sim.launches(L_GENPUB)) == [(0, 20000), (1, 20000)]
    ed.set_device_count(0)
    assert ed.device_count() == 4
    assert L.eddsa_b200_set_device_count(5) == EINVAL
    # verify with mutated rows over all four devices, ragged messages, result identical to the checker
    n = 50000
    sec, pub, msgs, off, sig = make_signed(cpu, r, n, max_len=40)
    bad_sig, bad_pub = mutate(r, sig, pub, 0.1)
    sim.reset()
    eq(ed.ed25519_verify_batch(bad_sig, bad_pub, msgs, off, 0), cpu.verify(bad_sig, bad_pub, msgs, off, 0), "verify over four devices")
    sim.clean()
    assert {d for d, _, _ in sim.launches(L_VERIFY)} == {0, 1, 2, 3}
    assert L.cudasim_current_device() == 3
    # one shard fails (an allocation on whichever device asks third): the call reports it, the next call is fine
    ed.shutdown()
    L.cudasim_fail(API_MALLOC_HOST, 3)
    ok, off64 = np.zeros(n, np.uint8), np.ascontiguousarray(off, np.uint64)
    assert L.ed25519_verify_batch(n, ok.ctypes.data, bad_sig.ctypes.data, bad_pub.ctypes.data, msgs.ctypes.data, off64.ctypes.data, 0) == 2   # cudaErrorMemoryAllocation
    assert b"cudaMallocHost" in L.eddsa_b200_last_error() and sim.pending() == 0
    L.cudasim_clear_faults()
    eq(ed.ed25519_verify_batch(bad_sig, bad_pub, msgs, off, 0), cpu.verify(bad_sig, bad_pub, msgs, off, 0), "verify after a failed shard")
    sim.clean()
    # a single operation runs on the first configured device and leaves the caller's device alone
    sim.reset()
    assert ed.ed25519_verify(bytes(sig[0]), bytes(pub[0]), bytes(msgs[int(off[0]):int(off[1])]))
    assert [d for d, _, _ in sim.launches()] == [0] and L.cudasim_current_device() == 3


def scenario_device_list():
    """EDDSA_B200_DEVICES="2,0": the shards go to device 2 and device 0, in that order."""
    assert os.environ.get("EDDSA_B200_DEVICES") == "2,0"
    sim = Sim()
    ed = sim.ed
    r = rng(5)
    assert ed.device_count() == 2
    n = 50000
    a, b = rand_rows(r, n), rand_rows(r, n)
    a[:25000, 0] = 1
    a[25000:, 0] = 2
    sim.reset()
    out = ed.fe_selftest(a, b, 2)
    check_fe_add(out, a, b, range(0, n, 211))
    sim.clean()
    assert sorted((d, m) for d, _, m in sim.launches(L_FE_TEST)) == [(0, 25000), (2, 25000)]
    assert sim.live()[0] > 0
    # only devices 2 and 0 have contexts
    ed.shutdown()
    assert sim.live() == (0, 0)


def scenario_scrub():
    """No copy of a secret input or output survives a call in any buffer the library owns (staging slots on both sides,
    kernel scratch) — with EDDSA_B200_DEBUG_NO_SCRUB=1 (negative control) the same search finds them."""
    from cpu_ref import best_cpu_impl
    negative = os.environ.get("EDDSA_B200_DEBUG_NO_SCRUB") == "1"
    sim, cpu = Sim(), best_cpu_impl()
    ed, L = sim.ed, sim.L
    r = rng(6)
    n = 3000
    sec, pub, msgs, off, sig = make_signed(cpu, r, n, fixed_len=20)
    pts = rand_rows(r, n)
    sample = list(range(0, n, 97)) + [n - 1]

    def residue(rows):
        return sim.find([rows[i] for i in sample])

    found = {}
    ed.ed25519_genpub_batch(sec)
    found["genpub"] = residue(sec)
    ed.ed25519_sign_batch(sec, pub, msgs, None, 20)
    found["sign"] = residue(sec)
    out = ed.x25519_batch(sec, pts)
    found["x25519"] = residue(sec)
    found["x25519 out"] = residue(out)
    ed.x25519_base_batch(sec)
    found["x25519_base"] = residue(sec)
    out = ed.sk_ed25519_to_x25519_batch(sec)
    found["sk_convert"] = residue(sec)
    found["sk_convert out"] = residue(out)
    # page-locked caller memory: nothing is staged on the host, the device slots are still wiped
    ps, pp, po = sim.user_array(sec.nbytes, K_PINNED), sim.user_array(pts.nbytes, K_PINNED), sim.user_array(sec.nbytes, K_PINNED)
    ps[0][:] = sec.reshape(-1)
    pp[0][:] = pts.reshape(-1)
    assert L.x25519_batch(n, po[1], ps[1], pp[1]) == 0
    eq(po[0].reshape(-1, 32), cpu.x25519(sec, pts), "x25519 from page-locked memory")
    found["x25519 pinned"] = residue(sec) + residue(po[0].reshape(-1, 32))
    sim.clean()
    # public data is NOT wiped (the search is live): signatures stay in the staging slots after a verify
    ed.ed25519_verify_batch(sig, pub, msgs, None, 20)
    assert residue(sig) > 0
    if negative:
        assert all(v > 0 for v in found.values()), found
    else:
        assert all(v == 0 for v in found.values()), found
    # one device, staging of the last call
    assert len(ed.peek_staging(0, 0, 64)) == 64


def _verify_case(sim, cpu, r, n):
    sec, pub, msgs, off, sig = make_signed(cpu, r, n, max_len=90)
    bad_sig, bad_pub = mutate(r, sig, pub, 0.2)
    return bad_sig, bad_pub, msgs, off, cpu.verify(bad_sig, bad_pub, msgs, off, 0)


def scenario_failures():
    """Every runtime call host.c makes fails once, at every position, during a multi-chunk call and during context creation:
    the call reports the error (never a wrong result), secrets do not linger, nothing leaks, and the next call works."""
    from cpu_ref import best_cpu_impl, Oracle
    assert os.environ.get("CUDASIM_SMS") == "1" and os.environ.get("CUDASIM_RESIDENT") == "32"
    sim, cpu = Sim(), best_cpu_impl()
    ed, L = sim.ed, sim.L
    r = rng(7)
    n = 140
    vsig, vpub, vmsgs, voff, vwant = _verify_case(sim, cpu, r, n)           # a wave is 32: chunks of 32, 32, 64, 12 — every slot is reused
    sec = rand_rows(r, 70000)                                               # sk conversion (secret in AND out): chunks of 65536 + 4464
    ok = np.zeros(n, np.uint8)
    outs = np.zeros_like(sec)
    voff64 = np.ascontiguousarray(voff, np.uint64)
    orc = Oracle()

    def run_verify():
        ok[:] = 9
        return L.ed25519_verify_batch(n, ok.ctypes.data, vsig.ctypes.data, vpub.ctypes.data, vmsgs.ctypes.data, voff64.ctypes.data, 0)

    def run_secret():
        outs[:] = 0
        return L.sk_ed25519_to_x25519_batch(len(sec), outs.ctypes.data, sec.ctypes.data)

    assert run_secret() == 0
    want_out = outs.copy()
    for i in range(0, len(sec), 2003):
        assert bytes(want_out[i]) == orc.sk_to_x25519(bytes(sec[i]))
    assert run_verify() == 0 and (ok == vwant).all()
    tested = lost = 0           # lost: scratch blocks whose cudaFreeAsync was made to fail (nothing the library could do)
    for fresh_context in (False, True):
        for api in range(16):
            nth = 0
            while True:
                nth += 1
                if fresh_context:
                    ed.shutdown()
                    assert sim.live()[0] == lost, f"leak after shutdown: {sim.live()} before {API_NAMES[api]} call {nth}"
                L.cudasim_fail(api, nth)
                rc_v = run_verify()
                rc_g = run_secret() if rc_v == 0 else 0
                where = f"{API_NAMES[api]} call {nth}, fresh context {fresh_context}"
                if rc_v == 0 and rc_g == 0:
                    # the failure was not reached (or hit a call whose error is tolerated): results must be right
                    assert (ok == vwant).all() and (outs == want_out).all(), where
                    L.cudasim_clear_faults()
                    assert sim.errors() == 0, sim.first_error()
                    break
                tested += 1
                lost += api == API_FREE_ASYNC
                assert L.eddsa_b200_last_error() != b"", where
                assert sim.pending() == 0, f"{where}: {sim.pending()} operations left queued after a failed call"
                assert L.cudasim_current_device() == 0, where
                if rc_g:
                    hits = sim.find([sec[i] for i in range(0, len(sec), 101)] + [want_out[i] for i in range(0, len(sec), 101)])
                    assert hits == 0, f"{where}: {hits} secret keys left in library buffers after a failed secret-key call"
                L.cudasim_clear_faults()
                L.cudasim_clear_errors()        # a faulted run may have tripped bounds checks on poisoned data; start clean
                assert run_verify() == 0 and (ok == vwant).all(), f"verify after {where}"
                assert nth < 400, where
    assert run_secret() == 0 and (outs == want_out).all()
    sim.clean()
    assert tested > 60, tested
    print("failure positions exercised:", tested)


def scenario_threads():
    """Four host threads issue mixed batch and single calls at once (two devices): every result is right."""
    from cpu_ref import best_cpu_impl
    sim, cpu = Sim(), best_cpu_impl()
    ed = sim.ed
    r = rng(8)
    cases = []
    for t in range(4):
        n = 20000 + 1000 * t
        sec, pub, msgs, off, sig = make_signed(cpu, r, 1500 + 100 * t, max_len=60)
        bad_sig, bad_pub = mutate(r, sig, pub, 0.2)
        a, b = rand_rows(r, n), rand_rows(r, n)
        cases.append(dict(sec=sec, pub=pub, msgs=msgs, off=off, sig=sig, bad_sig=bad_sig, bad_pub=bad_pub,
                          want=cpu.verify(bad_sig, bad_pub, msgs, off, 0), a=a, b=b, x=cpu.x25519_base(sec[:300])))
    errs = []

    def work(c, t):
        try:
            for it in range(3):
                eq(ed.ed25519_verify_batch(c["bad_sig"], c["bad_pub"], c["msgs"], c["off"], 0), c["want"], f"thread {t} verify")
                eq(ed.ed25519_sign_batch(c["sec"], c["pub"], c["msgs"], c["off"], 0), c["sig"], f"thread {t} sign")
                check_fe_add(ed.fe_selftest(c["a"], c["b"], 2), c["a"], c["b"], range(0, len(c["a"]), 501))
                eq(ed.x25519_base_batch(c["sec"][:300]), c["x"], f"thread {t} x25519_base")
                assert ed.ed25519_genpub(bytes(c["sec"][it])) == bytes(c["pub"][it])
        except BaseException as e:      # noqa: BLE001 — reported by the main thread
            errs.append(e)

    th = [threading.Thread(target=work, args=(c, t)) for t, c in enumerate(cases)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errs, errs
    sim.clean()


def scenario_dev_api():
    """The device-pointer entry points: asynchronous on the caller's stream, scratch from the pool, argument checks."""
    from cpu_ref import best_cpu_impl
    sim, cpu = Sim(), best_cpu_impl()
    ed, L = sim.ed, sim.L
    r = rng(9)
    n = 2500
    sec, pub, msgs, off, sig = make_signed(cpu, r, n, max_len=70)
    bad_sig, bad_pub = mutate(r, sig, pub, 0.2)
    want = cpu.verify(bad_sig, bad_pub, msgs, off, 0)
    off64 = np.ascontiguousarray(off, np.uint64)

    def dev(arr):
        a, p = sim.user_array(arr.nbytes + 16, K_DEVICE)           # + 16: the kernels' 128-bit loads may run past the blob
        a[:arr.nbytes] = arr.view(np.uint8).reshape(-1)
        return a, p

    d_sig, d_pub, d_msgs, d_off, d_sec = dev(bad_sig), dev(bad_pub), dev(msgs), dev(off64), dev(sec)
    d_ok, d_out, d_sig2 = sim.user_array(n, K_DEVICE), sim.user_array(32 * n, K_DEVICE), sim.user_array(64 * n, K_DEVICE)
    s1, s2 = L.cudasim_stream_create(0), L.cudasim_stream_create(0)
    sim.reset()
    before = ed.launch_count()
    assert L.ed25519_verify_batch_dev(n, d_ok[1], d_sig[1], d_pub[1], d_msgs[1], d_off[1], 0, s1) == 0
    assert L.ed25519_genpub_batch_dev(n, d_out[1], d_sec[1], s2) == 0
    if os.environ.get("CUDASIM_SCHEDULE", "lazy") == "lazy":
        assert sim.pending() > 0 and (d_ok[0] == 0xCC).all()         # nothing has run: the calls only enqueue
    L.cudasim_sync_all()
    eq(d_ok[0], want, "verify_batch_dev")
    eq(d_out[0].reshape(-1, 32), pub, "genpub_batch_dev")
    assert ed.launch_count() - before == 5
    d_pub2 = dev(pub)
    assert L.ed25519_sign_batch_dev(n, d_sig2[1], d_sec[1], d_pub2[1], d_msgs[1], d_off[1], 0, None) == 0     # default stream
    assert L.x25519_base_batch_dev(n, d_out[1], d_sec[1], s1) == 0
    L.cudasim_sync_all()
    eq(d_sig2[0].reshape(-1, 64), sig, "sign_batch_dev")
    eq(d_out[0].reshape(-1, 32), cpu.x25519_base(sec), "x25519_base_batch_dev")
    assert L.x25519_batch_dev(n, d_out[1], d_sec[1], d_pub2[1], s2) == 0
    L.cudasim_sync_all()
    eq(d_out[0].reshape(-1, 32), cpu.x25519(sec, pub), "x25519_batch_dev")
    assert L.pk_ed25519_to_x25519_batch_dev(n, d_out[1], d_pub2[1], s2) == 0 and L.sk_ed25519_to_x25519_batch_dev(n, d_sig2[1], d_sec[1], s1) == 0
    L.cudasim_sync_all()
    eq(d_out[0].reshape(-1, 32), ed.pk_ed25519_to_x25519_batch(pub), "pk conversion, device API vs host API")
    sim.clean()
    st = sim.stats()
    assert st["pool_allocs"] == 3 and st["dev_allocs"] <= 6 + 2, st      # scratch of verify, genpub, sign from the pool
    # argument checks: nothing launched, EINVAL
    before = ed.launch_count()
    assert L.ed25519_verify_batch_dev(n, d_ok[1], d_sig[1] + 8, d_pub[1], d_msgs[1], d_off[1], 0, s1) == EINVAL
    assert L.ed25519_verify_batch_dev(n, d_ok[1], d_sig[1], None, d_msgs[1], d_off[1], 0, s1) == EINVAL
    assert L.ed25519_verify_batch_dev(n, d_ok[1], d_sig[1], d_pub[1], None, d_off[1], 0, s1) == EINVAL
    assert L.ed25519_genpub_batch_dev(n, d_out[1] + 4, d_sec[1], s1) == EINVAL
    assert L.ed25519_sign_batch_dev(n, d_sig2[1], d_sec[1], None, d_msgs[1], d_off[1], 0, s1) == EINVAL
    assert L.x25519_batch_dev(n, d_out[1], d_sec[1], None, s1) == EINVAL
    assert L.ed25519_verify_batch_dev(0, None, None, None, None, None, 0, s1) == 0
    assert L.ed25519_verify_batch_dev(n - 3, d_ok[1] + 3, d_sig[1], d_pub[1], d_msgs[1], d_off[1], 0, s1) == 0   # the flags: any alignment
    L.cudasim_sync_all()
    eq(d_ok[0][3:], want[:-3], "verify flags at an odd address")
    assert ed.launch_count() == before + 3 and sim.errors() == 0, sim.first_error()
    # batches larger than a pass reuse one scratch allocation of min(n, pass) records
    big = 2 * 2 * 512 * 16 + 100                                     # two simulated SMs: a pass is 16384 signatures
    reps = -(-big // n)
    t_sig, t_pub = np.tile(bad_sig, (reps, 1))[:big], np.tile(bad_pub, (reps, 1))[:big]
    fixed = r.integers(0, 256, size=big * 8, dtype=np.uint8)
    e_sig, e_pub, e_msgs, e_ok = dev(t_sig), dev(t_pub), dev(fixed), sim.user_array(big, K_DEVICE)
    sim.reset()
    assert L.ed25519_verify_batch_dev(big, e_ok[1], e_sig[1], e_pub[1], e_msgs[1], None, 8, s2) == 0
    L.cudasim_sync_all()
    assert not e_ok[0].any() and sim.stats()["pool_allocs"] == 1
    sim.clean()


def scenario_lifecycle():
    """init / shutdown / re-initialisation: nothing the library allocated survives a shutdown; the single-operation API and the
    obsolete aliases (reference eddsa.h:84-114) give the reference's results."""
    from cpu_ref import best_cpu_impl, Oracle
    sim, cpu, orc = Sim(), best_cpu_impl(), Oracle()
    ed, L = sim.ed, sim.L
    r = rng(10)
    ed.init()
    assert ed.device_count() == int(os.environ.get("CUDASIM_DEVICES", "4"))
    assert sim.live(K_PINNED) == (0, 0)                              # contexts without staging buffers
    sec, pub, msgs, off, sig = make_signed(cpu, r, 8, max_len=200)
    for i in range(8):
        m = bytes(msgs[int(off[i]):int(off[i + 1])])
        assert ed.ed25519_genpub(bytes(sec[i])) == bytes(pub[i])
        assert ed.ed25519_sign(bytes(sec[i]), bytes(pub[i]), m) == bytes(sig[i])
        assert ed.ed25519_verify(bytes(sig[i]), bytes(pub[i]), m)
        assert not ed.ed25519_verify(bytes(sig[i]), bytes(pub[i]), m + b"x")
        assert ed.x25519_base(bytes(sec[i])) == bytes(cpu.x25519_base(sec[i:i + 1])[0])
        assert ed.x25519(bytes(sec[i]), bytes(pub[i])) == bytes(cpu.x25519(sec[i:i + 1], pub[i:i + 1])[0])
        assert ed.pk_ed25519_to_x25519(bytes(pub[i])) == orc.pk_to_x25519(bytes(pub[i]))
        assert ed.sk_ed25519_to_x25519(bytes(sec[i])) == orc.sk_to_x25519(bytes(sec[i]))
    out32, out64 = ctypes.create_string_buffer(32), ctypes.create_string_buffer(64)
    m0 = bytes(msgs[int(off[0]):int(off[1])])
    L.eddsa_genpub(out32, bytes(sec[0]))
    assert out32.raw == bytes(pub[0])
    L.eddsa_sign(out64, bytes(sec[0]), bytes(pub[0]), m0, ctypes.c_size_t(len(m0)))
    assert out64.raw == bytes(sig[0])
    L.eddsa_verify.restype = ctypes.c_bool
    assert L.eddsa_verify(bytes(sig[0]), bytes(pub[0]), m0, ctypes.c_size_t(len(m0)))
    L.DH(out32, bytes(sec[0]), bytes(pub[1]))
    assert out32.raw == bytes(cpu.x25519(sec[0:1], pub[1:2])[0])
    L.eddsa_pk_eddsa_to_dh(out32, bytes(pub[0]))
    assert out32.raw == orc.pk_to_x25519(bytes(pub[0]))
    L.eddsa_sk_eddsa_to_dh(out32, bytes(sec[0]))
    assert out32.raw == orc.sk_to_x25519(bytes(sec[0]))
    # NULL data with length 0 is what the reference's callers pass for an empty message
    L.ed25519_sign(out64, bytes(sec[0]), bytes(pub[0]), None, 0)
    assert out64.raw == bytes(cpu.sign(sec[0:1], pub[0:1], np.zeros(1, np.uint8), None, 0)[0])
    assert L.ed25519_verify(out64.raw, bytes(pub[0]), None, 0)
    sim.clean()
    for round_ in range(3):
        assert sim.live()[0] > 0
        ed.shutdown()
        assert sim.live() == (0, 0) and sim.pending() == 0, sim.live()
        ed.shutdown()                                                # twice is harmless
        eq(ed.ed25519_genpub_batch(sec), pub, "genpub after a shutdown")
    # the tables the kernels read, through the diagnostic readers (checked against the big-integer model by test_host_sim)
    import edmodel as em
    em.check_comb_table(ed.comb_table(), 6)
    t = ed.verify_tables()
    assert t.shape == (2, 32769, 3, 32) and not t[0, 0, 2].any()
    sim.clean()


def scenario_copy_helpers():
    """Staging copies of 8 MB and more are split over helper threads (EDDSA_B200_COPY_THREADS=3); the helpers are stopped by a
    shutdown and re-created afterwards without replaying the last request of their predecessors."""
    assert os.environ.get("EDDSA_B200_COPY_THREADS") == "3"
    sim = Sim()
    ed = sim.ed
    r = rng(11)
    n = 1200000
    for round_ in range(3):
        a, b = rand_rows(r, n), rand_rows(r, n)
        sim.reset()
        out = ed.fe_selftest(a, b, 2)
        check_fe_add(out, a, b, list(range(0, n, 4001)) + [65535, 65536, 65536 + 262143, 65536 + 262144, n - 1])
        sim.clean()
        sizes = [x[2] for x in sim.launches(L_FE_TEST)]
        assert sizes[:3] == [65536, 262144, 300000] and sum(sizes) == n, sizes      # 262144 x 32 bytes = 8 MB: the helpers' threshold
        del a, b, out
        ed.shutdown()
        assert sim.live() == (0, 0)


def scenario_fuzz():
    """A random walk over the C-ABI: random operations, sizes, message layouts, page-locked / ordinary buffers, device counts,
    caller devices, shutdowns and injected runtime failures (seed: argv[2]).  Every successful call is checked against the
    CPU reference; every failed call must leave nothing queued, no secret behind, and a working library."""
    import hashlib
    from cpu_ref import best_cpu_impl
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    steps = int(sys.argv[3]) if len(sys.argv) > 3 else 60
    assert os.environ.get("CUDASIM_RESIDENT") == "32" and os.environ.get("CUDASIM_SMS") == "1"      # a verify wave is 32 signatures
    sim, cpu = Sim(), best_cpu_impl()
    ed, L = sim.ed, sim.L
    r = rng(1000 + seed)
    ndev = ed.device_count()
    pool = make_signed(cpu, r, 700, max_len=120)                     # material for sign / verify calls
    psec, ppub, pmsgs, poff, psig = pool
    log, lost_blocks = [], 0       # lost: scratch blocks whose cudaFreeAsync was made to fail (they stay allocated for good)

    def buf(arr, pinned):
        """The array as the caller's buffer: ordinary numpy memory or memory the simulator knows as page-locked."""
        arr = np.ascontiguousarray(arr)
        if not pinned:
            return arr, arr.ctypes.data, None
        a, p = sim.user_array(arr.nbytes, K_PINNED)
        a[:] = arr.view(np.uint8).reshape(-1)
        return a, p, p

    def sk_expected(sec):
        out = np.zeros_like(sec)
        for i, k in enumerate(sec):
            h = bytearray(hashlib.sha512(bytes(k)).digest()[:32])
            h[0] &= 248
            h[31] = (h[31] & 127) | 64
            out[i] = np.frombuffer(bytes(h), np.uint8)
        return out

    for step in range(steps):
        what = r.choice(["fe_add", "fe_add", "sk_conv", "sk_conv", "verify", "verify", "sign", "x25519_base", "shutdown", "devices", "dev_api"])
        if what == "shutdown":
            ed.shutdown()
            assert sim.live()[0] == lost_blocks, (step, sim.live(), lost_blocks)
            continue
        if what == "devices":
            ed.set_device_count(int(r.integers(0, ndev + 1)))
            continue
        caller_dev = int(r.integers(0, ndev))
        L.cudasim_set_device(caller_dev)
        if what == "dev_api":
            # the device-pointer entry points on the caller's current device and a stream of its own: verify + genpub
            n = int(r.choice([1, 33, 200]))
            lo = int(r.integers(0, 700 - n + 1))
            off = np.ascontiguousarray(poff[lo:lo + n + 1], np.uint64)
            bad_sig, bad_pub = mutate(r, psig[lo:lo + n], ppub[lo:lo + n], 0.25)
            want = cpu.verify(bad_sig, bad_pub, pmsgs, off, 0)
            devs = []

            def dev(arr, pad=16):
                arr = np.ascontiguousarray(arr)
                a, p = sim.user_array(arr.nbytes + pad, K_DEVICE, caller_dev)
                a[:arr.nbytes] = arr.view(np.uint8).reshape(-1)
                devs.append(p)
                return a, p

            d_sig, d_pub, d_msgs, d_off, d_sec = dev(bad_sig), dev(bad_pub), dev(pmsgs), dev(off), dev(psec[lo:lo + n])
            d_ok, d_out = dev(np.zeros(n, np.uint8), 0), dev(np.zeros((n, 32), np.uint8), 0)
            st = L.cudasim_stream_create(caller_dev)
            fail_api, fail_nth = (int(r.choice([API_POOL_ALLOC, API_LAUNCH, API_MALLOC])), int(r.integers(1, 3))) if r.random() < 0.3 else (-1, 0)
            if fail_api >= 0:
                L.cudasim_fail(fail_api, fail_nth)
            rc1 = L.ed25519_verify_batch_dev(n, d_ok[1], d_sig[1], d_pub[1], d_msgs[1], d_off[1], 0, st)
            rc2 = L.ed25519_genpub_batch_dev(n, d_out[1], d_sec[1], st)
            L.cudasim_clear_faults()
            L.cudasim_sync_all()
            where = f"seed {seed} step {step}: dev_api n={n} fail={fail_api, fail_nth} rc={rc1, rc2}"
            assert fail_api >= 0 or (rc1, rc2) == (0, 0), where
            if rc1 == 0:
                eq(d_ok[0][:n], want, where + " verify_batch_dev")
            if rc2 == 0:
                eq(d_out[0][:32 * n].reshape(-1, 32), ppub[lo:lo + n], where + " genpub_batch_dev")
            assert sim.pending() == 0 and sim.errors() == 0, where + " " + sim.first_error()
            assert L.cudasim_current_device() == caller_dev, where
            for p_ in devs:
                L.cudasim_user_free(p_)
            log.append((step, what, n, [], fail_api, fail_nth))
            continue
        fail_api, fail_nth = (int(r.integers(0, 16)), int(r.integers(1, 25))) if r.random() < 0.3 else (-1, 0)
        if fail_api == API_SET_DEVICE:
            fail_nth = 1            # a later cudaSetDevice is the one that RESTORES the caller's device: nothing could be done about that
        pins = [bool(r.integers(0, 2)) for _ in range(5)]
        frees, secrets = [], []
        if what == "fe_add":
            n = int(r.choice([0, 1, 777, 16384, 16385, 65537, 150001]))
            a, b = rand_rows(r, n), rand_rows(r, n)
            (A, pa, fa), (B, pb, fb), (O, po, fo) = buf(a, pins[0]), buf(b, pins[1]), buf(np.zeros_like(a), pins[2])
            frees += [fa, fb, fo]
            call = lambda: L.eddsa_b200_fe_selftest(n, po, pa, pb, 2)
            check = lambda: check_fe_add(O.reshape(-1, 32), a, b, sorted(set(int(x) for x in r.integers(0, n, 60))) + [0, n - 1] if n else [])
        elif what == "sk_conv":
            n = int(r.choice([1, 33, 5000, 16385, 70001]))
            sec = rand_rows(r, n)
            want = sk_expected(sec)
            (S, ps, fs), (O, po, fo) = buf(sec, pins[0]), buf(np.zeros_like(sec), pins[1])
            frees += [fs, fo]
            secrets = [sec[i] for i in range(0, n, max(1, n // 40))] + [want[i] for i in range(0, n, max(1, n // 40))]
            call = lambda: L.sk_ed25519_to_x25519_batch(n, po, ps)
            check = lambda: eq(O.reshape(-1, 32), want, "sk conversion")
        elif what == "x25519_base":
            n = int(r.choice([1, 40, 300]))
            sec = rand_rows(r, n)
            want = cpu.x25519_base(sec)
            (S, ps, fs), (O, po, fo) = buf(sec, pins[0]), buf(np.zeros_like(sec), pins[1])
            frees += [fs, fo]
            secrets = [sec[i] for i in range(0, n, 7)]
            call = lambda: L.x25519_base_batch(n, po, ps)
            check = lambda: eq(O.reshape(-1, 32), want, "x25519_base")
        else:
            n = int(r.choice([1, 31, 32, 33, 100, 257, 700]))
            lo = int(r.integers(0, 700 - n + 1))
            sec, pub, sig = psec[lo:lo + n], ppub[lo:lo + n], psig[lo:lo + n]
            if r.random() < 0.5:                                     # ragged, offsets not starting at zero
                off = np.ascontiguousarray(poff[lo:lo + n + 1], np.uint64)
                msgs, fixed = pmsgs, 0
                (OFF, poffp, foff) = buf(off, False)
                want_sig = sig
            else:
                fixed = int(r.choice([0, 1, 64, 200]))
                msgs, off, poffp = r.integers(0, 256, size=max(1, n * fixed), dtype=np.uint8), None, None
                want_sig = cpu.sign(sec, pub, msgs, None, fixed)
            (M, pm, fm) = buf(msgs, pins[3])
            frees += [fm]
            if what == "sign":
                (S, ps, fs), (P_, pp, fp), (O, po, fo) = buf(sec, pins[0]), buf(pub, pins[1]), buf(np.zeros((n, 64), np.uint8), pins[2])
                frees += [fs, fp, fo]
                secrets = [sec[i] for i in range(0, n, 9)]
                call = lambda: L.ed25519_sign_batch(n, po, ps, pp, pm, poffp, fixed)
                check = lambda: eq(O.reshape(-1, 64), want_sig, "sign")
            else:
                bad_sig, bad_pub = mutate(r, want_sig, pub, 0.25)
                want = cpu.verify(bad_sig, bad_pub, msgs, off, fixed)
                (S, ps, fs), (P_, pp, fp), (O, po, fo) = buf(bad_sig, pins[0]), buf(bad_pub, pins[1]), buf(np.full(n, 7, np.uint8), pins[2])
                frees += [fs, fp, fo]
                call = lambda: L.ed25519_verify_batch(n, po, ps, pp, pm, poffp, fixed)
                check = lambda: eq(O, want, "verify")
        log.append((step, what, n, pins, fail_api, fail_nth))
        if fail_api >= 0:
            L.cudasim_fail(fail_api, fail_nth)
        rc = call()
        where = f"seed {seed} step {step}: {log[-1]}"
        lost = fail_api == API_FREE_ASYNC and rc != 0
        if rc == 0:
            check()
            L.cudasim_clear_faults()
            assert sim.errors() == 0, where + " " + sim.first_error()
        else:
            assert fail_api >= 0 and L.eddsa_b200_last_error() != b"", where
            if secrets:
                assert sim.find(secrets) == 0, where + ": secrets left behind by a failed call"
            L.cudasim_clear_faults()
            L.cudasim_clear_errors()
            assert call() == 0, where + " (retry)"
            check()
        assert sim.pending() == 0, where
        assert L.cudasim_current_device() == caller_dev, where
        if secrets and os.environ.get("EDDSA_B200_DEBUG_NO_SCRUB") != "1":
            assert sim.find(secrets) == 0, where + ": secrets left behind"
        for p in frees:
            if p:
                L.cudasim_user_free(p)
        lost_blocks += bool(lost)
    ed.shutdown()
    assert sim.live()[0] == lost_blocks, (sim.live(), lost_blocks)
    print("steps:", len(log), "failures injected:", sum(1 for x in log if x[4] >= 0))


def scenario_real_kernels():
    """The REAL kernels and launchers (libeddsa_b200/csrc/kernels_*.cu, rewritten for the SIMT emulator of simt_emul.h: OS threads
    as lanes, rendezvous for __syncthreads / warp collectives / mma.sync, the PTX interpreter for the carry chains) behind the real
    host layer, on the reference's own vectors and the committed fixtures: passes, tiles sorted by message length, the verify
    permutation, the comb kernel with its tensor-core table lookup, shared inversions — all of it as shipped, without a GPU."""
    import golden_util as gu
    from cpu_ref import best_cpu_impl
    assert "sim_kernels" in SIM_SO and os.environ.get("EDDSA_B200_VERIFY_WAVES") == "1"
    sim, cpu = Sim(), best_cpu_impl()
    ed = sim.ed
    r = rng(21)
    # the reference's x25519 table (1024 rows, 508 of them with bit 255 set) and the edge cases: k_x25519, shared inversions of 32
    point, scalar, result = gu.x25519_kat()
    eq(ed.x25519_batch(scalar, point), result, "x25519 KAT table")
    point, scalar, result = gu.x25519_edge()
    eq(ed.x25519_batch(scalar, point), result, "x25519 edge cases")
    bs, bo = gu.x25519_base_kat()
    eq(ed.x25519_base_batch(bs), bo, "x25519_base fixture")                  # k_comb<1>
    # Ed25519 KAT: 1024 rows, message length = row index (a ragged batch: two tiles of 512 sorted by length)
    sec, pub, sig, msgs = gu.ed25519_kat()
    blob, off = gu.ragged(msgs)
    eq(ed.ed25519_genpub_batch(sec), pub, "genpub KAT")                      # k_expand_key + k_comb<0>
    eq(ed.ed25519_sign_batch(sec, pub, blob, off, 0), sig, "sign KAT")       # k_sign_nonce<1> + k_comb<0> + k_sign_finish<1>
    assert ed.ed25519_verify_batch(sig, pub, blob, off, 0).all()             # k_verify_scalars<1> + k_verify_points + k_verify
    sim.clean()
    # every adversarial row (22 classes incl. torsion): 2960 decisions, three passes of 1024 signatures
    asig, apub, amsgs, cls, expect = gu.verify_adv()
    ablob, aoff = gu.ragged(amsgs)
    got = ed.ed25519_verify_batch(asig, apub, ablob, aoff, 0)
    bad = [(i, int(cls[i])) for i in range(len(got)) if got[i] != expect[i]]
    assert not bad, bad[:10]
    # fixed-length messages (the non-ragged kernels), wrong-pub signing, key conversions
    wsec, wpub, wsig, wmsgs = gu.sign_wrongpub()
    eq(ed.ed25519_sign_batch(wsec, wpub, np.frombuffer(b"".join(wmsgs), np.uint8), None, 64), wsig, "sign with the caller's (wrong) pub")
    n = 1100
    fsec, fpub, fmsgs, _, fsig = make_signed(cpu, r, n, fixed_len=64)
    eq(ed.ed25519_sign_batch(fsec, fpub, fmsgs, None, 64), fsig, "sign, fixed 64-byte messages")
    bsig, bpub = mutate(r, fsig, fpub, 0.1)
    eq(ed.ed25519_verify_batch(bsig, bpub, fmsgs, None, 64), cpu.verify(bsig, bpub, fmsgs, None, 64), "verify, fixed 64-byte messages")
    # message lengths around the SHA-512 block boundaries and long ones, at every byte alignment of the blob (the 128-bit, the
    # unaligned-block and the byte-wise loaders of sha512.cuh), as one ragged batch
    lens = [0, 1, 55, 56, 63, 64, 111, 112, 127, 128, 129, 239, 240, 255, 256, 1023, 1025]
    lens = [l for l in lens for _ in range(2)] + [4096 + 7, 16384]
    pad = r.integers(0, 16, size=len(lens))                             # gaps between messages: arbitrary alignment
    eoff = np.zeros(len(lens) + 1, np.uint64)
    pos = 3
    starts = []
    for l, g in zip(lens, pad):
        starts.append(pos)
        pos += l + int(g)
    # offsets must be contiguous for the batch ABI: message i = blob[off[i] .. off[i+1]) — so the gaps become part of the NEXT
    # message's prefix here; alignment still varies because the lengths do
    eoff[0] = 3
    eoff[1:] = 3 + np.cumsum(np.array(lens, np.uint64) + pad.astype(np.uint64))
    eblob = r.integers(0, 256, size=int(eoff[-1]) + 1, dtype=np.uint8)
    esec = rand_rows(r, len(lens))
    epub = cpu.genpub(esec)
    esig = cpu.sign(esec, epub, eblob, eoff, 0)
    eq(ed.ed25519_sign_batch(esec, epub, eblob, eoff, 0), esig, "sign, block-boundary lengths at odd alignments")
    bsig2, bpub2 = mutate(r, esig, epub, 0.2)
    eq(ed.ed25519_verify_batch(bsig2, bpub2, eblob, eoff, 0), cpu.verify(bsig2, bpub2, eblob, eoff, 0), "verify, block-boundary lengths")
    edsk, edpk, xsk, xpk = gu.convert_kat()
    eq(ed.sk_ed25519_to_x25519_batch(edsk), xsk, "sk conversion")
    eq(ed.pk_ed25519_to_x25519_batch(edpk), xpk, "pk conversion")
    sim.clean()
    # the tables the device builds (k_wtab_base / k_wtab_build, k_comb_base / k_comb_rows / k_comb_layout)
    import edmodel as em
    em.check_comb_table(ed.comb_table(), 6)
    assert ed.launch_count() >= 36
    ed.shutdown()
    assert sim.live() == (0, 0)


def scenario_kernel_scrub():
    """The kernels wipe their own scratch: the secret scalar a = clamp(SHA512(sk)[0..31]) mod L that k_expand_key / k_sign_nonce hand
    to the comb, and the nonce r of a signature, are gone from the pool block when the call returns (CUDASIM_KEEP_FREED=1 keeps
    returned pool blocks searchable, as pool memory keeps its contents on the device).  With the wipes compiled out (argv[2] ==
    "expect-residue": a mutant of the kernel source built by the test) the same search finds them."""
    import hashlib
    from cpu_ref import best_cpu_impl
    from edmodel import L as ORDER
    assert "sim_kernels" in SIM_SO and os.environ.get("CUDASIM_KEEP_FREED") == "1"
    expect_residue = len(sys.argv) > 2 and sys.argv[2] == "expect-residue"
    sim, cpu = Sim(), best_cpu_impl()
    ed = sim.ed
    r = rng(22)
    n = 300
    sec, pub, msgs, off, sig = make_signed(cpu, r, n, fixed_len=48)

    def secret_scalar(sk):
        h = bytearray(hashlib.sha512(bytes(sk)).digest())
        h[0] &= 248
        h[31] = (h[31] & 127) | 64
        a = int.from_bytes(bytes(h[:32]), "little") % ORDER
        nonce_prefix = bytes(h[32:])
        return a, nonce_prefix

    scalars, nonces = [], []
    for i in range(n):
        a, prefix = secret_scalar(sec[i])
        scalars.append(np.frombuffer(a.to_bytes(32, "little"), np.uint8))
        rr = int.from_bytes(hashlib.sha512(prefix + bytes(msgs[48 * i:48 * i + 48])).digest(), "little") % ORDER
        nonces.append(np.frombuffer(rr.to_bytes(32, "little"), np.uint8))
    eq(ed.ed25519_genpub_batch(sec), pub, "genpub")
    left_genpub = sim.find(scalars)
    eq(ed.ed25519_sign_batch(sec, pub, msgs, None, 48), sig, "sign")
    left_sign = sim.find(scalars) + sim.find(nonces)
    left_keys = sim.find([sec[i] for i in range(n)])
    print("residue: genpub", left_genpub, "sign", left_sign, "keys", left_keys)
    assert left_keys == 0
    if expect_residue:
        assert left_genpub >= n and left_sign >= 2 * n
    else:
        assert left_genpub == 0 and left_sign == 0


def scenario_tsan_workload():
    """The workload of tools/host_sanitize.sh (the real kernels under ThreadSanitizer): ragged sign / verify (tile sort in shared memory,
    permutation counters, staging of the verify loop), genpub (comb table staging, exchange areas, mma rendezvous), x25519."""
    from cpu_ref import best_cpu_impl
    sim, cpu = Sim(), best_cpu_impl()
    ed = sim.ed
    r = rng(3)
    n = 700
    sec, pub, msgs, off, sig = make_signed(cpu, r, n, max_len=90)
    eq(ed.ed25519_genpub_batch(sec), pub, "genpub")
    eq(ed.ed25519_sign_batch(sec, pub, msgs, off, 0), sig, "sign")
    bs, bp = mutate(r, sig, pub, 0.2)
    eq(ed.ed25519_verify_batch(bs, bp, msgs, off, 0), cpu.verify(bs, bp, msgs, off, 0), "verify")
    pts = rand_rows(r, 200)
    eq(ed.x25519_batch(sec[:200], pts), cpu.x25519(sec[:200], pts), "x25519")
    eq(ed.x25519_base_batch(sec[:200]), cpu.x25519_base(sec[:200]), "x25519_base")
    assert sim.errors() == 0


def scenario_real_kernels_full_scalars():
    """EDDSA_B200_DEBUG_FULL_SCALARS=1 on the real kernels: every signature takes the full-length fallback (rho, tau) = (1, t) of the
    half-size-scalar verification — 64 windows instead of 33 — and every adversarial decision stays the same."""
    import golden_util as gu
    assert "sim_kernels" in SIM_SO and os.environ.get("EDDSA_B200_DEBUG_FULL_SCALARS") == "1"
    sim = Sim()
    ed = sim.ed
    asig, apub, amsgs, cls, expect = gu.verify_adv()
    pick = list(range(0, len(asig), 4)) + [i for i in range(len(asig)) if cls[i] >= 16]
    ablob, aoff = gu.ragged([amsgs[i] for i in pick])
    got = ed.ed25519_verify_batch(asig[pick], apub[pick], ablob, aoff, 0)
    bad = [(pick[k], int(cls[pick[k]])) for k in range(len(pick)) if got[k] != expect[pick[k]]]
    assert not bad, bad[:10]
    sim.clean()


def scenario_real_kernels_structured():
    """The rare branches of the scalar code on the real kernels, checked against Python integers and the CPU reference (never
    against another build of the same headers): half_gcd (k_sc_selftest ops 3 and 4) on structured challenges that reach every
    branch class of tests/structured_inputs.py, the verify loop's 16-bit recoding (op 5) on digit-run values, and x25519_base
    (k_comb<1>: signed radix-64 recoding + tensor-core lookup) on scalars whose clamped value mod L has structured digits."""
    import structured_inputs as si
    from cpu_ref import best_cpu_impl
    assert "sim_kernels" in SIM_SO
    sim, cpu = Sim(), best_cpu_impl()
    ed = sim.ed
    rows = lambda vals: np.frombuffer(b"".join(v.to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32)
    val = lambda a: [int.from_bytes(a[i].tobytes(), "little") for i in range(len(a))]
    ts = si.half_gcd_inputs()
    counts = si.class_counts(ts)
    print("half_gcd inputs by branch class:", counts)
    assert all(counts[k] >= m for k, m in si.MIN_CLASS_COUNT.items()), counts
    a = rows(ts)
    z = np.zeros_like(a)
    taus, rhos = val(ed.sc_selftest(a, z, z, 3)), ed.sc_selftest(a, z, z, 4)
    for i, t in enumerate(ts):
        want_r, want_ta, info = si.half_gcd_model(t)
        w = rhos[i].view(np.uint32)
        r = int.from_bytes(rhos[i, :24].tobytes(), "little")
        assert w[6] == 0 and w[7] in (0, 1), (t, w)
        r = -r if w[7] else r
        assert (r, taus[i]) == (want_r, want_ta), (t, info, r, taus[i], want_r, want_ta)
    xs = si.recode_window_values(n_random=300)
    es = val(ed.sc_selftest(rows(xs), np.zeros((len(xs), 32), np.uint8), np.zeros((len(xs), 32), np.uint8), 5))
    for x, e in zip(xs, es):
        ds = si.window_digits(e)
        assert all(-2**15 <= d < 2**15 for d in ds) and sum(d << (16 * k) for k, d in enumerate(ds)) == x, (x, e)
    scal, targets, unreachable = si.comb_batch(n_random=300)
    print(f"comb targets: {sum(t is not None for t in targets)} reachable through x25519_base, {unreachable} dropped")
    sa = np.frombuffer(b"".join(scal), np.uint8).reshape(-1, 32)
    got = ed.x25519_base_batch(sa)
    eq(got, cpu.x25519_base(sa), "x25519_base with structured comb digits, against the CPU reference")
    picked = [i for i, t in enumerate(targets) if t is not None][:25]
    for i in picked:
        assert got[i].tobytes() == si.x25519_base_model(targets[i]), (i, targets[i])
    sim.clean()


def scenario_real_kernels_opcount():
    """Field operations the REAL verify kernels execute per signature, counted by the emulator (a lane of the loop kernel runs its
    warp's maximum window count, as on the device): the figure the integer-multiply roofline of bench.py is computed from."""
    import bench
    from cpu_ref import best_cpu_impl
    assert "sim_kernels" in SIM_SO
    sim, cpu = Sim(), best_cpu_impl()
    ed, L = sim.ed, sim.L
    r = rng(23)
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
    base = 512
    sec, pub, msgs, off, sig = make_signed(cpu, r, base, fixed_len=64)
    reps = n // base
    sec, pub, sig, msgs = np.tile(sec, (reps, 1)), np.tile(pub, (reps, 1)), np.tile(sig, (reps, 1)), np.tile(msgs, reps)
    # different challenges for every row: distinct messages need distinct signatures — sign on the emulated kernels themselves
    msgs = r.integers(0, 256, size=n * 64, dtype=np.uint8)
    sig = ed.ed25519_sign_batch(sec, pub, msgs, None, 64)
    ed.init()
    m, s = ctypes.c_ulonglong(), ctypes.c_ulonglong()
    L.edg_emul_counts(ctypes.byref(m), ctypes.byref(s), 1)
    assert ed.ed25519_verify_batch(sig, pub, msgs, None, 64).all()
    L.edg_emul_counts(ctypes.byref(m), ctypes.byref(s), 1)
    per_m, per_s = m.value / n, s.value / n
    nwin = (per_m - 267) / 28
    model_m, model_s = bench.OURS_FM["verify"]
    wide = 72 * per_m + 44 * per_s
    print(f"verify on the real kernels, {n} signatures: {per_m:.1f} M + {per_s:.1f} S per signature = {nwin:.2f} windows per lane; "
          f"{wide:.0f} wide multiplies (bench.py model: {model_m:.1f} M + {model_s:.1f} S = {72 * model_m + 44 * model_s:.0f})")
    assert abs((per_s - 494) / 16 - nwin) < 1e-6                         # both counts describe the same window count
    assert abs(wide / (72 * model_m + 44 * model_s) - 1) < 0.01          # the roofline's work figure, within 1 %
    if len(sys.argv) > 3 and sys.argv[3] == "all":
        # the operations with a shared inversion: bench.py's ours_fm(op, n) with the emulated device's resident threads (2 SMs: 1024
        # comb threads, 1024 ladder threads) must give exactly what the kernels execute
        resident = {"genpub": 1024, "sign": 1024, "x25519_base": 1024, "x25519": 1024}
        k = 8192
        ksec = rand_rows(r, k)
        kpub = cpu.genpub(ksec)
        kmsg = r.integers(0, 256, size=k * 64, dtype=np.uint8)
        pts = rand_rows(r, k)
        runs = {"genpub": lambda: ed.ed25519_genpub_batch(ksec), "sign": lambda: ed.ed25519_sign_batch(ksec, kpub, kmsg, None, 64),
                "x25519_base": lambda: ed.x25519_base_batch(ksec), "x25519": lambda: ed.x25519_batch(ksec[:4096], pts[:4096])}
        for op, fn in runs.items():
            cnt = 4096 if op == "x25519" else k
            L.edg_emul_counts(ctypes.byref(m), ctypes.byref(s), 1)
            fn()
            L.edg_emul_counts(ctypes.byref(m), ctypes.byref(s), 1)
            mm, ss = bench.OURS_FM_SINGLE[op]
            share = cnt / resident[op]
            want = (mm - 11 + 11 / share + 3, ss - 254 + 254 / share)
            print(f"{op}: {m.value / cnt:.3f} M + {s.value / cnt:.3f} S per operation on the real kernels, inversion shared by {share:.0f}; "
                  f"bench.py's formula: {want[0]:.3f} M + {want[1]:.3f} S")
            assert abs(m.value / cnt - want[0]) < 1e-6 and abs(s.value / cnt - want[1]) < 1e-6, op


def scenario_no_device():
    """No usable device: the batch calls report it (there is no CPU path to fall back to)."""
    assert os.environ.get("CUDASIM_DEVICES") == "0"
    sim = Sim()
    L = sim.L
    buf = np.zeros(64, np.uint8)
    assert L.ed25519_genpub_batch(2, buf.ctypes.data, buf.ctypes.data) == 100          # cudaErrorNoDevice
    assert b"no usable CUDA device" in L.eddsa_b200_last_error()
    assert L.ed25519_verify_batch_dev(2, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, None, 4, None) == 100
    assert L.eddsa_b200_init() == 100 and L.eddsa_b200_device_count() == 0
    L.eddsa_b200_shutdown()
    if len(sys.argv) > 2 and sys.argv[2] == "abort":
        out = ctypes.create_string_buffer(32)
        L.ed25519_genpub(out, bytes(32))                             # void function, cannot report: must abort()
        print("NOT REACHED")


SCENARIOS = {k[len("scenario_"):]: v for k, v in list(globals().items()) if k.startswith("scenario_")}

if __name__ == "__main__":
    SCENARIOS[sys.argv[1]]()
    print("OK", sys.argv[1])
