"""TEST INFRASTRUCTURE: the settle-site corpus (tests/golden/verify_settle.bin) through the real kernels and the real host
layer on the SIMT emulator, with the settle probe (settle_probe.py) applied to the emulator's copy of the headers.  Run by
tests/test_verify_settle.py in a fresh interpreter each:

    CUDASIM_SO=<probed kernels library> python tests/host_sim/settle_scenarios.py rows|lanes

Prints the per-site counts of the run; fails unless every site is taken and every output is 1.
"""
import ctypes
import os
import sys

import numpy as np

from sim_scenarios import K_DEVICE, Sim

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "golden"))
import make_verify_settle as corpus_file  # noqa: E402

MLEN = 32


def _arrays(rows):
    return tuple(np.array([np.frombuffer(r[k], np.uint8) for r in rows]) for k in range(3))


def _counts(L, sites):
    hits, alone = np.zeros(sites, np.uint64), np.zeros(sites, np.uint64)
    L.edg_probe_counts(ctypes.c_void_p(hits.ctypes.data), ctypes.c_void_p(alone.ctypes.data), 1)
    return hits, alone


def _check(L, what):
    hits, alone = _counts(L, corpus_file.SITES)
    print(f"{what}: taken {hits.tolist()}, alone {alone.tolist()}")
    assert (hits > 0).all() and (alone > 0).all(), (what, "sites not taken", np.nonzero(alone == 0)[0].tolist())


def scenario_rows():
    """Every corpus row through the host API of ed25519_verify_batch (k_verify: 33 windows in every warp)."""
    sim = Sim()
    ed, L = sim.ed, sim.L
    sig, pub, msg = _arrays(corpus_file.load()[0])
    _counts(L, corpus_file.SITES)
    ok = ed.ed25519_verify_batch(sig, pub, msg, None, MLEN)
    assert ok.all(), np.nonzero(ok != 1)[0]
    _check(L, "k_verify")
    sim.clean()


def scenario_lanes():
    """Every corpus lane through the device API of ed25519_verify_zip215_batched_dev under EDDSA_B200_DEBUG_NO_FALLBACK=1,
    lane l of warp w holding corpus lane 32 w + l (cyclically) at rows 32 K w + l + 32 r."""
    assert os.environ.get("EDDSA_B200_DEBUG_NO_FALLBACK") == "1"
    sim = Sim()
    ed, L = sim.ed, sim.L
    _, pool, lanes, seed = corpus_file.load()
    K = ed.VERIFY_BATCH_ROWS
    warps = (len(lanes) + 31) // 32
    idx = np.zeros(32 * K * warps, np.int64)
    for q in range(32 * warps):
        for r, k in enumerate(lanes[q % len(lanes)][3]):
            idx[32 * K * (q // 32) + q % 32 + 32 * r] = k
    sig, pub, msg = (a[idx] for a in _arrays(pool))
    n = len(sig)

    def dev(arr):
        a, ptr = sim.user_array(arr.nbytes, K_DEVICE)
        a[:] = np.ascontiguousarray(arr).view(np.uint8).reshape(-1)
        return ptr

    d_ok, d_okp = sim.user_array(n, K_DEVICE)
    _counts(L, corpus_file.SITES)
    assert L.ed25519_verify_zip215_batched_dev(n, d_okp, dev(sig), dev(pub), dev(msg), None, MLEN, ed._seed(seed), None) == 0
    L.cudasim_sync_all()
    assert d_ok.all(), np.nonzero(d_ok != 1)[0]
    _check(L, "k_verify_batched")
    sim.clean()


SCENARIOS = {k[len("scenario_"):]: v for k, v in list(globals().items()) if k.startswith("scenario_")}

if __name__ == "__main__":
    SCENARIOS[sys.argv[1]]()
    print("OK", sys.argv[1])
