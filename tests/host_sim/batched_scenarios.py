"""TEST INFRASTRUCTURE: scenarios for batched ZIP215 verification (ed25519_verify_zip215_batched / _dev), run by
tests/test_verify_batched.py in a fresh interpreter each, with the simulator control surface of sim_scenarios.py:

    CUDASIM_SO=<library> python tests/host_sim/batched_scenarios.py <scenario> [args]

Libraries: libeddsa_sim_kernels.so (the real kernels on the SIMT emulator) and libeddsa_sim.so (the mock kernels, which have no
batched launcher).  Results are checked against the big-integer models of tests/verify_policy_model.py and
tests/verify_batched_model.py.
"""
import os
import sys

import numpy as np

from sim_scenarios import EINVAL, K_DEVICE, SIM_SO, Sim

SEED = bytes(range(7, 39))
PASS = 512                      # CUDASIM_SMS=1, CUDASIM_RESIDENT=32: 1 SM x 32 x 16 waves


def _groups(n, k):
    """Group of each row of one device-API call: pass, warp within the pass, lane."""
    i = np.arange(n)
    return (i // PASS) * PASS + (i % PASS) // (32 * k) * 32 + i % 32


def scenario_real_kernels_verify_batched():
    """The real kernels (k_verify_scalars<., true>, k_verify_points<ZIP215>, k_verify_batched, k_verify_list) on every fixture and
    generated row, after a warp of valid rows holding a cancelling pair, through the device API: the output is the model's ZIP215.  argv[2] == "no_fallback" (with
    EDDSA_B200_DEBUG_NO_FALLBACK=1): every row of a group holding an invalid included row is 0, the others are ZIP215's."""
    import verify_batched_model as bm
    import verify_policy_model as vm
    assert "sim_kernels" in SIM_SO and os.environ.get("CUDASIM_SMS") == "1" and os.environ.get("CUDASIM_RESIDENT") == "32"
    no_fallback = len(sys.argv) > 2 and sys.argv[2] == "no_fallback"
    assert no_fallback == (os.environ.get("EDDSA_B200_DEBUG_NO_FALLBACK") == "1")
    sim = Sim()
    ed, L = sim.ed, sim.L
    rows, want, cls = vm.all_rows()
    # a warp of valid rows in front (32 K), with a cancelling pair at 0 and 32 (one group), which only random weights reject
    nf = 32 * ed.VERIFY_BATCH_ROWS
    valid = [r for r, d in zip(rows, want) if d[vm.ZIP215]][:nf]
    assert len(valid) == nf
    a, b = bm.cancelling_pair(*valid[0][:3], *valid[1][:3])
    front = [r[:3] + (-1,) for r in valid]
    front[0], front[32] = a + (-1,), b + (-1,)
    rows = front + list(rows)
    want = np.concatenate([vm.decide_rows(front), want])
    cls = np.concatenate([np.full(nf, -1), cls])
    zip_ok = want[:, vm.ZIP215].astype(bool)
    assert not zip_ok[0] and not zip_ok[32]
    sig, pub, blob, off = vm.as_arrays(rows)
    n = len(sig)

    def dev(arr):
        a, ptr = sim.user_array(arr.nbytes + 16, K_DEVICE)
        a[:arr.nbytes] = arr.view(np.uint8).reshape(-1)
        return ptr

    d_sig, d_pub, d_blob, d_off = dev(sig), dev(pub), dev(blob), dev(np.ascontiguousarray(off, np.uint64))
    d_ok, d_okp = sim.user_array(n, K_DEVICE)
    seed = ed._seed(SEED)
    assert L.ed25519_verify_zip215_batched_dev(n, d_okp, d_sig, d_pub, d_blob, d_off, 0, seed, None) == 0
    L.cudasim_sync_all()
    got = d_ok[:n].astype(bool)
    expect = zip_ok
    if no_fallback:
        g = _groups(n, ed.VERIFY_BATCH_ROWS)
        invalid = np.array([bm.included(r[0], r[1]) for r in rows]) & ~zip_ok
        failing = np.zeros(g.max() + 1, bool)
        failing[g[invalid]] = True
        expect = zip_ok & ~failing[g]
        assert failing.any() and expect.any()
    bad = np.nonzero(got != expect)[0]
    if len(bad):
        print("MISMATCH", [(int(i), int(cls[i]), int(got[i])) for i in bad[:10]])
    assert not len(bad)
    print(f"{n} rows, {int(got.sum())} accepted, as the model{' (raw batch equations)' if no_fallback else ''}")
    sim.clean()


def scenario_argument_checks():
    """On the real kernels: n = 0 is a no-op, misaligned device arrays are refused, and a failing getrandom(2) (seed = NULL;
    argv[2] == "getrandom_fails", under a preloaded getrandom that fails) returns EINVAL — nothing launched in each case."""
    assert "sim_kernels" in SIM_SO
    sim = Sim()
    ed, L = sim.ed, sim.L
    buf = np.zeros(4096, np.uint8)
    p = buf.ctypes.data
    before = ed.launch_count()
    seed = ed._seed(SEED)
    assert L.ed25519_verify_zip215_batched(0, p, p, p, p, None, 4, seed) == 0
    assert L.ed25519_verify_zip215_batched_dev(0, p, p, p, p, None, 4, seed, None) == 0
    assert L.ed25519_verify_zip215_batched_dev(2, p, p + 1, p, p, None, 4, seed, None) == EINVAL
    if len(sys.argv) > 2 and sys.argv[2] == "getrandom_fails":
        assert L.ed25519_verify_zip215_batched(2, p, p, p, p, None, 4, None) == EINVAL
        assert b"getrandom" in L.eddsa_b200_last_error()
        assert L.ed25519_verify_zip215_batched_dev(2, p, p, p, p, None, 4, None, None) == EINVAL
        assert b"getrandom" in L.eddsa_b200_last_error()
    assert ed.launch_count() == before
    sim.clean()


def scenario_no_batched_launcher():
    """Launchers without the batched check (the simulator's mock kernels): both entry points return EINVAL before any work."""
    assert SIM_SO.endswith("libeddsa_sim.so")
    sim = Sim()
    ed, L = sim.ed, sim.L
    buf = np.zeros(256, np.uint8)
    p = buf.ctypes.data
    before = ed.launch_count()
    for seed in (ed._seed(SEED), None):
        assert L.ed25519_verify_zip215_batched(2, p, p, p, p, None, 4, seed) == EINVAL
        assert b"no launcher" in L.eddsa_b200_last_error()
        assert L.ed25519_verify_zip215_batched_dev(2, p, p, p, p, None, 4, seed, None) == EINVAL
    assert ed.launch_count() == before
    sim.clean()


SCENARIOS = {k[len("scenario_"):]: v for k, v in list(globals().items()) if k.startswith("scenario_")}

if __name__ == "__main__":
    SCENARIOS[sys.argv[1]]()
    print("OK", sys.argv[1])
