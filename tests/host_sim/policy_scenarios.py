"""TEST INFRASTRUCTURE: scenarios for the verify acceptance rules (ed25519_verify_policy_batch / _dev), run by
tests/test_verify_policy.py in a fresh interpreter each, like those of sim_scenarios.py, whose simulator control surface (Sim)
they use:

    CUDASIM_SO=<library> python tests/host_sim/policy_scenarios.py <scenario> [args]

Libraries: libeddsa_sim_policy.so (host.c + cudasim_policy.cpp: the simulator's mock kernels and a mock of the rule-aware
launcher), libeddsa_sim.so (the mock kernels alone, which implement only the reference's rule) and libeddsa_sim_kernels.so (the
real kernels on the SIMT emulator, or a mutant of them).  Results are checked against the big-integer model of
tests/verify_policy_model.py.
"""
import os
import sys

import numpy as np

from sim_scenarios import EINVAL, K_DEVICE, L_VERIFY, SIM_SO, Sim, eq


def scenario_verify_policy():
    """ed25519_verify_policy_batch / _dev behind the real host layer (mock kernels: the host build of ops.cuh): unknown rules are
    refused before any work, rule 0 is ed25519_verify_batch, and every rule holds across chunks, passes and two shards with
    ragged offsets — checked against the big-integer model of tests/verify_policy_model.py on the fixture and generated rows."""
    import verify_policy_model as vm
    assert "sim_policy" in SIM_SO and os.environ.get("CUDASIM_DEVICES") == "2" and os.environ.get("CUDASIM_RESIDENT") == "32"
    sim = Sim()
    ed, L = sim.ed, sim.L
    rows, want, _ = vm.all_rows()
    buf = np.zeros(256, np.uint8)
    p = buf.ctypes.data
    before = ed.launch_count()
    for bad in (-1, 3):
        for n in (0, 2):
            assert L.ed25519_verify_policy_batch(n, p, p, p, p, None, 4, bad) == EINVAL
            assert b"unknown verify policy" in L.eddsa_b200_last_error()
            assert L.ed25519_verify_policy_batch_dev(n, p, p, p, p, None, 4, bad, None) == EINVAL
            assert b"unknown verify policy" in L.eddsa_b200_last_error()
    assert ed.launch_count() == before and sim.stats()["kernels"] == 0
    # 4 x the rows (> 16 384: two shards), ragged; a pass is 1 SM x 32 x 16 waves = 512 signatures
    reps = 4
    sig, pub, blob, off = vm.as_arrays(rows * reps)
    n = len(sig)
    assert n > 16384
    sim.reset()
    got = {pol: ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, pol) for pol in vm.POLICIES}
    for pol in vm.POLICIES:
        bad = np.nonzero(got[pol] != np.tile(want[:, pol], reps))[0]
        assert not len(bad), (vm.NAMES[pol], bad[:10])
    eq(ed.ed25519_verify_batch(sig, pub, blob, off, 0), got[vm.REFERENCE], "policy 0 vs ed25519_verify_batch")
    launches = sim.launches(L_VERIFY)
    assert {d for d, _, _ in launches} == {0, 1} and len(launches) >= 8, launches[:20]
    sim.clean()
    # device API: one call of more than a pass (several passes in one launcher call), on a stream of the caller
    sig, pub, blob, off = vm.as_arrays(rows)
    n = len(sig)
    off64 = np.ascontiguousarray(off, np.uint64)

    def dev(arr):
        a, ptr = sim.user_array(arr.nbytes + 16, K_DEVICE)
        a[:arr.nbytes] = arr.view(np.uint8).reshape(-1)
        return ptr

    d_sig, d_pub, d_blob, d_off = dev(sig), dev(pub), dev(blob), dev(off64)
    d_ok, d_okp = sim.user_array(n + 1, K_DEVICE)
    s1 = L.cudasim_stream_create(0)
    for pol in vm.POLICIES:
        assert L.ed25519_verify_policy_batch_dev(n, d_okp + 1, d_sig, d_pub, d_blob, d_off, 0, pol, s1) == 0
        L.cudasim_sync_all()
        bad = np.nonzero(d_ok[1:] != want[:, pol])[0]
        assert not len(bad), (vm.NAMES[pol], "device API", bad[:10])
    sim.clean()


def scenario_real_kernels_verify_policy():
    """The three acceptance rules on the REAL kernels (k_verify_points<POLICY>, k_verify<COFACTORED>) behind the real host layer:
    the fixture rows and the generated rows of tests/verify_policy_model.py, decided like the big-integer model.  argv[2] (optional):
    one rule name; argv[3] (optional): the classes to run, comma-separated — what the kernel mutants of tests/test_verify_policy.py
    run.  A disagreement prints MISMATCH."""
    import verify_policy_model as vm
    assert "sim_kernels" in SIM_SO
    sim = Sim()
    ed = sim.ed
    rows, want, cls = vm.all_rows()
    pols = [p for p in vm.POLICIES if len(sys.argv) <= 2 or vm.NAMES[p] == sys.argv[2]]
    pick = np.arange(len(rows))
    if len(sys.argv) > 3:
        pick = np.nonzero(np.isin(cls, [int(c) for c in sys.argv[3].split(",")]))[0]
    sig, pub, blob, off = vm.as_arrays([rows[i] for i in pick])
    for pol in pols:
        got = ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, pol)
        bad = np.nonzero(got != want[pick, pol])[0]
        if len(bad):
            print("MISMATCH", vm.NAMES[pol], [(int(pick[i]), int(cls[pick[i]]), int(got[i])) for i in bad[:10]])
        assert not len(bad)
        print(f"{vm.NAMES[pol]}: {len(pick)} rows, {int(got.sum())} accepted, as the model")
    sim.clean()



def scenario_reference_launchers_only():
    """Launchers that implement only the reference's rule (the simulator's mock kernels): STRICT and ZIP215 are refused with
    EDDSA_B200_EINVAL before any work, through both entry points; the reference's rule still runs."""
    import verify_policy_model as vm
    assert SIM_SO.endswith("libeddsa_sim.so")
    sim = Sim()
    ed, L = sim.ed, sim.L
    rows, want, _ = vm.all_rows()
    sig, pub, blob, off = vm.as_arrays(rows[:300])
    buf = np.zeros(256, np.uint8)
    p = buf.ctypes.data
    before = ed.launch_count()
    for pol in (vm.STRICT, vm.ZIP215):
        assert L.ed25519_verify_policy_batch(2, p, p, p, p, None, 4, pol) == EINVAL
        assert b"no launcher" in L.eddsa_b200_last_error()
        assert L.ed25519_verify_policy_batch_dev(2, p, p, p, p, None, 4, pol, None) == EINVAL
    assert ed.launch_count() == before
    eq(ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, vm.REFERENCE), want[:300, vm.REFERENCE], "reference rule")
    sim.clean()


SCENARIOS = {k[len("scenario_"):]: v for k, v in list(globals().items()) if k.startswith("scenario_")}

if __name__ == "__main__":
    SCENARIOS[sys.argv[1]]()
    print("OK", sys.argv[1])
