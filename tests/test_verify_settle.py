"""Every pending-carry settle of the verify window loops, taken by valid signatures (tests/golden/verify_settle.bin).

EDG_VERIFY_STEP (ops.cuh) computes groups of 2-4 independent public-data field operations, ORs their pending-carry flags
and settles the flagged results in one rarely taken branch: 28 settle sites in 8 groups, shared by ed25519_verify_loop
and ed25519_verify_batched_loop.  On random data 11 of the sites are never reached, so a settle of the wrong kind, of the
wrong result, or a flag missing from its group's OR would reject a valid signature that no other test presents.  The
corpus holds, per site, an honest signature (and a batched lane of 8 honest rows) that takes the site with no other flag of
its group set.  Here, without a GPU, on the site probe of tests/host_sim/settle_probe.py:
  * both host builds of the headers (portable paths; device paths with their PTX interpreted) take every site in both
    loops, with identical per-site counts and the site bitmaps recorded in the corpus;
  * every row is valid under the compiled reference, the policy model under each rule and libsodium, and the host builds
    accept it under each rule; every lane's raw equation holds in the batched model and in the host builds;
  * every single-site mutant (a settle that does not run, a flag left out of its group's OR) rejects a corpus row and a
    corpus lane;
  * on the SIMT emulator, the real kernels behind the real host layer, probed the same way, take every site: the rows
    through ed25519_verify_batch and the lanes through ed25519_verify_zip215_batched_dev without the fallback, every
    output 1.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import verify_batched_model as bm
import verify_policy_model as vm

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "host_sim"))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_verify_settle as corpus_file  # noqa: E402
import settle_probe  # noqa: E402

SITES = settle_probe.SITES
ALL = (1 << SITES) - 1
POLICIES = (vm.REFERENCE, vm.STRICT, vm.ZIP215)


@pytest.fixture(scope="module")
def corpus():
    rows, pool, lanes, seed = corpus_file.load()
    lane_rows = [[pool[k] for k in sel] for _, _, _, sel in lanes]
    return rows, lane_rows, lanes, seed


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    out = {}
    for flavour in ("host", "device"):
        lib = ctypes.CDLL(settle_probe.build(str(tmp_path_factory.mktemp("settle_" + flavour)), flavour))
        lib.sp_init()
        assert lib.sp_sites() == SITES and lib.sp_lane_rows() == bm.K
        out[flavour] = lib
    return out


def verify(lib, sig, pub, msg, policy=vm.REFERENCE):
    taken, alone = ctypes.c_uint32(), ctypes.c_uint32()
    ok = lib.sp_verify(sig, pub, msg, ctypes.c_uint64(len(msg)), policy, ctypes.byref(taken), ctypes.byref(alone))
    return ok, taken.value, alone.value


def batched(lib, rows, seed):
    off = np.zeros(len(rows) + 1, np.uint64)
    off[1:] = np.cumsum([len(m) for _, _, m in rows])
    taken, alone = ctypes.c_uint32(), ctypes.c_uint32()
    ok = lib.sp_batched(b"".join(s for s, _, _ in rows), b"".join(p for _, p, _ in rows), b"".join(m for _, _, m in rows),
                        ctypes.c_void_p(off.ctypes.data), seed, ctypes.byref(taken), ctypes.byref(alone))
    return ok, taken.value, alone.value


def counts(lib):
    hits, alone = np.zeros(SITES, np.uint64), np.zeros(SITES, np.uint64)
    lib.edg_probe_counts(ctypes.c_void_p(hits.ctypes.data), ctypes.c_void_p(alone.ctypes.data), 1)
    return hits, alone


def union(masks):
    u = 0
    for m in masks:
        u |= m
    return u


def test_corpus_takes_every_site_alone(corpus):
    rows, lane_rows, lanes, _ = corpus
    assert union(r[5] for r in rows) == ALL, "a site no row takes alone"
    assert union(ln[2] for ln in lanes) == ALL, "a site no lane takes alone"
    assert all(len(r) == bm.K and len(set(map(id, r))) == bm.K for r in lane_rows)


def test_both_host_builds_take_every_site(libs, corpus):
    """Per-site counts over the corpus: no zero in either loop, the same in both builds, the corpus's bitmaps per row/lane."""
    rows, lane_rows, lanes, seed = corpus
    per = {}
    for flavour, lib in libs.items():
        counts(lib)
        for sig, pub, msg, _, taken, alone in rows:
            assert verify(lib, sig, pub, msg) == (1, taken, alone), flavour
        row_counts = counts(lib)
        for lane, (_, taken, alone, _) in zip(lane_rows, lanes):
            assert batched(lib, lane, seed) == (1, taken, alone), flavour
        lane_counts = counts(lib)
        per[flavour] = (row_counts, lane_counts)
        for name, (hits, alone) in (("ed25519_verify_loop", row_counts), ("ed25519_verify_batched_loop<8>", lane_counts)):
            print(f"{flavour:6s} {name}: taken {hits.tolist()}, alone {alone.tolist()}")
            assert (hits > 0).all() and (alone > 0).all(), (flavour, name, np.nonzero(alone == 0)[0])
    for a, b in zip(per["host"], per["device"]):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_rows_are_valid_under_every_rule(libs, corpus, cpu):
    rows = corpus[0]
    sig = np.array([np.frombuffer(r[0], np.uint8) for r in rows])
    pub = np.array([np.frombuffer(r[1], np.uint8) for r in rows])
    msg = np.array([np.frombuffer(r[2], np.uint8) for r in rows])
    assert cpu.verify(sig, pub, msg, None, 32).all(), "the compiled reference rejects a corpus row"
    for s, p, m, idx, _, _ in rows:
        assert vm.decisions(s, p, m) == (1, 1, 1), idx
        assert vm.libsodium_decision(s, p, m) == 1, idx
        for policy in POLICIES:
            assert verify(libs["host"], s, p, m, policy)[0] == 1, (idx, policy)


def test_lane_equations_hold(libs, corpus):
    _, lane_rows, lanes, seed = corpus
    for lane, meta in zip(lane_rows, lanes):
        assert all(bm.included(s, p) for s, p, _ in lane) and bm.lane_holds(lane, seed), meta[0]
        assert batched(libs["host"], lane, seed)[0] == 1, meta[0]


@pytest.mark.parametrize("kind", ["settle_skipped", "flag_dropped"])
def test_every_single_site_mutant_is_caught(libs, corpus, kind):
    """For each site: its settle not run, or its flag left out of its group's OR.  Each mutant rejects a corpus row (per-
    signature loop) and makes a corpus lane's equation fail (batched loop).  Only rows and lanes that take the site can
    change, so those are the ones run."""
    rows, lane_rows, lanes, seed = corpus
    lib = libs["host"]
    missed = []
    try:
        for site in range(SITES):
            lib.sp_mutant(site if kind == "settle_skipped" else -1, site if kind == "flag_dropped" else -1)
            row_fails = sum(verify(lib, s, p, m)[0] == 0 for s, p, m, _, taken, _ in rows if taken >> site & 1)
            lane_fails = sum(batched(lib, ln, seed)[0] == 0 for ln, meta in zip(lane_rows, lanes) if meta[1] >> site & 1)
            if not row_fails or not lane_fails:
                missed.append((site, row_fails, lane_fails))
    finally:
        lib.sp_mutant(-1, -1)
    assert not missed, f"{kind}: sites whose mutant no row or no lane catches (site, failing rows, failing lanes): {missed}"
    s, p, m = rows[0][:3]
    assert verify(lib, s, p, m)[0] == 1


# ---- the real kernels behind the real host layer on the SIMT emulator, probe applied to the emulator's headers ----
HS = os.path.join(HERE, "host_sim")
EMUL = {"CUDASIM_DEVICES": "1", "CUDASIM_SMS": "1", "CUDASIM_RESIDENT": "32"}


@pytest.fixture(scope="module")
def probed_kernels(tmp_path_factory):
    """libeddsa_sim_kernels.so with kernels_verify built from a probed copy of the rewritten headers."""
    subprocess.run(["make", "-s", "-j4", "-C", HS], check=True)
    tmp = tmp_path_factory.mktemp("settle_emul")
    gen = tmp / "csrc"
    settle_probe.probe_tree(os.path.join(os.path.dirname(HERE), "libeddsa_b200", "csrc"), str(gen), ptx=True)
    obj, so = str(tmp / "kernels_verify.o"), str(tmp / "libeddsa_sim_kernels_probed.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-D__CUDA_ARCH__=1000", "-D__CUDACC__",
                    "-DEDG_EMUL_COUNT", "-I" + os.path.join(HS, "fake_cuda"), "-include", os.path.join(HS, "simt_emul.h"),
                    "-c", str(gen / "kernels_verify.cu.cpp"), "-o", obj], check=True)
    subprocess.run(["g++", "-shared", "-o", so, os.path.join(HS, "cudasim_real.o"), os.path.join(HS, "host_sim.o"),
                    os.path.join(HS, "_ptx", "kernels_x25519.o"), os.path.join(HS, "_ptx", "kernels_fixedbase.o"), obj, "-lpthread",
                    "-Wl,--allow-multiple-definition"], check=True)
    return so


@pytest.mark.parametrize("scenario", ["rows", "lanes"])
def test_real_kernels_on_the_simt_emulator_take_every_site(probed_kernels, scenario):
    """rows: ed25519_verify_batch over the corpus rows (k_verify).  lanes: ed25519_verify_zip215_batched_dev with every lane
    where k_verify_batched reads it, under EDDSA_B200_DEBUG_NO_FALLBACK=1.  Every site taken, every output 1."""
    env = {k: v for k, v in os.environ.items() if not k.startswith(("CUDASIM_", "EDDSA_B200_"))}
    env.update(EMUL, CUDASIM_SO=probed_kernels)
    if scenario == "lanes":
        env["EDDSA_B200_DEBUG_NO_FALLBACK"] = "1"
    res = subprocess.run([sys.executable, os.path.join(HS, "settle_scenarios.py"), scenario], env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, timeout=1800)
    print(res.stdout[-2000:])
    assert res.returncode == 0 and f"OK {scenario}" in res.stdout, res.stdout[-3000:]
