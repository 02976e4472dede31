"""The verify acceptance rules without a GPU (ed25519_verify_policy_batch / _dev; REFERENCE, STRICT = RFC 8032 with canonical
encodings as libsodium decides, ZIP215 = Zcash's ZIP 215):

- the big-integer model of tests/verify_policy_model.py against the compiled reference's decisions (the fixtures' expect
  column) and against libsodium (PyNaCl), and its per-class acceptance counts on the fixtures;
- the host build of ops.cuh (tests/host_sim/verify_policy_host.cpp, both flavours of tests/test_host_sim.py) deciding every row
  like the model under each rule;
- the host layer on the CUDA runtime simulator (tests/host_sim/cudasim_policy.cpp, policy_scenarios.py): unknown rules refused,
  rule 0 = ed25519_verify_batch, every rule across chunks, passes and shards with ragged offsets, through both new entry points;
  and, linked against launchers without the rules, STRICT and ZIP215 refused;
- the real kernels on the SIMT emulator, and three kernel mutants that scenario must catch.
"""
import collections
import ctypes
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import verify_policy_model as vm

HERE = os.path.dirname(os.path.abspath(__file__))
HS = os.path.join(HERE, "host_sim")

# per fixture class: rows, accepted under REFERENCE, STRICT, ZIP215 ("other": classes 1-4, 12-15 and 19, rejected by every rule)
CLASS_TABLE = {0: (88, 88, 88, 88), 5: (1024, 960, 0, 0), 6: (51, 13, 0, 14), 7: (234, 0, 0, 234), 10: (624, 73, 0, 624),
               11: (96, 22, 22, 96), 16: (18, 18, 18, 18), 17: (70, 0, 0, 70), 18: (54, 54, 0, 0), "other": (701, 0, 0, 0)}


@pytest.fixture(scope="module")
def model():
    return vm.all_rows()


def test_model_reference_rule_is_the_compiled_reference(model):
    """On all 2 960 fixture rows the model's REFERENCE decision is the compiled reference's (the fixtures' expect column)."""
    rows, want, cls = model
    fx, expect = vm.fixture_rows()
    assert len(fx) == 2960
    assert (want[:len(fx), vm.REFERENCE] == expect).all(), np.nonzero(want[:len(fx), vm.REFERENCE] != expect)[0][:10]


def test_model_strict_rule_is_libsodium(model):
    """STRICT decides like libsodium's crypto_sign_open on every fixture row and every generated row."""
    pytest.importorskip("nacl.bindings")
    rows, want, cls = model
    lib = np.array([vm.libsodium_decision(s, p, m) for s, p, m, _ in rows], np.uint8)
    bad = np.nonzero(lib != want[:, vm.STRICT])[0]
    assert not len(bad), [(int(i), int(cls[i]), int(lib[i])) for i in bad[:10]]


def test_per_class_acceptance_on_the_fixtures(model):
    rows, want, cls = model
    n = len(vm.fixture_rows()[0])
    got = collections.defaultdict(lambda: np.zeros(4, np.int64))
    for c, d in zip(cls[:n], want[:n]):
        got[int(c) if int(c) in CLASS_TABLE else "other"] += [1, *d]
    assert {k: tuple(int(x) for x in v) for k, v in got.items()} == CLASS_TABLE
    assert tuple(want[:n].sum(axis=0)) == (1228, 128, 1144)


def test_generated_rows(model):
    """What each generated class is built to show (the generator itself asserts the minimum row counts)."""
    rows, want, cls = model
    dec = lambda c: want[cls == c]
    for c in (vm.G_TORSION_R, vm.G_SMALL_R_ENCODING):            # accepted by ZIP215 only
        assert (dec(c) == (0, 0, 1)).all(), c
    assert not dec(vm.G_ZIP_ONLY_S_PLUS_L).any()                   # ... and with S + L by none
    mixed = dec(vm.G_MIXED_ORDER_KEY)
    assert (mixed[:, 1] == mixed[:, 0]).all() and mixed[:, 2].all() and 0 < mixed[:, 0].sum() < len(mixed)
    s = np.array([int.from_bytes(r[0][32:], "little") for r, c in zip(rows, cls) if c == vm.G_S_BOUNDARY])
    b = dec(vm.G_S_BOUNDARY)
    assert (b[:, 1:][s >= vm.L] == 0).all()                        # the range check of STRICT and ZIP215
    ident = np.array([r[1] == vm.em.enc((0, 1)) for r, c in zip(rows, cls) if c == vm.G_S_BOUNDARY])
    assert b[ident, 0].all() and (b[ident, 2] == (s[ident] < vm.L)).all() and not b[ident, 1].any()
    assert {vm.L - 1, vm.L, vm.L + 1, 2**253, 2**256 - 1} <= set(int(x) for x in s)


@pytest.fixture(scope="module", params=["host", "device"])
def ops(request):
    from test_host_sim import _build
    lib = _build("verify_policy_host", request.param)
    lib.hs_verify_policy.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint64, ctypes.c_int]
    return lib


def test_host_build_decides_like_the_model(ops, model):
    """ops.cuh compiled for the host (and its device paths on the PTX interpreter, every seventh row): every rule, every row."""
    rows, want, cls = model
    step = 7 if ops.device_paths else 1
    for i in range(0, len(rows), step):
        s, p, m, _ = rows[i]
        got = tuple(ops.hs_verify_policy(s, p, m, len(m), pol) for pol in vm.POLICIES)
        assert got == tuple(want[i]), (i, int(cls[i]), got, tuple(want[i]))


def _scenario(name, env, args=(), so=None, timeout=900):
    e = {k: v for k, v in os.environ.items() if not k.startswith(("CUDASIM_", "EDDSA_B200_"))}
    e.update(env)
    if so:
        e["CUDASIM_SO"] = so
    return subprocess.run([sys.executable, os.path.join(HS, "policy_scenarios.py"), name, *args], env=e, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=timeout)


@pytest.fixture(scope="module")
def simlibs(tmp_path_factory):
    """The simulator libraries of tests/host_sim/Makefile, and libeddsa_sim_policy.so: host.c + cudasim_policy.cpp (the mock kernels
    and a mock of the rule-aware launcher)."""
    subprocess.run(["make", "-s", "-j4", "-C", HS], check=True)
    d = tmp_path_factory.mktemp("sim_policy")
    obj, so = str(d / "cudasim_policy.o"), str(d / "libeddsa_sim_policy.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-Wno-unknown-pragmas", "-I/usr/local/cuda/include", "-c",
                    os.path.join(HS, "cudasim_policy.cpp"), "-o", obj], check=True)
    subprocess.run(["g++", "-shared", "-o", so, obj, os.path.join(HS, "host_sim.o"), "-lpthread"], check=True)
    return {"policy": so, "mock": os.path.join(HS, "libeddsa_sim.so"), "kernels": os.path.join(HS, "libeddsa_sim_kernels.so")}


def test_entry_points_on_the_simulator(simlibs):
    """EINVAL for rules -1 and 3 (also for n = 0, before any work); rule 0 = ed25519_verify_batch; all three rules over two shards,
    passes of 512 signatures and ragged offsets, host and device API."""
    res = _scenario("verify_policy", {"CUDASIM_DEVICES": "2", "CUDASIM_SMS": "1", "CUDASIM_RESIDENT": "32"}, so=simlibs["policy"])
    assert res.returncode == 0 and "OK verify_policy" in res.stdout, res.stdout[-3000:]


def test_launchers_without_the_rules_refuse_them(simlibs):
    """Linked against launchers that implement only the reference's rule, the host layer refuses STRICT and ZIP215 with EINVAL."""
    res = _scenario("reference_launchers_only", {"CUDASIM_DEVICES": "1"}, so=simlibs["mock"])
    assert res.returncode == 0 and "OK reference_launchers_only" in res.stdout, res.stdout[-3000:]


def test_real_kernels_on_the_simt_emulator(simlibs):
    """k_verify_points<POLICY> and k_verify<COFACTORED> as shipped: every fixture and generated row under each rule."""
    res = _scenario("real_kernels_verify_policy", {"CUDASIM_DEVICES": "1"}, so=simlibs["kernels"])
    assert res.returncode == 0 and "OK real_kernels_verify_policy" in res.stdout, res.stdout[-3000:]


# (what is changed in ops.cuh, the exact text, its replacement, the rule and the classes the scenario runs to notice it)
KERNEL_MUTANTS = [
    ("the S < L check dropped", "good = 0u - sc_below_L(s);", "good = 0xffffffffu;", "strict", "5"),
    ("the small-order test reads 7Q instead of 8Q",
     "        ge_add_cached<true>(Q, Q, c1, true);              // k*Q = (k-1)*Q + Q\n        ge_to_cached<true>(c, Q);\n",
     "        ge_p3 N;\n        ge_add_cached<true>(N, Q, c1, true);\n        ge_to_cached<true>(c, N);\n        if (k < 8) Q = N;\n",
     "strict", "6,10"),
    ("two cofactor doublings instead of three", "const int last = COFACTORED && j < 0 ? 3 :", "const int last = COFACTORED && j < 0 ? 2 :",
     "zip215", "17,101"),
]


@pytest.mark.parametrize("index", range(len(KERNEL_MUTANTS)), ids=[m[0] for m in KERNEL_MUTANTS])
def test_emulator_scenario_catches_kernel_mutants(simlibs, tmp_path, index):
    what, old, new, rule, classes = KERNEL_MUTANTS[index]
    gen = os.path.join(HS, "_ptx", "libeddsa_b200", "csrc")
    mut = tmp_path / "csrc"
    shutil.copytree(gen, mut)
    src = (mut / "ops.cuh").read_text()
    assert src.count(old) == 1, what
    (mut / "ops.cuh").write_text(src.replace(old, new))
    obj, so = str(tmp_path / "kernels_verify.o"), str(tmp_path / "libeddsa_sim_kernels_mutant.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-D__CUDA_ARCH__=1000", "-D__CUDACC__",
                    "-DEDG_EMUL_COUNT", "-I" + os.path.join(HS, "fake_cuda"), "-include", os.path.join(HS, "simt_emul.h"),
                    "-c", str(mut / "kernels_verify.cu.cpp"), "-o", obj], check=True)
    subprocess.run(["g++", "-shared", "-o", so, os.path.join(HS, "cudasim_real.o"), os.path.join(HS, "host_sim.o"),
                    os.path.join(HS, "_ptx", "kernels_x25519.o"), os.path.join(HS, "_ptx", "kernels_fixedbase.o"), obj, "-lpthread",
                    "-Wl,--allow-multiple-definition"], check=True)
    res = _scenario("real_kernels_verify_policy", {"CUDASIM_DEVICES": "1"}, args=(rule, classes), so=so)
    assert res.returncode != 0 and "MISMATCH " + rule in res.stdout, (what, res.stdout[-3000:])
