"""Batched ZIP215 verification without a GPU: the big-integer model of the lane equation (tests/verify_batched_model.py)
decides "every included row is ZIP215-valid" on every generated layout; a cancelling pair of invalid rows passes only under
unit weights; the public constants agree across header, binding and kernels; and on the CUDA runtime simulator the real
kernels decide every fixture and generated row like ZIP215 (and, without the fallback, like the raw lane equations), the
entry points check their arguments and a failing getrandom(2) before any work, and launcher sets without the batched
check refuse it."""
import os
import re
import shutil
import subprocess
import sys

import pytest

import verify_batched_model as bm
import verify_policy_model as vm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = bytes(range(32))


@pytest.fixture(scope="module")
def lanes():
    rows, want, _ = vm.all_rows()
    return bm.layouts(rows, want)


def test_layouts_cover_every_case(lanes):
    assert any(not bm.all_valid(lane) for lane in lanes)
    assert any(all(bm.included(s, p) for s, p, _ in lane) and bm.all_valid(lane) for lane in lanes)
    assert any(not all(bm.included(s, p) for s, p, _ in lane) and bm.all_valid(lane) for lane in lanes)
    assert any(len(lane) < bm.K for lane in lanes)


def test_lane_equation_is_all_included_rows_valid(lanes):
    for i, lane in enumerate(lanes):
        assert bm.lane_holds(lane, SEED) == bm.all_valid(lane), i


def test_cancelling_pair_needs_random_weights():
    rows, want, _ = vm.all_rows()
    valid = [r[:3] for r, d in zip(rows, want) if d[vm.ZIP215] and d[vm.REFERENCE]]
    a, b = bm.cancelling_pair(*valid[0], *valid[1])
    assert not vm.decisions(*a)[vm.ZIP215] and not vm.decisions(*b)[vm.ZIP215]
    assert bm.lane_holds([a, b], unit_weights=True)
    assert not bm.lane_holds([a, b], SEED)


def test_weights_depend_on_the_row_only():
    rows, _, _ = vm.all_rows()
    s, p, m, _ = rows[0]
    z = bm.weight(SEED, s, p, m)
    assert z & 1 and 0 < z < 2 ** 128 and z == bm.weight(SEED, s, p, m)
    assert z != bm.weight(bytes(32), s, p, m)


def test_batch_rows_agree():
    import libeddsa_b200 as ed
    hdr = open(os.path.join(ROOT, "include", "eddsa_batch.h")).read()
    ops = open(os.path.join(ROOT, "libeddsa_b200", "csrc", "ops.cuh")).read()
    h = int(re.search(r"#define EDDSA_B200_VERIFY_BATCH_ROWS (\d+)", hdr).group(1))
    k = int(re.search(r"#define EDG_VBATCH_K (\d+)", ops).group(1))
    assert h == k == ed.VERIFY_BATCH_ROWS == bm.K


# ---- the host layer and the real kernels on the CUDA runtime simulator (tests/host_sim/batched_scenarios.py) ----
HS = os.path.join(ROOT, "tests", "host_sim")
EMUL = {"CUDASIM_DEVICES": "1", "CUDASIM_SMS": "1", "CUDASIM_RESIDENT": "32"}


def _scenario(name, env, so, args=(), timeout=1800):
    e = {k: v for k, v in os.environ.items() if not k.startswith(("CUDASIM_", "EDDSA_B200_"))}
    e.update(env)
    e["CUDASIM_SO"] = so
    return subprocess.run([sys.executable, os.path.join(HS, "batched_scenarios.py"), name, *args], env=e, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=timeout)


@pytest.fixture(scope="module")
def simlibs():
    subprocess.run(["make", "-s", "-j4", "-C", HS], check=True)
    return {"mock": os.path.join(HS, "libeddsa_sim.so"), "kernels": os.path.join(HS, "libeddsa_sim_kernels.so")}


@pytest.mark.parametrize("mode", ["fallback", "no_fallback"])
def test_real_kernels_on_the_simt_emulator(simlibs, mode):
    """Every fixture and generated row through the real kernels: ZIP215 exactly; under EDDSA_B200_DEBUG_NO_FALLBACK=1 the raw
    equations, zero on exactly the groups that hold an invalid included row."""
    env = dict(EMUL, **({"EDDSA_B200_DEBUG_NO_FALLBACK": "1"} if mode == "no_fallback" else {}))
    res = _scenario("real_kernels_verify_batched", env, simlibs["kernels"], [mode])
    assert res.returncode == 0 and "OK real_kernels_verify_batched" in res.stdout, res.stdout[-3000:]


def test_argument_checks_and_getrandom_failure(simlibs, tmp_path):
    """n = 0, misaligned arrays and a failing getrandom(2) (a preloaded getrandom returning ENOSYS) launch nothing."""
    res = _scenario("argument_checks", EMUL, simlibs["kernels"])
    assert res.returncode == 0 and "OK argument_checks" in res.stdout, res.stdout[-3000:]
    src, shim = tmp_path / "getrandom_fails.c", tmp_path / "getrandom_fails.so"
    src.write_text("#include <errno.h>\n#include <sys/types.h>\n"
                   "ssize_t getrandom(void *b, size_t n, unsigned f) { (void)b; (void)n; (void)f; errno = ENOSYS; return -1; }\n")
    subprocess.run(["gcc", "-shared", "-fPIC", "-o", str(shim), str(src)], check=True)
    res = _scenario("argument_checks", dict(EMUL, LD_PRELOAD=str(shim)), simlibs["kernels"], ["getrandom_fails"])
    assert res.returncode == 0 and "OK argument_checks" in res.stdout, res.stdout[-3000:]


def test_launchers_without_the_batched_check_refuse_it(simlibs):
    res = _scenario("no_batched_launcher", {"CUDASIM_DEVICES": "1"}, simlibs["mock"])
    assert res.returncode == 0 and "OK no_batched_launcher" in res.stdout, res.stdout[-3000:]


# (what is changed in ops.cuh, the exact text, its replacement); each must make the raw-equation scenario fail
KERNEL_MUTANTS = [
    ("the cofactor doublings removed", "const int last = j < 0 ? 3 :", "const int last = j < 0 ? 0 :"),
    ("every weight forced to 1", "    z[0] |= 1u;\n", "    z[0] = 1u; z[1] = 0u; z[2] = 0u; z[3] = 0u;\n"),
    ("excluded rows not masked", "const int dg = ((incl >> r_) & 1u) ?", "const int dg = 1 ?"),
    ("the base digits of the neighbouring lane", "    sc_reduce512(es, acc);\n",
     "    sc_reduce512(es, acc);\n    for (int i = 0; i < 8; i++) es[i] = __shfl_sync(0xffffffffu, es[i], (threadIdx.x + 1) & 31);\n"),
]


@pytest.mark.parametrize("index", range(len(KERNEL_MUTANTS)), ids=[m[0] for m in KERNEL_MUTANTS])
def test_emulator_scenario_catches_kernel_mutants(simlibs, tmp_path, index):
    what, old, new = KERNEL_MUTANTS[index]
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
    res = _scenario("real_kernels_verify_batched", dict(EMUL, EDDSA_B200_DEBUG_NO_FALLBACK="1"), so, ["no_fallback"])
    assert res.returncode != 0 and "MISMATCH" in res.stdout, (what, res.stdout[-3000:])
