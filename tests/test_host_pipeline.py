"""The host layer (libeddsa_b200/csrc/host.c: sharding over devices, worker threads, chunk schedule, staging slots, event
dependencies, scrubbing of secrets, error paths, the single-operation API) exercised WITHOUT a GPU: host.c is linked, unchanged,
against a simulator of the CUDA runtime (tests/host_sim/cudasim.cpp — lazily executing streams, bounds-checked memory, failure
injection; its "kernels" run the per-thread operation bodies of ops.cuh compiled for the host) and driven through the product's
own ctypes binding.  Every scenario (tests/host_sim/sim_scenarios.py) runs in a fresh interpreter and checks results against the
CPU reference.  This is test infrastructure only: the simulator lives under tests/ and the product has no CPU path.

The mutants at the end prove the simulator has teeth: host.c with one dependency, synchronisation or scrub removed must FAIL the
scenario that covers it.
"""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
HS = os.path.join(HERE, "host_sim")
HOST_C = os.path.join(os.path.dirname(HERE), "libeddsa_b200", "csrc", "host.c")


_PREFETCHED = {}       # (scenario, env items, args) -> future: the scenario runs of this module, started three at a time in the background


def _key(name, env, args, so=None):
    return (name, tuple(sorted((env or {}).items())), tuple(args), so)


def _run(name, env=None, args=(), so=None, timeout=600):
    e = {k: v for k, v in os.environ.items() if not k.startswith(("CUDASIM_", "EDDSA_B200_"))}
    e.update(env or {})
    if so:
        e["CUDASIM_SO"] = so
    return subprocess.run([sys.executable, os.path.join(HS, "sim_scenarios.py"), name, *args], env=e, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=timeout)


def run_scenario(name, env=None, args=(), so=None, timeout=600):
    fut = _PREFETCHED.pop(_key(name, env, args, so), None)
    return fut.result() if fut else _run(name, env, args, so, timeout)


@pytest.fixture(scope="module")
def simlib():
    """Builds the simulator library and starts every scenario run of this module in the background (each is its own
    process; three at a time), so that the tests mostly collect results."""
    import concurrent.futures
    subprocess.run(["make", "-s", "-j4", "-C", HS], check=True)
    pool = concurrent.futures.ThreadPoolExecutor(max_workers=3)
    for name, env, args in _planned_runs():
        _PREFETCHED[_key(name, env, args)] = pool.submit(_run, name, env, args)
    for name, env in REAL_KERNEL_RUNS:
        _PREFETCHED[_key(name, env, (), KERNELS_SO)] = pool.submit(_run, name, env, (), KERNELS_SO)
    _PREFETCHED[_key("real_kernels_opcount", {"CUDASIM_DEVICES": "1"}, ("2048",), KERNELS_SO)] = pool.submit(
        _run, "real_kernels_opcount", {"CUDASIM_DEVICES": "1"}, ("2048",), KERNELS_SO)
    import tempfile
    scratch = tempfile.mkdtemp(prefix="eddsa_mutants_")
    for index in range(len(MUTANTS)):
        _PREFETCHED[("mutant", index)] = pool.submit(_mutant_job, index, os.path.join(scratch, str(index)))
    yield os.path.join(HS, "libeddsa_sim.so")
    for fut in _PREFETCHED.values():
        fut.cancel()
    pool.shutdown(wait=True)
    import shutil
    shutil.rmtree(scratch, ignore_errors=True)


SCENARIOS = {
    "all_ops": {"CUDASIM_DEVICES": "1"},
    "chunks": {"CUDASIM_DEVICES": "1", "CUDASIM_SMS": "1"},
    "budget": {"CUDASIM_DEVICES": "1", "EDDSA_B200_CHUNK_MB": "1"},
    "multi": {"CUDASIM_DEVICES": "4"},
    "device_list": {"CUDASIM_DEVICES": "4", "EDDSA_B200_DEVICES": "2,0"},
    "scrub": {"CUDASIM_DEVICES": "1"},
    "failures": {"CUDASIM_DEVICES": "1", "CUDASIM_SMS": "1", "CUDASIM_RESIDENT": "32"},
    "threads": {"CUDASIM_DEVICES": "2"},
    "dev_api": {"CUDASIM_DEVICES": "1"},
    "lifecycle": {"CUDASIM_DEVICES": "4"},
    "copy_helpers": {"CUDASIM_DEVICES": "1", "EDDSA_B200_COPY_THREADS": "3"},
    "no_device": {"CUDASIM_DEVICES": "0"},
}


# the REAL kernels and launchers on the SIMT emulator (host_sim/simt_emul.h) behind the same host layer and simulator
KERNELS_SO = os.path.join(HS, "libeddsa_sim_kernels.so")
# (the all_ops and lifecycle scenarios and the other stream schedules pass on it too; left out of the suite for time: ~30 s each)
REAL_KERNEL_RUNS = [("real_kernels", {"CUDASIM_DEVICES": "1", "EDDSA_B200_VERIFY_WAVES": "1"}),
                    ("real_kernels_full_scalars", {"CUDASIM_DEVICES": "1", "EDDSA_B200_DEBUG_FULL_SCALARS": "1"}),
                    ("real_kernels_structured", {"CUDASIM_DEVICES": "1"})]

OTHER_SCHEDULES = [(n, sch) for n in ("chunks", "budget", "multi", "threads", "dev_api", "failures") for sch in ("others-first", "eager", "random")
                   if n != "failures" or sch == "others-first"]        # the failure sweep: the two adversarial schedules only (12 s each)
WALKS = [(1, "lazy", 3), (2, "others-first", 4), (3, "random", 2), (6, "lazy", 3)]


def _walk_env(seed, schedule, devices):
    env = {"CUDASIM_DEVICES": str(devices), "CUDASIM_SMS": "1", "CUDASIM_RESIDENT": "32", "CUDASIM_SCHEDULE": schedule}
    if seed % 3 == 0:
        env["EDDSA_B200_CHUNK_MB"] = "1"
    return env


def _planned_runs():
    """In the order the tests below ask for them."""
    for name in SCENARIOS:
        yield name, SCENARIOS[name], ()
    for name, schedule in OTHER_SCHEDULES:
        yield name, dict(SCENARIOS[name], CUDASIM_SCHEDULE=schedule), ()
    for seed, schedule, devices in WALKS:
        yield "fuzz", _walk_env(seed, schedule, devices), (str(seed), "60")
    yield "scrub", dict(SCENARIOS["scrub"], EDDSA_B200_DEBUG_NO_SCRUB="1"), ()
    yield "no_device", SCENARIOS["no_device"], ("abort",)


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_host_layer_on_the_simulator(simlib, name):
    """Lazy streams: an operation runs only when something waits for it — the most adversarial legal schedule."""
    res = run_scenario(name, SCENARIOS[name])
    assert res.returncode == 0 and f"OK {name}" in res.stdout, res.stdout[-3000:]


@pytest.mark.parametrize("name,schedule", OTHER_SCHEDULES)
def test_host_layer_under_other_schedules(simlib, name, schedule):
    """The same scenarios with every other stream running as far as it can before the awaited one advances (work without a
    dependency runs EARLY — the complement of the lazy schedule), with everything executing at once, and with a random
    interleaving of the streams."""
    res = run_scenario(name, dict(SCENARIOS[name], CUDASIM_SCHEDULE=schedule))
    assert res.returncode == 0 and f"OK {name}" in res.stdout, res.stdout[-3000:]


@pytest.mark.parametrize("name,env", REAL_KERNEL_RUNS, ids=[n + "-" + e.get("CUDASIM_SCHEDULE", "lazy") for n, e in REAL_KERNEL_RUNS])
def test_real_kernels_on_the_simt_emulator(simlib, name, env):
    """kernels_*.cu as shipped — kernel launches and inline PTX rewritten (ptx_rewrite.py), lanes as OS threads with real
    rendezvous for __syncthreads, the warp collectives and mma.sync (simt_emul.h) — behind the real host layer: the reference's
    x25519 table, the Ed25519 KAT with ragged messages, all 2 960 adversarial verify decisions, wrong-pub signing, conversions,
    the device-built tables, SHA block-boundary lengths at odd alignments, the full-length fallback.  Bit-exact, without a GPU."""
    res = run_scenario(name, env, so=KERNELS_SO)
    assert res.returncode == 0 and f"OK {name}" in res.stdout, res.stdout[-3000:]


def test_roofline_work_figure_counted_on_the_real_kernels(simlib):
    """Field operations per signature executed by the shipped verify kernels (a lane runs its warp's maximum window count after the
    permutation), counted by the emulator: within 1 % of the figure bench.py's integer-multiply roofline uses (16 384 signatures:
    130 991 vs 130 992 wide multiplies, profiles/r02_notes.md)."""
    res = run_scenario("real_kernels_opcount", {"CUDASIM_DEVICES": "1"}, args=("2048",), so=KERNELS_SO)
    assert res.returncode == 0 and "OK real_kernels_opcount" in res.stdout, res.stdout[-3000:]


def test_kernels_wipe_their_scratch(simlib, tmp_path):
    """The secret scalars the hash kernels hand to the comb through pool scratch are wiped by the kernels themselves (searched for
    in the returned pool blocks); a mutant of kernels_fixedbase.cu with the three wipes removed leaves every one of them behind."""
    env = {"CUDASIM_DEVICES": "1", "CUDASIM_KEEP_FREED": "1"}
    res = run_scenario("kernel_scrub", env, so=KERNELS_SO)
    assert res.returncode == 0 and "OK kernel_scrub" in res.stdout, res.stdout[-3000:]
    gen = os.path.join(HS, "_ptx", "libeddsa_b200", "csrc")
    src = open(os.path.join(gen, "kernels_fixedbase.cu.cpp")).read()
    for wipe in ("wipe_words8(scalars + 8 * i0);", "wipe_words8(a_in + 8 * i);", "wipe_words8(r_in + 8 * i);"):
        assert src.count(wipe) == 1, wipe
        src = src.replace(wipe, "(void)0;")
    mutant = tmp_path / "kernels_fixedbase.cu.cpp"
    mutant.write_text(src)
    obj, so = str(tmp_path / "kernels_fixedbase.o"), str(tmp_path / "libeddsa_sim_kernels_nowipe.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-D__CUDA_ARCH__=1000", "-D__CUDACC__",
                    "-I" + os.path.join(HS, "fake_cuda"), "-I" + gen, "-include", os.path.join(HS, "simt_emul.h"), "-c", str(mutant), "-o", obj], check=True)
    subprocess.run(["g++", "-shared", "-o", so, os.path.join(HS, "cudasim_real.o"), os.path.join(HS, "host_sim.o"), os.path.join(HS, "_ptx", "kernels_x25519.o"),
                    obj, os.path.join(HS, "_ptx", "kernels_verify.o"), "-lpthread", "-Wl,--allow-multiple-definition"], check=True)
    res = run_scenario("kernel_scrub", env, args=("expect-residue",), so=so)
    assert res.returncode == 0 and "OK kernel_scrub" in res.stdout, res.stdout[-3000:]


@pytest.mark.parametrize("seed,schedule,devices", WALKS)
def test_random_walk_over_the_c_abi(simlib, seed, schedule, devices):
    """Random operations, sizes, layouts, page-locked / ordinary buffers, device counts, shutdowns and injected failures
    (tools/host_fuzz_campaign.sh runs the long version: 400 runs x 100 steps, profiles/r02_notes.md)."""
    res = run_scenario("fuzz", _walk_env(seed, schedule, devices), args=(str(seed), "60"))
    assert res.returncode == 0 and "OK fuzz" in res.stdout, res.stdout[-3000:]


def test_host_layer_under_sanitizers(simlib, tmp_path):
    """host.c, the simulator and the host build of the operation bodies compiled with AddressSanitizer + UBSan: no invalid access
    (a caller buffer written after the call returned would show up here), no undefined arithmetic."""
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], stdout=subprocess.PIPE, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan is not installed")
    root = os.path.dirname(HERE)
    san = ["-g", "-O1", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fPIC"]
    inc = ["-I" + os.path.join(root, "include"), "-I/usr/local/cuda/include"]
    so = str(tmp_path / "libeddsa_sim_san.so")
    subprocess.run(["gcc", *san, "-std=gnu11", "-fvisibility=hidden", "-DEDDSA_BUILD", *inc, "-c", HOST_C, "-o", str(tmp_path / "host.o")], check=True)
    subprocess.run(["g++", *san, "-std=c++17", "-Wno-unknown-pragmas", *inc, "-c", os.path.join(HS, "cudasim.cpp"), "-o", str(tmp_path / "cudasim.o")], check=True)
    subprocess.run(["g++", "-shared", "-fsanitize=address,undefined", "-o", so, str(tmp_path / "cudasim.o"), str(tmp_path / "host.o"), "-lpthread"], check=True)
    for name in ("all_ops", "budget"):
        env = dict(SCENARIOS[name], LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0")
        res = run_scenario(name, env, so=so)
        assert res.returncode == 0 and f"OK {name}" in res.stdout and "runtime error" not in res.stdout, res.stdout[-3000:]


def test_scrub_negative_control(simlib):
    """With the scrubbing switched off the same search finds the secrets: the scrub is what removes them."""
    res = run_scenario("scrub", dict(SCENARIOS["scrub"], EDDSA_B200_DEBUG_NO_SCRUB="1"))
    assert res.returncode == 0 and "OK scrub" in res.stdout, res.stdout[-3000:]


def test_single_operation_without_a_device_aborts(simlib):
    """The void functions of eddsa.h cannot report an error and there is no CPU fallback: they abort."""
    res = run_scenario("no_device", SCENARIOS["no_device"], args=("abort",))
    assert res.returncode == -6 and "NOT REACHED" not in res.stdout and "no usable CUDA device" in res.stdout, (res.returncode, res.stdout[-2000:])


# (what is removed from host.c, the exact text, its replacement, the scenario that must notice)
MUTANTS = [
    ("kernels do not wait for their chunk's input copies",
     "            CU(cudaStreamWaitEvent(c->kstream, c->in_ready[s], 0));\n", "", "chunks"),
    ("the result copy does not wait for the kernels",
     "            CU(cudaStreamWaitEvent(c->stream[s], c->k_done[s], 0));\n", "", "chunks"),
    ("a slot is reused without waiting for the chunk that used it",
     "        if (slot[s].inflight) { /* retire the chunk that used this slot */\n            CU(cudaEventSynchronize(c->done[s]));\n",
     "        if (slot[s].inflight) { /* retire the chunk that used this slot */\n", "chunks"),
    ("the last chunks are handed out without waiting for them",
     "            cudaError_t e = rc ? cudaSuccess : cudaEventSynchronize(c->done[s]);\n", "            cudaError_t e = cudaSuccess;\n", "all_ops"),
    ("buffers are re-allocated while chunks are in flight",
     "                if (slot[k].inflight) {\n                    CU(cudaEventSynchronize(c->done[k]));\n                    retire_slot(c, j, &slot[k], k, pin_out, 1);\n                }\n",
     "                slot[k].inflight = 0;\n", "budget"),
    ("message offsets are not rebased to the chunk",
     "ho[i] = (unsigned long long)(j->off[pos + i] - j->off[pos]);", "ho[i] = (unsigned long long)j->off[pos + i];", "budget"),
    ("the device copy of the secret keys is not wiped",
     "        if (secret_in) CU(cudaMemsetAsync(c->d_in[s], 0, m * j->in_item[0], c->stream[s]));", "", "scrub"),
    ("the staged host copy of the secret keys is not wiped",
     "    if (sl->staged_secret && !g_no_scrub) memset(c->h_in[s], 0, m * j->in_item[0]);\n", "", "scrub"),
    ("secret outputs stay in the host slot",
     "        if (op_secret_out(j->op) && !g_no_scrub) memset(c->h_out[s], 0, m * j->out_item);\n", "", "scrub"),
    ("the caller's current device is not restored",
     "    if (prev_dev >= 0 && prev_dev != c->dev) cudaSetDevice(prev_dev);\n", "", "multi"),
    ("a failed call returns while chunks are still in flight",
     "                cudaDeviceSynchronize();        /* the younger chunks", "                ;        /* the younger chunks", "failures"),
    ("keys staged by the chunk that failed are not wiped",
     "            if (c->h_in[k]) memset(c->h_in[k], 0, c->in_cap);\n", "", "failures"),
    ("shards overlap by one item",
     "        sh[g].hi = j->n * (size_t)(g + 1) / ndev;", "        sh[g].hi = j->n * (size_t)(g + 1) / ndev + (g + 1 < ndev);", "multi"),
]


def _mutant_job(index, workdir):
    """Builds host.c with one change and runs the covering scenario under the two adversarial schedules; returns None when a
    run failed (the mutant was caught), else a description."""
    what, old, new, scenario = MUTANTS[index]
    src = open(HOST_C).read()
    if src.count(old) != 1:
        return f"host.c changed: the text of mutant '{what}' must occur exactly once"
    os.makedirs(workdir, exist_ok=True)
    mutant_c, obj, so = os.path.join(workdir, "host.c"), os.path.join(workdir, "host.o"), os.path.join(workdir, "libeddsa_sim_mutant.so")
    with open(mutant_c, "w") as f:
        f.write(src.replace(old, new))
    inc = ["-I" + os.path.join(os.path.dirname(HERE), "include"), "-I" + os.path.join(os.path.dirname(HOST_C)), "-I/usr/local/cuda/include"]
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-fPIC", "-fvisibility=hidden", "-DEDDSA_BUILD", *inc, "-c", mutant_c, "-o", obj], check=True)
    subprocess.run(["g++", "-shared", "-o", so, os.path.join(HS, "cudasim.o"), obj, "-lpthread"], check=True)
    for schedule in ("lazy", "others-first"):
        if _run(scenario, dict(SCENARIOS[scenario], CUDASIM_SCHEDULE=schedule), so=so).returncode != 0:
            return None
    return f"the '{scenario}' scenario did not notice that {what}"


@pytest.mark.parametrize("index", range(len(MUTANTS)), ids=[m[0] for m in MUTANTS])
def test_simulator_catches_host_layer_mutants(simlib, tmp_path, index):
    fut = _PREFETCHED.pop(("mutant", index), None)
    verdict = fut.result() if fut else _mutant_job(index, str(tmp_path))
    assert verdict is None, verdict
