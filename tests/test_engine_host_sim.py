"""The engine's HOST logic on a box without a GPU.

csrc/engine.cu holds no device code: node-table builds (class-sorted records, the HRW2 blob, per-node policy state), directory sizing
and growth, the bounded-load round protocol, the place_batch / check_address_batch flows and every extern "C" entry point are plain
C++ around CUDA runtime calls and kernel launchers.  Here that file (with resolver.cu and durable.cu -- the very sources nvcc builds
into the product) is compiled with g++ against

  * tests/cpp/hostsim/cuda_runtime.h -- a synchronous stand-in for the ~45 runtime calls it makes ("device" memory is malloc'ed), and
  * tests/cpp/hostsim/launchers.cpp  -- plain restatements of what each kernel launcher of csrc/kernels.cuh is specified to do,

into tests/_build/librio_cuda_hostsim.so, and the `-m gpu` test modules are run against it UNCHANGED in a child pytest (plugin
tests/hostsim_plugin.py swaps the library path of the Python mirror).  What passing means: the host side builds the right tables,
sizes and grows the directory correctly, takes the right round decisions and reports the right errors -- for every scenario the GPU
suite has.  What it does NOT mean: anything about the CUDA kernels; those are proven on the GPU box against the oracle.  This is test
infrastructure, kept under tests/: the product has no CPU path (tests/test_abi.py::test_no_gpu_means_loud_failure_not_fallback) and
its loader has no switch for this library.
"""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rio_rs_b200", "csrc")
SIM = os.path.join(ROOT, "tests", "cpp", "hostsim")
TCPP = os.path.join(ROOT, "tests", "cpp")
OUT = os.path.join(ROOT, "tests", "_build")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
PRODUCT = [os.path.join(CSRC, f) for f in ("engine.cu", "resolver.cu", "durable.cu")]
DOUBLES = [os.path.join(SIM, "launchers.cpp")]

pytestmark = pytest.mark.skipif(GXX is None, reason="no host C++ compiler")


@pytest.fixture(scope="module")
def hostsim_so():
    os.makedirs(OUT, exist_ok=True)
    so = os.path.join(OUT, "librio_cuda_hostsim.so")
    deps = PRODUCT + DOUBLES + [os.path.join(SIM, "cuda_runtime.h")] + [os.path.join(CSRC, h) for h in ("kernels.cuh", "spec.cuh", "trie_table.hpp")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call([GXX, "-std=c++17", "-O2", "-g", "-fPIC", "-shared", "-Wall", "-Wextra", "-Werror", "-I" + SIM, "-x", "c++"] + PRODUCT + DOUBLES +
                              ["-o", so, "-ldl", "-lpthread"])
    return so


def test_the_doubles_cover_every_launcher_and_nothing_in_the_product_knows_them():
    decl = set(re.findall(r"\b((?:launch_[a-z0-9_]+)|assign_wave_objects|trie_wave_objects|trie_upload_level_constants|affinity_umma_[a-z_]+)\s*\(",
                          open(os.path.join(CSRC, "kernels.cuh")).read()))
    have = set(re.findall(r"^(?:void|bool|uint32_t|uint64_t)\s+([a-z0-9_]+)\s*\(", open(DOUBLES[0]).read(), flags=re.M))
    assert decl <= have, decl - have
    for dirpath, _, files in os.walk(os.path.join(ROOT, "rio_rs_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                assert "hostsim" not in open(os.path.join(dirpath, f), errors="replace").read(), f
    for f in ("bench.py", "__graft_entry__.py", os.path.join("include", "rio_cuda.h"), os.path.join("include", "rio_cuda_dev.h")):
        assert "hostsim" not in open(os.path.join(ROOT, f)).read(), f     # neither the bench nor the driver's entry points can reach it


def test_gpu_test_bodies_pass_on_the_engine_host_logic(hostsim_so):
    """tests/test_gpu_parity.py, test_gpu_hrw2.py, test_gpu_integration.py and test_gpu_affinity.py, unchanged, against the host-sim
    library: every scenario but the 10 M x 1024 flat grid (10^10 pair hashes: minutes on a CPU) -- including all 10 M objects under
    HRW2.  The affinity double has no tensor cores, so there every affinity case takes the CUDA-core branch and must equal the fp32
    fmaf restatement of the oracle exactly; compaction, the capacity fallback, chunking and the counters are the engine's own."""
    env = dict(os.environ)
    env["RIO_HOSTSIM_LIBRARY"] = hostsim_so
    env["PYTHONPATH"] = os.path.join(ROOT, "tests") + os.pathsep + env.get("PYTHONPATH", "")
    mods = [os.path.join(ROOT, "tests", m) for m in ("test_gpu_parity.py", "test_gpu_hrw2.py", "test_gpu_integration.py", "test_gpu_affinity.py")]
    cmd = [sys.executable, "-m", "pytest"] + mods + ["-m", "gpu", "-p", "hostsim_plugin", "-q", "-x", "-p", "no:cacheprovider", "-k", "not test_full_size_10m_x_1024_properties"]
    try:
        import pytest_timeout  # noqa: F401  (a test blocked inside a C call is only stopped by the thread method)

        cmd += ["--timeout=180", "--timeout-method=thread"]
    except ImportError:
        pass
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    m = re.search(r"(\d+) passed", r.stdout)
    assert m and int(m.group(1)) >= 95 and "failed" not in r.stdout, tail


@pytest.mark.parametrize("harness,args", [("backend_conformance.cpp", []), ("durable_conformance.cpp", ["TMP"]), ("resolver_stress.cpp", ["8", "60"])])
def test_cpp_harnesses_on_the_engine_host_logic_under_sanitizers(tmp_path, harness, args):
    """The C++ conformance harnesses of the GPU box (trait mirror, durable write-through, resolver queue) linked with engine.cu itself
    + the doubles into ONE executable under AddressSanitizer + UBSan: the engine's host code runs its real paths (string-level calls,
    directory growth, place_batch, recover) with every heap access checked."""
    exe = str(tmp_path / "harness")
    cmd = [GXX, "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-I" + SIM, "-I" + ROOT, "-x", "c++"] + PRODUCT + DOUBLES + \
          [os.path.join(TCPP, harness), "-o", exe, "-ldl", "-lpthread"]
    try:
        subprocess.check_call(cmd)
    except subprocess.CalledProcessError:
        pytest.skip("this toolchain has no ASan/UBSan runtime")
    r = subprocess.run([exe] + [str(tmp_path) if a == "TMP" else a for a in args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "all passed" in r.stdout, r.stdout[-1500:] + r.stderr[-3000:]
    assert "AddressSanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-3000:]


def test_abi_fuzz_on_the_engine_host_logic_under_sanitizers(tmp_path):
    """tests/cpp/abi_fuzz.cpp: random sequences of C-ABI calls with ordinary, boundary and wrong arguments (NULL buffers, indices out of
    range, sets used in the wrong order, tiny output buffers, membership changes in the middle of bounded calls) against engine.cu under
    ASan + UBSan; every call must answer with a status, never with a crash, and the directory must keep answering like
    LocalObjectPlacement.  (This harness found the heap overflow in the masked-table build that
    test_membership_touched_between_the_two_halves_of_a_bounded_call now pins.)"""
    exe = str(tmp_path / "abi_fuzz")
    cmd = [GXX, "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-I" + SIM, "-I" + ROOT, "-x", "c++"] + PRODUCT + DOUBLES + \
          [os.path.join(TCPP, "abi_fuzz.cpp"), "-o", exe, "-ldl", "-lpthread"]
    try:
        subprocess.check_call(cmd)
    except subprocess.CalledProcessError:
        pytest.skip("this toolchain has no ASan/UBSan runtime")
    for seed in (1, 6, 24, 31):
        r = subprocess.run([exe, str(seed), "2500"], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "abi fuzz: all passed" in r.stdout, "seed %d\n" % seed + r.stdout[-1500:] + r.stderr[-4000:]


def test_one_handle_shared_by_many_threads_under_tsan(tmp_path):
    """tests/cpp/abi_threads.cpp: 8 threads x random C-ABI calls on ONE handle (string calls, batched calls, membership flapping, bounded
    calls on private sets, a shared resolver) against engine.cu under ThreadSanitizer: "re-entrant and thread-safe per handle"."""
    exe = str(tmp_path / "abi_threads")
    cmd = [GXX, "-std=c++17", "-O1", "-g", "-fsanitize=thread", "-I" + SIM, "-I" + ROOT, "-x", "c++"] + PRODUCT + DOUBLES + [os.path.join(TCPP, "abi_threads.cpp"), "-o", exe, "-ldl", "-lpthread"]
    try:
        subprocess.check_call(cmd)
    except subprocess.CalledProcessError:
        pytest.skip("this toolchain has no TSan runtime")
    env = dict(os.environ)
    env["TSAN_OPTIONS"] = "halt_on_error=1"
    r = subprocess.run([exe, "8", "300"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and "abi threads: all passed" in r.stdout and "ThreadSanitizer" not in r.stderr, r.stdout[-1500:] + r.stderr[-4000:]


def test_durable_provider_fuzz_with_restarts(tmp_path):
    """tests/cpp/durable_fuzz.cpp: random update / remove / clean_server / batched update / written-through place_batch / member
    deaths / crash-and-recover sequences on the native durable provider (durable.cu over engine.cu, real libsqlite3) against a shadow
    map with the reference's semantics; after every restart the recovered directory must hold exactly the shadow's rows."""
    import ctypes

    try:
        ctypes.CDLL("libsqlite3.so.0")
    except OSError:
        pytest.skip("libsqlite3 is not installed")
    exe = str(tmp_path / "durable_fuzz")
    cmd = [GXX, "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-I" + SIM, "-I" + ROOT, "-x", "c++"] + PRODUCT + DOUBLES + \
          [os.path.join(TCPP, "durable_fuzz.cpp"), "-o", exe, "-ldl", "-lpthread"]
    try:
        subprocess.check_call(cmd)
    except subprocess.CalledProcessError:
        pytest.skip("this toolchain has no ASan/UBSan runtime")
    for seed in (1, 2, 3):
        r = subprocess.run([exe, str(tmp_path), str(seed), "1200"], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "durable fuzz: all passed" in r.stdout, "seed %d\n" % seed + r.stdout[-1500:] + r.stderr[-4000:]


@pytest.mark.parametrize("world,solver", [(2, "hrw2"), (4, "hrw"), (8, "hrw2"), (8, "hrw")])
def test_multi_rank_host_path_in_one_process(hostsim_so, world, solver):
    """tests/hostsim_multirank.py: `world` ranks of the engine as threads of one process, windows attached through the same
    rio_cuda_comm_ipc_* calls a multi-process run uses: bounded calls whose spill rounds fire, three calls in flight, leave / join,
    global counters -- every rank's shard equal to the oracle on the GLOBAL key set, up to the 8 ranks no GPU box was free for."""
    env = dict(os.environ)
    env["RIO_HOSTSIM_LIBRARY"] = hostsim_so
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "hostsim_multirank.py"), str(world), solver], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0 and "multirank ok" in r.stdout, r.stdout[-1500:] + r.stderr[-3000:]
