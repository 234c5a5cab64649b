"""Builds the C++ conformance harness against the C++ mirror of the trait and runs it (GPU), and checks on CPU that it
compiles and links against librio_cuda.so."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """Compiles tests/cpp/<name>.cpp against librio_cuda.so into a temporary directory (the checkout may be read-only), once per
    module, and returns the executable's path."""
    from rio_rs_b200 import build

    build.build()
    out = tmp_path_factory.mktemp("cpp_harness")
    libdir = os.path.join(ROOT, "rio_rs_b200")
    built = {}

    def get(name="backend_conformance"):
        if name not in built:
            exe = str(out / name)
            src = os.path.join(ROOT, "tests", "cpp", name + ".cpp")
            subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-o", exe, src, "-L" + libdir, "-lrio_cuda", "-Wl,-rpath," + libdir])
            built[name] = exe
        return built[name]

    return get


def test_cpp_mirror_compiles_and_links(harness):
    assert os.path.exists(harness())


@pytest.mark.gpu
def test_cpp_backend_conformance_on_gpu(harness):
    r = subprocess.run([harness()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all passed" in r.stdout


def test_cpp_durable_harness_compiles_and_links(harness):
    assert os.path.exists(harness("durable_conformance"))


@pytest.mark.gpu
def test_cpp_durable_conformance_on_gpu(harness, tmp_path):
    """The reference's SqliteObjectPlacement tests + restart recovery + the written-through place_batch, through the C ABI
    (rio_cuda_durable_*, libsqlite3.so.0 dlopen'ed): SURVEY 8(f) row 3 below the language bindings."""
    r = subprocess.run([harness("durable_conformance"), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "durable: all passed" in r.stdout
