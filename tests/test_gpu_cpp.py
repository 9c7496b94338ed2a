"""The C++ host mirror (include/caf_b200.hpp) restating caf_rust/tests/test.rs, compiled with g++ against the in-tree
libcaf_b200.so and executed on the GPU."""
import os
import shutil
import subprocess

import pytest

from caf_cookoff_b200 import _lib
from conftest import DATA, ROOT

@pytest.fixture(scope="module")
def out_dir(tmp_path_factory):
    """Where the native programs are built: outside the repository tree, which may be read-only."""
    return tmp_path_factory.mktemp("native")


def _build(out_dir):
    gxx = shutil.which("g++")
    assert gxx, "g++ is required for the C++ mirror test"
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(out_dir / "test_rs")
    cmd = [gxx, "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_rs.cpp"),
           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"]
    subprocess.check_call(cmd)
    return exe


def test_cpp_mirror_compiles_without_gpu(out_dir):
    """CPU check: the header-only mirror and the C ABI header compile and link against the built library."""
    assert os.path.exists(_build(out_dir))


@pytest.mark.gpu
def test_cpp_restatement_of_test_rs(out_dir):
    res = subprocess.run([_build(out_dir), DATA], capture_output=True, text=True, timeout=300)
    print(res.stdout[-3000:], res.stderr[-2000:])
    assert res.returncode == 0
    assert "all tests passed" in res.stdout
    assert "Frequency offset: 69.0Hz" in res.stdout and "Time offset: 202 samples (4.208ms)" in res.stdout


def _build_cli(out_dir):
    gxx = shutil.which("g++")
    assert gxx, "g++ is required for the CLI"
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(out_dir / "caf_cli")
    subprocess.check_call([gxx, "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "caf_cli.cpp"),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    return exe


def test_cli_builds_and_parses_arguments(out_dir):
    """CPU: tools/caf_cli (main.rs:10-32 with the arguments its TODO asks for) builds, documents itself and rejects
    bad command lines without touching a GPU."""
    CLI = _build_cli(out_dir)
    assert "usage: caf_cli NEEDLE.c64 HAYSTACK.c64" in subprocess.run([CLI, "--help"], capture_output=True, text=True).stdout
    assert subprocess.run([CLI, "only_one.c64"], capture_output=True, text=True).returncode == 2
    assert subprocess.run([CLI, "a", "b", "--bogus"], capture_output=True, text=True).returncode == 2
    assert subprocess.run([CLI, "/nonexistent_a", "/nonexistent_b"], capture_output=True, text=True).returncode == 1


@pytest.mark.gpu
def test_cli_prints_what_main_rs_prints(tmp_path, out_dir):
    import numpy as np
    CLI = _build_cli(out_dir)
    a, b = os.path.join(DATA, "chirp_0_raw.c64"), os.path.join(DATA, "chirp_0_T+202samp_F+69.25Hz.c64")
    res = subprocess.run([CLI, a, b], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    assert res.stdout == "Frequency offset: 69.0Hz\nTime offset: 202 samples (4.208ms)\n"            # main.rs:29-31
    # the same report with both files loaded through pinned memory straight onto the GPU (read_file_c64_dev, caf_peak_dev)
    res = subprocess.run([CLI, a, b, "--device-load"], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    assert res.stdout == "Frequency offset: 69.0Hz\nTime offset: 202 samples (4.208ms)\n"
    assert subprocess.run([CLI, "/nonexistent_a", b, "--device-load"], capture_output=True, text=True, timeout=120).returncode == 1
    # a finer grid, as caf_rust/tests/test.rs uses, and the surface dumped the way caf.go:14-29 dumps it
    dump = str(tmp_path / "surf.bin")
    res = subprocess.run([CLI, a, b, "--fstep", "0.25", "--dump", dump], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and "Frequency offset: 69.2Hz" in res.stdout and "Time offset: 202 samples" in res.stdout
    surf = np.fromfile(dump, dtype="<f8").reshape(800, 8192)
    assert np.unravel_index(surf.argmax(), surf.shape) == (677, 202)
    # the sibling programs' reports on their own pair (main.go:13-35, caf.py:126-146)
    a4, b4 = os.path.join(DATA, "chirp_4_raw.c64"), os.path.join(DATA, "chirp_4_T+70samp_F+82.89Hz.c64")
    res = subprocess.run([CLI, a4, b4, "--layout", "go"], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and res.stdout.startswith("caf result: 70 samples 83 hz")
    res = subprocess.run([CLI, a4, b4, "--layout", "python"], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and res.stdout.startswith("amb_surf (400, 4096) float64 -> 70 83")


def test_native_programs_fail_loudly_without_a_gpu(out_dir):
    """CPU box only: the CLI and the C++ restatement of test.rs stop with the library's ENODEVICE message and a
    non-zero exit code — neither has (or falls back to) a CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the failure path is exercised on the CPU-only box")
    BIN, CLI = _build(out_dir), _build_cli(out_dir)
    a, b = os.path.join(DATA, "chirp_0_raw.c64"), os.path.join(DATA, "chirp_0_T+202samp_F+69.25Hz.c64")
    res = subprocess.run([CLI, a, b], capture_output=True, text=True, timeout=120)
    assert res.returncode == 1 and res.stdout == ""
    assert "status -5" in res.stderr and "no CPU fallback" in res.stderr
    res = subprocess.run([BIN, DATA], capture_output=True, text=True, timeout=120)
    assert res.returncode != 0 and "all tests passed" not in res.stdout
    assert "no CPU fallback" in res.stdout + res.stderr
