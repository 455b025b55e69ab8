"""The Hadamard-product accumulation prover of the C++ host mirror (ASForHadamardProducts::prove / verify / decide in accumulation_b200/host/ark_mirror.hpp)
driven by a compiled harness (tests/host/hp_prove_tests.cpp): CPU suite: it compiles against include/accmsm.h and refuses to run
without a GPU; GPU suite: every scenario passes on a single-device and on a 2-device group ctx."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host", "hp_prove_tests.cpp")
EXE = os.path.join(ROOT, "tests", "host", "hp_prove_tests")


def build_harness():
    from accumulation_b200 import build
    from oracle import cref
    build.build(); cref.build()
    deps = [SRC, os.path.join(ROOT, "accumulation_b200", "host", "ark_mirror.hpp"), os.path.join(ROOT, "include", "accmsm.h"),
            os.path.join(ROOT, "oracle", "oracle.h")]
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        lib_dirs = [os.path.join(ROOT, "accumulation_b200"), os.path.join(ROOT, "oracle")]
        cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-o", EXE, SRC, f"-L{lib_dirs[0]}", f"-L{lib_dirs[1]}", "-l:libaccmsm.so",
               "-l:liboracle.so", f"-Wl,-rpath,{lib_dirs[0]}", f"-Wl,-rpath,{lib_dirs[1]}", "-fopenmp", "-pthread"]
        subprocess.check_call(cmd)
    return EXE


def test_hp_prove_harness_builds_and_refuses_without_gpu():
    exe = build_harness()
    p = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert p.returncode == 3 and "NO_GPU" in p.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("devices", ["", "0,0"] + (["0,1"] if os.environ.get("ACCMSM_HAVE_2_GPUS") else []))
def test_cpp_hp_prove_scenarios(devices):
    exe = build_harness()
    p = subprocess.run([exe], capture_output=True, text=True, timeout=600, env=dict(os.environ, ACCMSM_TEST_DEVICES=devices))
    print(p.stdout[-4000:])
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    assert "FAIL" not in p.stdout and p.stdout.count("PASS") == 24
