"""feature::FPFHEstimation, registration::match_features and registration::RANSACRegistration through the C++ facade
(include/sycl_points/algorithms/feature/fpfh.hpp, include/sycl_points/algorithms/registration/ransac_registration.hpp):
they compile with plain g++ against libspx.so with no CUDA / SYCL / Eigen include, and on a GPU
tests/cpp/test_global_registration.cpp runs descriptors, matching and RANSAC."""
import os
import subprocess

import pytest

from test_cpp_facade import ROOT, compile_cpp

HEADERS = ("algorithms/feature/fpfh.hpp", "algorithms/registration/ransac_registration.hpp")


@pytest.fixture(scope="module")
def global_exe():
    return compile_cpp("tests/cpp/test_global_registration.cpp", "test_global_registration")


def test_global_facade_compiles_without_cuda_sycl_or_eigen(global_exe):
    assert os.access(global_exe, os.X_OK)
    for h in HEADERS:
        text = open(os.path.join(ROOT, "include", "sycl_points", h)).read()
        for banned in ("cuda_runtime", "<cuda", "<sycl/", "<CL/", "<Eigen/"):
            assert banned not in text, (h, banned)
        assert "not a verified drop-in" in text, h  # each header states that its interface is libspx's own


@pytest.mark.gpu
def test_global_facade_on_gpu(global_exe):
    r = subprocess.run([global_exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])
    assert " 0 failed" in r.stdout
