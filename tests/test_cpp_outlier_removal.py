"""filter::OutlierRemoval through the C++ facade (include/sycl_points/algorithms/filter/outlier_removal_filter.hpp):
it compiles with plain g++ against libspx.so with no CUDA / SYCL / Eigen include, and on a GPU
tests/cpp/test_outlier_removal.cpp runs the square-plus-far-point case and the radius cases."""
import os
import subprocess

import pytest

from test_cpp_facade import ROOT, compile_cpp

HEADERS = ("algorithms/filter/outlier_removal_filter.hpp", "algorithms/filter/gather_attributes.hpp")


@pytest.fixture(scope="module")
def outlier_exe():
    return compile_cpp("tests/cpp/test_outlier_removal.cpp", "test_outlier_removal")


def test_outlier_facade_compiles_without_cuda_sycl_or_eigen(outlier_exe):
    assert os.access(outlier_exe, os.X_OK)
    for h in HEADERS:
        text = open(os.path.join(ROOT, "include", "sycl_points", h)).read()
        for banned in ("cuda_runtime", "<cuda", "<sycl/", "<CL/", "<Eigen/"):
            assert banned not in text, (h, banned)
    # the header states that its interface is libspx's own
    assert "not a verified drop-in" in open(os.path.join(ROOT, "include", "sycl_points", HEADERS[0])).read()


@pytest.mark.gpu
def test_outlier_facade_on_gpu(outlier_exe):
    r = subprocess.run([outlier_exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])
    assert " 0 failed" in r.stdout
