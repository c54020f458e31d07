"""segmentation::PlaneSegmentation through the C++ facade
(include/sycl_points/algorithms/segmentation/plane_segmentation.hpp): it compiles with plain g++ against libspx.so with
no CUDA / SYCL / Eigen include, and on a GPU tests/cpp/test_plane.cpp runs a plane with clutter and non-finite rows."""
import os
import subprocess

import pytest

from test_cpp_facade import ROOT, compile_cpp

HEADER = "algorithms/segmentation/plane_segmentation.hpp"


@pytest.fixture(scope="module")
def plane_exe():
    return compile_cpp("tests/cpp/test_plane.cpp", "test_plane")


def test_plane_facade_compiles_without_cuda_sycl_or_eigen(plane_exe):
    assert os.access(plane_exe, os.X_OK)
    text = open(os.path.join(ROOT, "include", "sycl_points", HEADER)).read()
    for banned in ("cuda_runtime", "<cuda", "<sycl/", "<CL/", "<Eigen/"):
        assert banned not in text, banned
    assert "not a verified drop-in" in text  # the header states that its interface is libspx's own


@pytest.mark.gpu
def test_plane_facade_on_gpu(plane_exe):
    r = subprocess.run([plane_exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])
    assert " 0 failed" in r.stdout
