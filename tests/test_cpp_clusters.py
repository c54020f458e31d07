"""segmentation::EuclideanClustering through the C++ facade
(include/sycl_points/algorithms/segmentation/euclidean_clustering.hpp): it compiles with plain g++ against libspx.so
with no CUDA / SYCL / Eigen include, and on a GPU tests/cpp/test_clusters.cpp runs a chain and a bridged comb."""
import os
import subprocess

import pytest

from test_cpp_facade import ROOT, compile_cpp

HEADER = "algorithms/segmentation/euclidean_clustering.hpp"


@pytest.fixture(scope="module")
def clusters_exe():
    return compile_cpp("tests/cpp/test_clusters.cpp", "test_clusters")


def test_clustering_facade_compiles_without_cuda_sycl_or_eigen(clusters_exe):
    assert os.access(clusters_exe, os.X_OK)
    text = open(os.path.join(ROOT, "include", "sycl_points", HEADER)).read()
    for banned in ("cuda_runtime", "<cuda", "<sycl/", "<CL/", "<Eigen/"):
        assert banned not in text, banned
    assert "not a verified drop-in" in text  # the header states that its interface is libspx's own


@pytest.mark.gpu
def test_clustering_facade_on_gpu(clusters_exe):
    r = subprocess.run([clusters_exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-2000:])
    assert " 0 failed" in r.stdout
