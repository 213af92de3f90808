"""The reference's OWN test suite (/root/reference/tests/*.cpp|*.cu, 48 gtest cases), compiled
UNCHANGED against this repository's headers and libspmv_b200.so (tests/ref_suite/Makefile; a
stand-in gtest header replaces the GoogleTest the reference downloads at configure time,
/root/reference/CMakeLists.txt:32-50).  This is the C++ drop-in proof SURVEY 4 / 7 step 3 asks for:
an object file written against include/spmv/*.h links against the new library and behaves --
CudaBuffer<T>, CUDA_CHECK, benchmark_from_json and the by-value C++ structs included.

CPU test: build the binary (when the reference tree is present) and run the 22 cases that never touch a
device.  GPU test: run all 48.  The reference's test sources are not part of this repository, so both tests
skip where the binary could not be built.  Expected deviation, documented in SURVEY F10: SpMVUnitTest.EmptyMatrix
expects SUCCESS from spmv_csr(csr_create(0,0,0), ..., vec_size = 1) although the reference itself returns
INVALID_DIMENSION (0 != 1, src/spmv_kernels.cu:224-226) -- it fails on the reference too, and a faithful
drop-in must fail it the same way."""
import os
import re
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SUITE = os.path.join(HERE, "ref_suite")
BINARY = os.path.join(SUITE, "_build", "spmv_tests")
CONTROL = os.path.join(SUITE, "_build", "spmv_tests_ref")  # same test objects + the unmodified reference library

# cases that never reach the CUDA runtime (SURVEY 4)
CPU_ONLY = [
    "CommonTest.ErrorStringConversion", "CudaBufferTest.DefaultConstruction", "CudaBufferTest.ZeroSizeConstruction",
    "CSRPropertyTest.DenseToSparseRoundTrip", "CSRPropertyTest.ElementLookupCorrectness",
    "CSRPropertyTest.SerializationRoundTrip", "CSRUnitTest.EmptyMatrix", "CSRUnitTest.AllZeroMatrix",
    "CSRUnitTest.SingleElementMatrix", "ELLPropertyTest.DenseToSparseRoundTrip", "ELLPropertyTest.PaddingCorrectness",
    "ELLPropertyTest.ColumnMajorLayout", "ELLPropertyTest.SerializationRoundTrip", "ELLUnitTest.FromCSR",
    "KernelSelectorPropertyTest.SelectorValidity", "KernelSelectorUnitTest.ShortRowsSelectScalar",
    "KernelSelectorUnitTest.UniformRowsSelectVector", "KernelSelectorUnitTest.SkewedRowsSelectMergePath",
    "KernelSelectorUnitTest.LargeVectorUsesTexture", "SpMVUnitTest.KernelSelector", "BandwidthUnitTest.ZeroElapsedTime",
    "BenchmarkUnitTest.JSONFormat",
]
# Cases that fail on the REFERENCE ITSELF (checked on the GPU against the control binary below):
#   SpMVUnitTest.EmptyMatrix            SURVEY F10 (vec_size 1 != num_cols 0 -> INVALID_DIMENSION)
#   BenchmarkPropertyTest.JSONRoundTrip benchmark_to_json prints 6 fixed decimals (src/benchmark.cu:187-202);
#                                       kernel times of 10..100-row matrices are ~0.005 ms, so only 3-4
#                                       significant digits survive and EXPECT_FLOAT_EQ (4 ULP) cannot hold
EXPECTED_DEVIATIONS = {"SpMVUnitTest.EmptyMatrix", "BenchmarkPropertyTest.JSONRoundTrip"}
TOTAL_CASES = 48


def build():
    p = subprocess.run(["make", "-C", SUITE, "-j", "8"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0, p.stdout[-4000:]


def run(filter_=None, timeout=900, binary=BINARY):
    cmd = [binary] + ([f"--gtest_filter={filter_}"] if filter_ else [])
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout, cwd="/tmp")
    ok = re.findall(r"^\[       OK \] (\S+)", p.stdout, re.M)
    failed = sorted(set(re.findall(r"^\[  FAILED  \] (\S+)$", p.stdout, re.M)))
    return p, ok, failed


def test_reference_tests_compile_and_link_unchanged_cpu_cases_pass(sp):
    if os.path.exists("/root/reference/tests/test_spmv.cu"):
        build()
    if not os.path.exists(BINARY):
        pytest.skip("tests/ref_suite/_build/spmv_tests not built (reference tree absent)")
    listing = subprocess.run([BINARY, "--gtest_list_tests"], stdout=subprocess.PIPE, text=True, cwd="/tmp").stdout.split()
    assert len(listing) == TOTAL_CASES and set(CPU_ONLY) <= set(listing)
    p, ok, failed = run(":".join(CPU_ONLY))
    assert p.returncode == 0 and not failed, p.stdout[-3000:]
    assert sorted(ok) == sorted(CPU_ONLY)
    # the binary resolves the API from OUR library, not from a reference build
    ldd = subprocess.run(["ldd", BINARY], stdout=subprocess.PIPE, text=True).stdout
    assert "libspmv_b200.so" in ldd and "libspmv_ref" not in ldd


@pytest.mark.gpu
def test_reference_suite_on_the_gpu(sp, cuda):
    if not os.path.exists(BINARY):
        pytest.skip("tests/ref_suite/_build/spmv_tests not built (reference tree absent)")
    p, ok, failed = run()
    print(p.stdout[-2500:])
    assert set(failed) <= EXPECTED_DEVIATIONS, p.stdout[-6000:]
    assert len(ok) + len(failed) == TOTAL_CASES
    assert len(ok) >= TOTAL_CASES - len(EXPECTED_DEVIATIONS)
    if "SpMVUnitTest.EmptyMatrix" in failed:  # the failure is the reference's own: error_code -1, not a crash
        assert re.search(r"actual: -1 vs 0", p.stdout), p.stdout[-3000:]
    # control arm: the same test objects linked against the unmodified reference library.  Whatever fails
    # here must fail there too -- a drop-in may not fail a case the reference passes.
    if os.path.exists(CONTROL):
        pc, ok_c, failed_c = run(binary=CONTROL)
        print("reference control arm failed:", failed_c)
        assert len(ok_c) + len(failed_c) == TOTAL_CASES
        assert set(failed) <= set(failed_c), (failed, failed_c)
