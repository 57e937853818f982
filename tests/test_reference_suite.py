"""The reference's OWN test program (test/runTests.cpp, unmodified; compiled from where it lies by
`make -C oracle reftests` into the git-ignored oracle/_ref/) run against this engine: against the
CPU emulation of the kernels here, against the product library on the GPU box."""
import os
import subprocess

import pytest

from edlib_b200._ffi import REPO

REFBIN = os.path.join(REPO, "oracle", "_ref")


def _build_if_possible():
    if os.path.isdir("/root/reference"):
        subprocess.run(["make", "-s", "-C", os.path.join(REPO, "edlib_b200", "csrc")], check=True)
        subprocess.run(["make", "-s", "-C", os.path.join(REPO, "tests", "emul")], check=True)
        subprocess.run(["make", "-s", "-C", os.path.join(REPO, "oracle"), "reftests"], check=True)


def test_reference_runtests_on_emulated_kernels():
    _build_if_possible()
    exe = os.path.join(REFBIN, "runTests_emul")
    if not os.path.exists(exe):
        pytest.skip("reference test binary not built (no /root/reference here)")
    out = subprocess.run([exe, "25"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:]
    assert out.stdout.count("25/25") == 6 and "All specific tests passed!" in out.stdout


@pytest.mark.gpu
def test_reference_runtests_on_gpu():
    exe = os.path.join(REFBIN, "runTests_b200")
    if not os.path.exists(exe):
        pytest.skip("reference test binary did not travel")
    out = subprocess.run([exe, "40"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:]
    assert out.stdout.count("40/40") == 6 and "All specific tests passed!" in out.stdout


HELLO = r'''
#include <stdio.h>
#include "edlib.h"

int main(void) {
    EdlibAlignResult r = edlibAlign("hello", 5, "world!", 6, edlibDefaultAlignConfig());
    printf("status %d, edit distance %d\n", r.status, r.editDistance);
    edlibFreeAlignResult(r);
    return r.status;
}
'''


@pytest.mark.gpu
def test_reference_hello_world_on_gpu(tmp_path):
    """The reference's hello-world example in C: a plain C caller of include/edlib.h, linked against the product library."""
    exe = str(tmp_path / "hello")
    lib = os.path.join(REPO, "edlib_b200", "lib")
    subprocess.run(["gcc", "-x", "c", "-std=c99", "-I", os.path.join(REPO, "include"), "-o", exe, "-", "-L" + lib, "-ledlib_b200",
                    "-Wl,-rpath," + lib], input=HELLO, text=True, check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout == "status 0, edit distance 5\n"
