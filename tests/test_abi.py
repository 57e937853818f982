"""CPU tests of the drop-in boundary: the product library loads without a GPU, exports every
symbol that include/*.h declares, and fails loudly (no CPU fallback) when no device exists."""
import ctypes as C
import os
import re
import subprocess

import cases
from edlib_b200._ffi import REPO, AlignConfig, AlignResult, EqualityPair, product_path


def declared_symbols():
    names = set()
    for h in ("edlib.h", "edlib_b200.h"):
        src = open(os.path.join(REPO, "include", h)).read()
        names.update(re.findall(r"EDLIB_API[^;(]*?\b(edlib\w+)\s*\(", src))
    return names


def test_library_exports_every_declared_symbol():
    subprocess.run(["make", "-s", "-C", os.path.join(REPO, "edlib_b200", "csrc")], check=True)
    lib = C.CDLL(product_path())
    names = declared_symbols()
    assert {"edlibAlign", "edlibAlignBatch", "edlibNewAlignConfig", "edlibDefaultAlignConfig",
            "edlibFreeAlignResult", "edlibAlignmentToCigar"} <= names
    for n in names:
        assert hasattr(lib, n), n


def test_struct_layout_matches_reference_abi(tmp_path):
    # sizes measured on the reference build (SURVEY.md section 2.1)
    assert C.sizeof(EqualityPair) == 2 and C.sizeof(AlignConfig) == 32 and C.sizeof(AlignResult) == 48
    code = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "edlib.h"
    int main(void) {
        printf("%zu %zu %zu %zu %zu %zu %d %d %d %d\n", sizeof(EdlibEqualityPair), sizeof(EdlibAlignConfig),
               sizeof(EdlibAlignResult), offsetof(EdlibAlignResult, endLocations), offsetof(EdlibAlignResult, alignment),
               offsetof(EdlibAlignConfig, additionalEqualities), EDLIB_MODE_HW, EDLIB_TASK_PATH, EDLIB_CIGAR_EXTENDED,
               EDLIB_EDOP_MISMATCH);
        return 0;
    }'''
    exe = str(tmp_path / "edlib_abi_probe")
    subprocess.run(["gcc", "-x", "c", "-std=c99", "-I", os.path.join(REPO, "include"), "-o", exe, "-"],
                   input=code, text=True, check=True)
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()
    assert out == ["2", "32", "48", "8", "32", "16", "2", "2", "1", "3"]


def test_fails_loudly_without_gpu_or_runs_on_gpu():
    """No device => EDLIB_STATUS_ERROR (never a silent CPU answer)."""
    import torch
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "from edlib_b200._ffi import EdlibLib, product_path\n"
        "lib = EdlibLib(product_path(), has_batch=True)\n"
        "print(lib.lib.edlibB200Available(), lib.align(b'ACGT', b'ACCT')['status'])\n"
    ) % REPO
    out = subprocess.run(["python", "-c", code], capture_output=True, text=True, check=True).stdout.split()
    if torch.cuda.is_available():
        assert out == ["1", "0"]
    else:
        assert out == ["0", "1"]


def test_host_only_helpers():
    lib = C.CDLL(product_path())
    lib.edlibAlignmentToCigar.restype = C.c_void_p
    lib.edlibAlignmentToCigar.argtypes = [C.POINTER(C.c_ubyte), C.c_int, C.c_int]
    ops = bytes([0, 0, 1, 1, 1, 2, 1, 1, 3, 0, 0])  # reference test/runTests.cpp:506-533
    buf = (C.c_ubyte * len(ops))(*ops)
    assert C.string_at(lib.edlibAlignmentToCigar(buf, len(ops), 1)) == b"2=3I1D2I1X2="
    assert C.string_at(lib.edlibAlignmentToCigar(buf, len(ops), 0)) == b"2M3I1D2I3M"
    assert lib.edlibAlignmentToCigar(buf, len(ops), 7) is None
    lib.edlibDefaultAlignConfig.restype = AlignConfig
    cfg = lib.edlibDefaultAlignConfig()
    assert (cfg.k, cfg.mode, cfg.task, cfg.additionalEqualitiesLength) == (-1, 0, 0, 0)


def test_cigar_strings_match_the_reference_on_random_scripts():
    """edlibAlignmentToCigar (one-pass, word-at-a-time run detection) against the reference build's strings (stored as
    fingerprints): random edit scripts of every length around the word boundaries, both formats, long runs, bad
    operation codes."""
    from edlib_b200._ffi import EdlibLib
    emul = os.path.join(REPO, "tests", "emul", "libedlib_emul.so")
    subprocess.run(["make", "-s", "-C", os.path.join(REPO, "tests", "emul")], check=True)
    # pure host formatting: the product library answers it without a GPU, so both builds of eb_capi.cpp are checked
    for mine in (EdlibLib(emul, has_batch=True), EdlibLib(product_path(), has_batch=True)):
        check_cigar_strings(mine)


def check_cigar_strings(mine):
    from helpers import digest, golden_digests
    expected = golden_digests()["cigar"]
    n = 0
    for case, ((ops, bad), exp) in enumerate(zip(cases.cigar_scripts(12, 3000), expected)):
        for fmt in (0, 1):
            if bad:
                # The reference indexes its 4-entry table with the bad code before it looks at it (edlib.cpp:321) and only
                # checks codes that open a run (edlib.cpp:334), so its answer there is undefined; the header's contract is
                # "NULL on error", which is what this library returns for a bad code at any position.
                assert mine.cigar(ops, fmt) is None, (case, len(ops), fmt, ops[:40])
        if not bad:
            got = [mine.cigar(ops, fmt) for fmt in (0, 1)]
            assert digest(got) == exp, (case, len(ops), ops[:40], [g[:80] for g in got])
        n += 1
    assert n == len(expected) == 3000
