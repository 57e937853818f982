"""Generates tests/golden/ref_digests.json: fingerprints (helpers.digest) of what the UNMODIFIED reference computes on the
seeded inputs of the tests that compare with it -- every result field of the oracle-pinning cases, the CIGAR strings of
random edit scripts, and the normalised output of the reference's edlib-aligner for every option set of
tests/test_aligner_cli.py.  Needs the reference build (`make -C oracle ref reftests` with the reference sources):

    python tests/golden/make_ref_digests.py
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import cases  # noqa: E402
import test_aligner_cli  # noqa: E402
from helpers import digest, ref  # noqa: E402
from edlib_b200._ffi import REPO  # noqa: E402


def main():
    R = ref()
    out = {"source": "reference edlib v1.2.6 (commit 0ddc23e) built by oracle/Makefile"}
    out["oracle_random"] = [digest(R.align(c["q"], c["t"], c["k"], c["mode"], c["task"], c["eqs"]))
                            for c in cases.single_pair_cases(101, 4000)]
    out["oracle_hirschberg"] = [digest(R.align(c["q"], c["t"], c["k"], c["mode"], c["task"])) for c in cases.hirschberg_cases(7, 40)]
    # a bad operation code has no defined answer in the reference (see test_abi.py)
    out["cigar"] = [None if bad else digest([R.cigar(ops, fmt) for fmt in (0, 1)]) for ops, bad in cases.cigar_scripts(12, 3000)]
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(REPO, "oracle", "_ref", "edlib-aligner_ref")
        out["aligner"] = {key: digest(value) for key, value in test_aligner_cli.aligner_outputs(exe, tmp)}
    with open(os.path.join(HERE, "ref_digests.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print({k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
