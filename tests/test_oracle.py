"""CPU tests: the oracle restatement is pinned against the reference build's answers, stored as golden vectors
(tests/golden/ref_vectors.json) and as fingerprints of every result field (tests/golden/ref_digests.json)."""
import json
import os

import cases
from helpers import digest, golden_digests, oracle
from edlib_b200._ffi import MODES, TASKS

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_vectors.json")


def test_known_answers_oracle():
    O = oracle()
    for q, t, mode, task, k, eqs, exp in cases.KNOWN:
        r = O.align(q, t, k, MODES[mode], TASKS[task], eqs)
        for key, val in exp.items():
            if key == "cigar":
                assert O.cigar(r["alignment"]) == val
            else:
                assert r[key] == val, (q, t, mode, key, r)


def test_cigar_formats():
    O = oracle()
    ops = bytes([0, 0, 1, 1, 1, 2, 1, 1, 3, 0, 0])  # runTests.cpp:506-533
    assert O.cigar(ops, 1) == "2=3I1D2I1X2="
    assert O.cigar(ops, 0) == "2M3I1D2I3M"
    assert O.cigar(b"", 1) == ""
    assert O.cigar(bytes([0, 4]), 1) is None


def test_golden_vectors_oracle():
    O = oracle()
    with open(GOLDEN) as f:
        gold = json.load(f)
    assert len(gold["cases"]) > 200
    for c in gold["cases"]:
        eqs = [(bytes.fromhex(a), bytes.fromhex(b)) for a, b in c["eqs"]] if c["eqs"] else None
        r = O.align(bytes.fromhex(c["q"]), bytes.fromhex(c["t"]), c["k"], c["mode"], c["task"], eqs)
        exp = dict(c["expect"])
        exp["alignment"] = bytes.fromhex(exp["alignment"]) if exp.get("alignment") is not None else None
        assert r == exp, c


def test_oracle_vs_reference_random():
    """Every result field of 4,000 seeded cases against the fingerprints of the reference build's answers."""
    O = oracle()
    expected = golden_digests()["oracle_random"]
    got = [digest(O.align(c["q"], c["t"], c["k"], c["mode"], c["task"], c["eqs"])) for c in cases.single_pair_cases(101, 4000)]
    assert len(got) == len(expected) == 4000
    assert [i for i, (g, e) in enumerate(zip(got, expected)) if g != e] == []


def test_oracle_vs_reference_hirschberg_regime():
    """Paths beyond the reference's 1 MiB stored-matrix rule (edlib.cpp:1188-1211)."""
    O = oracle()
    expected = golden_digests()["oracle_hirschberg"]
    got = [digest(O.align(c["q"], c["t"], c["k"], c["mode"], c["task"])) for c in cases.hirschberg_cases(7, 40)]
    assert len(got) == len(expected) == 40
    assert [i for i, (g, e) in enumerate(zip(got, expected)) if g != e] == []
