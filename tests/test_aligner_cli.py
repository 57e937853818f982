"""The batched command-line aligner (apps/aligner/aligner.cpp over edlibAlignBatch) must print what the
reference's edlib-aligner prints (reference apps/aligner/aligner.cpp, built unmodified into
oracle/_ref/edlib-aligner_ref by `make -C oracle reftests`), for every option combination, except the
progress counter and the timing line.  What the reference printed is stored as fingerprints in
tests/golden/ref_digests.json (generator tests/golden/make_ref_digests.py)."""
import json
import os
import random
import subprocess

import pytest

from edlib_b200._ffi import REPO
from helpers import digest, mutate, rand_seq

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_digests.json")
OPTION_SETS = [["-m", "HW"], ["-m", "NW", "-l"], ["-m", "SHW", "-l", "-k", "30"], ["-m", "HW", "-p", "-f", "CIG_EXT"],
               ["-m", "HW", "-p"], ["-m", "NW", "-p", "-f", "CIG_STD"], ["-m", "HW", "-n", "5", "-l"],
               ["-m", "HW", "-n", "3", "-k", "8", "-p", "-f", "CIG_EXT"], ["-m", "SHW", "-n", "2"],
               [], ["-s"], ["-m", "HW", "-s", "-p"], ["-m", "HW", "-r", "2", "-l"], ["-m", "SHW", "-p", "-f", "CIG_STD", "-k", "40"],
               ["-m", "NW", "-p", "-f", "NICE", "-k", "0"], ["-m", "HW", "-k", "0", "-l"], ["-m", "NW", "-n", "1", "-p"]]
# wrong usage: same messages and exit codes (argv[0] differs in the usage text)
ERROR_SETS = [["-m", "XX"], ["-f", "SAM", "-p"], ["-m", "HW", "no-such-queries.fasta"], ["-m", "HW", "Q", "no-such-target.fasta"], ["-m", "HW", "onlyone"],
              ["-z"]]


def write_fasta(path, seqs):
    with open(path, "w") as f:
        for i, s in enumerate(seqs):
            f.write(">seq%d some description\n" % i)
            for a in range(0, len(s), 70):
                f.write(s[a:a + 70].decode() + "\n")


def make_inputs(tmp):
    rng = random.Random(77)
    t = rand_seq(rng, 20000, b"ACGT")
    qs = []
    for i in range(60):
        a = rng.randrange(0, len(t) - 400)
        qs.append(mutate(rng, t[a:a + rng.choice([60, 150, 300])], rng.choice([0.0, 0.03, 0.1]), b"ACGT"))
    qs.append(rand_seq(rng, 120, b"ACGT"))
    qf, tf = os.path.join(tmp, "q.fasta"), os.path.join(tmp, "t.fasta")
    write_fasta(qf, qs)
    write_fasta(tf, [t])
    return qf, tf


def normalised(exe, opts, qf, tf):
    return strip_progress(subprocess.run([exe] + opts + [qf, tf], capture_output=True, text=True, check=True).stdout)


def strip_progress(text):
    """stdout lines without the progress counter and the timing line."""
    return [l for l in text.replace("\r", "\n").split("\n") if not l.startswith("Cpu time") and not (l and l.replace("/", "").isdigit())]


def aligner_outputs(exe, tmp):
    """What `exe` prints for every option set and odd input, in a fixed order: [(key, normalised output)]."""
    qf, tf = make_inputs(tmp)
    out = [("opts " + " ".join(opts), normalised(exe, opts, qf, tf)) for opts in OPTION_SETS]
    # FASTA reading: wrapped lines, blank lines, lower case and other letters, blanks inside a line, an empty record, CRLF line
    # ends, no header, an empty file, a header alone, no newline at the end, several records in the target file
    odd = {"odd": ">q1\nACGTACGTAC\nGTAC\n\n>q2 desc\nacgtnnACGT\n>q3\n\n>q4\nAC GT\tAC\n", "crlf": ">q1\r\nACGTAC\r\nGT\r\n>q2\r\nTTGACC\r\n",
           "nohdr": "ACGT\nACGT\n", "empty": "", "hdr": ">only header\n", "noeol": ">q1\nACGT"}
    small_t = os.path.join(tmp, "small_t.fasta")
    with open(small_t, "w") as f:
        f.write(">t\nACGTACGTACGTACGGTACCAGT\nACGTTTGACCA\n")
    for name, text in odd.items():
        path = os.path.join(tmp, name + ".fasta")
        with open(path, "w", newline="") as f:
            f.write(text)
        for opts in (["-m", "HW", "-l"], ["-m", "NW", "-p", "-f", "CIG_EXT"]):
            r = subprocess.run([exe] + opts + [path, small_t], capture_output=True, text=True)
            out.append(("fasta %s %s" % (name, " ".join(opts)), [r.returncode, strip_progress(r.stdout)]))
    # first record of a multi-record target file
    out.append(("multi-record target", normalised(exe, ["-m", "HW"], small_t, os.path.join(tmp, "odd.fasta"))))
    for opts in ERROR_SETS:
        args = [qf if a == "Q" else a for a in opts]
        if not any(a.endswith(".fasta") or a == "onlyone" for a in opts):
            args += [qf, tf]
        elif opts[-1] == "no-such-queries.fasta":
            args += [tf]
        r = subprocess.run([exe] + args, capture_output=True, text=True)
        usage = [l for l in r.stderr.replace(exe, "PROG").splitlines() if l.startswith("Usage:")]  # the option help is worded differently
        out.append(("usage " + " ".join(opts), [r.returncode, r.stdout, usage]))
    return out


def compare(mine, tmp_path):
    """Every output of `mine` against the fingerprint of what the reference's edlib-aligner printed for it."""
    with open(GOLDEN) as f:
        expected = json.load(f)["aligner"]
    got = aligner_outputs(mine, str(tmp_path))
    assert [key for key, _ in got] == list(expected)
    for key, value in got:
        assert digest(value) == expected[key], (key, value[:12])


def test_aligner_matches_reference_on_emulated_kernels(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(REPO, "tests", "emul"), "libedlib_emul.so", "edlib-aligner"], check=True)
    compare(os.path.join(REPO, "tests", "emul", "edlib-aligner"), tmp_path)


@pytest.mark.gpu
def test_aligner_matches_reference_on_gpu(tmp_path):
    compare(os.path.join(REPO, "edlib_b200", "lib", "edlib-aligner"), tmp_path)
