"""Real-data parity on the reference's own test data (E. coli DH1 genome, 4,630,707 bp; reads and mutated prefixes of
50 bp .. 10 kbp shipped next to it): the data travel as fixtures (edlib_b200/data/e_coli_DH1.2bit,
tests/golden/ecoli_reads.json with the reference build's answers; generator tests/golden/make_real_data.py), so the
same checks run on the CPU emulation here and on the GPU box, where /root/reference does not exist.

SURVEY.md 8c's measured values are asserted on top of the fixture (they pin the fixture itself)."""
import json
import os

import pytest

import parity
from edlib_b200 import workloads

HERE = os.path.dirname(os.path.abspath(__file__))

# SURVEY.md 8c, measured from the reference: file -> (editDistance, end locations)
SURVEY = {
    "mason_illumina_reads/50bp/e_coli_DH1_illumina_1x50.fasta": (0, [2646428]),
    "mason_illumina_reads/100bp/e_coli_DH1_illumina_1x100.fasta": (0, [2646478]),
    "mason_illumina_reads/250bp/e_coli_DH1_illumina_1x250.fasta": (0, [2646628]),
    "mason_illumina_reads/500bp/e_coli_DH1_illumina_1x500.fasta": (3, [2646878]),
    "mason_illumina_reads/10kbp/e_coli_DH1_illumina_1x10000.fasta": (87, [2656389]),
    "mason_illumina_reads/50bp/mutated_80_perc.fasta": (13, [2646427, 2646429, 2646430, 2646431]),
    "mason_illumina_reads/100bp/mutated_60_perc.fasta": (37, [2646472, 2646473, 3531981]),
    "mason_illumina_reads/10kbp/mutated_60_perc.fasta": (3980, [2656385, 2656386, 2656387]),
}


def fixture():
    with open(os.path.join(HERE, "golden", "ecoli_reads.json")) as f:
        fx = json.load(f)
    genome = workloads.ecoli_genome().tobytes()
    assert len(genome) == fx["genome_length"] == 4630707
    for name, (ed, ends) in SURVEY.items():
        assert fx["reads"][name]["editDistance"] == ed and fx["reads"][name]["endLocations"] == ends, name
    return genome, fx["reads"]


def check(lib, genome, reads, names):
    seqs = [reads[n]["seq"].encode("ascii") for n in names]
    st, res = lib.align_batch(seqs, [genome] * len(seqs), -1, 2, 1)
    assert st == 0
    for n, r in zip(names, res):
        exp = reads[n]
        assert (r["editDistance"], r["endLocations"], r["startLocations"], r["alphabetLength"]) == \
               (exp["editDistance"], exp["endLocations"], exp["startLocations"], exp["alphabetLength"]), (n, str(r)[:300])
        assert r["numLocations"] == len(exp["endLocations"]) and r["alignment"] is None


def test_ecoli_short_reads_hw_locations_on_emulated_kernels():
    """Reads and mutated prefixes of at most 256 bp as ONE HW batch over the genome (the config-2 shape, candidate
    filter at production settings) through the CPU emulation of the kernels."""
    from test_engine_emul import load_emul
    genome, reads = fixture()
    names = sorted(n for n in reads if 0 < len(reads[n]["seq"]) <= 256)
    assert len(names) >= 20
    check(load_emul(), genome, reads, names)


@pytest.mark.gpu
def test_ecoli_all_reads_hw_locations_on_gpu():
    """Every read of the data set -- 50 bp to 10 kbp, 60 % to 100 % identity -- as ONE HW batch over the genome on
    the GPU: short reads through the seed filter, long ones through the chunked / seeded warp kernel."""
    from helpers import product
    lib = product()
    assert lib.lib.edlibB200Available() == 1
    genome, reads = fixture()
    check(lib, genome, reads, sorted(reads))


def test_phage_nw_distances_config1():
    """BASELINE configs[0] and its siblings: mutated phage genomes vs the phage genome (94 kbp), NW, k = -1
    (band doubling on the warp kernel): SURVEY.md 8c's measured reference values.  The reference's test data travel as
    tests/golden/phage_nw.fasta.xz (generator tests/golden/make_phage.py)."""
    import lzma
    from test_engine_emul import load_emul

    with lzma.open(os.path.join(HERE, "golden", "phage_nw.fasta.xz")) as f:
        lines = f.read().split(b"\n")
    seqs = dict(zip((l[1:].decode() for l in lines[0::2]), lines[1::2]))
    target = seqs["Enterobacteria_phage_1"]
    assert len(target) == 94481
    lib = load_emul()
    for pc, ed in ((99, 990), (97, 2977), (94, 6042), (90, 9506)):
        q = seqs["mutated_%d_perc" % pc]
        r = lib.align(q, target, -1, 0, 0)
        assert r["editDistance"] == ed and r["endLocations"] == [94480] and r["startLocations"] is None, (pc, r)
