"""Writes tests/golden/phage_nw.fasta.xz from the reference's own test DATA: the Enterobacteria phage 1 genome
(94,481 bp) and its 99 / 97 / 94 / 90 % mutated copies (test_data/Enterobacteria_Phage_1), one record each,
one line per sequence, xz-compressed (the copies share most of their text, so the file stays small).

    python tests/golden/make_phage.py <checkout of the reference>
"""
import lzma
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
NAMES = ["Enterobacteria_phage_1"] + ["mutated_%d_perc" % pc for pc in (99, 97, 94, 90)]


def read_fasta(path):
    with open(path, "rb") as f:
        return b"".join(l.strip() for l in f if not l.startswith(b">"))


def main(ref_root):
    d = os.path.join(ref_root, "test_data", "Enterobacteria_Phage_1")
    text = b"".join(b">%s\n%s\n" % (n.encode(), read_fasta(os.path.join(d, n + ".fasta"))) for n in NAMES)
    with open(os.path.join(HERE, "phage_nw.fasta.xz"), "wb") as f:
        f.write(lzma.compress(text, preset=9 | lzma.PRESET_EXTREME))


if __name__ == "__main__":
    main(sys.argv[1])
