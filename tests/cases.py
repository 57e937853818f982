"""Seeded case generators shared by the CPU (emulation) and GPU parity tests."""
import random

from helpers import mutate, rand_seq


def single_pair_cases(seed, count):
    """Small mixed cases: every mode/task, explicit and free k, odd alphabets, equalities,
    empty sequences, query lengths around the 32/64-bit word boundaries."""
    rng = random.Random(seed)
    for _ in range(count):
        asz = rng.choice([1, 2, 4, 4, 4, 10, 20])
        alpha = bytes(rng.sample(range(256), asz))
        m = rng.choice([0, 1, 2, 5, 31, 32, 33, 63, 64, 65, 100, 128, 129, 150, 200]) if rng.random() < 0.5 else rng.randrange(0, 300)
        if rng.random() < 0.4:
            t = rand_seq(rng, rng.randrange(0, 600), alpha)
            q = rand_seq(rng, m, alpha)
        else:
            t = rand_seq(rng, rng.randrange(1, 800), alpha)
            if len(t) > 1:
                a = rng.randrange(0, len(t))
                b = rng.randrange(a, min(len(t), a + 300))
                q = mutate(rng, t[a:b], rng.choice([0.0, 0.03, 0.1, 0.3]), alpha)
            else:
                q = rand_seq(rng, m, alpha)
        mode = rng.randrange(3)
        task = rng.randrange(3)
        k = rng.choice([-1, -1, 0, 1, 2, 5, 10, 50, 1000])
        eqs = None
        if rng.random() < 0.2 and asz >= 2:
            eqs = [(bytes([rng.choice(alpha)]), bytes([rng.choice(alpha)])) for _ in range(rng.randrange(1, 4))]
        yield dict(q=q, t=t, k=k, mode=mode, task=task, eqs=eqs)


def batch_cases(seed, count):
    """Batches that share a few targets (the reference's own batch shape, aligner.cpp:162-170)."""
    rng = random.Random(seed)
    for _ in range(count):
        asz = rng.choice([1, 2, 4, 4, 4, 10])
        alpha = bytes(rng.sample(range(256), asz))
        targets = [rand_seq(rng, rng.choice([rng.randrange(1, 200), rng.randrange(200, 3000)]), alpha)
                   for _ in range(rng.randrange(1, 4))]
        npairs = rng.choice([5, 40, 100, 300])
        qs, ts = [], []
        for _ in range(npairs):
            t = rng.choice(targets)
            if rng.random() < 0.5 and len(t) > 2:
                a = rng.randrange(0, len(t))
                b = rng.randrange(a, min(len(t), a + rng.choice([20, 150, 250, 400])))
                q = mutate(rng, t[a:b], rng.choice([0.0, 0.03, 0.1, 0.3]), alpha)
            else:
                q = rand_seq(rng, rng.choice([0, 1, 31, 32, 33, 64, 100, 150, 256, 257, 300]), alpha)
            qs.append(q)
            ts.append(t)
        mode = rng.randrange(3)
        task = rng.randrange(3)
        k = rng.choice([-1, -1, 0, 2, 10, 50, 1000])
        eqs = None
        if rng.random() < 0.2 and asz >= 2:
            eqs = [(bytes([rng.choice(alpha)]), bytes([rng.choice(alpha)])) for _ in range(rng.randrange(1, 4))]
        yield dict(qs=qs, ts=ts, k=k, mode=mode, task=task, eqs=eqs)


def long_cases(seed, count):
    """Queries taller than one 1024-row window: sliding band, strips, k doubling."""
    rng = random.Random(seed)
    for _ in range(count):
        alpha = bytes(rng.sample(range(256), rng.choice([2, 4, 4, 10])))
        kind = rng.randrange(4)
        if kind == 0:
            n = rng.choice([1100, 2100, 3000, 5000, 9000])
            t = rand_seq(rng, n, alpha)
            q = mutate(rng, t, rng.choice([0.01, 0.03, 0.1]), alpha)
            mode, k = 0, rng.choice([-1, 50, 200, 500, 2000])
        elif kind == 1:
            n = rng.choice([3000, 6000])
            t = rand_seq(rng, n, alpha)
            a = rng.randrange(0, n - 2600)
            q = mutate(rng, t[a:a + rng.choice([1030, 1100, 2500])], 0.05, alpha)
            mode, k = rng.choice([1, 2]), rng.choice([-1, 100, 1000])
        elif kind == 2:
            q = rand_seq(rng, rng.choice([8200, 9000, 17000]), alpha)
            t = rand_seq(rng, rng.randrange(50, 400), alpha)
            mode, k = rng.randrange(3), -1
        else:
            q = rand_seq(rng, rng.randrange(1025, 4000), alpha)
            t = rand_seq(rng, rng.randrange(1025, 4000), alpha)
            mode, k = 0, rng.choice([-1, 100, 3000])
        yield dict(q=q, t=t, k=k, mode=mode, task=rng.choice([0, 1]), eqs=None)


def path_cases(seed, count):
    """PATH beyond the reference's 1 MiB stored-matrix rule (Hirschberg, edlib.cpp:1188-1211):
    short query vs long target (runTests.cpp random shapes), similar long pairs, infix reads."""
    rng = random.Random(seed)
    for _ in range(count):
        alpha = bytes(rng.sample(range(256), rng.choice([2, 4, 4, 10])))
        kind = rng.random()
        if kind < 0.3:
            q = rand_seq(rng, rng.randrange(50, 350), alpha)
            t = rand_seq(rng, rng.randrange(9000, 14000), alpha)
        elif kind < 0.7:
            t = rand_seq(rng, rng.randrange(800, 4000), alpha)
            q = mutate(rng, t, rng.choice([0.01, 0.05, 0.2, 0.5]), alpha)
        else:
            n = rng.randrange(2000, 12000)
            t = rand_seq(rng, n, alpha)
            a = rng.randrange(0, n - 600)
            q = mutate(rng, t[a:a + rng.randrange(300, 2000)], 0.1, alpha)
        yield dict(q=q, t=t, k=-1, mode=rng.choice([0, 0, 1, 2]), task=2, eqs=None)


def filter_cases(seed, count):
    """HW batches of reads (>= 48 bp) over one shared target: clean hits, hits above the filter
    thresholds, unrelated reads, exact copies inside repeated target segments (several far-apart or
    neighbouring candidate ranges, equal-score hits in different windows), tandem-repeat targets
    (range lists that saturate), explicit and free k -- every branch of the two-stage candidate filter."""
    rng = random.Random(seed)
    yield filter_edge_case(seed)
    for _ in range(count - 1):
        alpha = rng.choice([b"ACGT", b"ACGT", b"ACGT", b"ACGTN", b"ACDEFGHIKLMNPQRSTVWY", b"AC"])
        shape = rng.random()
        if shape < 0.12:  # tandem repeat with a few mutations: candidates everywhere
            unit = rand_seq(rng, rng.choice([5, 13, 31, 50]), alpha)
            t = mutate(rng, unit * (rng.choice([6000, 20000]) // len(unit)), 0.01, alpha)
        else:
            t = rand_seq(rng, rng.choice([3000, 8000, 20000]), alpha)
            if shape < 0.45:  # a segment copied to several places (some close to each other)
                seg = t[100:100 + rng.choice([200, 600])]
                for _c in range(rng.choice([1, 2, 4])):
                    at = rng.randrange(0, len(t))
                    t = t[:at] + (mutate(rng, seg, 0.01, alpha) if rng.random() < 0.5 else seg) + t[at:]
        qs = []
        for _ in range(rng.choice([8, 40, 100])):
            L = rng.choice([48, 64, 80, 96, 100, 128, 150, 150, 200, 256])
            r = rng.random()
            if r < 0.7:
                a = rng.randrange(0, len(t) - L - 10)
                q = mutate(rng, t[a:a + L + 8], rng.choice([0, 0.02, 0.05, 0.12, 0.3]), alpha)[:L]
            elif r < 0.85:
                q = rand_seq(rng, L, alpha)
            else:
                a = rng.randrange(0, max(1, len(t) - L))
                q = t[a:a + L]
            if len(q) < L:
                q = q + rand_seq(rng, L - len(q), alpha)
            qs.append(q)
        yield dict(qs=qs, ts=[t] * len(qs), k=rng.choice([-1, -1, 3, 10, 40]), mode=2, task=rng.randrange(3), eqs=None)


def filter_edge_case(seed):
    """Deterministic corner cases of the window planning: reads taken from the very start and the very end
    of the target (windows clipped at column 0 / n-1), reads hanging over either end, a read longer than what
    is left of the target, exact duplicates far apart and back to back (equal-score hits in several windows,
    long end-location lists), a read equal to a tandem stretch (saturation), one unrelated read."""
    rng = random.Random(seed * 7919 + 1)
    alpha = b"ACGT"
    unit = rand_seq(rng, 11, alpha)
    body = rand_seq(rng, 6000, alpha)
    dup = body[2000:2150]
    t = body[:4000] + dup + dup + body[4000:] + unit * 40 + rand_seq(rng, 500, alpha)
    n = len(t)
    qs = [t[:150], t[:90], t[n - 150:], t[n - 70:],                              # flush with either end
          rand_seq(rng, 20, alpha) + t[:130], t[n - 130:] + rand_seq(rng, 20, alpha),  # hanging over the ends
          t[n - 200:] + rand_seq(rng, 56, alpha),                                # longer than what is left
          dup, mutate(rng, dup, 0.03, alpha), dup[10:140],                       # three copies of the same stretch
          (unit * 40)[:150], (unit * 40)[5:125],                                 # tandem repeat
          rand_seq(rng, 150, alpha), t[3000:3100], mutate(rng, t[1000:1256], 0.05, alpha)[:256]]
    return dict(qs=qs, ts=[t] * len(qs), k=[-1, 12, 3][seed % 3], mode=2, task=seed % 3, eqs=None)


def stream_cases(seed, count):
    """HW batches shaped like read sets (lengths within two neighbouring word classes, one shared target): what
    edlibAlignBatch streams in slices when the batch is large (the tests lower the size limits).  Includes bytes
    that do not occur in the target (they get the one extra code of a streamed batch), reads too short for any
    seed, unrelated reads, reads hanging over the ends of the target, repeats, bounded and free k, all tasks."""
    rng = random.Random(seed)
    for it in range(count):
        alpha = rng.choice([b"ACGT", b"ACGT", b"ACGT", b"ACGTN", b"ACDEFGHIKLMNPQRSTVWY", b"AC"])
        foreign = bytes(b for b in b"NXZ#" if b not in alpha)
        n = rng.choice([3000, 8000, 20000])
        t = rand_seq(rng, n, alpha)
        if rng.random() < 0.4:  # a segment copied to several places
            seg = t[100:100 + rng.choice([200, 600])]
            for _c in range(rng.choice([1, 2, 4])):
                at = rng.randrange(0, len(t))
                t = t[:at] + (mutate(rng, seg, 0.01, alpha) if rng.random() < 0.5 else seg) + t[at:]
        lo, hi = rng.choice([(100, 150), (129, 160), (40, 64), (150, 150), (225, 256), (20, 32)])
        qs = []
        for _ in range(rng.choice([70, 200, 500])):
            L = rng.randrange(lo, hi + 1)
            r = rng.random()
            if r < 0.7:
                a = rng.randrange(0, len(t) - L - 10)
                q = mutate(rng, t[a:a + L + 8], rng.choice([0, 0.02, 0.05, 0.12, 0.3]), alpha)[:L]
            elif r < 0.8:
                q = rand_seq(rng, L, alpha)
            elif r < 0.9:  # hanging over either end of the target
                q = (rand_seq(rng, 10, alpha) + t[:L])[:L] if rng.random() < 0.5 else (t[len(t) - L + 10:] + rand_seq(rng, 10, alpha))[:L]
            else:
                a = rng.randrange(0, max(1, len(t) - L))
                q = t[a:a + L]
            if len(q) < L:
                q = q + rand_seq(rng, L - len(q), alpha)
            if rng.random() < 0.15:  # bytes the target does not hold
                q = bytearray(q)
                for _x in range(rng.choice([1, 2, 5])):
                    q[rng.randrange(len(q))] = rng.choice(foreign)
                q = bytes(q)
            qs.append(q)
        yield dict(qs=qs, ts=[t] * len(qs), k=rng.choice([-1, -1, 3, 10, 40]), mode=2, task=(it + seed) % 3, eqs=None)


def long_hw_cases(seed, count):
    """HW batches of LONG queries (300 .. 2600 rows) over one long-ish target: the seed levels with doubling thresholds
    (distances below and above 64 / 128), sliding warp windows, unrelated and heavily mutated queries (chunked sweeps
    with 2m halos), repeats (saturated seeds, many end locations), queries hanging over the ends, bounded k; all
    tasks.  The tests lower the target-length limits so that these small targets take the long-query path."""
    rng = random.Random(seed)
    for it in range(count):
        alpha = rng.choice([b"ACGT", b"ACGT", b"ACGTN", b"ACDEFGHIKLMNPQRSTVWY"])
        n = rng.choice([12000, 20000, 30000, 45000])
        t = rand_seq(rng, n, alpha)
        if rng.random() < 0.5:  # a long segment copied elsewhere (equal-score hits far apart), or a tandem stretch
            if rng.random() < 0.6:
                seg = t[500:500 + rng.choice([600, 1500])]
                at = rng.randrange(3000, len(t))
                t = t[:at] + seg + t[at:]
            else:
                unit = rand_seq(rng, rng.choice([7, 40]), alpha)
                at = rng.randrange(0, len(t))
                t = t[:at] + unit * (1200 // len(unit)) + t[at:]
        qs = []
        for _ in range(rng.choice([3, 6])):
            L = rng.choice([300, 700, 1100, 1500, 2600, 3400])
            r = rng.random()
            if r < 0.65:
                a = rng.randrange(0, len(t) - L - 50)
                q = mutate(rng, t[a:a + L + 40], rng.choice([0, 0.01, 0.04, 0.08, 0.15]), alpha)[:L]
            elif r < 0.75:
                q = rand_seq(rng, L, alpha)
            elif r < 0.85:
                q = (rand_seq(rng, 30, alpha) + t[:L])[:L] if rng.random() < 0.5 else (t[len(t) - L + 30:] + rand_seq(rng, 30, alpha))[:L]
            else:
                a = rng.randrange(0, max(1, len(t) - L))
                q = t[a:a + L]
            if len(q) < L:
                q = q + rand_seq(rng, L - len(q), alpha)
            qs.append(q)
        yield dict(qs=qs, ts=[t] * len(qs), k=rng.choice([-1, -1, 30, 100, 400]), mode=2, task=(it + seed) % 3, eqs=None)


def pairwise_cases(seed, count):
    """Batches of short queries each with its OWN target (pairwise comparison shape): the lane-per-
    alignment kernel with per-job targets, all modes and tasks, odd alphabets, equalities."""
    rng = random.Random(seed)
    for _ in range(count):
        alpha = bytes(rng.sample(range(256), rng.choice([2, 4, 4, 20])))
        qs, ts = [], []
        for _ in range(rng.choice([10, 60, 150])):
            t = rand_seq(rng, rng.randrange(1, 500), alpha)
            if rng.random() < 0.6 and len(t) > 5:
                a = rng.randrange(0, len(t) - 1)
                q = mutate(rng, t[a:a + rng.randrange(1, 257)], rng.choice([0, 0.05, 0.3]), alpha)[:256]
            else:
                q = rand_seq(rng, rng.choice([0, 1, 33, 64, 100, 200, 256]), alpha)
            qs.append(q)
            ts.append(t)
        eqs = [(bytes([alpha[0]]), bytes([alpha[1]]))] if rng.random() < 0.2 else None
        yield dict(qs=qs, ts=ts, k=rng.choice([-1, -1, 2, 20]), mode=rng.randrange(3), task=rng.randrange(3), eqs=eqs)


# Hand vectors with known answers from the reference's own tests (SURVEY.md section 8c):
# bindings/python/test.py:6-73 and test/runTests.cpp:427-570, plus API probes measured on the
# reference build.  (query, target, mode, task, k, equalities) -> expected fields.
KNOWN = [
    (b"telephone", b"elephant", "NW", "path", -1, None,
     dict(editDistance=3, endLocations=[7], startLocations=[0], alphabetLength=8, cigar="1I5=1X1=1X")),
    (b"AACG", b"TCAACCTG", "HW", "path", -1, None,
     dict(editDistance=1, endLocations=[4, 5], startLocations=[2, 2], cigar="3=1I")),
    (b"TAAGGATGGTCCCATTC", b"AAGGGGTCTCATATC", "NW", "path", -1, None,
     dict(editDistance=5, endLocations=[14], cigar="1I4=2I4=1X3=1D2=")),
    (b"AA", b"B", "HW", "path", -1, None,
     dict(editDistance=2, endLocations=[-1, 0], startLocations=[0, 0], cigar="2I")),
    (b"AA", b"B", "SHW", "path", -1, None, dict(editDistance=2)),
    (b"ACGT", b"", "NW", "distance", -1, None, dict(editDistance=4, endLocations=[-1])),
    (b"", b"ACGT", "NW", "distance", -1, None, dict(editDistance=4, endLocations=[3])),
    (b"", b"ACGT", "HW", "path", -1, None, dict(editDistance=0, endLocations=[-1], startLocations=None, alignment=None)),
    (b"GCATATCAATAAGCGGAGGA", b"TAACAAGGTTTCCGTAGGTGAACCTGCGGAAGGATCATTATTGAATTATATCTT", "HW", "locations", -1,
     [(b"R", b"A"), (b"R", b"G"), (b"M", b"A"), (b"M", b"C"), (b"W", b"A"), (b"W", b"T")], dict()),
]


def hirschberg_cases(seed, count):
    """PATH of long pairs (query x target beyond the reference's 1 MiB stored-matrix rule, edlib.cpp:1188-1211): short
    queries in long targets and mutated copies, alphabets of 2, 4 and 10 symbols, every mode."""
    rng = random.Random(seed)
    for _ in range(count):
        alpha = bytes(rng.sample(range(256), rng.choice([2, 4, 10])))
        if rng.random() < 0.5:
            q = rand_seq(rng, rng.randrange(50, 350), alpha)
            t = rand_seq(rng, rng.randrange(9000, 14000), alpha)
        else:
            t = rand_seq(rng, rng.randrange(1500, 4000), alpha)
            q = mutate(rng, t, rng.choice([0.02, 0.2]), alpha)
        mode = rng.choice([0, 0, 1, 2])
        yield dict(q=q, t=t, k=-1, mode=mode, task=2, eqs=None)


def cigar_scripts(seed, count):
    """Edit scripts for edlibAlignmentToCigar: every length around the word boundaries, runs of every length, and now
    and then a bad operation code.  Yields (ops, bad)."""
    rng = random.Random(seed)
    for _ in range(count):
        n = rng.choice([0, 1, 2, 7, 8, 9, 15, 16, 17, 31, 33, 64, 150, 151, 1000, 1500, 5000])
        style = rng.randrange(4)
        if style == 0:
            ops = bytes(rng.choice([0, 0, 0, 0, 0, 0, 1, 2, 3]) for _ in range(n))
        elif style == 1:
            ops = bytes([rng.randrange(4)]) * n
        elif style == 2:
            ops = b"".join(bytes([rng.randrange(4)]) * rng.randrange(1, 40) for _ in range(n // 8 + 1))[:n]
        else:
            ops = bytes(rng.randrange(4) for _ in range(n))
        bad = rng.random() < 0.03 and n > 0
        if bad:
            ops = bytearray(ops)
            ops[rng.randrange(n)] = rng.choice([4, 7, 255])
            ops = bytes(ops)
        yield ops, bad


def big_batch_case(seed, num=140_000, target_len=4000):
    """One HW batch large enough for the multi-threaded host paths (classification, seed-stage
    outcomes, end-location assembly): short reads of two word classes over one target, with empty
    queries, unrelated reads and a few queries beyond the lane kernels mixed in."""
    rng = random.Random(seed)
    alpha = b"ACGT"
    t = rand_seq(rng, target_len, alpha)
    qs = []
    for i in range(num):
        r = rng.random()
        L = rng.choice([40, 48, 60, 70])
        if r < 0.001:
            q = b""
        elif r < 0.0015:
            a = rng.randrange(0, target_len - 400)
            q = mutate(rng, t[a:a + 300], 0.05, alpha)
        elif r < 0.9:
            a = rng.randrange(0, target_len - L - 8)
            q = mutate(rng, t[a:a + L + 6], rng.choice([0, 0.03, 0.08]), alpha)[:L]
        else:
            q = rand_seq(rng, L, alpha)
        qs.append(q)
    return dict(qs=qs, ts=[t] * num, k=rng.choice([-1, 6]), mode=2, task=rng.choice([0, 1]), eqs=None)


def tied_ends_cases(seed, count):
    """HW read sets whose reads tie on MANY neighbouring end columns (homopolymer and short-period tandem stretches
    inside a random target): one window of the candidate filter then holds more than its inline end columns, so the
    overflow list of the window sweeps and its assembly (device reduction, host-driven stages) are exercised; reads
    across the borders of the stretches and plain reads ride along."""
    from helpers import mutate, rand_seq
    rng = random.Random(seed)
    for it in range(count):
        parts, marks = [], []
        at = 0
        for _ in range(rng.randrange(2, 5)):
            u = rand_seq(rng, rng.randrange(1500, 4000), b"ACGT")
            parts.append(u)
            at += len(u)
            unit = rng.choice([b"A", b"T", b"AC", b"GGC", b"ACGTTGCA"])
            rep = unit * (rng.randrange(60, 420) // len(unit))
            marks.append((at, len(rep)))
            parts.append(rep)
            at += len(rep)
        parts.append(rand_seq(rng, 2000, b"ACGT"))
        t = b"".join(parts)
        qs = []
        for _ in range(rng.randrange(40, 90)):
            m = rng.choice([24, 32, 40, 40, 64, 100, 150, 200, 256])
            kind = rng.randrange(4)
            if kind == 0:      # inside a stretch
                a, ln = rng.choice(marks)
                s = a + rng.randrange(0, max(1, ln - m))
            elif kind == 1:    # across a border of a stretch
                a, ln = rng.choice(marks)
                s = max(0, (a if rng.random() < 0.5 else a + ln) - rng.randrange(1, m))
            else:
                s = rng.randrange(0, len(t) - m)
            q = mutate(rng, t[s:s + m], rng.choice([0.0, 0.0, 0.02, 0.05]), b"ACGT")
            if q:
                qs.append(q)
        yield dict(qs=qs, ts=[t] * len(qs), k=rng.choice([-1, -1, 2, 5, 20]), mode=2, task=(it + seed) % 3, eqs=None)


def band_cases(seed, count):
    """Pairwise NW batches of long queries (2,100 .. 12,000 rows) with a bound k or with k = -1 (doubling): the k-banded
    sweeps run on the thread-per-alignment band kernel (eb_core.h: band_job) at several window sizes; targets are
    mutated copies (some beyond the bound), some with a long insertion or deletion so that the band sits off the
    main diagonal, protein-sized alphabets included."""
    from helpers import mutate, rand_seq
    rng = random.Random(seed)
    for it in range(count):
        alpha = rng.choice([b"ACGT", b"ACGT", b"ACGTN", b"ACDEFGHIKLMNPQRSTVWY"])
        k = rng.choice([-1, 0, 1, 40, 90, 200, 500, 900])
        qs, ts = [], []
        for _ in range(rng.randrange(3, 9)):
            m = rng.choice([2100, 3000, 4097, 6000, 10000, 12000])
            q = rand_seq(rng, m, alpha)
            t = mutate(rng, q, rng.choice([0.0, 0.005, 0.02, 0.03, 0.06]) if k > 1 or k < 0 else rng.choice([0.0, 0.0, 0.0002]), alpha)
            shift = rng.choice([0, 0, 0, 17, 150, 400])
            if shift and rng.random() < 0.5:
                at = rng.randrange(0, len(t))
                t = t[:at] + rand_seq(rng, shift, alpha) + t[at:]
            elif shift:
                at = rng.randrange(0, max(1, len(t) - shift))
                t = t[:at] + t[at + shift:]
            qs.append(q)
            ts.append(t)
        yield dict(qs=qs, ts=ts, k=k, mode=0, task=rng.choice([0, 1]), eqs=None)


def equality_read_cases(seed, count):
    """HW read sets with additional equalities: case folding (a TRANSITIVE relation: the engine gives equal bytes one
    code and runs its plain-equality fast paths, seed filter included) and, every third batch, a wildcard on top of it
    (N equals A and C, which differ: the table path)."""
    from helpers import mutate, rand_seq
    rng = random.Random(seed)
    for it in range(count):
        t = rand_seq(rng, rng.randrange(3000, 9000), b"ACGT")
        qs = []
        for _ in range(rng.randrange(40, 120)):
            m = rng.choice([33, 64, 100, 150, 200])
            s = rng.randrange(0, len(t) - m)
            q = bytearray(mutate(rng, t[s:s + m], rng.choice([0.0, 0.02, 0.05]), b"ACGT"))
            for i in range(len(q)):
                if rng.random() < 0.3:
                    q[i] = q[i] + 32  # lower case
                elif it % 3 == 2 and rng.random() < 0.03:
                    q[i] = ord("N")
            if q:
                qs.append(bytes(q))
        eqs = [(b"A", b"a"), (b"C", b"c"), (b"g", b"G"), (b"T", b"t")]
        if it % 3 == 2:
            eqs += [(b"N", b"A"), (b"N", b"C"), (b"N", b"a"), (b"N", b"c")]
        yield dict(qs=qs, ts=[t] * len(qs), k=rng.choice([-1, -1, 6, 20]), mode=2, task=(it + seed) % 3, eqs=eqs)


def small_k_cases(seed, count):
    """HW read sets with the tightest bounds (k = 0, 1, 2): exact and nearly exact copies of target substrings, so the
    filter works with thresholds t = 0, 1, 2 -- at t = 0 the only alignment of interest runs along the TOP diagonal of
    its verification window (regression: the early exit of hopeless windows once discarded exactly those)."""
    from helpers import mutate, rand_seq
    rng = random.Random(seed)
    for it in range(count):
        alpha = rng.choice([b"ACGT", b"ACGT", b"ACGTN", b"ABCDEFGHIJKLMNOPQRST"])
        t = rand_seq(rng, rng.randrange(400, 6000), alpha)
        qs = []
        for _ in range(rng.randrange(30, 90)):
            m = rng.choice([20, 33, 64, 100, 148, 150, 200, 256])
            s = rng.randrange(0, len(t) - m)
            q = bytearray(t[s:s + m])
            for _ in range(rng.choice([0, 0, 0, 1, 2, 3])):   # a few single-symbol edits
                kind, at = rng.randrange(3), rng.randrange(len(q))
                if kind == 0:
                    q[at] = rng.choice(alpha)
                elif kind == 1:
                    q.insert(at, rng.choice(alpha))
                elif len(q) > 1:
                    del q[at]
            qs.append(bytes(q))
        yield dict(qs=qs, ts=[t] * len(qs), k=[0, 1, 2, 0][it % 4], mode=2, task=(it + seed) % 3, eqs=None)


BOUNDARY_LENGTHS = [0, 1, 2, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, 255, 256, 257, 300, 511, 512, 513, 1000, 2049]


def boundary_mix_cases(seed, count):
    """Batches whose query AND target lengths sit on the 32/64-bit word boundaries (0, 1, 31..33, 63..65, ... 2049), over
    one shared target (up to 70 kbp) or one target per query, with alphabets of 1, 2, 4, 27 and 256 symbols, every mode
    and task, bounds from 0 to 1000 and now and then a few equality pairs: queries are random, mutated substrings, or
    mutated prefixes / suffixes of their target."""
    from helpers import mutate, rand_seq
    rng = random.Random(seed)
    for _ in range(count):
        alpha = rng.choice([b"ACGT", b"AC", b"A", bytes(range(33, 60)), bytes(range(256))])
        n = rng.choice([1, 2, 7, 40, 130, 300])
        if rng.random() < 0.5:
            ts = [rand_seq(rng, rng.choice(BOUNDARY_LENGTHS + [5000, 20000, 70000]), alpha)] * n
        else:
            ts = [rand_seq(rng, rng.choice(BOUNDARY_LENGTHS), alpha) for _ in range(n)]
        qs = []
        for t in ts:
            style = rng.randrange(4)
            m = rng.choice(BOUNDARY_LENGTHS[:rng.choice([12, 18, len(BOUNDARY_LENGTHS)])])
            if style == 0 or not t:
                q = rand_seq(rng, m, alpha)
            elif style == 1:
                at = rng.randrange(len(t))
                q = mutate(rng, t[at:at + m], rng.choice([0, 0.02, 0.1, 0.3]), alpha)
            elif style == 2:
                q = mutate(rng, t[:m], 0.05, alpha)
            else:
                q = mutate(rng, t[-m:] if m else b"", 0.05, alpha)
            qs.append(q)
        eqs = None
        if rng.random() < 0.15:
            eqs = [(bytes([rng.choice(alpha)]), bytes([rng.choice(alpha)])) for _ in range(rng.randrange(1, 5))]
        yield dict(qs=qs, ts=ts, k=rng.choice([-1, -1, 0, 1, 2, 5, 20, 64, 100, 1000]), mode=rng.randrange(3), task=rng.randrange(3), eqs=eqs)
