#!/usr/bin/env python3
"""
Generate the golden fixtures under tests/golden/ from the REFERENCE ITSELF.

Needs the reference checkout (builds oracle/_ref on the fly):

    python tests/golden/make_golden.py [fixture function ...]      (default: all of them)

Everything written here is input/output pairs of the reference's own compiled code
(cutadapt._align, _kmer_finder, qualtrim, kmer_heuristic, adapters) plus the per-read
coordinates of the reference's golden files tests/cut/illumina.info.txt and
illumina5.info.txt, so that the tests need neither the reference nor oracle/_ref.
Seeds are fixed; re-running reproduces the files byte for byte.
"""
import gzip
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
from oracle import build_ref  # noqa: E402
from util import batch_digest, canon, digest, random_locate_cases  # noqa: E402

build_ref.import_ref()
from cutadapt._align import Aligner, PrefixComparer, SuffixComparer, edit_environment  # noqa: E402
from cutadapt.align import hamming_environment  # noqa: E402
from cutadapt._kmer_finder import KmerFinder  # noqa: E402
from cutadapt.kmer_heuristic import create_positions_and_kmers  # noqa: E402
from cutadapt.qualtrim import quality_trim_index, nextseq_trim_index, poly_a_trim_index, expected_errors  # noqa: E402
from cutadapt import adapters as RA  # noqa: E402
from cutadapt import _match_tables as RT  # noqa: E402

REF_TESTS = "/root/reference/tests"


def dump(name, obj):
    path = os.path.join(HERE, name)
    data = json.dumps(obj, separators=(",", ":"), sort_keys=True).encode()
    with open(path, "wb") as raw:
        with gzip.GzipFile(fileobj=raw, mode="wb", mtime=0, filename="") as f:
            f.write(data)
    print(f"{name}: {len(obj) if hasattr(obj, '__len__') else ''} entries, {os.path.getsize(path)} bytes")


def rnd(rng, alpha, n):
    return "".join(rng.choice(alpha) for _ in range(n))


def mutate(rng, piece, alpha, n_edits):
    piece = list(piece)
    for _ in range(n_edits):
        if not piece:
            break
        p = rng.randrange(len(piece))
        r = rng.random()
        if r < 0.4:
            piece[p] = rng.choice(alpha)
        elif r < 0.7:
            del piece[p]
        else:
            piece.insert(p, rng.choice(alpha))
    return "".join(piece)


def locate_kat():
    rng = random.Random(1001)
    cases = []
    # the reference's own known-answer tests (tests/test_align.py:69-146, 256-261, 326-413)
    fixed = [
        ("", "", 0, 0, False, False, 1, 0),
        ("CCAGTCCTCT", "CCAGTCCTTTCCTGAGAGT", 0.3, 8, False, False, 1, 1),
        ("TCGATC", "TCGATGC", 1.5 / 6, 8, False, False, 1, 1),
        ("GCCGAACTTCTTAGACTGCCTTAAGGACGT", "CAAATCACCAGAAGGCGCCTAACTTCTTAGACTGCC", 0.1, 14, False, False, 1, 1),
        ("TTTT", "CCTTTT", 0.25, 14, False, False, 1, 1),
        ("TTTTTT", "CCTTTT", 0.25, 14, False, False, 1, 1),
        ("TTT", "CCTTTT", 1 / 3, 14, False, False, 1, 1),
        ("AAAAAAAAAAAAAAAAA", "ACAGAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA", 0.0, 14, False, False, 1, 1),
        ("CTGAATT", "AAAAAAACTGAATTAAAA", 0.0, 14, False, False, 1, 1),
        ("NNNCTGAATT", "AAAAAAACTGAATTAAAA", 0.1, 14, True, False, 1, 1),
        ("ACGTNNNN", "TTTTACGTACGT", 0.2, 11, True, False, 1, 1),
        ("ATNGNA", "CCATCGTACC", 0.0, 15, True, False, 1, 1),
        ("ATRGNA", "CCATAGTACC", 0.0, 15, True, True, 1, 1),
    ]
    for ref, q, rate, flags, wr, wq, ic, mo in fixed:
        cases.append([ref, q, rate, flags, wr, wq, ic, mo])
    for _ in range(4000):
        alpha = rng.choice(["ACGT", "ACGT", "AC", "ACGTN", "ACGTacgtNn", "ACGTRYKMSWN", "A"])
        m = rng.randint(1, 28)
        ref = rnd(rng, alpha, m)
        wr, wq = rng.random() < 0.3, rng.random() < 0.2
        if wr and set(ref.upper()) <= {"N"}:
            continue
        rate = rng.choice([0, 0.05, 0.1, 0.15, 0.2, 0.25, 0.34, 0.5])
        flags = rng.choice([14, 11, 15, 8, 2, 9, 6, rng.randint(0, 15)])
        ic = rng.choice([1, 1, 1, 1, 100000, 2])
        mo = rng.randint(1, 5)
        n = rng.randint(0, 70)
        q = rnd(rng, alpha, n)
        if rng.random() < 0.7:
            piece = ref if rng.random() < 0.6 else ref[rng.randint(0, m // 2) : rng.randint(m // 2, m)]
            piece = mutate(rng, piece, alpha, rng.choice([0, 0, 1, 2]))
            pos = rng.choice([0, len(q), rng.randint(0, len(q))])
            q = q[:pos] + piece + q[pos:]
        cases.append([ref, q, rate, flags, wr, wq, ic, mo])
    out = []
    for ref, q, rate, flags, wr, wq, ic, mo in cases:
        res = Aligner(ref, rate, flags, wr, wq, ic, mo).locate(q)
        out.append([ref, q, rate, flags, wr, wq, ic, mo, list(res) if res is not None else None])
    dump("locate_kat.json.gz", out)


def comparer_kat():
    rng = random.Random(1002)
    out = []
    for _ in range(1200):
        alpha = rng.choice(["ACGT", "ACGTN", "ACGTacgtn", "ACGTRYN"])
        m = rng.randint(1, 20)
        ref = rnd(rng, alpha, m)
        wr, wq = rng.random() < 0.4, rng.random() < 0.3
        if wr and ref.count("N") - ref.count("n") == m:
            continue
        rate = rng.choice([0, 0.1, 0.2, 0.3, 0.5, 1.0])
        mo = rng.randint(1, 6)
        q = rnd(rng, alpha, rng.randint(0, 30))
        if rng.random() < 0.5:
            q = mutate(rng, ref[: rng.randint(0, m)], alpha, rng.choice([0, 1])) + q
        if rng.random() < 0.5:
            q = q + mutate(rng, ref[rng.randint(0, m) :], alpha, rng.choice([0, 1]))
        try:
            p = PrefixComparer(ref, rate, wr, wq, mo).locate(q)
            s = SuffixComparer(ref, rate, wr, wq, mo).locate(q)
        except ValueError:
            continue
        out.append([ref, q, rate, wr, wq, mo, list(p) if p else None, list(s) if s else None])
    dump("comparer_kat.json.gz", out)


def kmer_kat():
    rng = random.Random(1003)
    heur = []
    for _ in range(400):
        L = rng.randint(1, 40)
        ad = rnd(rng, "ACGT" if rng.random() < 0.8 else "ACGTN", L)
        mo = rng.randint(1, min(L, 8))
        er = rng.choice([0, 0.05, 0.1, 0.15, 0.2, 0.3, 0.5])
        b, f, i = rng.choice([(1, 0, 1), (0, 1, 1), (1, 1, 1), (1, 0, 0), (0, 1, 0)])
        try:
            res = create_positions_and_kmers(ad, mo, er, bool(b), bool(f), bool(i))
        except NotImplementedError:
            res = "NotImplementedError"
        else:
            res = sorted(([s, e, sorted(k)] for s, e, k in res),
                         key=lambda x: (x[0], -(10**9) if x[1] is None else x[1], x[2]))
        heur.append([ad, mo, er, b, f, i, res])
    present = []
    for _ in range(300):
        alpha = rng.choice(["ACGT", "ACGTN", "ACGTacgtn", "ACGTRYN"])
        sets = []
        for _ in range(rng.randint(1, 4)):
            kmers = [rnd(rng, alpha if rng.random() < 0.5 else "ACGT", rng.randint(1, 12)) for _ in range(rng.randint(1, 7))]
            start, stop = rng.choice([(0, None), (-rng.randint(1, 20), None), (0, rng.randint(1, 20)),
                                      (rng.randint(0, 10), None), (-15, -3), (2, -2)])
            sets.append([start, stop, kmers])
        rw, qw = rng.random() < 0.4, rng.random() < 0.3
        kf = KmerFinder([(s, e, k) for s, e, k in sets], rw, qw)
        reads = []
        for _ in range(12):
            n = rng.randint(0, 45)
            read = rnd(rng, alpha, n)
            if rng.random() < 0.5 and n > 0:
                kmer = rng.choice(rng.choice(sets)[2])
                pos = rng.choice([0, max(0, n - len(kmer)), rng.randint(0, n)])
                read = read[:pos] + kmer + read[pos + len(kmer) :]
            if any(stop is not None and stop > len(read) for _, stop, _ in sets):
                continue  # the reference scans past the end of the string here (undefined)
            reads.append([read, bool(kf.kmers_present(read))])
        present.append([sets, rw, qw, reads])
    dump("kmer_kat.json.gz", {"heuristic": heur, "present": present})


def qualtrim_kat():
    rng = random.Random(1004)
    out = []
    for _ in range(1500):
        n = rng.randint(0, 60)
        base = rng.choice([33, 33, 64])
        q = "".join(chr(base + rng.choice([0, 2, 2, 5, 10, 15, 20, 25, 30, 35, 40])) for _ in range(n))
        cf, cb = rng.choice([0, 0, 5, 10, 20, 30]), rng.choice([0, 10, 20, 20, 30])
        out.append([q, cf, cb, base, list(quality_trim_index(q, cf, cb, base))])
    # the reference's own fixtures for -q (tests/data/lowqual.fastq, test_commandline.py:246-248)
    with open(os.path.join(REF_TESTS, "data", "lowqual.fastq")) as f:
        lines = f.read().split("\n")
    for i in range(3, len(lines), 4):
        q = lines[i]
        out.append([q, 0, 10, 33, list(quality_trim_index(q, 0, 10, 33))])
    dump("qualtrim_kat.json.gz", out)


TYPES = ["FrontAdapter", "RightmostFrontAdapter", "BackAdapter", "RightmostBackAdapter", "AnywhereAdapter",
         "NonInternalFrontAdapter", "NonInternalBackAdapter", "PrefixAdapter", "SuffixAdapter"]


def trim_scans_kat():
    """nextseq_trim_index and poly_a_trim_index (qualtrim.pyx:76-169) incl. the reference's own test cases."""
    from types import SimpleNamespace

    rng = random.Random(1021)
    nextseq, polya = [], []
    # the reference's own known-answer test (tests/test_qualtrim.py:7-15): expected 0 and 33
    for seq, qual, cutoff in [("", "", 22),
                              ("TCTCGTATGCCGTCTTATGCTTGAAAAAAAAAAGGGGGGGGGGGGGGGGGNNNNNNNNNNNGGNGG",
                               "AA//EAEE//A6///E//A//EA/EEEEEEAEA//EEEEEEEEEEEEEEE###########EE#EA", 22)]:
        nextseq.append([seq, qual, cutoff, 33, nextseq_trim_index(SimpleNamespace(sequence=seq, qualities=qual), cutoff, 33)])
    assert [x[4] for x in nextseq] == [0, 33]
    for _ in range(1500):
        n = rng.randint(0, 160)
        seq = rnd(rng, rng.choice(["ACGT", "ACGTN", "GGGA", "acgtG"]), n)
        if rng.random() < 0.4 and n:
            t = rng.randint(1, n)
            seq = seq[: n - t] + "G" * t
        qual = "".join(chr(33 + rng.choice([2, 2, 10, 15, 20, 25, 30, 37, 41])) for _ in range(n))
        cutoff = rng.choice([0, 5, 10, 20, 25, 30])
        base = rng.choice([33, 33, 64])
        nextseq.append([seq, qual, cutoff, base, nextseq_trim_index(SimpleNamespace(sequence=seq, qualities=qual), cutoff, base)])
    # the reference's own known-answer tests (tests/test_qualtrim.py:18-62)
    tails = [("", ""), ("GGGGGGGGAAAGAAGAAGAAGAAGAAGAAG", ""), ("TTTAGA", ""), ("TTTAGAA", ""), ("TTTAG", "AAA"),
             ("TCAAGAAGTCCTTTACCAGCTTTC", "AAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA"),
             ("TCAAGAAGTCCTTTACCAGCTTTC", "AAATAAAAAAAAAAAAAAAAAAAAAAAAAAAAA"),
             ("GCAGATCACCTT", "AAAAAAAAAAAAAAAAAAAAAAAAAAAATAAA"), ("GCAGATCACCTT", "AAAAAAAAAAAAAAAAAAAAAAAAAAAAT"),
             ("GCAGATCACCTT", "AAAAAAAAAAAAAAAAAAAAAAAAAAAATCG"), ("GCAGATCACCTAT", "AAAACAAAAAAACAAAAAAAACAAAAAA"),
             ("TTTT", "AAATAAAA"), ("GGGGGGGGAAAGAAGAAGAAGAAGAAGAAG", "AAA")]
    for seq, tail in tails:
        assert poly_a_trim_index(seq + tail) == len(seq)
        polya.append([seq + tail, False, len(seq)])
    heads = [("", ""), ("", "GGGGGGGGAAAGAAGAAGAAGAAGAAGAAG"), ("", "TGTCCC"), ("", "TTGTCCC"), ("TTT", "GTCCC"),
             ("TTTTTTTTTTTTTTTTTTTTT", "CAAGAAGTCCCCAGCTTTC"),
             ("TTTATTTTTTTTTTTTTTTTTTTTTTTTTTTTT", "CAAGAAGTCCTTTACCAGCTTTC"),
             ("TTTTTATTTTTTTTTTTTTTTTTTTTTTTTTT", "GCAGATCACCTT"), ("ATTTTTTTTTTTTTTTTTTTTTTTTTTTT", "GCAGATCACCTT"),
             ("AGCTTTTTTTTTTTTTTTTTTTTTTTTTTTT", "GCAGATCACCTT"), ("TTTTGTTTTTTTGTTTTTTTTGTTTTTT", "GCAGATCACCTAT"),
             ("TTTATTTT", "AAAA"), ("TTT", "GGGGGGGGAAAGAAGAAGAAGAAGAAGAAG")]
    for head, seq in heads:
        assert poly_a_trim_index(head + seq, revcomp=True) == len(head)
        polya.append([head + seq, True, len(head)])
    for _ in range(1500):
        n = rng.randint(0, 160)
        seq = rnd(rng, rng.choice(["ACGT", "ACGTN", "AAAC", "TTTG", "acgtA"]), n)
        if rng.random() < 0.5:
            tail = mutate(rng, "A" * rng.randint(0, 60), "ACGT", rng.choice([0, 0, 1, 2, 4]))
            seq = seq + tail
        if rng.random() < 0.5:
            head = mutate(rng, "T" * rng.randint(0, 60), "ACGT", rng.choice([0, 0, 1, 2, 4]))
            seq = head + seq
        for rc in (False, True):
            polya.append([seq, rc, poly_a_trim_index(seq, rc)])
    # expected_errors: FP64, results stored as float.hex() so that the comparison is bit-exact.
    # Single-character strings expose the reference's table SCORE_TO_ERROR_RATE itself.
    ee = []
    enc = lambda quals: "".join(chr(q + 33) for q in quals)  # noqa: E731
    for quals in [[], [10], [20], [30], [10, 10], [10, 20], [20, 10], [10, 10, 10], [10, 20, 30], [10, 10, 20, 30, 40]]:
        ee.append([enc(quals), 33, expected_errors(enc(quals)).hex()])          # tests/test_qualtrim.py:65-82
    for q in range(94):
        ee.append([chr(33 + q), 33, expected_errors(chr(33 + q)).hex()])
    for _ in range(1500):
        n = rng.randint(0, 200)
        base = rng.choice([33, 33, 64])
        qual = "".join(chr(base + rng.choice([2, 2, 10, 15, 20, 25, 30, 37, 41, rng.randint(0, 126 - base)])) for _ in range(n))
        ee.append([qual, base, expected_errors(qual, base).hex()])
    dump("trim_scans_kat.json.gz", {"nextseq": nextseq, "polya": polya, "expected_errors": ee})


def match_desc(m):
    if m is None:
        return None
    if hasattr(m, "front_match"):
        return ["Linked", match_desc(m.front_match), match_desc(m.back_match)]
    return [type(m).__name__, m.astart, m.astop, m.rstart, m.rstop, m.score, m.errors]


def adapters_kat():
    rng = random.Random(1005)
    out = []

    def make(alpha):
        t = rng.choice(TYPES)
        seq = rnd(rng, alpha, rng.randint(3, 34))
        if set(seq) <= {"N"}:
            seq = "A" + seq
        kw = dict(max_errors=rng.choice([0, 0.1, 0.1, 0.15, 0.2, 0.3, 1, 2]), min_overlap=rng.randint(1, 6),
                  read_wildcards=rng.random() < 0.2, adapter_wildcards=rng.random() < 0.7,
                  indels=rng.random() < 0.8)
        if t in ("FrontAdapter", "BackAdapter", "RightmostFrontAdapter", "RightmostBackAdapter") and rng.random() < 0.2:
            kw["force_anywhere"] = True
        return t, seq, kw

    for _ in range(260):
        alpha = rng.choice(["ACGT", "ACGT", "ACGTN", "ACGTacgtn"])
        adalpha = rng.choice(["ACGT", "ACGT", "ACGTN", "ACGTRYN"])
        specs, objs, ad_seqs = [], [], []
        for _ in range(rng.choice([1, 1, 2, 3, 5])):
            if rng.random() < 0.2:
                while True:
                    t1, s1, k1 = make(adalpha)
                    if t1 in ("FrontAdapter", "NonInternalFrontAdapter", "PrefixAdapter"):
                        break
                while True:
                    t2, s2, k2 = make(adalpha)
                    if t2 in ("BackAdapter", "NonInternalBackAdapter", "SuffixAdapter"):
                        break
                fq, bq = rng.random() < 0.5, rng.random() < 0.5
                specs.append(["Linked", [t1, s1, k1], [t2, s2, k2], fq, bq])
                objs.append(RA.LinkedAdapter(getattr(RA, t1)(s1, name="f", **k1), getattr(RA, t2)(s2, name="b", **k2), fq, bq, "lnk"))
                ad_seqs += [s1, s2]
            else:
                t, s, k = make(adalpha)
                specs.append([t, s, k])
                objs.append(getattr(RA, t)(s, name="x", **k))
                ad_seqs.append(s)
        multi = RA.MultipleAdapters(objs)
        reads = []
        for _ in range(16):
            q = rnd(rng, alpha, rng.randint(0, 80))
            for _ in range(rng.choice([0, 1, 1, 2])):
                ad = rng.choice(ad_seqs)
                piece = ad if rng.random() < 0.6 else ad[rng.randint(0, len(ad) // 2) : rng.randint(len(ad) // 2, len(ad))]
                piece = "".join(c if c in "ACGT" else rng.choice("ACGT") for c in piece)
                piece = mutate(rng, piece, alpha, rng.choice([0, 0, 1, 2]))
                pos = rng.choice([0, len(q), rng.randint(0, len(q))])
                q = q[:pos] + piece + q[pos:]
            reads.append([q, match_desc(multi.match_to(q))])
        out.append({"adapters": specs, "reads": reads})
    dump("adapters_kat.json.gz", out)


def index_kat():
    """AdapterIndex / IndexedPrefixAdapters / IndexedSuffixAdapters (adapters.py:1289-1571)."""
    rng = random.Random(1013)
    out = []
    while len(out) < 120:
        prefix = rng.random() < 0.5
        cls = "PrefixAdapter" if prefix else "SuffixAdapter"
        members = []
        for _ in range(rng.choice([1, 2, 3, 5, 8])):
            seq = rnd(rng, "ACGT", rng.randint(4, 22))
            kw = dict(max_errors=rng.choice([0, 0.1, 0.15, 0.2, 1, 2]), indels=rng.random() < 0.6,
                      min_overlap=rng.choice([1, 3, len(seq)]))
            members.append([seq, kw])
        objs = [getattr(RA, cls)(s, name="x", **k) for s, k in members]
        if not all(RA.AdapterIndex.is_acceptable(a, prefix) for a in objs):
            continue
        if any(int(len(s) * a.max_error_rate) >= len(s) for (s, _), a in zip(members, objs)):
            continue
        indexed = (RA.IndexedPrefixAdapters if prefix else RA.IndexedSuffixAdapters)(objs)
        specs = [["Indexed", prefix, members]]
        parts = [indexed]
        if rng.random() < 0.4:
            extra = [rng.choice(["BackAdapter", "FrontAdapter"]), rnd(rng, "ACGT", 12), dict(max_errors=0.1)]
            specs.insert(rng.choice([0, 1]), extra)
            obj = getattr(RA, extra[0])(extra[1], name="x", **extra[2])
            parts = [obj, indexed] if specs[0] is extra else [indexed, obj]
        multi = RA.MultipleAdapters(parts)
        reads = []
        for _ in range(40):
            body = rnd(rng, "ACGT", rng.randint(0, 40))
            ad = mutate(rng, rng.choice(members)[0], "ACGTN", rng.choice([0, 0, 1, 1, 2, 3]))
            r = rng.random()
            if r < 0.1:
                q = body
            elif r < 0.2:
                q = ad[: rng.randint(0, len(ad))] if prefix else ad[rng.randint(0, len(ad)):]
            else:
                q = ad + body if prefix else body + ad
            if rng.random() < 0.1:
                q = q.lower()
            if q and rng.random() < 0.05:
                pos = rng.randrange(len(q))
                q = q[:pos] + rng.choice("RYXn") + q[pos + 1:]
            reads.append([q, match_desc(multi.match_to(q))])
        ix = indexed._index
        out.append({"adapters": specs, "reads": reads, "n_keys": len(ix._index),
                    "lengths": list(ix._lengths), "ambiguous": ix._ambiguous})
    dump("index_kat.json.gz", out)


def info_file_kat():
    """Per-read coordinates pinned by the reference's golden files tests/cut/*.info.txt."""
    out = {}
    # test_info_file.py:14-32: -a adapt=GCCGAACTTCTTAGACTGCCTTAAGGACGT on illumina.fastq.gz
    with gzip.open(os.path.join(REF_TESTS, "data", "illumina.fastq.gz"), "rt") as f:
        lines = f.read().split("\n")
    reads = {lines[i][1:]: (lines[i + 1], lines[i + 3]) for i in range(0, len(lines) - 3, 4)}
    rows = []
    with open(os.path.join(REF_TESTS, "cut", "illumina.info.txt")) as f:
        for line in f:
            cols = line.rstrip("\n").split("\t")
            name = cols[0]
            seq = reads[name][0]
            if cols[1] == "-1":
                rows.append([seq, None])
            else:
                rows.append([seq, [int(cols[1]), int(cols[2]), int(cols[3])]])
    out["illumina"] = {"adapter": "GCCGAACTTCTTAGACTGCCTTAAGGACGT", "rows": rows}
    # test_info_file.py:35-55: --times 2 -a adapt=GCCGAACTTCTTA -a adapt2=GACTGCCTTAAGGACGT on illumina5.fastq
    with open(os.path.join(REF_TESTS, "data", "illumina5.fastq")) as f:
        lines = f.read().split("\n")
    reads = {lines[i][1:]: lines[i + 1] for i in range(0, len(lines) - 3, 4)}
    per_read = {}
    order = []
    with open(os.path.join(REF_TESTS, "cut", "illumina5.info.txt")) as f:
        for line in f:
            cols = line.rstrip("\n").split("\t")
            name = cols[0]
            if name not in per_read:
                per_read[name] = []
                order.append(name)
            if cols[1] != "-1":
                per_read[name].append([int(cols[1]), int(cols[2]), int(cols[3]), cols[7]])
    out["illumina5"] = {
        "adapters": [["adapt", "GCCGAACTTCTTA"], ["adapt2", "GACTGCCTTAAGGACGT"]],
        "rows": [[reads[name], per_read[name]] for name in order],
    }
    dump("info_file_kat.json.gz", out)


def env_kat():
    rng = random.Random(1006)
    out = []
    for _ in range(40):
        t = rnd(rng, "ACGT", rng.randint(1, 8))
        k = rng.randint(0, 2)
        out.append([t, k, sorted(map(list, edit_environment(t, k))), sorted(map(list, hamming_environment(t, k)))])
    dump("environment_kat.json.gz", out)


def dp_debug_kat():
    """Aligner.enable_debug(): the printed cost and score matrices of the reference for a few searches."""
    rng = random.Random(77)
    out = []
    for trial in range(40):
        ref = rnd(rng, rng.choice(["ACGT", "ACGTN"]), rng.randint(3, 14))
        q = mutate(rng, ref, "ACGT", rng.choice([0, 1, 2]))
        q = rnd(rng, "ACGT", rng.randint(0, 8)) + q + rnd(rng, "ACGT", rng.randint(0, 8))
        rate = rng.choice([0.1, 0.2, 0.3])
        flags = rng.choice([14, 11, 15, 8, 2, 0])
        wr = "N" in ref and rng.random() < 0.7
        mo = rng.randint(1, 3)
        try:
            al = Aligner(ref, rate, flags, wr, False, 1, mo)
        except ValueError:
            continue
        al.enable_debug()
        res = al.locate(q)
        out.append([ref, q, rate, flags, wr, mo, list(res) if res else None, str(al.dpmatrix), str(al.scorematrix)])
    dump("dp_debug_kat.json.gz", out)


def tables():
    import base64

    enc = lambda b: base64.b64encode(b).decode()  # noqa: E731
    out = {"acgt": enc(RT._acgt_table()), "iupac": enc(RT._iupac_table()), "upper": enc(RT._upper_table())}
    for rw in (0, 1):
        for qw in (0, 1):
            out[f"lookup_{rw}{qw}"] = [enc(x) for x in RT.matches_lookup(bool(rw), bool(qw))]
    dump("tables.json.gz", out)


# ---- the reference's answers for the tests that compared with the reference itself ----------------------------------

GATE_READS = 100_000      # reads compared with the reference per configuration in tests/test_gpu_gate.py
GATE_SAMPLE = 10_000      # of which the answers are stored; the rest are pinned by a digest


def reference_suite_kat():
    """Every call the reference's own tests/test_kmer_heuristic.py makes into cutadapt.kmer_heuristic, with the
    reference's result, per test (replayed against this package by tests/test_reference_suite.py)."""
    import pytest
    from cutadapt import kmer_heuristic as KH

    tests, current, depth = [], [None], [0]

    def recorded(name, fn):
        def call(*args, **kwargs):
            depth[0] += 1
            try:
                result = fn(*args, **kwargs)
            finally:
                depth[0] -= 1
            if depth[0] == 0 and current[0] is not None:
                current[0]["calls"].append([name, list(args), kwargs, canon(result)])
            return result
        return call

    for name in ("kmer_chunks", "minimize_kmer_search_list", "create_back_overlap_searchsets", "create_positions_and_kmers"):
        setattr(KH, name, recorded(name, getattr(KH, name)))

    class Recorder:
        @pytest.hookimpl(hookwrapper=True)
        def pytest_runtest_call(self, item):
            mark = item.get_closest_marker("timeout")
            current[0] = {"test": item.name, "timeout": mark.args[0] if mark else None, "calls": []}
            yield
            tests.append(current[0])
            current[0] = None

    path = os.path.join(REF_TESTS, "test_kmer_heuristic.py")
    assert pytest.main([path, "-q", "--noconftest", "-p", "no:cacheprovider"], plugins=[Recorder()]) == 0
    assert all(t["calls"] for t in tests)
    dump("reference_suite_kat.json.gz", {"test_kmer_heuristic.py": tests})


def reference_random_kat():
    """Aligner.locate and quality_trim_index of the reference on tests/util.py's random_locate_cases()."""
    answers = []
    cases = list(random_locate_cases())
    for ref, rate, flags, wr, wq, ic, mo, queries, qs in cases:
        al = Aligner(ref, rate, flags, wr, wq, ic, mo)
        locs = [al.locate(q) for q in queries]
        answers.append([[list(r) if r else None for r in locs], list(quality_trim_index(qs, 5, 20))])
    dump("reference_random_kat.json.gz", {"cases_digest": digest(cases), "answers": answers})


def _index_rows(idx, reads):
    rows = []
    for r in reads:
        m = idx.match_to(r)
        rows.append(None if m is None else [int(m.adapter.name[2:]), m.astart, m.astop, m.rstart, m.rstop, m.score, m.errors])
    return rows


def index_reference_kat():
    """IndexedPrefixAdapters of the 96 barcodes of configuration 5, with and without indels: the keys of its index and
    its matches on 3000 reads of the configuration (every 50th with an N in the barcode)."""
    from cutadapt_b200.configs import config5_barcodes, make_config_batch, to_strings

    bcs = config5_barcodes()
    b = make_config_batch(5, 3000, seed=77)
    b["seq"][::50, 3] = ord("N")
    out = {"reads_digest": batch_digest(b)}
    for key, indels in (("indels", True), ("hamming", False)):
        idx = RA.IndexedPrefixAdapters([RA.PrefixAdapter(s, max_errors=0.1, indels=indels, name=f"bc{i}")
                                        for i, s in enumerate(bcs)])
        out[key] = {"keys": sorted(idx._index._index), "lengths": list(idx._index._lengths),
                    "rows": _index_rows(idx, to_strings(b["seq"]))}
    dump("index_reference_kat.json.gz", out)


def gate_reference_kat():
    """The reference's matches on the first GATE_READS reads (configuration 4: GATE_READS / 2 pairs) of each benchmark
    configuration, drawn on the CPU: the first GATE_SAMPLE answers and the digest of all of them."""
    from cutadapt.qualtrim import quality_trim_index as qtrim
    from cutadapt_b200 import configs as CF

    def coords(m):
        return None if m is None else [m.astart, m.astop, m.rstart, m.rstop, m.score, m.errors]

    def entry(rows):
        return {"digest": digest(rows), "sample": rows[:GATE_SAMPLE]}

    out = {}
    for cfg in (2, 3, 4, 5):
        e = CF.CONFIG_ERROR_RATE[cfg]
        b = CF.make_config_batch(cfg, GATE_READS // 2 if cfg == 4 else GATE_READS, device="cpu")
        reads = CF.to_strings(b["seq"])
        res = {"n": len(reads), "reads_digest": batch_digest(b)}
        if cfg == 2:
            ra = RA.BackAdapter(CF.CONFIG2_ADAPTER, max_errors=e, min_overlap=3, name="adapter")
            res["seq"] = entry([coords(ra.match_to(r)) for r in reads])
        elif cfg == 3:
            objs = [RA.BackAdapter(s, max_errors=e, min_overlap=3, name=f"a{i}") for i, s in enumerate(CF.CONFIG3_BACK)]
            objs.append(RA.LinkedAdapter(RA.PrefixAdapter(CF.CONFIG3_LINKED[0], max_errors=e, min_overlap=3, name="lf"),
                                         RA.BackAdapter(CF.CONFIG3_LINKED[1], max_errors=e, min_overlap=3, name="lb"),
                                         True, False, "linked"))
            rmulti = RA.MultipleAdapters(objs)
            res["seq"] = entry([match_desc(rmulti.match_to(r)) for r in reads])
        elif cfg == 4:
            for skey, qkey, adapter in (("seq", "qual", CF.CONFIG4_R1), ("seq2", "qual2", CF.CONFIG4_R2)):
                ra = RA.BackAdapter(adapter, max_errors=e, min_overlap=3, name="x")
                rows = []
                for r, q in zip(CF.to_strings(b[skey]), CF.to_strings(b[qkey])):
                    s, t = qtrim(q, 0, 20, 33)
                    rows.append([s, t, coords(ra.match_to(r[s:t]))])
                res[skey] = entry(rows)
        else:
            idx = RA.IndexedPrefixAdapters([RA.PrefixAdapter(s, max_errors=e, min_overlap=3, indels=True, name=f"bc{i}")
                                            for i, s in enumerate(CF.config5_barcodes())])
            res["seq"] = entry(_index_rows(idx, reads))
        out[str(cfg)] = res
    dump("gate_reference_kat.json.gz", out)


def parity_reference_kat():
    """BackAdapter AGATCGGAAGAGC (e = 0.1) of the reference on the first 3000 reads of make_reads(10000, config=1)
    (tests/test_gpu_parity.py)."""
    from cutadapt_b200.synth import make_reads

    reads = make_reads(10000, config=1)[0][:3000]
    ra = RA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a")
    rows = []
    for read in reads:
        m = ra.match_to(read)
        rows.append(None if m is None else [m.astart, m.astop, m.rstart, m.rstop, m.score, m.errors])
    dump("parity_reference_kat.json.gz", {"reads_digest": digest(reads), "rows": rows})


def statistics_reference_kat():
    """The reference's AdapterStatistics fed with its own matches on the reads of tests/_dist_worker.workload()
    (the four adapters built there): per adapter and end, errors as [length, errors, count] and adjacent_bases."""
    from _dist_worker import workload

    reads, _ = workload()
    robjs = [RA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a"), RA.FrontAdapter("ACGTTGCATTGAC", max_errors=0.1, name="f"),
             RA.AnywhereAdapter("CTGTCTCTTATACACATCT", max_errors=0.1, name="w"),
             RA.LinkedAdapter(RA.PrefixAdapter("GTTCAGAGTTCTACAGTCCGACGATC", max_errors=0.1, name="lf"),
                              RA.BackAdapter("TGGAATTCTCGGGTGCCAAGG", max_errors=0.1, name="lb"), False, False, "linked")]
    rmulti = RA.MultipleAdapters(robjs)
    rstats = {id(a): a.create_statistics() for a in robjs}
    for read in reads:
        m = rmulti.match_to(read)
        if m is not None:
            rstats[id(m.adapter)].add_match(m)
    adapters = []
    for a in robjs:
        ends = []
        for end in rstats[id(a)].end_statistics():
            ends.append(None if end is None else {
                "errors": sorted([length, e, n] for length, d in end.errors.items() for e, n in d.items()),
                "adjacent_bases": sorted([base, n] for base, n in end.adjacent_bases.items())})
        adapters.append(ends)
    dump("statistics_reference_kat.json.gz", {"reads_digest": digest(reads), "adapters": adapters})


FIXTURES = [locate_kat, comparer_kat, kmer_kat, qualtrim_kat, trim_scans_kat, adapters_kat, index_kat, info_file_kat,
            env_kat, dp_debug_kat, tables, reference_suite_kat, reference_random_kat, index_reference_kat,
            gate_reference_kat, parity_reference_kat, statistics_reference_kat]


if __name__ == "__main__":
    wanted = sys.argv[1:]
    for fn in FIXTURES:
        if not wanted or fn.__name__ in wanted:
            fn()
