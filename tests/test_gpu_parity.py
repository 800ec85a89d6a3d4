"""
GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the oracle, the
committed golden vectors and -- at benchmark-like sizes -- size-independent properties.
Integer/byte/index work: the bar is bit-exact equality.
"""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from cutadapt_b200 import _lib as L  # noqa: E402
from oracle import oracle  # noqa: E402
from util import digest, golden, build_adapters, match_desc, random_reads  # noqa: E402

FIELDS = ("astart", "astop", "rstart", "rstop", "score", "errors")


def rec_tuple(r):
    return None if r["adapter"] < 0 else [int(r[f]) for f in FIELDS]


def run_set(adapters, groups, reads, quals=None, **kw):
    spec = L.AdapterSetSpec(adapters, groups)
    aset = L.AdapterSet(spec)
    data, offsets = L.pack_strings(reads)
    qd = L.pack_strings(quals)[0] if quals is not None else None
    return aset.process(data, offsets, qd, L.make_params(**kw))


# ---- the three native functions through their reference-shaped Python API --------------------


def test_aligner_locate_golden():
    from cutadapt_b200._align import Aligner

    cases = golden("locate_kat.json.gz")
    # group by aligner parameters so that each adapter set is uploaded once
    by_params = {}
    for ref, q, rate, flags, wr, wq, ic, mo, expected in cases:
        by_params.setdefault((ref, rate, flags, wr, wq, ic, mo), []).append((q, expected))
    for (ref, rate, flags, wr, wq, ic, mo), items in by_params.items():
        al = Aligner(ref, rate, flags, wr, wq, ic, mo)
        got = al.locate_batch([q for q, _ in items])
        for (q, expected), g in zip(items, got):
            assert (list(g) if g is not None else None) == expected, (ref, q, rate, flags, wr, wq, ic, mo)


def test_aligner_debug_matrices_golden():
    """Aligner.enable_debug() / .dpmatrix / .scorematrix through cg_locate_debug, against the reference's printouts."""
    from cutadapt_b200._align import Aligner

    for ref, q, rate, flags, wr, mo, expected, dp_text, score_text in golden("dp_debug_kat.json.gz"):
        al = Aligner(ref, rate, flags, wr, False, 1, mo)
        plain = al.locate(q)
        assert al.dpmatrix is None
        al.enable_debug()
        res = al.locate(q)
        assert (list(res) if res else None) == expected == (list(plain) if plain else None)
        assert str(al.dpmatrix) == dp_text and str(al.scorematrix) == score_text, (ref, q, flags)


def test_reference_known_answer_tests():
    """tests/test_align.py:69-146 of the reference, verbatim expectations."""
    from cutadapt_b200._align import Aligner
    from cutadapt_b200.adapters import Where

    assert Aligner("", 0, flags=0, min_overlap=0).locate("") == (0, 0, 0, 0, 0, 0)
    assert Aligner("CCAGTCCTCT", 0.3, flags=Where.PREFIX).locate("CCAGTCCTTTCCTGAGAGT") == (0, 10, 0, 10, 8, 1)
    assert Aligner("TCGATC", 1.5 / 6, flags=Where.PREFIX).locate("TCGATGC") == (0, 6, 0, 6, 4, 1)
    assert Aligner("GCCGAACTTCTTAGACTGCCTTAAGGACGT", 0.1, flags=Where.BACK).locate(
        "CAAATCACCAGAAGGCGCCTAACTTCTTAGACTGCC") == (0, 20, 16, 36, 18, 1)
    assert Aligner("TTTT", 0.25, flags=Where.BACK).locate("CCTTTT") == (0, 4, 2, 6, 4, 0)
    assert Aligner("TTTTTT", 0.25, flags=Where.BACK).locate("CCTTTT") == (0, 4, 2, 6, 4, 0)
    assert Aligner("TTT", 1 / 3, flags=Where.BACK).locate("CCTTTT")[:4] == (0, 3, 2, 5)
    assert Aligner("CTGAATT", 0.1, flags=Where.BACK).locate("AAAAAAA") is None
    with pytest.raises(ValueError):
        Aligner("ACGT", 0.1).locate("AC\xe4GT")


def test_comparers_golden():
    from cutadapt_b200._align import PrefixComparer, SuffixComparer

    for ref, q, rate, wr, wq, mo, p, s in golden("comparer_kat.json.gz"):
        got = PrefixComparer(ref, rate, wr, wq, mo).locate(q)
        assert (list(got) if got else None) == p, ("prefix", ref, q)
        got = SuffixComparer(ref, rate, wr, wq, mo).locate(q)
        assert (list(got) if got else None) == s, ("suffix", ref, q)


def test_kmer_finder_golden():
    from cutadapt_b200._kmer_finder import KmerFinder

    for sets, rw, qw, reads in golden("kmer_kat.json.gz")["present"]:
        kf = KmerFinder([(s, e, k) for s, e, k in sets], rw, qw)
        got = kf.kmers_present_batch([r for r, _ in reads])
        assert list(map(bool, got)) == [e for _, e in reads], (sets, rw, qw)
    kf = KmerFinder([(0, None, ["ACGT"])])
    assert kf.kmers_present("ttacgttt") is True and kf.kmers_present("ttacttt") is False
    with pytest.raises(ValueError):
        kf.kmers_present("AC\xe4GT")


def test_quality_trim_golden():
    from cutadapt_b200.qualtrim import quality_trim_index, quality_trim_index_batch, HasNoQualities

    cases = golden("qualtrim_kat.json.gz")
    by = {}
    for q, cf, cb, base, expected in cases:
        by.setdefault((cf, cb, base), []).append((q, expected))
    for (cf, cb, base), items in by.items():
        got = quality_trim_index_batch([q for q, _ in items], cf, cb, base)
        assert got.tolist() == [e for _, e in items]
    assert quality_trim_index("IIII####", 0, 20) == (0, 4)
    with pytest.raises(HasNoQualities):
        quality_trim_index(None, 0, 20)


def test_trim_scans_golden():
    """nextseq_trim_index / poly_a_trim_index on the device == the reference (incl. its own KATs)."""
    from types import SimpleNamespace
    from cutadapt_b200 import qualtrim as Q

    g = golden("trim_scans_kat.json.gz")
    by_param = {}
    for seq, qual, cutoff, base, expected in g["nextseq"]:
        by_param.setdefault((cutoff, base), []).append((seq, qual, expected))
    for (cutoff, base), rows in by_param.items():
        got = Q.nextseq_trim_index_batch([r[0] for r in rows], [r[1] for r in rows], cutoff, base)
        assert got.tolist() == [r[2] for r in rows]
    s = SimpleNamespace(sequence="TCTCGTATGCCGTCTTATGCTTGAAAAAAAAAAGGGGGGGGGGGGGGGGGNNNNNNNNNNNGGNGG",
                        qualities="AA//EAEE//A6///E//A//EA/EEEEEEAEA//EEEEEEEEEEEEEEE###########EE#EA")
    assert Q.nextseq_trim_index(s, cutoff=22) == 33          # tests/test_qualtrim.py:10-15
    with pytest.raises(Q.HasNoQualities):
        Q.nextseq_trim_index(SimpleNamespace(sequence="ACGT", qualities=None), 20)
    for rc in (False, True):
        rows = [(seq, e) for seq, r, e in g["polya"] if bool(r) == rc]
        got = Q.poly_a_trim_index_batch([r[0] for r in rows], rc)
        assert got.tolist() == [r[1] for r in rows]
    assert Q.poly_a_trim_index("TTTAG" + "AAA") == 5 and Q.poly_a_trim_index("TTT" + "GTCCC", revcomp=True) == 3
    # expected_errors: FP64 with the reference's summation order -> bit-identical doubles
    for base in (33, 64):
        rows = [(q, e) for q, b, e in g["expected_errors"] if b == base]
        got = Q.expected_errors_batch([r[0] for r in rows], base)
        assert [float(x).hex() for x in got] == [r[1] for r in rows]
    assert Q.expected_errors("5") == pytest.approx(0.01)        # tests/test_qualtrim.py:72
    with pytest.raises(ValueError):
        Q.expected_errors("II I")                               # ' ' is below base 33


# ---- adapter classes ------------------------------------------------------------------------


def test_adapter_classes_golden():
    """Every adapter type, linked and multiple adapters: reference match_to() results."""
    import cutadapt_b200.adapters as PA

    for case in golden("adapters_kat.json.gz"):
        multi = build_adapters(PA, case["adapters"])
        reads = [r for r, _ in case["reads"]]
        got = multi.match_to_batch(reads)
        for (read, expected), m in zip(case["reads"], got):
            assert match_desc(m) == expected, (case["adapters"], read)


def test_indexed_adapters_golden():
    """IndexedPrefixAdapters / IndexedSuffixAdapters: reference AdapterIndex.match_to() results."""
    import cutadapt_b200.adapters as PA

    for case in golden("index_kat.json.gz"):
        multi = build_adapters(PA, case["adapters"])
        reads = [r for r, _ in case["reads"]]
        got = multi.match_to_batch(reads)
        for (read, expected), m in zip(case["reads"], got):
            assert match_desc(m) == expected, (case["adapters"], read)


def test_config5_demultiplex_96_anchored_barcodes():
    """BASELINE config 5 shape: 96 anchored 5' barcodes through the device index == the same
    adapters evaluated one by one (MultipleAdapters semantics, adapters.py:1265-1286) whenever
    the best hit is unique; every index hit is a true within-k barcode occurrence."""
    import cutadapt_b200.adapters as PA

    rng = random.Random(96)
    barcodes = set()
    while len(barcodes) < 96:
        barcodes.add("".join(rng.choice("ACGT") for _ in range(10)))
    barcodes = sorted(barcodes)
    pre = [PA.PrefixAdapter(b, max_errors=1, indels=False, name=f"bc{i}") for i, b in enumerate(barcodes)]
    indexed = PA.IndexedPrefixAdapters(pre)
    plain = PA.MultipleAdapters(pre)
    reads = []
    for _ in range(20000):
        bc = list(rng.choice(barcodes))
        if rng.random() < 0.3:
            bc[rng.randrange(10)] = rng.choice("ACGTN")
        if rng.random() < 0.1:
            bc = [rng.choice("ACGT") for _ in range(10)]
        reads.append("".join(bc) + "".join(rng.choice("ACGT") for _ in range(140)))
    got = indexed.match_to_batch(reads)
    ref = plain.match_to_batch(reads)
    n_hit = 0
    for read, g, r in zip(reads, got, ref):
        has_n = "N" in read[:10]
        if g is None:
            # either nothing matches or the key was ambiguous between two barcodes (an N is looked
            # up as A, adapters.py:1535-1551, which can make the looked-up key ambiguous or absent)
            if r is not None and not has_n:
                same = [b for b in barcodes if sum(x != y for x, y in zip(b, read[:10])) == r.errors]
                assert len(same) > 1
            continue
        n_hit += 1
        assert r is not None
        assert (g.rstart, g.rstop) == (0, 10)
        assert g.errors >= r.errors if has_n else g.errors == r.errors
        assert sum(x != y for x, y in zip(g.adapter.sequence, read[:10])) == g.errors
    assert n_hit > 15000
    # ... and the index path equals the oracle's own index (built from the oracle's Hamming spheres), record by record
    data = np.frombuffer("".join(reads).encode(), dtype=np.uint8)
    offsets = np.arange(len(reads) + 1, dtype=np.int64) * 150
    exp = oracle.oracle_index_process(barcodes, 0.1, False, True, data, offsets, [a.descriptor() for a in pre])
    for i, g in enumerate(got):
        if g is None:
            assert exp["adapter"][i] < 0, i
        else:
            e = exp[i]
            assert (barcodes.index(g.adapter.sequence), g.astart, g.astop, g.rstart, g.rstop, g.score, g.errors) == \
                (int(e["adapter"]), int(e["astart"]), int(e["astop"]), int(e["rstart"]), int(e["rstop"]), int(e["score"]),
                 int(e["errors"])), i


def test_match_objects_behave_like_the_reference():
    """tests/test_adapters.py:38-76 (leftmost rule) and Match.trimmed / statistics plumbing."""
    import cutadapt_b200.adapters as PA

    adapter = PA.BackAdapter("ACGT", max_errors=0.0, min_overlap=3, name="a")
    m = adapter.match_to("TTTACGTCCCACGT")      # two exact occurrences: the leftmost wins
    assert (m.rstart, m.rstop, m.errors) == (3, 7, 0)
    assert m.trimmed("TTTACGTCCCACGT") == "TTT" and m.adjacent_base() == "T"
    assert m.removed_sequence_length() == 11
    stats = adapter.create_statistics()
    stats.add_match(m)
    assert stats.end.errors[11][0] == 1 and stats.end.adjacent_bases["T"] == 1
    front = PA.FrontAdapter("AAAA", max_errors=0.25, name="f")
    m = front.match_to("CCAAAATCCCC")
    assert isinstance(m, PA.RemoveBeforeMatch) and m.trimmed("CCAAAATCCCC") == "TCCCC"
    assert m.removed_sequence_length() == 6
    assert PA.BackAdapter("GGGGGGGG", name="n").match_to("ACACACAC") is None
    linked = PA.LinkedAdapter(PA.PrefixAdapter("AAAA", name="p"), PA.BackAdapter("TTTT", name="b"), True, False, "lnk")
    lm = linked.match_to("AAAACCCCTTTTGG")
    assert lm.front_match.rstop == 4 and lm.back_match.rstart == 4 and lm.trimmed("AAAACCCCTTTTGG") == "CCCC"
    assert linked.match_to("CCCCAAAATTTT") is None            # required front adapter missing


def test_info_file_coordinates_of_the_reference():
    """Per-read errors/rstart/rstop of tests/cut/illumina.info.txt and illumina5.info.txt."""
    import cutadapt_b200.adapters as PA

    data = golden("info_file_kat.json.gz")
    il = data["illumina"]
    adapter = PA.BackAdapter(il["adapter"], max_errors=0.1, min_overlap=3, name="adapt")
    got = adapter.match_to_batch([s for s, _ in il["rows"]])
    for (seq, expected), m in zip(il["rows"], got):
        assert (None if m is None else [m.errors, m.rstart, m.rstop]) == expected, seq
    il5 = data["illumina5"]
    multi = PA.MultipleAdapters([PA.BackAdapter(s, max_errors=0.1, min_overlap=3, name=n) for n, s in il5["adapters"]])
    aset = multi.adapter_set()
    seqs = [s for s, _ in il5["rows"]]
    d, o = L.pack_strings(seqs)
    recs, _ = aset.process(d, o, None, L.make_params(times=2))
    for i, (seq, expected) in enumerate(il5["rows"]):
        rows = []
        cur = seq
        for r in range(2):
            m = multi.matches_from_records(recs[i, r], cur)
            if m is None:
                break
            rows.append([m.errors, m.rstart, m.rstop, m.adapter.name])
            cur = m.trimmed(cur)
        assert rows == expected, seq


# ---- the fused batch path against the oracle ---------------------------------------------------


def test_config1_10k_single_adapter_bit_exact():
    """BASELINE config 1/2 shape: 150 bp, one 3' adapter AGATCGGAAGAGC, e=0.1."""
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_reads

    reads, _ = make_reads(10000, config=1)
    adapter = PA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a")
    d = adapter.descriptor()
    got, _ = run_set([d], None, reads)
    exp, _ = oracle.oracle_process([d], None, reads)
    assert (got == exp).all()
    assert 4500 < int((got["adapter"] >= 0).sum()) < 5500
    # and the reference itself on the first 3000 reads (parity_reference_kat)
    g = golden("parity_reference_kat.json.gz")
    assert digest(reads[:3000]) == g["reads_digest"]
    for read, rec, expected in zip(reads, got[:, 0, 0], g["rows"]):
        assert rec_tuple(rec) == expected, read


def test_config3_five_adapters_iupac_linked():
    """BASELINE config 3 shape: 5 adapters incl. IUPAC wildcards, an N-run and a linked adapter, e=0.15."""
    import cutadapt_b200.adapters as PA

    rng = random.Random(3)
    seqs = ["AGATCGGAAGAGC", "CTGTCTCTTATACACATCT", "VCCGAMCYUCKHRKDCUBBCNUWNSGHCGU",
            "AGATCGGAAGAGCNNNNNNNNATCTCGTATGCC"]
    objs = [PA.BackAdapter(s, max_errors=0.15, name=f"a{i}") for i, s in enumerate(seqs)]
    objs.append(PA.LinkedAdapter(PA.PrefixAdapter("GTTCAGAGTTCTACAGTCCGACGATC", max_errors=0.15, name="f"),
                                 PA.BackAdapter("TGGAATTCTCGGGTGCCAAGG", max_errors=0.15, name="b"),
                                 True, False, "linked"))
    multi = PA.MultipleAdapters(objs)
    reads = random_reads(rng, seqs + ["GTTCAGAGTTCTACAGTCCGACGATC", "TGGAATTCTCGGGTGCCAAGG"], 6000, "ACGT", 150)
    reads += random_reads(rng, seqs, 500, "ACGTN", 150)
    singles, groups, _ = multi._flatten()
    descs = [s.descriptor() for s in singles]
    got, _ = run_set(descs, groups, reads)
    exp, _ = oracle.oracle_process(descs, groups, reads)
    assert (got == exp).all()
    assert int((got["adapter"][:, 0, :] >= 0).any(axis=1).sum()) > 1000


def test_config4_quality_trim_then_adapter():
    """BASELINE config 4 shape: -q 20 fused in front of a 33-mer 3' adapter; qualities staged too."""
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_reads

    ad = "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA"
    reads, quals = make_reads(8000, config=4, with_qualities=True, adapter=ad)
    d = PA.BackAdapter(ad, max_errors=0.1, name="a").descriptor()
    got, qt = run_set([d], None, reads, quals, quality_trim=True, cutoff_front=0, cutoff_back=20)
    exp, eqt = oracle.oracle_process([d], None, reads, quals, quality_trim=True, cutoff_back=20)
    assert (qt == eqt).all() and (got == exp).all()
    assert int((qt[:, 1] < 150).sum()) > 500


def test_fused_nextseq_trim_then_quality_trim_then_adapter():
    """--nextseq-trim fused in front of -q and the adapter search (cli.py:940-953 order)."""
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_reads

    ad = "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA"
    reads, quals = make_reads(6000, config=4, with_qualities=True, adapter=ad)
    rng = random.Random(4)
    reads = [r[:-t] + "G" * t if (t := rng.choice([0, 0, 5, 20])) else r for r in reads]   # dark cycles
    for descs, groups in (([PA.BackAdapter(ad, max_errors=0.1, name="a").descriptor()], None),
                          ([PA.BackAdapter(ad, max_errors=0.1, name="a").descriptor(),
                            PA.BackAdapter("CTGTCTCTTATACACATCT", max_errors=0.1, name="b").descriptor()], None)):
        for qt in (False, True):
            got, gqt = run_set(descs, groups, reads, quals, quality_trim=qt, cutoff_front=0, cutoff_back=20, nextseq_cutoff=20)
            exp, eqt = oracle.oracle_process(descs, groups, reads, quals, quality_trim=qt, cutoff_back=20, nextseq_cutoff=20)
            assert (gqt == eqt).all() and (got == exp).all(), (len(descs), qt)
            assert int((gqt[:, 1] < 150).sum()) > 1500


def test_random_adapter_sets_against_oracle():
    """All adapter types, wildcards, --no-indels (wide cells), rounds, quality trimming."""
    import cutadapt_b200.adapters as PA
    from util import spec_of

    rng = random.Random(11)
    types = ["FrontAdapter", "RightmostFrontAdapter", "BackAdapter", "RightmostBackAdapter", "AnywhereAdapter",
             "NonInternalFrontAdapter", "NonInternalBackAdapter", "PrefixAdapter", "SuffixAdapter"]
    for trial in range(40):
        ads, objs = [], []
        for _ in range(rng.choice([1, 2, 3])):
            seq = "".join(rng.choice("ACGT" if rng.random() < 0.7 else "ACGTNRY") for _ in range(rng.randint(4, 30)))
            if set(seq) <= {"N"}:
                seq = "A" + seq
            kw = dict(max_errors=rng.choice([0, 0.1, 0.15, 0.2, 0.3]), min_overlap=rng.randint(1, 5),
                      read_wildcards=rng.random() < 0.2, indels=rng.random() < 0.8)
            objs.append(getattr(PA, rng.choice(types))(seq, name="x", **kw))
            ads.append(seq)
        multi = PA.MultipleAdapters(objs)
        spec = spec_of(multi)
        reads = random_reads(rng, ads, 300, rng.choice(["ACGT", "ACGTN", "ACGTacgtn"]), 120)
        quals = ["".join(chr(33 + rng.choice([2, 2, 15, 30, 38])) for _ in r) for r in reads]
        times = rng.choice([1, 2])
        qtrim = rng.random() < 0.5
        got, qt = run_set(spec.adapters, spec.groups, reads, quals if qtrim else None, quality_trim=qtrim,
                          cutoff_front=5, cutoff_back=20, times=times)
        exp, eqt = oracle.oracle_process(spec.adapters, spec.groups, reads, quals, qtrim, 5, 20, 33, times)
        assert (got == exp).all(), [repr(o) for o in objs]
        if qtrim:
            assert (qt == eqt).all()


def test_edge_cases_empty_ragged_long():
    import cutadapt_b200.adapters as PA

    d = PA.BackAdapter("AGATCGGAAGAGC", name="a").descriptor()
    reads = ["", "A", "AGA", "AGATCGGAAGAGC", "", "T" * 300 + "AGATCGGAAGAGC", "ACGT" * 50, "", "AGAT"]
    got, _ = run_set([d], None, reads)
    exp, _ = oracle.oracle_process([d], None, reads)
    assert (got == exp).all()
    # only empty reads: nothing to stage at all
    got, _ = run_set([d], None, ["", "", ""])
    assert (got["adapter"] == -1).all()
    # a single read / exactly one tile / one more than a tile
    for n in (1, 128, 129, 257):
        reads = ["ACGTACGTAGATCGGAAGAGCAAAA"] * n
        got, _ = run_set([d], None, reads)
        assert (got["rstart"][:, 0, 0] == 8).all() and (got["errors"] == 0).all()
    # very long reads take the generic (wide-cell, unstaged) kernel; 40 kb > packed-cell origin range
    rng = random.Random(2)
    long_reads = ["".join(rng.choice("ACGT") for _ in range(40000)) + "AGATCGGAAGAGC" + "ACGT" * 10,
                  "".join(rng.choice("ACGT") for _ in range(5000))]
    got, _ = run_set([d], None, long_reads)
    exp, _ = oracle.oracle_process([d], None, long_reads)
    assert (got == exp).all() and got["rstart"][0, 0, 0] == 40000
    # the same ragged batches through the multi-pass schedule (two adapters + a linked adapter), plus
    # reads longer than 511 (wider scan groups) and long enough for the generic fallback of every pass
    multi = PA.MultipleAdapters([
        PA.BackAdapter("AGATCGGAAGAGC", name="a"), PA.FrontAdapter("TTGACCGATTAC", name="b"),
        PA.LinkedAdapter(PA.PrefixAdapter("ACGTACGT", name="f"), PA.BackAdapter("GGCATTCAGG", name="g"), True, False, "l")])
    singles, groups, _ = multi._flatten()
    descs = [s.descriptor() for s in singles]
    reads = ["", "A", "AGA", "AGATCGGAAGAGC", "", "T" * 300 + "AGATCGGAAGAGC", "ACGT" * 50, "", "AGAT",
             "ACGTACGT" + "C" * 700 + "GGCATTCAGG" + "A" * 30, "TTGACCGATTAC" + "G" * 1500, "N" * 40,
             "acgtacgt" + "t" * 20 + "ggcattcagg"] + long_reads
    got, _ = run_set(descs, groups, reads)
    exp, _ = oracle.oracle_process(descs, groups, reads)
    assert (got == exp).all()
    got, _ = run_set(descs, groups, ["", ""])
    assert (got["adapter"] == -1).all()


def test_non_ascii_reads_raise_like_the_reference():
    import cutadapt_b200.adapters as PA

    d = PA.BackAdapter("AGATCGGAAGAGC", name="a").descriptor()
    spec = L.AdapterSetSpec([d])
    aset = L.AdapterSet(spec)
    data = np.frombuffer(b"ACGT\xe4CGTAGATCGGAAGAGC", dtype=np.uint8)
    offsets = np.array([0, data.size], dtype=np.int64)
    with pytest.raises(ValueError):
        aset.process(data, offsets)
    # and the context is usable afterwards
    got, _ = run_set([d], None, ["ACGTAGATCGGAAGAGC"])
    assert got["rstart"][0, 0, 0] == 4
    # every schedule reports it: one-phase kernels, a comparer-only set (cooperative tile check), multi-pass
    import os
    d2 = PA.PrefixAdapter("ACGT", indels=False, name="p").descriptor()
    for descs, env in (([d], "general"), ([d], "block"), ([d2], None), ([d, d2], None)):
        if env:
            os.environ["CUTADAPT_B200_KERNEL"] = env
        try:
            with pytest.raises(ValueError):
                L.AdapterSet(L.AdapterSetSpec(descs)).process(data, offsets)
        finally:
            os.environ.pop("CUTADAPT_B200_KERNEL", None)


def test_large_batch_properties():
    """
    2 M reads (several pipeline chunks and both lanes): properties that do not need the oracle --
    idempotence (trimmed reads no longer contain a full adapter), determinism across batch
    splits, and agreement with the oracle on a strided sample.
    """
    import torch
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_read_tensor

    n = 2_000_000
    seq, _ = make_read_tensor(n, config=2, device="cuda")
    host = seq.cpu().numpy().reshape(-1)
    offsets = np.arange(n + 1, dtype=np.int64) * 150
    d = PA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a").descriptor()
    aset = L.AdapterSet(L.AdapterSetSpec([d]))
    full, _ = aset.process(host, offsets)
    # the same reads in two halves give the same records
    half = n // 2 + 77
    a, _ = aset.process(host[: half * 150], offsets[: half + 1])
    b, _ = aset.process(host[half * 150:], offsets[half:] - half * 150)
    assert (np.concatenate([a, b]) == full).all()
    # oracle on a strided sample
    idx = np.arange(0, n, 997)
    sample = [host[i * 150:(i + 1) * 150].tobytes().decode() for i in idx]
    exp, _ = oracle.oracle_process([d], None, sample)
    assert (full[idx] == exp).all()
    # idempotence: after trimming, an exact full-length adapter can no longer be found
    hit = full["adapter"][:, 0, 0] >= 0
    assert 0.45 < hit.mean() < 0.56
    rstart = np.where(hit, full["rstart"][:, 0, 0], 150)
    keep = np.arange(150)[None, :] < rstart[:200000, None]
    trimmed = np.where(keep, host[: 200000 * 150].reshape(-1, 150), ord("X")).reshape(-1)
    again, _ = aset.process(np.ascontiguousarray(trimmed), offsets[:200001])
    exact = (again["adapter"][:, 0, 0] >= 0) & (again["errors"][:, 0, 0] == 0) & (again["astop"][:, 0, 0] == 13)
    assert not exact.any()


def test_compressed_transfer_is_lossless(monkeypatch):
    """
    cg_process_batch sends large batches as a base-6 stream + exception list (cg_hostpack.h).  Records must
    equal those of the raw transfer and the oracle's, for ragged reads with lower case, IUPAC, 'N' and
    arbitrary ASCII bytes, with and without qualities; the stream must be about a third of the bytes.
    """
    import cutadapt_b200.adapters as PA

    rng = random.Random(11)
    n = 150_000
    reads, quals = [], []
    for i in range(n):
        ln = rng.choice((0, 1, 2, 3, 17, 75, 150, 150, 150, 151, 301))
        kind = i % 50
        alphabet = "ACGT" if kind < 30 else ("ACGTN" if kind < 49 else "ACGTNacgtnRYKMSWX.*-z")
        r = "".join(rng.choice(alphabet) for _ in range(ln))
        if ln > 40 and rng.random() < 0.5:
            cut = rng.randrange(10, ln - 5)
            ad = "AGATCGGAAGAGCACACGTC"
            if rng.random() < 0.02:
                ad = ad.lower()
            r = (r[:cut] + ad + r)[:ln]
        reads.append(r)
        quals.append("".join(chr(33 + rng.randrange(2, 41)) for _ in range(ln)))
    descs = [PA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a").descriptor(),
             PA.FrontAdapter("NACGTTGCA", max_errors=0.2, name="b").descriptor()]
    for dset, kw, use_q in (([descs[0]], {}, False), (descs, {"times": 2}, False),
                            ([descs[0]], {"quality_trim": True, "cutoff_back": 20}, True)):
        aset = L.AdapterSet(L.AdapterSetSpec(dset))
        data, offsets = L.pack_strings(reads)
        qd = L.pack_strings(quals)[0] if use_q else None
        aset.ctx.transfer_bytes(reset=True)
        monkeypatch.setenv("CUTADAPT_B200_H2D_PACK", "all")
        packed, qt_p = aset.process(data, offsets, qd, L.make_params(**kw))
        h2d_packed, d2h = aset.ctx.transfer_bytes(reset=True)
        monkeypatch.setenv("CUTADAPT_B200_H2D_PACK", "0")
        raw, qt_r = aset.process(data, offsets, qd, L.make_params(**kw))
        h2d_raw, _ = aset.ctx.transfer_bytes(reset=True)
        monkeypatch.setenv("CUTADAPT_B200_H2D_PACK", "1")      # adaptive split: part compressed, part raw
        for _ in range(2):
            mixed, _ = aset.process(data, offsets, qd, L.make_params(**kw))
            assert (mixed == raw).all()
        aset.ctx.transfer_bytes(reset=True)
        assert (packed == raw).all()
        if use_q:
            assert (qt_p == qt_r).all()
        assert d2h >= packed.nbytes
        if not use_q:
            assert h2d_packed < 0.6 * h2d_raw, (h2d_packed, h2d_raw)
        idx = list(range(0, n, 41))
        exp, eqt = oracle.oracle_process(dset, None, [reads[i] for i in idx],
                                         [quals[i] for i in idx] if use_q else None, **kw)
        assert (packed[idx] == exp).all()
    monkeypatch.delenv("CUTADAPT_B200_H2D_PACK")
    # an offset array that does not start at 0, with an unaligned first read
    aset = L.AdapterSet(L.AdapterSetSpec([descs[0]]))
    data, offsets = L.pack_strings(reads)
    skip = 1234
    a, _ = aset.process(data, offsets[skip:])
    b, _ = aset.process(data, offsets)
    assert (a == b[skip:]).all()


def test_device_resident_api_and_statistics():
    """cg_process_batch_device on torch tensors + the statistics vector against a numpy recount."""
    import ctypes as C
    import torch
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_read_tensor
    from cutadapt_b200.pipeline import DeviceBatch, stats_layout

    n = 300_000
    seq, qual = make_read_tensor(n, config=4, device="cuda", with_qualities=True)
    multi = PA.MultipleAdapters([PA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a")])
    batch = DeviceBatch(multi, quality_cutoff=(0, 20))
    res = batch.run(seq.reshape(-1), torch.arange(n + 1, device="cuda", dtype=torch.int64) * 150, qual.reshape(-1),
                    max_read_len=150)
    recs = res.matches.cpu().numpy().view(L.MATCH_DTYPE).reshape(n, 1, 1)
    qt = res.qtrim.cpu().numpy().reshape(n, 2)
    host = seq.cpu().numpy().reshape(-1)
    hq = qual.cpu().numpy().reshape(-1)
    offsets = np.arange(n + 1, dtype=np.int64) * 150
    exp, eqt = batch.adapter_set.process(host, offsets, hq, batch.params)
    assert (recs == exp).all() and (qt == eqt).all()
    stats = batch.statistics(res).cpu().numpy()
    lay = stats_layout(1, 150, 3)
    assert stats[0] == n and stats[1] == n * 150
    hit = recs["adapter"][:, 0, 0] >= 0
    assert stats[2] == hit.sum()
    assert stats[3] == (150 - (qt[:, 1] - qt[:, 0])).sum()
    removed = (qt[:, 1] - qt[:, 0]) - recs["rstart"][:, 0, 0]
    assert stats[4] == removed[hit].sum()
    from cutadapt_b200.pipeline import end_block, adapter_statistics_from_vector
    from util import hostsim_statistics

    adjacent, hist = end_block(stats, lay, 0, 1)           # the 3' end of the one adapter
    assert hist.sum() == hit.sum() and end_block(stats, lay, 0, 0)[1].sum() == 0
    L_, E_ = 20, 0
    assert hist[L_, E_] == ((removed == L_) & (recs["errors"][:, 0, 0] == E_) & hit).sum()
    # adjacent bases: the character in front of the match in the quality-trimmed read
    pos = qt[:, 0] + recs["rstart"][:, 0, 0] - 1
    base = np.where(hit & (recs["rstart"][:, 0, 0] > 0), host.reshape(n, 150)[np.arange(n), np.clip(pos, 0, 149)], 0)
    for k, c in enumerate(b"ACGT"):
        assert adjacent[k] == (hit & (base == c)).sum()
    assert adjacent.sum() == hit.sum()
    # read lengths after trimming
    final = np.where(hit, recs["rstart"][:, 0, 0], qt[:, 1] - qt[:, 0])
    assert (stats[lay["lengths"]:lay["lengths"] + 151] == np.bincount(final, minlength=151)).all()
    # the whole vector equals the host build of the same per-read function, and rebuilds the statistics objects
    reads = [host[i * 150:(i + 1) * 150].tobytes().decode() for i in range(20000)]
    sub = batch.statistics(batch.run(seq[:20000].reshape(-1), torch.arange(20001, device="cuda", dtype=torch.int64) * 150,
                                     qual[:20000].reshape(-1), max_read_len=150)).cpu().numpy()
    assert (sub == hostsim_statistics(reads, recs[:20000], qt[:20000], 1, 150, 3)).all()
    st = adapter_statistics_from_vector(stats, multi, 150, 3)[0]
    assert sum(st.end.lengths.values()) == hit.sum() and st.end.adjacent_bases["A"] == adjacent[0]


@pytest.mark.parametrize("jit", ["0", "1"])
def test_statistics_fused_into_the_pass_equal_the_statistics_kernel(jit, monkeypatch):
    """cg_process_batch_device_stats: the first stage counts the reads it settles, the task list supplies the rest --
    the vector must equal cg_stats_accumulate_device on the records, for 3' / 5' / anywhere adapters, with and without
    quality trimming, ragged reads, several sub-batches, interpreted and specialised first stage; sets the fused
    path does not cover (two adapters) take the kernel and give the same."""
    import torch
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_read_tensor
    from cutadapt_b200.pipeline import DeviceBatch

    monkeypatch.setenv("CUTADAPT_B200_JIT", jit)
    monkeypatch.setenv("CUTADAPT_B200_FUSED_STATS", "1")
    monkeypatch.setenv("CUTADAPT_B200_SUB_READS", "70000")
    n = 200_000
    seq, qual = make_read_tensor(n, config=4, device="cuda", with_qualities=True)
    rng = np.random.default_rng(5)
    lens = torch.from_numpy(rng.integers(0, 151, n)).cuda()
    lens[::7] = 150
    offsets = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    offsets[1:] = torch.cumsum(lens, 0)
    # ragged copy: read i = the first lens[i] characters of row i
    keep = (torch.arange(150, device="cuda")[None, :] < lens[:, None])
    rseq = torch.cat([seq[keep], torch.zeros(64, dtype=torch.uint8, device="cuda")])
    rqual = torch.cat([qual[keep], torch.zeros(64, dtype=torch.uint8, device="cuda")])
    cases = [([PA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a")], None),
             ([PA.BackAdapter("AGATCGGAAGAGCACACGTCTGAACTCCAGTCA", max_errors=0.1, name="a")], (0, 20)),
             ([PA.FrontAdapter("GATCGGAAGAGCA", max_errors=0.1, name="f")], (5, 15)),
             ([PA.AnywhereAdapter("AGATCGGAAGAGC", max_errors=0.2, name="w")], None),
             ([PA.BackAdapter("AGATCGGAAGAGC", name="a"), PA.BackAdapter("CACGTCTGAACTC", name="b")], (0, 20))]
    for ads, qc in cases:
        batch = DeviceBatch(PA.MultipleAdapters(ads), quality_cutoff=qc)
        for sq, ql, offs in ((seq.reshape(-1), qual.reshape(-1), torch.arange(n + 1, device="cuda", dtype=torch.int64) * 150),
                             (rseq, rqual, offsets)):
            res = batch.run(sq, offs, ql if qc else None, max_read_len=150)
            want = batch.statistics(res, 150, 3)
            res2, got = batch.run_with_statistics(sq, offs, ql if qc else None, max_read_len=150, max_len=150, kmax=3)
            assert torch.equal(res.matches, res2.matches)
            assert torch.equal(got, want), (ads, qc, torch.nonzero(got != want)[:5].tolist())
            # a histogram narrower than the reads: everything beyond lands in the last bin, in both paths
            want40 = batch.statistics(res, 40, 1)
            _, got40 = batch.run_with_statistics(sq, offs, ql if qc else None, max_read_len=150, max_len=40, kmax=1)
            assert torch.equal(got40, want40)


def test_both_kernel_schedules_agree():
    """The two-phase kernel (default for one adapter) and the one-phase kernel give identical records."""
    import os
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_reads

    rng = random.Random(8)
    cases = [(PA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a"), make_reads(20000, config=2)[0]),
             (PA.FrontAdapter("GTTCAGAGTTCTACAGTCCGACGATC", max_errors=0.15, name="f"), None),
             (PA.AnywhereAdapter("CTGTCTCTTATACACATCT", max_errors=0.2, name="w"), None),
             (PA.BackAdapter("AGATCGGAAGAGCNNNNNNNNATCTCGTATGCC", max_errors=0.1, name="n"), None),
             (PA.RightmostFrontAdapter("ACGTTGCATT", max_errors=0.1, name="r"), None)]
    for adapter, reads in cases:
        if reads is None:
            reads = random_reads(rng, [adapter.sequence], 5000, "ACGT", rng.choice([100, 150, 400]))
        d = adapter.descriptor()
        exp, _ = oracle.oracle_process([d], None, reads)
        got, _ = run_set([d], None, reads)                       # default: split scan/DP pipeline
        assert (got == exp).all(), ("default", repr(adapter))
        for variant in ("general", "block", "warp"):             # the fused kernels
            os.environ["CUTADAPT_B200_KERNEL"] = variant
            try:
                other, _ = run_set([d], None, reads)
            finally:
                del os.environ["CUTADAPT_B200_KERNEL"]
            assert (other == exp).all(), (variant, repr(adapter))
        os.environ["CUTADAPT_B200_SCAN"] = "shiftand"           # split pipeline with the shift-and first stage
        try:
            other, _ = run_set([d], None, reads)
        finally:
            del os.environ["CUTADAPT_B200_SCAN"]
        assert (other == exp).all(), ("shiftand", repr(adapter))


def test_specialised_first_stage_matches_the_interpreter_and_the_oracle(monkeypatch):
    """
    The run-time specialisation of the first stage (cg_jit.cpp: the plane program written out as calls with literal
    arguments, compiled with NVRTC) must give the records of the precompiled interpreter kernel and of the oracle.
    """
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_reads

    rng = random.Random(5)
    for trial, seq in enumerate(["AGATCGGAAGAGC", "AGATCGGAAGAGCACACGTCTGAACTCCAGTCA", "CTGTCTCTTATACACATCT", "TGGAATTCTCGGGTGCCAAGG"]):
        ad = PA.BackAdapter(seq, max_errors=0.1, min_overlap=3, name="x")
        d = ad.descriptor()
        reads, quals = make_reads(30000, config=2, seed=100 + trial, with_qualities=True, adapter=seq)
        reads += random_reads(rng, [seq], 3000, "ACGTNacgt", 200 if trial == 2 else 130)
        quals += ["".join(chr(33 + rng.choice([2, 20, 30, 38])) for _ in r) for r in reads[30000:]]
        qt = trial % 2 == 1
        kw = dict(quality_trim=qt, cutoff_front=0, cutoff_back=20)
        exp, eqt = oracle.oracle_process([d], None, reads, quals if qt else None, quality_trim=qt, cutoff_back=20)
        monkeypatch.setenv("CUTADAPT_B200_JIT", "0")
        plain, _ = run_set([d], None, reads, quals if qt else None, **kw)
        monkeypatch.setenv("CUTADAPT_B200_JIT", "1")
        aset = L.AdapterSet(L.AdapterSetSpec([d]))
        data, offsets = L.pack_strings(reads)
        qd = L.pack_strings(quals)[0] if qt else None
        got, gqt = aset.process(data, offsets, qd, L.make_params(**kw))
        assert aset.jit_status() == 1, L.last_error()
        assert "plane_chain_step<W>" in aset.jit_source(5 if max(map(len, reads)) <= 160 else 8, qt)
        assert (got == exp).all() and (plain == exp).all() and (not qt or (gqt == eqt).all()), seq


def test_bitplane_first_stage_kernel_against_oracle():
    """
    cg_pscan_kernel (bit-plane first stage of plain A/C/G/T 3' adapters) + the exact path behind it: ragged reads of
    0..256 characters (both plane widths) and longer ones (the batch falls back to the shift-and scan), N / lower
    case / other letters, several adapter copies, with and without fused quality trimming.
    """
    import cutadapt_b200.adapters as PA

    rng = random.Random(99)
    for trial in range(24):
        m = rng.choice([8, 13, 13, 20, 33, 33, 50])
        seq = "AGATCGGAAGAGC" if trial == 0 else "".join(rng.choice("ACGT") for _ in range(m))
        ad = PA.BackAdapter(seq, max_errors=rng.choice([0.05, 0.1, 0.1, 0.2]), min_overlap=rng.randint(1, 5), name="x")
        d = ad.descriptor()
        alpha = rng.choice(["ACGT", "ACGTN", "ACGTNacgtn", "ACGTRYKMEUXacgt"])
        max_len = rng.choice([100, 150, 150, 160, 240, 256, 500])
        reads = random_reads(rng, [seq], 3000, alpha, max_len - len(seq) - 2 if max_len <= 256 else max_len)
        if max_len <= 256:
            reads = [r[:max_len] for r in reads]
        for _ in range(3000):
            ins = rng.randint(0, max_len)
            r = ("".join(rng.choice(alpha) for _ in range(ins)) + seq + "".join(rng.choice("ACGT") for _ in range(max_len)))[:max_len]
            reads.append(r.lower() if rng.random() < 0.1 else r)
        quals = ["".join(chr(33 + rng.choice([2, 2, 20, 30, 38])) for _ in r) for r in reads]
        qt = trial % 3 == 0
        got, gqt = run_set([d], None, reads, quals if qt else None, quality_trim=qt, cutoff_front=5, cutoff_back=20)
        exp, eqt = oracle.oracle_process([d], None, reads, quals if qt else None, quality_trim=qt, cutoff_front=5, cutoff_back=20)
        assert (not qt or (gqt == eqt).all()) and (got == exp).all(), (trial, repr(ad), max_len)


def test_multipass_schedule_agrees_with_one_phase_and_oracle():
    """Adapter sets on the multi-pass schedule (per-adapter pipelines + cg_select_kernel) == the one-phase
    kernel == the oracle, incl. linked adapters, long/wildcard adapters (bit-vector plan) and quality trimming."""
    import os
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_reads

    rng = random.Random(88)
    reads0, quals0 = make_reads(6000, config=3, with_qualities=True)
    five = [PA.BackAdapter(s, max_errors=0.15, name=f"a{i}") for i, s in enumerate(
        ["AGATCGGAAGAGC", "CTGTCTCTTATACACATCT", "VCCGAMCYUCKHRKDCUBBCNUWNSGHCGU", "AGATCGGAAGAGCNNNNNNNNATCTCGTATGCC"])]
    five.append(PA.LinkedAdapter(PA.PrefixAdapter("GTTCAGAGTTCTACAGTCCGACGATC", max_errors=0.15, name="f"),
                                 PA.BackAdapter("TGGAATTCTCGGGTGCCAAGG", max_errors=0.15, name="b"), True, False, "l"))
    sets = [PA.MultipleAdapters(five)]
    for _ in range(6):
        ads = ["".join(rng.choice("ACGT") for _ in range(rng.randint(8, 60))) for _ in range(rng.randint(2, 4))]
        objs = [rng.choice([PA.BackAdapter, PA.FrontAdapter, PA.AnywhereAdapter, PA.SuffixAdapter, PA.NonInternalBackAdapter])(
            a, max_errors=rng.choice([0.05, 0.1, 0.2]), name="x") for a in ads]
        if rng.random() < 0.6:
            objs.append(PA.LinkedAdapter(PA.FrontAdapter(ads[0][:14], max_errors=0.1), PA.BackAdapter(ads[1], max_errors=0.1),
                                         rng.random() < 0.5, rng.random() < 0.5, "l"))
        sets.append(PA.MultipleAdapters(objs))
    for k, multi in enumerate(sets):
        singles, groups, _ = multi._flatten()
        descs = [s.descriptor() for s in singles]
        if k == 0:
            reads, quals = reads0, quals0
        else:
            reads = random_reads(rng, [s.sequence for s in singles], 3000, "ACGT", 150)
            quals = ["".join(chr(33 + rng.choice([2, 2, 15, 30, 38])) for _ in r) for r in reads]
        for qt in (False, True):
            kw = dict(quality_trim=True, cutoff_front=5, cutoff_back=20) if qt else {}
            exp, eqt = oracle.oracle_process(descs, groups, reads, quals if qt else None, qt, 5 if qt else 0, 20 if qt else 0)
            got, gqt = run_set(descs, groups, reads, quals if qt else None, **kw)
            assert (got == exp).all(), ("multipass", k, qt)
            if qt:
                assert (gqt == eqt).all()
            os.environ["CUTADAPT_B200_KERNEL"] = "general"
            try:
                other, _ = run_set(descs, groups, reads, quals if qt else None, **kw)
            finally:
                del os.environ["CUTADAPT_B200_KERNEL"]
            assert (other == exp).all(), ("general", k, qt)

