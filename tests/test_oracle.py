"""
The oracle against the reference: every function of oracle/cutadapt_oracle.c is pinned to the
golden vectors generated from the reference's own compiled code (tests/golden/make_golden.py).
"""
import random

import pytest

from oracle import oracle
from util import batch_digest, digest, golden, match_desc, build_adapters, random_locate_cases


def test_locate_golden():
    cases = golden("locate_kat.json.gz")
    assert len(cases) > 3000
    for ref, q, rate, flags, wr, wq, ic, mo, expected in cases:
        got = oracle.locate(ref, q, rate, flags, wr, wq, ic, mo)
        assert (list(got) if got is not None else None) == expected, (ref, q, rate, flags, wr, wq, ic, mo)


def test_reference_known_answers():
    # tests/test_align.py:74-107 in the reference
    assert oracle.locate("CCAGTCCTCT", "CCAGTCCTTTCCTGAGAGT", 0.3, 8) == (0, 10, 0, 10, 8, 1)
    assert oracle.locate("TCGATC", "TCGATGC", 1.5 / 6, 8) == (0, 6, 0, 6, 4, 1)
    assert oracle.locate("GCCGAACTTCTTAGACTGCCTTAAGGACGT", "CAAATCACCAGAAGGCGCCTAACTTCTTAGACTGCC", 0.1, 14) == (
        0, 20, 16, 36, 18, 1)
    assert oracle.locate("", "", 0, 0, min_overlap=0) == (0, 0, 0, 0, 0, 0)
    assert oracle.locate("TTTT", "CCTTTT", 0.25, 14) == (0, 4, 2, 6, 4, 0)


def test_comparers_golden():
    for ref, q, rate, wr, wq, mo, p, s in golden("comparer_kat.json.gz"):
        got = oracle.prefix_compare(ref, q, rate, wr, wq, mo)
        assert (list(got) if got else None) == p, ("prefix", ref, q)
        got = oracle.suffix_compare(ref, q, rate, wr, wq, mo)
        assert (list(got) if got else None) == s, ("suffix", ref, q)


def test_kmers_present_golden():
    for sets, rw, qw, reads in golden("kmer_kat.json.gz")["present"]:
        tables = oracle.KmerTables([(s, e, k) for s, e, k in sets], rw, qw)
        for read, expected in reads:
            assert tables.present(read) == expected, (sets, rw, qw, read)


def test_quality_trim_golden():
    for q, cf, cb, base, expected in golden("qualtrim_kat.json.gz"):
        assert list(oracle.quality_trim_index(q, cf, cb, base)) == expected, (q, cf, cb, base)


def test_non_ascii_is_an_error():
    with pytest.raises(ValueError):
        oracle.locate("ACGT", "AC\xe4GT", 0.1)


def test_info_file_coordinates():
    """Per-read coordinates of the reference's golden file tests/cut/illumina.info.txt."""
    from cutadapt_b200.kmer_heuristic import create_positions_and_kmers

    data = golden("info_file_kat.json.gz")["illumina"]
    adapter = data["adapter"]
    tables = oracle.KmerTables(create_positions_and_kmers(adapter, 3, 0.1, True, False), False, False)
    n_hits = 0
    for seq, expected in data["rows"]:
        res = oracle.locate(adapter, seq, 0.1, 14, min_overlap=3) if tables.present(seq) else None
        if expected is None:
            assert res is None, seq
        else:
            n_hits += 1
            assert [res[5], res[2], res[3]] == expected, seq
    assert n_hits > 30


def test_against_reference_random():
    """Aligner.locate / quality_trim_index of the reference on 3000 random cases (answers: reference_random_kat)."""
    g = golden("reference_random_kat.json.gz")
    cases = list(random_locate_cases())
    assert digest(cases) == g["cases_digest"] and len(cases) == len(g["answers"])
    for (ref, rate, flags, wr, wq, ic, mo, queries, qs), (locs, qt) in zip(cases, g["answers"]):
        for q, expected in zip(queries, locs):
            got = oracle.locate(ref, q, rate, flags, wr, wq, ic, mo)
            assert (list(got) if got is not None else None) == expected, (ref, q, rate, flags)
        assert list(oracle.quality_trim_index(qs, 5, 20)) == qt, qs


def test_oracle_composition_matches_golden_adapters():
    """oracle_process (prefilter + locate + best-of / linked) against reference match_to results."""
    import cutadapt_b200.adapters as PA
    from util import spec_of
    import numpy as np

    for case in golden("adapters_kat.json.gz"):
        multi = build_adapters(PA, case["adapters"])
        spec = spec_of(multi)
        reads = [r for r, _ in case["reads"]]
        recs, _ = oracle.oracle_process(spec.adapters, spec.groups, reads)
        if recs.shape[2] == 1 and spec.slots == 2:
            pass
        for i, (read, expected) in enumerate(case["reads"]):
            got = match_desc(multi.matches_from_records(recs[i, 0], read))
            assert got == expected, (case["adapters"], read)


def test_trim_scans_golden():
    """nextseq_trim_index / poly_a_trim_index of the oracle == the reference (incl. its own KATs)."""
    g = golden("trim_scans_kat.json.gz")
    for seq, qual, cutoff, base, expected in g["nextseq"]:
        assert oracle.nextseq_trim_index(seq, qual, cutoff, base) == expected, (seq, qual, cutoff, base)
    for seq, revcomp, expected in g["polya"]:
        assert oracle.poly_a_trim_index(seq, revcomp) == expected, (seq, revcomp)
    for qual, base, expected in g["expected_errors"]:           # bit-exact doubles
        assert oracle.expected_errors(qual, base).hex() == expected, (qual, base)
    assert oracle.expected_errors("II!I ", 33) < 0             # a character below the base


def test_fastq_oracle_reproduces_the_reference_command_line_goldens():
    """
    oracle.oracle_fastq_trim (parse -> modifiers -> filters -> format) against the expected output files of
    the reference's own command-line tests (the case list in tests/golden/fastq_kat.json.gz names test and command line).
    """
    from util import fastq_cases, fastq_case_adapters, fastq_case_kwargs, spec_of
    import cutadapt_b200.adapters as PA

    cases = fastq_cases()
    assert len(cases) >= 17
    for c in cases:
        ads = fastq_case_adapters(c["options"])
        descs = groups = None
        if ads:
            spec = spec_of(PA.MultipleAdapters(ads))
            descs, groups = spec.adapters, spec.groups
        got, counters = oracle.oracle_fastq_trim(c["input_bytes"], descs, groups, **fastq_case_kwargs(c["options"]))
        assert got == c["expected_bytes"], c["name"]
        assert counters["n_records"] >= counters["n_written"]
    with pytest.raises(oracle.FastqFormatError):
        oracle.parse_fastq(b"@r\nACGT\n+\nII\n")
    with pytest.raises(oracle.FastqFormatError):
        oracle.parse_fastq(b"@r\nACGT\n+\n")


def test_paired_fastq_oracle_reproduces_the_reference_goldens():
    """oracle.oracle_fastq_trim_paired against the expected files of the reference's tests/test_paired.py."""
    from util import fastq_paired_cases, oracle_paired

    cases = fastq_paired_cases()
    assert len(cases) >= 16
    for c in cases:
        o1, o2, c1, c2 = oracle_paired(oracle, c["options"], *c["input_bytes"])
        assert [o1, o2] == c["expected_bytes"], c["name"]
        assert c1["n_written"] == c2["n_written"] <= c1["n_records"] == c2["n_records"]


def test_demultiplex_oracle_reproduces_the_reference_golden():
    from util import fastq_demux_case, spec_of
    import cutadapt_b200.adapters as PA

    c = fastq_demux_case()
    ads = [PA.BackAdapter(seq, max_errors=0.1, min_overlap=3, name=name) for name, seq in c["adapters"]]
    spec = spec_of(PA.MultipleAdapters(ads))
    got = oracle.oracle_fastq_demux(c["input_bytes"], spec.adapters, spec.groups, [a.name for a in ads])
    assert got == c["expected"]


def test_fastq_oracle_reproduces_the_fasta_goldens_of_the_reference():
    """32 more command-line known answers of the reference (anchored / non-internal / linked adapters, --no-indels,
    -N, --match-read-wildcards, --trim-n, --poly-a, --max-n ...) whose vectors are FASTA: the oracle must reproduce
    the expected sequences (tests/golden/make_fastq_golden.py stores them as FASTQ with constant qualities)."""
    from util import golden, fastq_file, adapter_from_spec, fastq_case_kwargs, spec_of
    import cutadapt_b200.adapters as PA

    cases = golden("fastq_kat.json.gz")["fasta_cases"]
    assert len(cases) >= 30
    for c in cases:
        o = c["options"]
        params = dict(max_errors=o.get("error_rate", 0.1), min_overlap=o.get("min_overlap", 3),
                      adapter_wildcards=not o.get("no_wildcards", False), read_wildcards=o.get("read_wildcards", False),
                      indels=not o.get("no_indels", False))
        ads = [adapter_from_spec(spec, kind, name=f"a{i}", **params) for i, (kind, spec) in enumerate(o["specs"])]
        descs = groups = None
        if ads:
            spec = spec_of(PA.MultipleAdapters(ads))
            descs, groups = spec.adapters, spec.groups
        got, _ = oracle.oracle_fastq_trim(fastq_file(f"fa_{c['name']}.in.fastq"), descs, groups, **fastq_case_kwargs(o))
        assert got == fastq_file(f"fa_{c['name']}.out.fastq"), (c["name"], c["command"])


def test_packed_batch_loop_equals_the_per_read_composition():
    """oracle_process_packed (the C loop the 10^6-read gate tests use) == oracle_process on every adapter type."""
    import numpy as np
    import cutadapt_b200.adapters as PA
    from cutadapt_b200 import _lib as L
    from util import random_reads

    rng = random.Random(12)
    for trial in range(25):
        ads = ["".join(rng.choice("ACGT") for _ in range(rng.randint(5, 40))) for _ in range(rng.randint(1, 4))]
        types = [PA.BackAdapter, PA.FrontAdapter, PA.AnywhereAdapter, PA.RightmostFrontAdapter, PA.RightmostBackAdapter,
                 PA.PrefixAdapter, PA.SuffixAdapter, PA.NonInternalBackAdapter]
        objs = [rng.choice(types)(a, max_errors=rng.choice([0.1, 0.2]), indels=rng.random() < 0.8, name="a") for a in ads]
        if rng.random() < 0.4:
            objs.append(PA.LinkedAdapter(PA.PrefixAdapter(ads[0][:10], max_errors=0.2), PA.BackAdapter(ads[-1], max_errors=0.1),
                                         rng.random() < 0.5, rng.random() < 0.5, "l"))
        multi = PA.MultipleAdapters(objs)
        singles, groups, _ = multi._flatten()
        descs = [s.descriptor() for s in singles]
        reads = random_reads(rng, ads, 300, rng.choice(["ACGT", "ACGTN"]), 120)
        quals = ["".join(chr(33 + rng.choice([2, 2, 15, 30, 38])) for _ in r) for r in reads]
        qt, times = rng.random() < 0.5, rng.choice([1, 1, 2, 3])
        nx = rng.choice([None, None, 20])
        a, aq = oracle.oracle_process(descs, groups, reads, quals, qt, 5, 20, 33, times, nextseq_cutoff=nx)
        data, offs = L.pack_strings(reads)
        qd, _ = L.pack_strings(quals)
        b, bq = oracle.oracle_process_packed(descs, groups, data, offs, qd, qt, 5, 20, 33, times, nextseq_cutoff=nx,
                                             threads=rng.choice([1, 3]))
        assert (a == b).all() and (aq == bq).all(), trial


def test_neighbourhoods_and_index_golden():
    """edit_environment / hamming_sphere / AdapterIndex of the oracle against the reference's own (goldens)."""
    for t, k, ee, he in golden("environment_kat.json.gz"):
        assert sorted(map(list, oracle.edit_environment(t, k))) == sorted(ee), (t, k)
        ham = [[s, e, len(t) - e] for e in range(k + 1) for s in oracle.hamming_sphere(t, e)]
        assert sorted(ham) == sorted(he), (t, k)
    import numpy as np
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.configs import config5_barcodes, make_config_batch, to_strings

    # the reference's IndexedPrefixAdapters of the 96 barcodes: index keys and matches (index_reference_kat)
    g = golden("index_reference_kat.json.gz")
    bcs = config5_barcodes()
    b = make_config_batch(5, 3000, seed=77)
    b["seq"][::50, 3] = ord("N")
    assert batch_digest(b) == g["reads_digest"]
    for key, indels in (("indels", True), ("hamming", False)):
        lengths, index = oracle.index_build(bcs, 0.1, indels)
        assert sorted(index) == g[key]["keys"] and lengths == g[key]["lengths"]
        host = b["seq"].numpy().reshape(-1)
        offs = np.arange(3001, dtype=np.int64) * 150
        descs = [PA.PrefixAdapter(s, max_errors=0.1, indels=indels, name=f"bc{i}").descriptor() for i, s in enumerate(bcs)]
        out = oracle.oracle_index_process(bcs, 0.1, indels, True, host, offs, descs)
        for r, rec, expected in zip(to_strings(b["seq"]), out, g[key]["rows"]):
            have = None if rec["adapter"] < 0 else [
                int(rec[f]) for f in ("adapter", "astart", "astop", "rstart", "rstop", "score", "errors")]
            assert have == expected, (key, r)
