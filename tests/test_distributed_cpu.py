"""
The N>1 path on CPU: two gloo ranks shard the reads, trim their shard (device functions compiled for
the host -- test infrastructure), reduce the statistics vector with the product's
``allreduce_statistics`` and must arrive at the single-process totals.
"""
import socket

import numpy as np


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_shard_range_partitions_exactly():
    from cutadapt_b200.pipeline import shard_range

    for n in (0, 1, 7, 128, 1000003):
        for world in (1, 2, 3, 8):
            bounds = [shard_range(n, r, world) for r in range(world)]
            assert bounds[0][0] == 0 and bounds[-1][1] == n
            assert all(bounds[i][1] == bounds[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in bounds]
            assert max(sizes) - min(sizes) <= 1


def test_two_rank_statistics_allreduce(tmp_path):
    import torch.multiprocessing as mp
    import _dist_worker
    import cutadapt_b200.adapters as PA
    from cutadapt_b200.synth import make_reads
    from util import hostsim_process, spec_of

    mp.spawn(_dist_worker.run, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0 = np.load(tmp_path / "rank0.npy")
    r1 = np.load(tmp_path / "rank1.npy")
    assert (r0 == r1).all()
    assert (np.load(tmp_path / "local0.npy") + np.load(tmp_path / "local1.npy") == r0).all()
    # single-process totals of the same reads
    reads, multi = _dist_worker.workload()
    spec = spec_of(multi)
    matches, _ = hostsim_process(spec, reads)
    total = _dist_worker.host_statistics(reads, matches, None, len(spec.adapters), 200, 3)
    assert (total == r0).all()
    assert r0[0] == len(reads) and 1500 < r0[2] < 3500
    # ... and the reduced vector rebuilds the per-adapter statistics objects: errors[length][errors] and adjacent
    # bases of every end, equal to feeding every Match to add_match() like the reference's AdapterCutter does
    from cutadapt_b200.pipeline import adapter_statistics_from_vector, stats_layout

    rebuilt = adapter_statistics_from_vector(r0, multi, 200, 3)
    fed = [a.create_statistics() for a in multi]
    by_adapter = {id(a): st for a, st in zip(multi, fed)}
    lengths = np.zeros(201, dtype=np.int64)
    for i, read in enumerate(reads):
        m = multi.matches_from_records(matches[i, 0], read)
        lengths[len(read) if m is None else len(m.trimmed(read))] += 1
        if m is not None:
            by_adapter[id(m.adapter)].add_match(m)
    assert len(rebuilt) == len(fed) == 4
    for a, b in zip(rebuilt, fed):
        for ea, eb in zip(a.end_statistics(), b.end_statistics()):
            assert (ea is None) == (eb is None)
            if ea is not None:
                assert ea.errors == eb.errors and ea.adjacent_bases == eb.adjacent_bases, a.name
    lay = stats_layout(len(spec.adapters), 200, 3)
    assert (r0[lay["lengths"]:lay["lengths"] + 201] == lengths).all()
    # against the reference itself: its AdapterStatistics fed with its own matches (statistics_reference_kat)
    from util import digest, golden

    g = golden("statistics_reference_kat.json.gz")
    assert digest(reads) == g["reads_digest"] and len(g["adapters"]) == len(rebuilt)
    for mine, ends in zip(rebuilt, g["adapters"]):
        for ea, eb in zip(mine.end_statistics(), ends):
            assert (ea is None) == (eb is None)
            if ea is not None:
                errors = {}
                for length, e, count in eb["errors"]:
                    errors.setdefault(length, {})[e] = count
                assert ea.errors == errors and ea.adjacent_bases == dict(eb["adjacent_bases"]), mine.name
    # the FASTQ counters of both ranks add up to the single-process totals
    import json
    from oracle import oracle

    f0, f1 = (json.load(open(tmp_path / f"fq{r}.json")) for r in (0, 1))
    assert f0["total"] == f1["total"]
    reads2, _ = make_reads(3001, config=2, seed=99)
    spec2 = spec_of(PA.MultipleAdapters([PA.BackAdapter("AGATCGGAAGAGC", max_errors=0.1, name="a")]))
    fq = "".join(f"@r{i}\n{r}\n+\n{'I' * len(r)}\n" for i, r in enumerate(reads2)).encode()
    _, whole = oracle.oracle_fastq_trim(fq, spec2.adapters, spec2.groups, minimum_length=100)
    for k, v in whole.items():
        assert f0["total"][k] == v == f0["local"][k] + f1["local"][k], k
    assert whole["n_written"] + whole["too_short"] == 3001 and whole["too_short"] > 100


def test_kept_intervals_compose_like_the_reference():
    """kept_intervals == applying QualityTrimmer then every Match.trimmed() (adapters.py:453-487)."""
    import random
    import cutadapt_b200.adapters as PA
    from cutadapt_b200 import _lib as L
    from cutadapt_b200.pipeline import kept_intervals
    from util import hostsim_process, spec_of, random_reads

    rng = random.Random(4)
    ads = ["ACGTTGCAAC", "TTGACCAGTA"]
    multi = PA.MultipleAdapters([PA.BackAdapter(ads[0], name="a"), PA.FrontAdapter(ads[1], name="b")])
    spec = spec_of(multi)
    reads = random_reads(rng, ads, 300, "ACGT", 90)
    quals = ["".join(chr(33 + rng.choice([2, 20, 35])) for _ in r) for r in reads]
    params = L.make_params(quality_trim=True, cutoff_front=0, cutoff_back=15, times=2)
    matches, qtrim = hostsim_process(spec, reads, quals, params)
    iv = kept_intervals(matches, qtrim, np.array([len(r) for r in reads]))
    for i, read in enumerate(reads):
        cur = read[qtrim[i, 0]:qtrim[i, 1]]
        for r in range(2):
            m = multi.matches_from_records(matches[i, r], cur)
            if m is None:
                break
            cur = m.trimmed(cur)
        assert read[iv[i, 0]:iv[i, 1]] == cur


def test_round_robin_runner_merges_chunks_in_order(tmp_path):
    """
    The multi-GPU chunk driver on CPU (gloo, 3 ranks, the FASTQ oracle as the per-chunk worker): chunk c goes to rank
    c mod 3, rank 0 writes the outputs in chunk order -- the file equals what one process writes (the contract of
    OrderedChunkWriter, runners.py:224-245), over more than 64 chunks including a short last round.
    """
    import io
    import torch.multiprocessing as mp
    import _dist_worker
    from cutadapt_b200.pipeline import read_fastq_chunks

    mp.spawn(_dist_worker.run_chunks, args=(3, _free_port(), str(tmp_path)), nprocs=3, join=True)
    merged = open(tmp_path / "merged.fastq", "rb").read()
    data, process = _dist_worker.chunk_workload()
    chunks = list(read_fastq_chunks(io.BytesIO(data), 24 * 1024))
    assert len(chunks) > 64 and len(chunks) % 3 != 0
    assert int(open(tmp_path / "chunks.txt").read()) == len(chunks)
    assert merged == b"".join(process(c) for c in chunks)
    assert merged == process(data)                   # and the chunking itself changes nothing
