"""Shared helpers of the test-suite (test infrastructure only)."""
import ctypes as C
import gzip
import hashlib
import json
import os
import random

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def golden(name):
    with gzip.open(os.path.join(HERE, "golden", name), "rt") as f:
        return json.load(f)


def digest(obj):
    """sha256 of the compact JSON form of `obj` (numpy integers count as ints): lets a fixture pin a list of answers
    too long to store."""
    return hashlib.sha256(json.dumps(obj, separators=(",", ":"), default=int).encode()).hexdigest()


def batch_digest(batch):
    """sha256 of the reads (and qualities) of a make_config_batch() result: pins the generator a fixture was made with."""
    h = hashlib.sha256()
    for key in ("seq", "qual", "seq2", "qual2"):
        if batch.get(key) is not None:
            h.update(np.ascontiguousarray(batch[key].cpu().numpy()).tobytes())
    return h.hexdigest()


def canon(x):
    """A result in a form that ignores the order of lists and sets but keeps the order inside tuples."""
    if isinstance(x, tuple):
        return [canon(v) for v in x]
    if isinstance(x, (list, set, frozenset)):
        return sorted((canon(v) for v in x), key=json.dumps)
    return x


def random_locate_cases():
    """(reference, max_error_rate, flags, wildcard_ref, wildcard_query, indel_cost, min_overlap, [4 queries],
    qualities) of the random oracle-against-reference test; tests/golden/reference_random_kat.json.gz holds the
    reference's answers."""
    rng = random.Random(77)
    for _ in range(3000):
        alpha = rng.choice(["ACGT", "AC", "ACGTN", "ACGTacgtNn", "ACGTRYKMN"])
        m = rng.randint(1, 20)
        ref = "".join(rng.choice(alpha) for _ in range(m))
        wr, wq = rng.random() < 0.3, rng.random() < 0.2
        if wr and set(ref.upper()) <= {"N"}:
            continue
        rate = rng.choice([0, 0.1, 0.2, 0.34, 0.5])
        flags, ic, mo = rng.randint(0, 15), rng.choice([1, 1, 100000, 3]), rng.randint(1, 4)
        queries = []
        for _ in range(4):
            q = "".join(rng.choice(alpha) for _ in range(rng.randint(0, 40)))
            if rng.random() < 0.5:
                pos = rng.randint(0, len(q))
                q = q[:pos] + ref[rng.randint(0, m // 2):] + q[pos:]
            queries.append(q)
        qs = "".join(chr(33 + rng.choice([0, 2, 10, 20, 30, 40])) for _ in range(rng.randint(0, 50)))
        yield ref, rate, flags, wr, wq, ic, mo, queries, qs


# ---- hostsim: the device functions compiled for the host (tests only) ------------------------

_hs = None


def hostsim_lib():
    global _hs
    if _hs is None:
        from cutadapt_b200 import _lib as L

        lib = C.CDLL(os.environ.get("CUTADAPT_B200_HOSTSIM_LIB") or os.path.join(HERE, "hostsim", "libhostsim.so"))
        lib.hs_last_error.restype = C.c_char_p
        lib.hs_process_batch.argtypes = [
            C.POINTER(L.cg_adapter_desc), C.c_int, C.POINTER(L.cg_group_desc), C.c_int, C.c_void_p,
            C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(L.cg_params), C.c_void_p, C.c_void_p, C.c_int,
        ]
        lib.hs_process_batch_indexed.argtypes = [
            C.POINTER(L.cg_adapter_desc), C.c_int, C.POINTER(L.cg_group_desc), C.c_int,
            C.POINTER(L.cg_index_desc), C.c_int, C.c_void_p,
            C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(L.cg_params), C.c_void_p, C.c_void_p, C.c_int,
        ]
        _hs = lib
    return _hs


def hostsim_process(spec, seqs, quals=None, params=None, force_wide=0):
    from cutadapt_b200 import _lib as L

    params = params or L.make_params()
    arr, n, garr, ng = spec.to_ctypes()
    data, offs = L.pack_strings(seqs)
    qd = L.pack_strings(quals)[0] if quals is not None else None
    times = max(1, params.times)
    out = np.zeros((len(seqs), times, spec.slots), dtype=L.MATCH_DTYPE)
    qt = np.zeros((len(seqs), 2), dtype=np.int32)
    iarr, ni = spec.index_ctypes()
    rc = hostsim_lib().hs_process_batch_indexed(
        arr, n, garr, ng, iarr, ni, data.ctypes.data, qd.ctypes.data if qd is not None else None, offs.ctypes.data,
        len(seqs), C.byref(params), out.ctypes.data, qt.ctypes.data, force_wide,
    )
    if rc:
        raise RuntimeError((rc, hostsim_lib().hs_last_error()))
    return out, qt


def hostsim_statistics(seqs, matches, qtrim, n_adapters, max_len=150, kmax=3):
    """The statistics vector of a batch computed by the host build of stats_read_core (what cg_stats_kernel runs)."""
    from cutadapt_b200 import _lib as L
    from cutadapt_b200.pipeline import stats_layout

    data, offs = L.pack_strings(seqs)
    out = np.zeros(stats_layout(n_adapters, max_len, kmax)["size"], dtype=np.int64)
    m = np.ascontiguousarray(matches)
    q = np.ascontiguousarray(qtrim, dtype=np.int32) if qtrim is not None else None
    rc = hostsim_lib().hs_statistics(C.c_void_p(data.ctypes.data), C.c_void_p(offs.ctypes.data), C.c_int64(len(seqs)),
                                     C.c_void_p(m.ctypes.data), C.c_void_p(q.ctypes.data) if q is not None else None,
                                     C.c_int(m.shape[1]), C.c_int(m.shape[2]), C.c_int(n_adapters), C.c_int(max_len),
                                     C.c_int(kmax), C.c_void_p(out.ctypes.data))
    assert rc == 0
    return out


def hostsim_plane_classes(spec, seqs):
    """Class of every read in the bit-plane first stage: 0 no match, 1 exact occurrence, 2 re-scan, 3 plan from the planes' hits, -1 n/a."""
    from cutadapt_b200 import _lib as L

    arr, n, garr, ng = spec.to_ctypes()
    data, offs = L.pack_strings(seqs)
    cls = np.zeros(len(seqs), dtype=np.int32)
    lib = hostsim_lib()
    rc = lib.hs_plane_classify(arr, n, garr, ng, C.c_void_p(data.ctypes.data), C.c_void_p(offs.ctypes.data),
                               C.c_int64(len(seqs)), C.c_void_p(cls.ctypes.data))
    if rc:
        raise RuntimeError((rc, lib.hs_last_error()))
    return cls


# ---- building adapters from the golden "adapters_kat" specs ----------------------------------


def build_adapters(module, specs):
    """Instantiate [type, seq, kwargs] / ["Linked", front, back, freq, breq] specs with `module`'s classes."""
    objs = []
    for spec in specs:
        if spec[0] == "Linked":
            _, (t1, s1, k1), (t2, s2, k2), fq, bq = spec
            front = getattr(module, t1)(s1, name="f", **k1)
            back = getattr(module, t2)(s2, name="b", **k2)
            objs.append(module.LinkedAdapter(front, back, fq, bq, "lnk"))
        elif spec[0] == "Indexed":
            _, prefix, members = spec
            cls = module.PrefixAdapter if prefix else module.SuffixAdapter
            parts = [cls(s, name="x", **k) for s, k in members]
            objs.append((module.IndexedPrefixAdapters if prefix else module.IndexedSuffixAdapters)(parts))
        else:
            t, s, k = spec
            objs.append(getattr(module, t)(s, name="x", **k))
    return module.MultipleAdapters(objs)


def match_desc(m):
    if m is None:
        return None
    if hasattr(m, "front_match"):
        return ["Linked", match_desc(m.front_match), match_desc(m.back_match)]
    return [type(m).__name__, m.astart, m.astop, m.rstart, m.rstop, m.score, m.errors]


def spec_of(multi):
    """AdapterSetSpec + bookkeeping for a cutadapt_b200 MultipleAdapters / adapter."""
    from cutadapt_b200 import _lib as L

    singles, groups, owners = multi._flatten()
    spec = L.AdapterSetSpec([s.descriptor() for s in singles], groups, multi._flatten_indexes())
    multi._device_set = (None, singles, owners)
    return spec


def random_reads(rng, adapters, n_reads, alpha="ACGT", max_len=80):
    reads = []
    for _ in range(n_reads):
        q = "".join(rng.choice(alpha) for _ in range(rng.randint(0, max_len)))
        for _ in range(rng.choice([0, 1, 1, 2])):
            ad = rng.choice(adapters)
            piece = ad if rng.random() < 0.6 else ad[rng.randint(0, len(ad) // 2): rng.randint(len(ad) // 2, len(ad))]
            piece = list(c if c in "ACGT" else rng.choice("ACGT") for c in piece)
            for _ in range(rng.choice([0, 0, 1, 2])):
                if piece:
                    p = rng.randrange(len(piece))
                    r = rng.random()
                    if r < 0.4:
                        piece[p] = rng.choice(alpha)
                    elif r < 0.7:
                        del piece[p]
                    else:
                        piece.insert(p, rng.choice(alpha))
            pos = rng.choice([0, len(q), rng.randint(0, len(q))])
            q = q[:pos] + "".join(piece) + q[pos:]
        reads.append(q)
    return reads


# ---- FASTQ known-answer cases of the reference's command-line tests (tests/golden/fastq_kat.json.gz) -----------------

_FASTQ_KAT = None


def fastq_file(name) -> bytes:
    """One fixture of tests/golden/fastq_kat.json.gz (made by tests/golden/make_fastq_golden.py)."""
    global _FASTQ_KAT
    if _FASTQ_KAT is None:
        _FASTQ_KAT = golden("fastq_kat.json.gz")
    return _FASTQ_KAT["files"][name].encode("latin-1")


def fastq_cases():
    fastq_file("small.in.fastq")
    cases = [dict(c) for c in _FASTQ_KAT["cases"]]
    for c in cases:
        c["input_bytes"] = fastq_file(c["name"] + ".in.fastq")
        c["expected_bytes"] = fastq_file(c["name"] + ".out.fastq")
    return cases


def fastq_case_adapters(options, key="adapters"):
    """The adapters of a case as the command line would build them (-e, -O, default 3): cutadapt_b200 objects."""
    import cutadapt_b200.adapters as PA

    kinds = {"back": PA.BackAdapter, "front": PA.FrontAdapter, "anywhere": PA.AnywhereAdapter}
    e = options.get("error_rate", 0.1)
    o = options.get("min_overlap", 3)
    out = []
    for i, spec in enumerate(options[key]):
        if spec[0] == "linked":        # ["linked", front sequence, back sequence]: -a FRONT...BACK (front not anchored)
            _, f, b = spec
            out.append(PA.LinkedAdapter(PA.FrontAdapter(f, max_errors=e, min_overlap=o, name=f"a{i}f"),
                                        PA.BackAdapter(b, max_errors=e, min_overlap=o, name=f"a{i}b"),
                                        False, False, f"a{i}"))
        else:
            out.append(kinds[spec[0]](spec[1], max_errors=e, min_overlap=o, name=f"a{i}"))
    return out


def fastq_paired_cases():
    fastq_file("small.in.fastq")
    cases = [dict(c) for c in _FASTQ_KAT["paired_cases"]]
    for c in cases:
        c["input_bytes"] = [fastq_file(f"paired_{c['name']}.in{k}.fastq") for k in (1, 2)]
        c["expected_bytes"] = [fastq_file(f"paired_{c['name']}.out{k}.fastq") for k in (1, 2)]
    return cases


def oracle_paired(oracle, options, data1, data2):
    """oracle.oracle_fastq_trim_paired for a paired case's options."""
    import cutadapt_b200.adapters as PA

    sets = []
    for key in ("adapters1", "adapters2"):
        ads = fastq_case_adapters(options, key)
        if ads:
            spec = spec_of(PA.MultipleAdapters(ads))
            sets.append((spec.adapters, spec.groups))
        else:
            sets.append((None, None))
    return oracle.oracle_fastq_trim_paired(
        data1, data2, sets[0][0], sets[0][1], sets[1][0], sets[1][1],
        fastq_case_kwargs(options["options1"]), fastq_case_kwargs(options["options2"]), options.get("pair_filter", "any"))


def fastq_case_kwargs(options):
    """Keyword arguments shared by oracle.oracle_fastq_trim and (renamed) pipeline.FastqTrimmer."""
    kw = {}
    if "quality_cutoff" in options:
        kw.update(quality_trim=True, cutoff_front=options["quality_cutoff"][0], cutoff_back=options["quality_cutoff"][1])
    for k in ("quality_base", "nextseq_cutoff", "max_expected_errors", "discard_trimmed", "discard_untrimmed",
              "minimum_length", "maximum_length", "max_n", "times", "cut", "poly_a", "length", "trim_n",
              "discard_casava", "action"):
        if k in options:
            kw[k] = options[k]
    return kw


def fastq_demux_case():
    """tests/test_commandline.py:581-601 of the reference (FASTA vectors stored as FASTQ, see make_fastq_golden.py)."""
    return dict(adapters=[("first", "AATTTCAGGAATT"), ("second", "GTTCTCTAGTTCT")],
                input_bytes=fastq_file("demux_twoadapters.in.fastq"),
                expected={n: fastq_file(f"demux_twoadapters.{n}.out.fastq") for n in ("first", "second", "unknown")})


# ---- adapter specification strings of the reference's command line (test helper) -------------------------------

def adapter_from_spec(spec, adapter_type, name=None, **params):
    """
    One -a / -g / -b value as the reference's command line builds it (src/cutadapt/parser.py:129-149, 221-365,
    440-550): placement restrictions ^ADAPTER / ADAPTER$ / XADAPTER / ADAPTERX, x{n} repeats, linked
    ADAPTER1...ADAPTER2 (-g requires both parts, -a only the anchored ones), ...ADAPTER / ADAPTER...; name=SEQ.
    Search parameters after ';' are not supported.  Returns a cutadapt_b200 adapter object.
    """
    import re
    import cutadapt_b200.adapters as PA

    def expand_braces(seq):
        return re.sub(r"(.)\{(\d+)\}", lambda m: m.group(1) * int(m.group(2)), seq)

    def parse(one, kind):
        nm = None
        if "=" in one:
            nm, one = one.split("=", 1)
        one = expand_braces(one.strip())
        if len(one.strip("X")) == 0:
            return nm, None, one, kind
        front = back = None
        if one.startswith("^"):
            front, one = "anchored", one[1:]
        if one.upper().startswith("X"):
            assert front is None
            front, one = "noninternal", one.lstrip("xX")
        if one.endswith("$"):
            back, one = "anchored", one[:-1]
        if one.upper().endswith("X"):
            assert back is None
            back, one = "noninternal", one.rstrip("xX")
        assert not (front and back)
        assert not (kind == "front" and back) and not (kind == "back" and front) and not (kind == "anywhere" and (front or back))
        return nm, front or back, one, kind

    def cls_of(kind, restriction):
        return {("front", None): PA.FrontAdapter, ("front", "anchored"): PA.PrefixAdapter,
                ("front", "noninternal"): PA.NonInternalFrontAdapter, ("back", None): PA.BackAdapter,
                ("back", "anchored"): PA.SuffixAdapter, ("back", "noninternal"): PA.NonInternalBackAdapter,
                ("anywhere", None): PA.AnywhereAdapter}[(kind, restriction)]

    spec1, middle, spec2 = spec.partition("...")
    if middle and spec1 and spec2:
        assert adapter_type != "anywhere"
        n1, r1, s1, _ = parse(spec1, "front")
        _, r2, s2, _ = parse(spec2, "back")
        required = (True, True) if adapter_type == "front" else (r1 is not None, r2 is not None)
        return PA.LinkedAdapter(cls_of("front", r1)(s1, name="linked_front", **params),
                                cls_of("back", r2)(s2, name="linked_back", **params),
                                required[0], required[1], name or n1 or "linked")
    if middle:
        assert adapter_type != "anywhere"
        if not spec1:
            assert adapter_type == "back"
            spec = spec2
        else:
            spec = spec1
            adapter_type = "front"
    nm, restriction, seq, kind = parse(spec, adapter_type)
    return cls_of(kind, restriction)(seq, name=name or nm or "adapter", **params)


def hostsim_jit_compile(spec, plane_words=5, has_qual=False):
    """(cubin size or error code, generated source, NVRTC log) of the run-time specialisation of the first stage
    (cg_jit.cpp) for this adapter set -- NVRTC compiles for sm_100a without a device."""
    lib = hostsim_lib()
    lib.hs_jit_compile.restype = C.c_long
    lib.hs_jit_compile.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_long,
                                   C.c_char_p, C.c_long]
    ads, na, groups, ng = spec.to_ctypes()
    src = C.create_string_buffer(1 << 20)
    log = C.create_string_buffer(1 << 16)
    n = lib.hs_jit_compile(C.cast(ads, C.c_void_p), na, C.cast(groups, C.c_void_p), ng, plane_words, int(has_qual), src,
                           len(src), log, len(log))
    return n, src.value.decode(), log.value.decode()
