"""
Parity at the gate BASELINE.md states: >= 10^6 synthetic reads per benchmark configuration against the C oracle
(oracle_process_packed: the oracle's per-read pass as one C loop, run from all host threads) and >= 10^5 against
the reference itself.  The reads are the generators of cutadapt_b200.configs (SURVEY.md section 8(d)).  The
reference's answers are stored (tests/golden/gate_reference_kat.json.gz, made by make_golden.py): they belong to the
first 10^5 reads each generator draws on the CPU, so that part of each test trims reads drawn on the CPU.
"""
import numpy as np
import pytest

from cutadapt_b200 import _lib as L
from oracle import oracle
from util import batch_digest, digest, golden, match_desc

pytestmark = pytest.mark.gpu

N_GATE = 1_000_000
N_REF = 100_000


def _flat(multi):
    singles, groups, owners = multi._flatten()
    multi._device_set = (None, singles, owners)        # lets matches_from_records() map records back to objects
    return [s.descriptor() for s in singles], groups


def _packed(t):
    host = np.ascontiguousarray(t.cpu().numpy()).reshape(-1)
    n, L_ = t.shape
    return host, np.arange(n + 1, dtype=np.int64) * L_


def _coords(rec):
    return None if rec["adapter"] < 0 else [int(rec[f]) for f in ("astart", "astop", "rstart", "rstop", "score", "errors")]


def _reference_batch(config):
    """The reads the stored reference answers of `config` belong to."""
    from cutadapt_b200.configs import make_config_batch

    ref = golden("gate_reference_kat.json.gz")[str(config)]
    assert ref["n"] == (N_REF // 2 if config == 4 else N_REF)
    b = make_config_batch(config, ref["n"], device="cpu")
    assert batch_digest(b) == ref["reads_digest"], "the generator no longer draws the reads the answers belong to"
    return b


def _assert_reference_rows(config, key, rows):
    """One row per read against the reference's: row by row over the stored sample, all rows through the digest."""
    ref = golden("gate_reference_kat.json.gz")[str(config)][key]
    for i, (have, want) in enumerate(zip(rows, ref["sample"])):
        assert have == want, (config, key, i)
    assert digest(rows) == ref["digest"], (config, key, "differs from the reference after the stored sample")


def test_gate_config2_one_adapter():
    from cutadapt_b200.configs import config_adapters, make_config_batch

    multi, _ = config_adapters(2)
    descs, groups = _flat(multi)
    seq = make_config_batch(2, N_GATE, device="cuda")["seq"]
    data, offsets = _packed(seq)
    aset = L.AdapterSet(L.AdapterSetSpec(descs, groups))
    got, _ = aset.process(data, offsets)
    exp, _ = oracle.oracle_process_packed(descs, groups, data, offsets)
    assert (got == exp).all()
    assert 0.45 < (got["adapter"][:, 0, 0] >= 0).mean() < 0.56
    got, _ = aset.process(*_packed(_reference_batch(2)["seq"]))
    _assert_reference_rows(2, "seq", [_coords(rec) for rec in got[:, 0, 0]])


def test_gate_config3_five_adapters():
    from cutadapt_b200.configs import config_adapters, make_config_batch, to_strings

    multi, _ = config_adapters(3)
    descs, groups = _flat(multi)
    seq = make_config_batch(3, N_GATE, device="cuda")["seq"]
    data, offsets = _packed(seq)
    aset = L.AdapterSet(L.AdapterSetSpec(descs, groups))
    got, _ = aset.process(data, offsets)
    exp, _ = oracle.oracle_process_packed(descs, groups, data, offsets)
    assert (got == exp).all()
    hit = (got["adapter"][:, 0, :] >= 0).any(axis=1)
    assert 0.4 < hit.mean() < 0.8
    # every construct is found: each of the five groups wins for a good share of the reads
    grp = got["info"][:, 0, :].max(axis=1) & 255
    for g in range(5):
        assert (hit & (grp == g)).mean() > 0.03, g
    seq = _reference_batch(3)["seq"]
    got, _ = aset.process(*_packed(seq))
    _assert_reference_rows(3, "seq", [match_desc(multi.matches_from_records(got[i, 0], read))
                                      for i, read in enumerate(to_strings(seq))])


def test_gate_config4_pairs_with_quality_trimming():
    from cutadapt_b200.configs import config_adapters, make_config_batch

    m1, m2 = config_adapters(4)
    n_pairs = N_GATE // 2
    b = make_config_batch(4, n_pairs, device="cuda")
    rb = _reference_batch(4)
    for multi, skey, qkey in ((m1, "seq", "qual"), (m2, "seq2", "qual2")):
        descs, groups = _flat(multi)
        data, offsets = _packed(b[skey])
        qdata, _ = _packed(b[qkey])
        aset = L.AdapterSet(L.AdapterSetSpec(descs, groups))
        params = L.make_params(quality_trim=True, cutoff_front=0, cutoff_back=20)
        got, gqt = aset.process(data, offsets, qdata, params)
        exp, eqt = oracle.oracle_process_packed(descs, groups, data, offsets, qdata, True, 0, 20)
        assert (gqt == eqt).all() and (got == exp).all(), skey
        assert 0.4 < (got["adapter"][:, 0, 0] >= 0).mean() < 0.6
        data, offsets = _packed(rb[skey])
        got, gqt = aset.process(data, offsets, _packed(rb[qkey])[0], params)
        _assert_reference_rows(4, skey, [[int(s), int(e), _coords(rec)] for (s, e), rec in zip(gqt, got[:, 0, 0])])


def test_gate_config5_barcode_index_with_indels():
    """96 anchored 5' barcodes, e = 0.1 with indels: the device index against the oracle's own index (built from the
    oracle's edit environment) on 10^6 reads, and against the reference's IndexedPrefixAdapters."""
    from cutadapt_b200.configs import config_adapters, config5_barcodes, make_config_batch

    multi, _ = config_adapters(5)
    seq = make_config_batch(5, N_GATE, device="cuda")["seq"]
    data, offsets = _packed(seq)
    singles, groups, _ = multi._flatten()
    spec = L.AdapterSetSpec([s.descriptor() for s in singles], groups, multi._flatten_indexes())
    aset = L.AdapterSet(spec)
    got, _ = aset.process(data, offsets)
    barcodes = config5_barcodes()
    exp = oracle.oracle_index_process(barcodes, 0.1, True, True, data, offsets, spec.adapters)
    assert (got["adapter"][:, 0, 0] == exp["adapter"]).all()
    for f in ("astart", "astop", "rstart", "rstop", "score", "errors"):
        assert (got[f][:, 0, 0] == exp[f]).all(), f
    assert 0.95 < (got["adapter"][:, 0, 0] >= 0).mean() < 0.995
    got, _ = aset.process(*_packed(_reference_batch(5)["seq"]))
    _assert_reference_rows(5, "seq", [None if rec["adapter"] < 0 else [int(rec["adapter"])] + _coords(rec)
                                      for rec in got[:, 0, 0]])
