"""
The reference's OWN test files replayed against this package.  tests/golden/make_golden.py ran each file against the
reference and recorded, per test, every call it made into the module under test with the reference's result (and
the test's time limit, if it has one); here the same calls go to cutadapt_b200's module and must give the same
results.  Results are compared as the reference's tests compare them: lists and sets without regard to order
(util.canon).  Only host-side modules are covered here -- the aligner, the k-mer finder and the adapter classes run
on the GPU library; their known answers are the other fixtures of tests/golden/.
"""
import importlib
import time

import pytest

from util import canon, golden

KAT = golden("reference_suite_kat.json.gz")
MODULES = {"test_kmer_heuristic.py": "cutadapt_b200.kmer_heuristic"}


@pytest.mark.parametrize("name", sorted(KAT))
def test_reference_test_file_passes_against_this_package(name):
    module = importlib.import_module(MODULES[name])
    tests = KAT[name]
    assert len(tests) >= 15
    for test in tests:
        t0 = time.perf_counter()
        for fn, args, kwargs, expected in test["calls"]:
            assert canon(getattr(module, fn)(*args, **kwargs)) == expected, (test["test"], fn, args, kwargs)
        if test["timeout"] is not None:
            assert time.perf_counter() - t0 < test["timeout"], test["test"]
