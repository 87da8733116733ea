"""CPU tier (with a Porechop checkout only): the REFERENCE'S OWN unittest suite (<checkout>/test/*.py, 85 CLI-level
tests -- SURVEY.md section 4) run against the two drop-ins, with the reference CLI on its own C++ as the baseline
(tests/refsuite/run_reference_suite.py).  The engine under the drop-ins is the product's own engine.cu + kernels.cuh in the
host simulation of tests/sim (`--engine sim`; `--engine oracle` uses the C restatement instead, `--engine cuda` the real
device on a GPU box that has a checkout).

  patch  (python -m porechop_b200)            every one of the 85 tests has the baseline's outcome -- including the three
                                              tests that fail against the reference itself at this commit (SURVEY 0.10)
  flat   (python -m porechop_b200.flat_cli)   identical except for tests that assert on the progress report printed to
                                              stdout / stderr, which the flat CLI does not reproduce (flat_cli.py docstring)
"""
import os
import sys

import pytest

from helpers import PORECHOP_CHECKOUT, ROOT

REF = PORECHOP_CHECKOUT
pytestmark = pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, 'test')) and
                                     os.path.exists(os.path.join(ROOT, 'oracle', '_ref', 'cpp_functions.so'))),
                                reason='needs a Porechop checkout (helpers.porechop_checkout) and oracle/_ref built from it')

# tests whose assertions include text of the reference's progress report (adapter table, "N / M reads ...", barcode table)
REPORT_TESTS = {
    'test_barcodes.TestBarcodes.test_barcodes_1', 'test_barcodes.TestBarcodes.test_barcodes_2',
    'test_barcodes.TestBarcodes.test_barcodes_3', 'test_barcodes.TestBarcodes.test_barcodes_4',
    'test_choose_barcodes.TestBarcodes.test_choose_forward', 'test_choose_barcodes.TestBarcodes.test_choose_reverse',
    'test_one_adapter_set.TestOneAdapterSet.test_adapter_threshold_1', 'test_one_adapter_set.TestOneAdapterSet.test_check_reads',
    'test_one_adapter_set.TestOneAdapterSet.test_piped_output', 'test_one_adapter_set.TestOneAdapterSet.test_verbosity_1_output',
    'test_one_adapter_set.TestOneAdapterSet.test_verbosity_2_output',
    'test_two_adapter_sets.TestTwoAdapterSets.test_check_reads_1', 'test_two_adapter_sets.TestTwoAdapterSets.test_check_reads_2',
    'test_two_adapter_sets.TestTwoAdapterSets.test_check_reads_3',
}


def test_reference_unittest_suite_outcomes_match_the_baseline():
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'refsuite'))
    try:
        import run_reference_suite as R
    finally:
        sys.path.pop(0)
    jobs = max(1, (os.cpu_count() or 2) - 1)
    base = R.run_mode('reference', 'oracle', REF, '', jobs)
    assert len(base) == 85
    failing = sorted(k for k, v in base.items() if v != 'ok')
    assert failing == ['test_albacore_directory.TestAlbacoreDirectory.test_albacore_directory_3',
                       'test_albacore_directory.TestAlbacoreDirectory.test_albacore_directory_all',
                       'test_albacore_directory.TestAlbacoreDirectory.test_albacore_directory_unclassified'], failing
    patch = R.run_mode('patch', 'sim', REF, '', jobs)         # the product's own engine code, in the host simulation (tests/sim)
    assert patch == base
    if os.environ.get('PB200_REFSUITE_FLAT', '0') != '1':
        return          # the flat CLI's run of the suite (another ~40 s; round 1: differs on exactly REPORT_TESTS) is opt-in;
                        # tests/test_flat_cli.py compares its output files with the reference CLI's in every run
    flat = R.run_mode('flat', 'sim', REF, '', jobs)
    assert sorted(flat) == sorted(base)
    differs = {k for k in base if flat[k] != base[k]}
    assert differs <= REPORT_TESTS, sorted(differs - REPORT_TESTS)
