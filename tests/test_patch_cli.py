"""CPU tier (authoring container only): the run-time drop-in `porechop_b200.patch` under the UNMODIFIED reference CLI.

The reference's own `main()` (porechop/porechop.py:33-79, imported from a Porechop checkout) runs its fixture inputs twice:
  baseline  its per-call path on the reference C++ (oracle/_ref/cpp_functions.so),
  patched   with `patch.install()`: one prefetch batch per phase, the original drivers unchanged.
Everything the CLI writes -- stdout (progress, verbose alignments, summaries) and every output file -- must be
byte-identical, and the patched run must not have fallen through to a per-call alignment (memo.misses == 0).

There is no GPU in this tier, so the engine's two entry points are replaced by the oracle for the duration of the
test (the oracle as checker, tests only); the same comparison against the real engine is tests/test_gpu_phases.py's
job through the golden vectors.  Skipped without a Porechop checkout.
"""
import contextlib
import ctypes
import io
import os
import sys
import types
import warnings

import numpy as np
import pytest

from helpers import PORECHOP_CHECKOUT, ROOT, oracle_batch, oracle_string

REF = PORECHOP_CHECKOUT
REF_SO = os.path.join(ROOT, 'oracle', '_ref', 'cpp_functions.so')
pytestmark = pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, 'porechop')) and os.path.exists(REF_SO)),
                                reason='needs a Porechop checkout (helpers.porechop_checkout) and oracle/_ref built from it')


def load_reference():
    """Import the reference package with `porechop.cpp_function_wrappers` bound to oracle/_ref/cpp_functions.so (the
    reference's wrapper insists on a .so inside its own read-only tree; nothing of the reference is modified)."""
    warnings.simplefilter('ignore')
    lib = ctypes.CDLL(REF_SO)
    lib.adapterAlignment.argtypes = [ctypes.c_char_p, ctypes.c_char_p] + [ctypes.c_int] * 4
    lib.adapterAlignment.restype = ctypes.c_void_p
    lib.freeCString.argtypes = [ctypes.c_void_p]

    def adapter_alignment(read_sequence, adapter_sequence, scoring_scheme_vals):
        p = lib.adapterAlignment(read_sequence.encode(), adapter_sequence.encode(), *scoring_scheme_vals)
        s = ctypes.cast(p, ctypes.c_char_p).value.decode()
        lib.freeCString(p)
        return s

    sys.path.insert(0, REF)
    try:
        stub = types.ModuleType('porechop.cpp_function_wrappers')
        stub.adapter_alignment = adapter_alignment
        import porechop
        sys.modules['porechop.cpp_function_wrappers'] = stub
        from porechop import porechop as P
        from porechop import adapters as A
    finally:
        sys.path.remove(REF)
    return porechop, P, A


@pytest.fixture(scope='module')
def porechop_modules():
    return load_reference()


def _run_cli(P, A, argv, out_dir):
    """reference main() in-process; returns (stdout text, {relative file name: bytes})."""
    for a in A.ADAPTERS:
        a.best_start_score, a.best_end_score = 0.0, 0.0
    os.makedirs(out_dir, exist_ok=True)
    old_argv, buf = sys.argv, io.StringIO()
    sys.argv = ['porechop'] + argv
    try:
        with contextlib.redirect_stdout(buf), warnings.catch_warnings():
            warnings.simplefilter('ignore')
            P.main()
    finally:
        sys.argv = old_argv
    files = {}
    for d, _, names in os.walk(out_dir):
        for nm in names:
            p = os.path.join(d, nm)
            files[os.path.relpath(p, out_dir)] = open(p, 'rb').read()
    return buf.getvalue(), files


def _oracle_engine(monkeypatch):
    from porechop_b200 import cpp_function_wrappers as W

    def batch(seq_buf, seq_off, ad_buf, ad_off, scoring, pair_seq=None, pair_adapter=None, out=None):
        return oracle_batch(np.asarray(seq_buf), np.asarray(seq_off), np.asarray(ad_buf), np.asarray(ad_off), list(scoring),
                            pair_seq, pair_adapter)
    monkeypatch.setattr(W, 'adapter_alignment_batch', batch)
    monkeypatch.setattr(W, 'adapter_alignment', lambda r, a, sc: oracle_string(r, a, list(sc)))


CASES = [
    ('one_set_v2', ['-i', 'test_one_adapter_set.fastq', '-o', '{out}/o.fastq', '-v', '2', '-t', '1']),
    ('one_set_lowmid', ['-i', 'test_one_adapter_set.fastq', '-o', '{out}/o.fasta', '-v', '3', '-t', '1',
                        '--middle_threshold', '70', '--min_split_read_size', '10']),
    ('two_sets_threads', ['-i', 'test_two_adapter_sets.fastq', '-o', '{out}/o.fastq', '-v', '1', '-t', '4']),
    ('barcodes', ['-i', 'test_barcodes.fastq', '-b', '{out}/bins', '-v', '2', '-t', '1']),
    ('barcodes_two', ['-i', 'test_barcodes.fastq', '-b', '{out}/bins', '-v', '0', '-t', '2', '--require_two_barcodes',
                      '--discard_middle']),
    ('nosplit', ['-i', 'test_format.fastq.gz', '-o', '{out}/o.fastq', '-v', '1', '-t', '1', '--no_split']),
]


@pytest.mark.parametrize('name,argv', CASES, ids=[c[0] for c in CASES])
def test_reference_cli_identical_with_patch(name, argv, porechop_modules, monkeypatch, tmp_path):
    porechop, P, A = porechop_modules
    from porechop_b200 import patch

    def args_for(out):
        return [a.replace('{out}', out) if '{out}' in a else
                (os.path.join(REF, 'test', a) if a.startswith('test_') else a) for a in argv]

    base_out, base_files = _run_cli(P, A, args_for(str(tmp_path / 'a')), str(tmp_path / 'a'))
    _oracle_engine(monkeypatch)
    memo = patch.install(porechop)
    try:
        got_out, got_files = _run_cli(P, A, args_for(str(tmp_path / 'b')), str(tmp_path / 'b'))
    finally:
        patch.uninstall(memo)
    # the two runs write to sibling directories .../a and .../b (same length, so column padding is unaffected)
    assert got_out.replace(str(tmp_path / 'b'), str(tmp_path / 'a')).replace('/b/bins', '/a/bins') == base_out
    assert sorted(got_files) == sorted(base_files) and len(base_files) >= 1
    for k in base_files:
        assert got_files[k] == base_files[k], k
    assert memo.misses == 0 and memo.hits > 0
    assert 2 <= memo.batches <= 12          # a handful of submits for the whole run, not one per alignment
