"""CPU tier (authoring container only): `python -m porechop_b200.flat_cli` against the UNMODIFIED reference CLI.

Both run in-process on the reference's fixture inputs and on this repo's synthetic edge-case FASTQs; every output file
must be byte-identical (gz outputs are compared after decompression).  The flat CLI takes its argument parser, adapter
table and policy functions from the reference package itself; only the data path differs (porechop_b200/fastq.py).
The oracle stands in for the engine (tests only).  Skipped without a Porechop checkout (helpers.porechop_checkout)."""
import contextlib
import gzip
import io
import os
import sys

import pytest

from helpers import load_golden
from test_patch_cli import REF, _oracle_engine, _run_cli, porechop_modules, pytestmark  # noqa: F401


def _flat_cli(A, argv, out_dir):
    from porechop_b200 import flat_cli
    for a in A.ADAPTERS:
        a.best_start_score, a.best_end_score = 0.0, 0.0
    os.makedirs(out_dir, exist_ok=True)
    old = sys.argv
    sys.argv = ['porechop'] + argv
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            flat_cli.main()
    finally:
        sys.argv = old
    files = {}
    for d, _, names in os.walk(out_dir):
        for nm in names:
            files[os.path.relpath(os.path.join(d, nm), out_dir)] = open(os.path.join(d, nm), 'rb').read()
    return files


def _plain(files):
    return {k: (gzip.decompress(v) if k.endswith('.gz') else v) for k, v in files.items()}


CASES = [
    ('one_set', 'test_one_adapter_set.fastq', ['-o', '{out}/o.fastq']),
    ('one_set_fasta_lowmid', 'test_one_adapter_set.fastq', ['-o', '{out}/o.fasta', '--middle_threshold', '70',
                                                            '--min_split_read_size', '10']),
    ('two_sets', 'test_two_adapter_sets.fastq', ['-o', '{out}/o.fastq', '--discard_middle']),
    ('barcodes', 'test_barcodes.fastq', ['-b', '{out}/bins']),
    ('barcodes_two_untrimmed', 'test_barcodes.fastq', ['-b', '{out}/bins', '--require_two_barcodes', '--untrimmed',
                                                       '--discard_unassigned']),
    ('gz_in_gz_out', 'test_format.fastq.gz', ['-o', '{out}/o.fastq.gz', '--no_split']),
    ('gz_in_bins', 'test_format_barcodes.fastq.gz', ['-b', '{out}/bins']),
    ('fasta_in_fastq_out', 'test_format.fasta', ['-o', '{out}/o.fastq']),
    ('fasta_gz_in_auto_out', 'test_format.fasta.gz', ['-o', '{out}/trimmed_reads', '--min_split_read_size', '100']),
    ('fasta_in_bins', 'test_choose_barcodes_1.fasta', ['-b', '{out}/bins']),
    ('fasta_gz_in_bins_gz', 'test_format_barcodes.fasta.gz', ['-b', '{out}/bins', '--discard_unassigned']),
    ('albacore_dir_bins', 'test_albacore_directory', ['-b', '{out}/bins']),
    ('albacore_dir_bins_opts', 'test_albacore_directory', ['-b', '{out}/bins', '--check_reads', '6', '--barcode_diff', '1',
                                                            '--discard_unassigned']),
    ('albacore_dir_single_out', 'test_albacore_directory', ['-o', '{out}/all.fasta']),
    ('empty_result_gz', 'INLINE:@only\n\n+\n\n', ['-o', '{out}/o.fastq.gz']),
    ('empty_result_plain', 'INLINE:@only\n\n+\n\n', ['-o', '{out}/o.fasta']),
    ('synthetic_edges', 'GOLDEN:input_fastq', ['-o', '{out}/o.fastq', '--min_split_read_size', '50']),
    ('synthetic_barcoded', 'GOLDEN:barcoded_fastq', ['-b', '{out}/bins', '--format', 'fasta']),
]


@pytest.mark.parametrize('name,input_name,argv', CASES, ids=[c[0] for c in CASES])
def test_flat_cli_writes_the_reference_cli_files(name, input_name, argv, porechop_modules, monkeypatch, tmp_path):  # noqa: F811
    porechop, P, A = porechop_modules
    if input_name.startswith('GOLDEN:') or input_name.startswith('INLINE:'):
        inp = str(tmp_path / 'in.fastq')
        with open(inp, 'w', newline='') as f:
            f.write(input_name[7:] if input_name.startswith('INLINE:') else load_golden('golden_emit.json')[input_name.split(':')[1]])
    else:
        inp = os.path.join(REF, 'test', input_name)

    def args_for(out):
        return ['-i', inp, '-v', '0', '-t', '1'] + [a.replace('{out}', out) for a in argv]
    _, base = _run_cli(P, A, args_for(str(tmp_path / 'a')), str(tmp_path / 'a'))
    _oracle_engine(monkeypatch)
    monkeypatch.syspath_prepend(REF)            # flat_cli imports `porechop` like a user would (already in sys.modules)
    got = _flat_cli(A, args_for(str(tmp_path / 'b')), str(tmp_path / 'b'))
    base, got = _plain(base), _plain(got)
    assert sorted(got) == sorted(base) and len(base) >= 1
    for k in base:
        assert got[k] == base[k], k


@pytest.mark.parametrize('chunk', [3000, 20000])
@pytest.mark.parametrize('input_name,argv', [('test_barcodes.fastq', ['-b', '{out}/bins', '--check_reads', '5']),
                                             ('test_format.fasta', ['-o', '{out}/o.fasta', '--check_reads', '7']),
                                             ('GOLDEN:input_fastq', ['-o', '{out}/o.fastq.gz', '--check_reads', '4',
                                                                     '--min_split_read_size', '50'])])
def test_flat_cli_streams_in_chunks(chunk, input_name, argv, porechop_modules, monkeypatch, tmp_path):  # noqa: F811
    """tiny chunks (many whole-record pieces, bins appended piece by piece): same files as the reference CLI."""
    monkeypatch.setenv('PB200_FLAT_CHUNK_BYTES', str(chunk))
    test_flat_cli_writes_the_reference_cli_files('chunked', input_name, argv, porechop_modules, monkeypatch, tmp_path)


@pytest.mark.parametrize('chunk', [3000, 1 << 20])
@pytest.mark.parametrize('input_name,argv', [('test_barcodes.fastq', ['-b', '{out}/bins']),
                                             ('test_two_adapter_sets.fastq', ['-o', '{out}/o.fastq']),
                                             ('GOLDEN:input_fastq', ['-o', '{out}/o.fastq', '--min_split_read_size', '50'])])
def test_flat_cli_phase_a_over_all_reads(chunk, input_name, argv, porechop_modules, monkeypatch, tmp_path):  # noqa: F811
    """PB200_CHECK_ALL_READS=1 (opt-in): Phase A streams over every read in bounded chunks -- same files as the reference
    CLI told to check more reads than the input holds; the flat CLI itself is given a --check_reads of 1, which the switch
    must override."""
    porechop, P, A = porechop_modules
    if input_name.startswith('GOLDEN:'):
        inp = str(tmp_path / 'in.fastq')
        with open(inp, 'w', newline='') as f:
            f.write(load_golden('golden_emit.json')[input_name.split(':')[1]])
    else:
        inp = os.path.join(REF, 'test', input_name)

    def args_for(out, check):
        return ['-i', inp, '-v', '0', '-t', '1', '--check_reads', str(check)] + [a.replace('{out}', out) for a in argv]
    _, base = _run_cli(P, A, args_for(str(tmp_path / 'a'), 1000000), str(tmp_path / 'a'))
    _oracle_engine(monkeypatch)
    monkeypatch.syspath_prepend(REF)
    monkeypatch.setenv('PB200_FLAT_CHUNK_BYTES', str(chunk))
    monkeypatch.setenv('PB200_CHECK_ALL_READS', '1')
    got = _flat_cli(A, args_for(str(tmp_path / 'b'), 1), str(tmp_path / 'b'))
    base, got = _plain(base), _plain(got)
    assert sorted(got) == sorted(base) and len(base) >= 1
    for k in base:
        assert got[k] == base[k], k


def _rank_worker(rank, world, port, argv, q):
    """one torchrun-style rank of the flat CLI on CPU: gloo for the barrier, the oracle as the engine (tests only)."""
    import numpy as np
    os.environ.update({'RANK': str(rank), 'LOCAL_RANK': str(rank), 'WORLD_SIZE': str(world), 'MASTER_ADDR': '127.0.0.1',
                       'MASTER_PORT': str(port), 'PB200_FLAT_CHUNK_BYTES': '6000'})
    try:
        from helpers import oracle_batch
        from test_patch_cli import load_reference
        load_reference()
        sys.path.insert(0, REF)
        from porechop_b200 import cpp_function_wrappers as W
        from porechop_b200 import flat_cli
        W.adapter_alignment_batch = lambda sb, so, ab, ao, sc, ps=None, pa=None, out=None: oracle_batch(
            np.asarray(sb), np.asarray(so), np.asarray(ab), np.asarray(ao), list(sc), ps, pa)
        sys.argv = ['porechop'] + argv
        with contextlib.redirect_stdout(io.StringIO()):
            flat_cli.main()
        q.put((rank, 'ok'))
    except BaseException as e:      # noqa: BLE001 -- report to the parent instead of hanging it
        q.put((rank, repr(e)))


@pytest.mark.parametrize('argv', [['-b', '{out}/bins', '--check_reads', '5'], ['-o', '{out}/o.fastq.gz', '--check_reads', '5'],
                                  ['-b', '{out}/bins', '--check_reads', '1000000', 'ALL_READS']],
                         ids=['bins', 'single_gz', 'bins_phase_a_all_reads'])
def test_flat_cli_two_ranks_gloo(argv, porechop_modules, tmp_path, monkeypatch):  # noqa: F811
    """world_size 2 on CPU (gloo): chunks alternate between the ranks, rank 0 stitches the pieces -- same files as the
    reference CLI, no leftovers."""
    import socket
    import torch.multiprocessing as mp
    porechop, P, A = porechop_modules
    inp = os.path.join(REF, 'test', 'test_barcodes.fastq')
    if 'ALL_READS' in argv:         # Phase A over every read: the ranks combine their per-set maxima (spawned ranks inherit the env)
        argv = [a for a in argv if a != 'ALL_READS']
        monkeypatch.setenv('PB200_CHECK_ALL_READS', '1')

    def args_for(out):
        return ['-i', inp, '-v', '0', '-t', '1'] + [a.replace('{out}', out) for a in argv]
    _, base = _run_cli(P, A, args_for(str(tmp_path / 'a')), str(tmp_path / 'a'))
    with socket.socket() as s_:
        s_.bind(('127.0.0.1', 0))
        port = s_.getsockname()[1]
    os.makedirs(str(tmp_path / 'b'), exist_ok=True)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, args_for(str(tmp_path / 'b')), q)) for r in range(2)]
    for p_ in procs:
        p_.start()
    results = dict(q.get(timeout=300) for _ in procs)
    for p_ in procs:
        p_.join(timeout=60)
    assert results == {0: 'ok', 1: 'ok'}
    got = {}
    for d, _, names in os.walk(str(tmp_path / 'b')):
        for nm in names:
            got[os.path.relpath(os.path.join(d, nm), str(tmp_path / 'b'))] = open(os.path.join(d, nm), 'rb').read()
    base, got = _plain(base), _plain(got)
    assert sorted(got) == sorted(base), sorted(got)
    for k in base:
        assert got[k] == base[k], k
