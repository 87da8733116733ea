"""CPU tier: the PRODUCT'S OWN engine -- engine.cu's host logic and every kernel of kernels.cuh, as written -- executed on
the host by tests/sim (a stand-in for the CUDA runtime and execution model: one fiber per CUDA thread, warp collectives as
rendezvous points; pbsim_cuda.h, build_sim.py), called through the product's ctypes wrapper and compared with the oracle.

tests/test_emulation.py checks the arithmetic of dp_core.cuh lane by lane; this file checks what that cannot see: the
kernels' orchestration (hot / careful chunks, trace addressing, staging rings, dynamic slot refill, task synthesis, the
two-pass launch sequences, the chunk pipeline of the host API) and every opt-in path of DESIGN.md section 5c end to end
through the C-ABI.  The simulated library is test infrastructure: nothing in porechop_b200/ builds or loads it."""
import os
import random
import sys

import numpy as np
import pytest

from helpers import DEFAULT, PORECHOP_CHECKOUT, ROOT, load_golden, oracle_batch
from test_oracle import SURVEY_EDGE, rebuild_fullread_inputs

sys.path.insert(0, os.path.join(ROOT, 'tests', 'sim'))

OPTION_DEFAULTS = {'h2d_pack': 0, 'tight_window': 1, 'profile': 1, 'direct_max': 160,
                   'chunk_tasks': 131072, 'pack_threads': 8, 'scratch_mb': 128, 'hbuf': 'auto'}


@pytest.fixture(scope='module')
def W():
    import sim_engine
    w = sim_engine.load()
    assert w.device_count() == 1
    return w


def _with(W, opts, fn):
    try:
        for k, v in opts.items():
            W.set_option(k, v)
        return fn()
    finally:
        for k in opts:
            W.set_option(k, OPTION_DEFAULTS[k])


def _windows(n, seed, ads=None):
    from porechop_b200 import workloads as wl
    yt, yb = ads or wl.nsk007()
    _, sw, ew = wl.synth_end_windows(n, yt, yb, seed=seed)
    return wl.windows_to_batch(sw), wl.windows_to_batch(ew)


def test_sim_legacy_strings_and_golden_pairs(W):
    for rd, ad, exp in SURVEY_EDGE:
        assert W.adapter_alignment(rd, ad, DEFAULT) == exp
    g = load_golden('golden_random.json')
    for rd, ad, sc, exp in g[:120]:
        assert W.adapter_alignment(rd, ad, sc) == exp
    by_scheme = {}
    for rd, ad, sc, exp in g[:1500]:
        by_scheme.setdefault(tuple(sc), []).append((rd, ad, exp))
    for sc, cases in by_scheme.items():                          # pair-list mode: every row-capacity class, generic int32 path
        sbuf, soff = W.pack_sequences([c[0] for c in cases])
        abuf, aoff = W.pack_sequences([c[1] for c in cases], offset_dtype=np.int32)
        idx = np.arange(len(cases), dtype=np.int32)
        recs = W.adapter_alignment_batch(sbuf, soff, abuf, aoff, list(sc), idx, idx)
        for k, c in enumerate(cases):
            assert W.format_record(recs[k]) == c[2], (sc, c[0], c[1])


def test_sim_end_windows_demux_cross_and_ragged(W):
    from porechop_b200 import workloads as wl
    yt, yb = wl.nsk007()
    (sb, so), (eb, eo) = _windows(1200, 3)
    for (buf, off), ad in (((sb, so), yt), ((eb, eo), yb)):
        abuf, aoff = wl.pack_adapters([ad])
        for opts in ({}, {'chunk_tasks': 500}, {'scratch_mb': 1}, {'hbuf': 'global'}):
            got = _with(W, opts, lambda: W.adapter_alignment_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING))
            assert np.array_equal(got, oracle_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING)), opts
    starts, ends = wl.demux_adapters()
    (sb, so), (eb, eo) = _windows(24, 5, (starts[5], ends[5]))
    for (buf, off), ads in (((sb, so), starts), ((eb, eo), ends)):        # all 356 adapters: every class, paired + odd adapters
        abuf, aoff = wl.pack_adapters(ads)
        got = W.adapter_alignment_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING)
        assert np.array_equal(got, oracle_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING))
    rng = random.Random(3)
    reads = ['', 'A', 'N' * 20, '-' * 20, 'acgu' * 10, yt, yt[5:], 'GG' + yt + 'GG', 'ACGT' * 300]
    reads += [''.join(rng.choice('ACGTN') for _ in range(rng.randint(1, 400))) for _ in range(120)]
    ads = ['', 'A', yt, 'GCAATACGTAACTGAACGAAGT', 'ACGT' * 10, 'N' * 5, 'ACGT' * 30, 'ACGT' * 60]
    sbuf, soff = W.pack_sequences(reads)
    abuf, aoff = W.pack_sequences(ads, offset_dtype=np.int32)
    for sc in ([3, -6, -5, -2], [3, -6, -5, -5], [2, -3, -2, -5], [3, -6, 1, -2]):      # the last one: generic int32 kernel
        got = W.adapter_alignment_batch(sbuf, soff, abuf, aoff, sc)
        assert np.array_equal(got, oracle_batch(sbuf, soff, abuf, aoff, sc)), sc


def test_sim_long_reads_two_pass_and_options(W):
    """score_kernel (dynamic slot refill, staging ring, longest-first order) -> window_tasks_kernel -> trace_kernel; the
    golden full-read cases incl. masked re-alignments; then the same reads with every second-pass / score-pass option."""
    from porechop_b200 import workloads as wl
    sc, cases = rebuild_fullread_inputs()
    reads = [c[0] for c in cases]
    ads = sorted(set(c[1] for c in cases))
    sbuf, soff = W.pack_sequences(reads)
    abuf, aoff = W.pack_sequences(ads, offset_dtype=np.int32)
    ps = np.arange(len(cases), dtype=np.int32)
    pa = np.array([ads.index(c[1]) for c in cases], dtype=np.int32)
    recs = W.adapter_alignment_batch(sbuf, soff, abuf, aoff, sc, ps, pa)
    for k, c in enumerate(cases):
        assert W.format_record(recs[k]) == c[2]
    yt, yb = wl.nsk007()
    full = wl.demux_adapters()[0][-1]
    buf, off = wl.synth_reads(10, yt, yb, seed=11, chimera_p=0.4, max_len=4000)
    rng = random.Random(2)
    short = [''.join(rng.choice('ACGTN') for _ in range(rng.randint(520, 900))) for _ in range(5)] + ['', 'ACGT' * 200]
    sb2, so2 = W.pack_sequences(short)
    buf = np.concatenate([buf, sb2]); off = np.concatenate([off, so2[1:] + off[-1]])
    sets = [s_ for s_ in wl.load_adapter_sets()['sets'] if s_['name'].endswith('(forward)')][:2]
    bcs = [s_['start'][1] for s_ in sets] + [s_['end'][1] for s_ in sets]
    for ads in ([yt, yb], [yt, yb, full], bcs):
        abuf, aoff = wl.pack_adapters(ads)
        for scheme in (wl.DEFAULT_SCORING, (3, -6, -5, -5)):
            exp = oracle_batch(buf, off, abuf, aoff, scheme)
            for opts in ({}, {'tight_window': 0}, {'profile': 0}, {'profile': 0, 'tight_window': 0},
                         {'h2d_pack': 1, 'chunk_tasks': 10}):
                got = _with(W, opts, lambda: W.adapter_alignment_batch(buf, off, abuf, aoff, scheme))
                assert np.array_equal(got, exp), (len(ads), scheme, opts)
    # BASELINE config 5 shape (bench.py --workload sweep): fixed-length reads x the 192 forward barcode sequences
    bcs = wl.forward_barcode_sequences()
    a5, o5 = wl.pack_adapters(bcs)
    for L in (500, 2000, 6000):
        b5, f5 = wl.synth_fixed_length_reads(3, L, bcs, seed=L)
        exp = oracle_batch(b5, f5, a5, o5, wl.DEFAULT_SCORING)
        for opts in ({}, {'profile': 0, 'tight_window': 0}):
            got = _with(W, opts, lambda: W.adapter_alignment_batch(b5, f5, a5, o5, wl.DEFAULT_SCORING))
            assert np.array_equal(got, exp), (L, opts)
    # one pass over multi-kb sequences with the bases staged in global scratch (no score pass)
    abuf, aoff = wl.pack_adapters([yt, yb])
    got = _with(W, {'hbuf': 'global', 'direct_max': 100000}, lambda: W.adapter_alignment_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING))
    assert np.array_equal(got, oracle_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING))


def test_sim_forced_two_pass_windows_small_classes_and_packed_upload(W):
    """150-column windows forced through the two-pass path (direct_max = 100: score pass -> bounded windows -> trace pass),
    both window bounds; global staging; h2d_pack over several chunks; one- / two-adapter and odd classes on ragged inputs;
    the demux cross product."""
    from porechop_b200 import workloads as wl
    yt, yb = wl.nsk007()
    (sb, so), (eb, eo) = _windows(1000, 19)
    for (buf, off), ad in (((sb, so), yt), ((eb, eo), yb)):
        abuf, aoff = wl.pack_adapters([ad])
        exp = oracle_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING)
        for opts in ({'direct_max': 100}, {'direct_max': 100, 'tight_window': 0}, {'hbuf': 'global'},
                     {'h2d_pack': 1, 'chunk_tasks': 300, 'pack_threads': 3}, {'direct_max': 100, 'h2d_pack': 1}):
            got = _with(W, opts, lambda: W.adapter_alignment_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING))
            assert np.array_equal(got, exp), opts
    starts, ends = wl.demux_adapters()
    (sb, so), _ = _windows(24, 6, (starts[5], ends[5]))
    abuf, aoff = wl.pack_adapters(starts)
    got = W.adapter_alignment_batch(sb, so, abuf, aoff, wl.DEFAULT_SCORING)
    assert np.array_equal(got, oracle_batch(sb, so, abuf, aoff, wl.DEFAULT_SCORING))
    rng = random.Random(17)
    reads = ['', 'A', 'N' * 120, '-' * 130, 'acgu' * 40, yt, 'GG' + yt + 'GG', 'ACGT' * 100]
    reads += [''.join(rng.choice('ACGTN') for _ in range(rng.randint(1, 500))) for _ in range(100)]
    ads = ['', 'A', yt, yb, 'ACGT' * 10, 'N' * 5, 'ACGT' * 30]
    rbuf, roff = W.pack_sequences(reads)
    abuf, aoff = W.pack_sequences(ads, offset_dtype=np.int32)
    for sc in ([3, -6, -5, -2], [3, -6, -5, -5], [5, -4, -8, -1]):
        exp = oracle_batch(rbuf, roff, abuf, aoff, sc)
        for opts in ({}, {'direct_max': 120}, {'direct_max': 120, 'profile': 0}):
            got = _with(W, opts, lambda: W.adapter_alignment_batch(rbuf, roff, abuf, aoff, sc))
            assert np.array_equal(got, exp), (sc, opts)
    (sb5, so5), _ = _windows(12, 6, (starts[5], ends[5]))
    for ads in (ends[:40], starts[:4], starts[:5], [yt, yb, starts[-1]]):
        abuf, aoff = wl.pack_adapters(ads)
        exp = oracle_batch(sb5, so5, abuf, aoff, wl.DEFAULT_SCORING)
        for opts in ({}, {'direct_max': 100}):
            got = _with(W, opts, lambda: W.adapter_alignment_batch(sb5, so5, abuf, aoff, wl.DEFAULT_SCORING))
            assert np.array_equal(got, exp), (len(ads), opts)
    for ads in (['ACGT' * 5], [yt], [yt, yb], ['ACGTTGCA' * 5, 'TTGACCA' * 5], ['ACGT' * 16], [yt, ''], ['N' * 22]):
        abuf, aoff = W.pack_sequences(ads, offset_dtype=np.int32)
        for sc in ([3, -6, -5, -2], [3, -6, -5, -5]):
            exp = oracle_batch(rbuf, roff, abuf, aoff, sc)
            for opts in ({}, {'direct_max': 200}):
                got = _with(W, opts, lambda: W.adapter_alignment_batch(rbuf, roff, abuf, aoff, sc))
                assert np.array_equal(got, exp), (ads, sc, opts)


def test_sim_multi_submit_and_device_resident_api(W):
    from porechop_b200 import workloads as wl
    yt, yb = wl.nsk007()
    starts, ends = wl.demux_adapters()
    (sb, so), (eb, eo) = _windows(1500, 3)
    (sb2, so2), (eb2, eo2) = _windows(60, 4, (starts[7], ends[7]))
    lbuf, loff = wl.synth_reads(6, yt, yb, seed=6, chimera_p=0.5, max_len=4000)
    batches = [(sb, so) + wl.pack_adapters([yt]), (eb, eo) + wl.pack_adapters([yb]),
               (sb2, so2) + wl.pack_adapters(starts[:20]),
               (np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.int64)) + wl.pack_adapters([yt]),
               (eb2, eo2) + wl.pack_adapters(ends[:13]), (lbuf, loff) + wl.pack_adapters([yt, yb]),
               (sb2, so2) + wl.pack_adapters(starts[40:47])]
    for opts in ({'chunk_tasks': 500}, {'chunk_tasks': 500, 'h2d_pack': 1, 'tight_window': 0, 'profile': 0}):
        got = _with(W, opts, lambda: W.adapter_alignment_batch_multi(batches, wl.DEFAULT_SCORING))
        for b, g in zip(batches, got):
            assert np.array_equal(g, oracle_batch(b[0], b[1], b[2], b[3], wl.DEFAULT_SCORING)), opts
    # device-resident API (device memory is host memory in the simulation): windows and long reads
    for buf, off, ads in ((sb, so, [yt]), (lbuf, loff, [yt, yb])):
        abuf, aoff = wl.pack_adapters(ads)
        buf, off = np.ascontiguousarray(buf), np.ascontiguousarray(off, dtype=np.int64)
        out = np.zeros(((len(off) - 1) * len(ads), 9), dtype=np.int32)
        for max_len in (int(np.diff(off).max()), -1):
            out[:] = 0
            W.adapter_alignment_batch_device(buf.ctypes.data, off.ctypes.data, len(off) - 1, len(buf), max_len, abuf, aoff,
                                             wl.DEFAULT_SCORING, out.ctypes.data, 0)
            W.synchronize()
            assert np.array_equal(out, oracle_batch(buf, off, abuf, aoff, wl.DEFAULT_SCORING))


def test_sim_end_decisions_and_flat_pipeline(W, monkeypatch):
    """adapterEndDecisions through the simulated engine (decide_kernel in the chunk pipeline) equals the host rule on the
    records; the flat pipeline's reference-CLI goldens with the simulated engine, records path and device decisions."""
    from porechop_b200 import fastq, hostio, workloads as wl
    from porechop_b200.align import _percent_exact
    starts, ends = wl.demux_adapters()
    ads_s = [starts[0], starts[3], starts[100], starts[150], 'ACGT', starts[-1]]
    ads_e = [ends[0], ends[100], ends[-1]]
    (sb, so), (eb, eo) = _windows(700, 8, (starts[100], ends[100]))
    rng = np.random.default_rng(4)

    def ragged(buf, off):
        lens = np.diff(off).copy()
        lens[::37] = 0
        lens[5::41] = rng.integers(1, 60, len(lens[5::41]))
        off2 = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        keep = np.repeat(np.arange(len(lens)) * 150, lens) + (np.arange(int(lens.sum())) - np.repeat(off2[:-1], lens))
        return np.ascontiguousarray(buf[keep]), off2
    (sb, so), (eb, eo) = ragged(sb, so), ragged(eb, eo)
    sa, sao = wl.pack_adapters(ads_s)
    ea, eao = wl.pack_adapters(ads_e)
    srec = W.adapter_alignment_batch(sb, so, sa, sao, wl.DEFAULT_SCORING).reshape(-1, len(ads_s), 9)
    erec = W.adapter_alignment_batch(eb, eo, ea, eao, wl.DEFAULT_SCORING).reshape(-1, len(ads_e), 9)
    scols, ecols = [2, 0, 5, 2], [1]
    for end_size, extra, thr, min_trim, opts in ((150, 2, 75.0, 4, {}), (150, 0, 90.0, 1, {'chunk_tasks': 900}),
                                                 (150, 5, 50.0, 10, {'h2d_pack': 1})):
        outs = _with(W, opts, lambda: W.adapter_end_decisions(
            [(sb, so, sa, sao, True, scols), (eb, eo, ea, eao, False, ecols)], wl.DEFAULT_SCORING, end_size, extra, thr,
            min_trim, want_records=True))
        for (trim, pairs, rec), full_rec, is_start, cols in ((outs[0], srec, True, scols), (outs[1], erec, False, ecols)):
            assert np.array_equal(rec.reshape(full_rec.shape), full_rec)
            assert np.array_equal(trim.astype(np.int64), hostio.end_trim(full_rec, is_start, end_size, extra, thr, min_trim))
            got = _percent_exact(pairs[:, :, 0], pairs[:, :, 1])
            assert np.array_equal(got, hostio.full_scores(full_rec, cols), equal_nan=True)
    with pytest.raises(W.EngineError) as e:                    # a window longer than end_size is refused before any launch
        W.adapter_end_decisions([(sb, so, sa, sao, True, [])], wl.DEFAULT_SCORING, 100, 2, 75.0, 4)
    assert 'error 102' in str(e.value)
    bad = so.copy(); bad[400] = bad[399] - 5
    with pytest.raises(W.EngineError) as e:                    # offsets are checked chunk by chunk while the pipeline runs
        _with(W, {'chunk_tasks': 600}, lambda: W.adapter_alignment_batch(sb, bad, sa, sao, wl.DEFAULT_SCORING))
    assert 'error 102' in str(e.value) and 'not monotone' in str(e.value)
    # the flat FASTQ pipeline on the simulated engine: reference-CLI output files, byte for byte
    import test_fastq_emit as T
    monkeypatch.setattr(fastq, 'W', W)
    for dd in (False, True):
        monkeypatch.setattr(fastq, 'DEVICE_DECISIONS', dd)
        T._run(T.CASES[0] if dd else T.CASES[1])
        T._run_demux(T.BARCODE_CASES[1] if dd else T.BARCODE_CASES[0])


# ---- the GPU tier's own test functions, run on the simulated engine -------------------------------------------------
# (same code, same sizes as on the B200; excluded: tests that need torch CUDA tensors, 10^6-read properties and threads)
GPU_PARITY = ['test_legacy_single_call_strings', 'test_golden_random_pair_list', 'test_golden_windows_cross',
              'test_golden_fullread_two_pass', 'test_synthetic_windows_vs_oracle', 'test_demux_cross_all_adapters_vs_oracle',
              'test_ragged_and_edge_inputs', 'test_long_reads_two_pass_vs_oracle', 'test_read_length_sweep_barcodes',
              'test_score_pass_with_and_without_query_profile', 'test_generic_int32_path', 'test_single_pass_long_windows_and_global_staging']
GPU_OPTIONS = ['test_packed_upload_windows_ragged_and_long_reads', 'test_tight_window_long_reads_and_forced_two_pass_windows',
               'test_multi_batch_submit_equals_single_calls',
               'test_end_decisions_on_device_equal_host_rule', 'test_bad_sequence_offsets_fail_cleanly_mid_pipeline',
               'test_query_profile_score_pass_equals_oracle', 'test_small_and_odd_classes_ragged_inputs_both_stagings',
               'test_global_staging_under_load_every_window_length_mod_4']


# the larger ones take minutes in the simulation (10 min for all): run with PB200_SIM_FULL=1; the dedicated tests above
# cover the same paths at smaller sizes.  Round 1, final build: all 33 tests of this file pass with PB200_SIM_FULL=1
# PB200_SIM_ASAN=1 (915 s).
SLOW = {'test_demux_cross_all_adapters_vs_oracle', 'test_multi_batch_submit_equals_single_calls',
        'test_end_decisions_on_device_equal_host_rule',
        'test_bad_sequence_offsets_fail_cleanly_mid_pipeline', 'test_query_profile_score_pass_equals_oracle',
        'test_small_and_odd_classes_ragged_inputs_both_stagings', 'test_global_staging_under_load_every_window_length_mod_4'}
FULL = os.environ.get('PB200_SIM_FULL', '0') == '1'


def _maybe_slow(name):
    if name in SLOW and not FULL:
        pytest.skip('minutes in the simulation: set PB200_SIM_FULL=1')


@pytest.mark.parametrize('name', GPU_PARITY)
def test_sim_runs_gpu_parity_test(W, name):
    _maybe_slow(name)
    import test_gpu_parity as T
    getattr(T, name)(W)


@pytest.mark.parametrize('name', GPU_OPTIONS)
def test_sim_runs_gpu_option_test(W, name):
    _maybe_slow(name)
    import test_gpu_zz_options as T
    getattr(T, name)(W)


@pytest.mark.parametrize('case_index', [0, 1, 2, 3])
def test_sim_runs_gpu_phase_drivers(W, monkeypatch, case_index):
    import test_gpu_phases as T
    from porechop_b200 import phases
    monkeypatch.setattr(phases, 'W', W)
    T.test_phases_match_reference(case_index)


@pytest.mark.skipif(os.environ.get('PB200_SIM_ASAN', '0') != '1', reason='2 minutes: set PB200_SIM_ASAN=1 (round 1: clean)')
def test_sim_engine_under_address_sanitizer():
    """tests/sim/asan_check.py: the simulated engine compiled with -fsanitize=address, default and opt-in paths once -- no
    out-of-bounds access of any kernel on the "device" heap blocks, the shared-memory arrays or the stacks."""
    import subprocess
    import build_sim
    lib = build_sim.build_asan()
    asan = subprocess.check_output(['gcc', '-print-file-name=libasan.so']).decode().strip()
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS='detect_leaks=0:detect_stack_use_after_return=0', PB200_SIM_ASAN_LIB=lib)
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'sim', 'asan_check.py')], env=env, capture_output=True, text=True)
    assert r.returncode == 0 and 'ASAN RUN COMPLETE' in r.stdout and 'DIFFERENT' not in r.stdout, r.stdout[-1500:] + r.stderr[-3000:]
    assert 'ERROR: AddressSanitizer' not in r.stderr


# ---- the two CLI drop-ins on the simulated engine (the other CPU tests of these files use the oracle as the engine) ----
def _sim_as_engine(W):
    def install(monkeypatch):
        from porechop_b200 import cpp_function_wrappers as real
        for name in ('adapter_alignment_batch', 'adapter_alignment', 'adapter_alignment_batch_multi', 'adapter_end_decisions'):
            monkeypatch.setattr(real, name, getattr(W, name))
    return install


@pytest.mark.skipif(not (PORECHOP_CHECKOUT and os.path.isdir(os.path.join(PORECHOP_CHECKOUT, 'porechop'))),
                    reason='needs a Porechop checkout (helpers.porechop_checkout)')
def test_sim_engine_under_the_unmodified_cli_and_the_flat_cli(W, monkeypatch, tmp_path):
    """tests/test_patch_cli.py and tests/test_flat_cli.py compare the drop-ins with the reference CLI byte for byte, with the
    oracle standing in for the engine; here the same comparisons run on the product's engine code (host simulation): the
    reference's stdout + output files under `python -m porechop_b200`, the output files of the flat CLI."""
    import test_flat_cli as F
    import test_patch_cli as P
    mods = P.load_reference()
    install = _sim_as_engine(W)
    monkeypatch.setattr(P, '_oracle_engine', install)
    monkeypatch.setattr(F, '_oracle_engine', install)
    for k, case in enumerate(P.CASES[:4]):
        P.test_reference_cli_identical_with_patch(case[0], case[1], mods, monkeypatch, tmp_path / ('p%d' % k))
    for k, case in enumerate(F.CASES[:5]):
        F.test_flat_cli_writes_the_reference_cli_files(case[0], case[1], case[2], mods, monkeypatch, tmp_path / ('f%d' % k))
