"""Pin the oracle (oracle/overlap_oracle.c) to the reference: SURVEY section-4 golden strings, the committed
golden fixtures (outputs of the unmodified reference C++), and the reference's stored strings for seeded random inputs
(checked against the live reference too when oracle/_ref exists)."""
import random

from helpers import abi_string, load_golden, oracle_lib, oracle_record, oracle_string, ref_lib

# SURVEY.md section 4: C-ABI strings captured from the reference build on test/test_one_adapter_set.fastq
Y_TOP = 'AATGTACTTCGTTCAGTTACGTATTGCT'
Y_BOTTOM = 'GCAATACGTAACTGAACGAAGT'
SURVEY_WINDOWS = {  # read number (1-based) -> (seq[:150] vs Y_Top, seq[-150:] vs Y_Bottom)
    1: ('94,129,0,27,8,61.538462,61.538462', '137,149,0,8,10,69.230769,34.615385'),
    2: ('0,27,0,27,75,96.428571,96.428571', '53,74,0,21,12,68.000000,68.000000'),
    3: ('0,0,27,27,3,100.000000,3.571429', '128,149,0,21,57,95.454545,95.454545'),
    4: ('0,11,16,27,27,91.666667,39.285714', '134,149,0,15,48,100.000000,72.727273'),
    7: ('0,5,22,27,18,100.000000,21.428571', '145,149,0,4,15,100.000000,22.727273'),
    8: ('0,19,8,27,60,100.000000,71.428571', '23,48,0,21,8,58.620690,58.620690'),
}
SURVEY_FULL = [(5, Y_BOTTOM, '3500,3521,0,21,66,100.000000,100.000000'), (6, Y_TOP, '4000,4027,0,27,75,96.428571,96.428571'),
               (9, Y_TOP, '1700,1727,0,27,84,100.000000,100.000000'), (9, Y_BOTTOM, '1500,1521,0,21,66,100.000000,100.000000')]
SURVEY_EDGE = [('', 'ACGT', '-1,0,-1,0,-2147483648,0.000000,0.000000'), ('ACGT', '', '-1,0,-1,0,-2147483648,0.000000,0.000000'),
               ('N' * 20, Y_TOP, '0,0,28,27,0,-nan,0.000000'), ('-' * 20, Y_TOP, '0,0,28,27,0,-nan,0.000000'),
               ('A', 'C', '0,0,1,0,0,-nan,0.000000'), ('A', 'A', '0,0,0,0,3,100.000000,100.000000'),
               ('ACGTTTTTTTTTTACGT', 'ACGT', '0,3,0,3,12,100.000000,100.000000'),
               ('TTTTACG', 'ACGT', '4,6,0,2,9,100.000000,75.000000')]


def fixture_reads():
    return [r for r in load_golden('fixture_reads.json') if r['file'] == 'test_one_adapter_set.fastq']


def test_survey_window_strings():
    reads = fixture_reads()
    for num, (s_exp, e_exp) in SURVEY_WINDOWS.items():
        seq = reads[num - 1]['seq']
        assert oracle_string(seq[:150], Y_TOP) == s_exp
        assert oracle_string(seq[-150:], Y_BOTTOM) == e_exp


def test_survey_fullread_strings():
    reads = fixture_reads()
    for num, ad, exp in SURVEY_FULL:
        assert oracle_string(reads[num - 1]['seq'], ad) == exp


def test_survey_edge_cases():
    for rd, ad, exp in SURVEY_EDGE:
        assert oracle_string(rd, ad) == exp


def test_golden_windows():
    g = load_golden('golden_windows.json')
    reads = load_golden('fixture_reads.json')
    n = 0
    for ri, kind, ai, exp in g['results']:
        seq = reads[ri]['seq']
        w = seq[:150] if kind == 'start' else seq[-150:]
        assert oracle_string(w, g['panel'][ai][1], g['scoring']) == exp
        n += 1
    assert n > 900


def rebuild_fullread_inputs():
    """Replay the masking rounds of make_golden.py to recover each masked input sequence."""
    g = load_golden('golden_fullread.json')
    reads = load_golden('fixture_reads.json')
    out = []
    cur = {}
    for ri, rnd, an, aseq, n_masked, exp in g['results']:
        key = (ri, an)
        seq = reads[ri]['seq'] if rnd == 0 else cur[key]
        assert seq.count('-') == n_masked
        out.append((seq, aseq, exp))
        parts = exp.split(',')
        rs, re_ = int(parts[0]), int(parts[1]) + 1
        cur[key] = seq[:rs] + '-' * (re_ - rs) + seq[re_:]
    return g['scoring'], out


def test_golden_fullread():
    sc, cases = rebuild_fullread_inputs()
    for seq, ad, exp in cases:
        assert oracle_string(seq, ad, sc) == exp


def test_golden_random():
    for rd, ad, sc, exp in load_golden('golden_random.json'):
        assert oracle_string(rd, ad, sc) == exp


def test_record_matches_string():
    from porechop_b200.align import record_string
    for rd, ad, sc, exp in load_golden('golden_random.json')[:400]:
        assert record_string(oracle_record(rd, ad, sc)) == exp


def live_cases():
    """1500 seeded (read, adapter, scoring) inputs; tests/golden/golden_live.json holds the reference's strings for them."""
    rng = random.Random(99)
    schemes = [[3, -6, -5, -2], [3, -6, -2, -2], [2, -3, -2, -5], [1, 0, -1, -1], [4, -5, -3, -3]]
    out = []
    for _ in range(1500):
        al = rng.choice(['AC', 'ACGT', 'ACGTN'])
        ad = ''.join(rng.choice(al) for _ in range(rng.randint(1, 60)))
        rd = ''.join(rng.choice(al) for _ in range(rng.randint(1, 300)))
        if rng.random() < 0.6:
            p = rng.randint(0, len(rd))
            rd = rd[:p] + ad[rng.randint(0, len(ad) // 2):] + rd[p:]
        out.append((rd, ad, rng.choice(schemes)))
    return out


def test_live_against_reference():
    """The oracle against the reference C++ on live_cases(): its stored strings, and the library itself when built."""
    g = load_golden('golden_live.json')
    cases = live_cases()
    assert len(g['results']) == len(cases)
    for (rd, ad, sc), exp in zip(cases, g['results']):
        assert abi_string(oracle_lib(), rd, ad, sc) == exp
        if ref_lib() is not None:
            assert abi_string(ref_lib(), rd, ad, sc) == exp
