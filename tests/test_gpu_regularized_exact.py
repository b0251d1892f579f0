"""The regularised whole-list DP on every SM (K9, csrc/regularized_exact.cu) against the flat C oracle
(reg_oracle.FlatOracleReg.square_split) and against the one-CTA kernel K6 (csrc/regularized_dp.cu), bit for bit on
P, prev, the split numbers, score and splits; the size dispatch of pasio_square_split_regularized; the public routes
(`exact`, `slidingwindow`, the CLI) that reach it."""
import io
import os
import subprocess
import sys

import numpy as np
import pytest

import reg_oracle as ro
import pasio_b200
from oracle import pasio_oracle as po
from pasio_b200 import _native, configure_splitter, synth
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from pasio_b200.process_bedgraph import split_bedgraph_stream
from pasio_b200.splitters.square_splitter import _identity, penalty_tables

pytestmark = pytest.mark.gpu

THREADS = max(1, min(32, os.cpu_count() or 1))
# (split-number multiplier, length multiplier, length function): test_gpu_regularized.PENALTY_CASES
PENALTY_CASES = [(3.0, 0, 'none'), (0, 1.5, 'revlog'), (0.75, 40.0, 'revlog'), (0, 0.001, 'none'), (2, 0, 'none'),
                 (-1.5, 3.0, 'revlog')]
K6, BY_SIZE, K9 = 0, 1, 2
THRESHOLD = 1025            # REG_EXACT_MIN_CANDIDATES of csrc/api.cu


def _far(length):
    """1 beyond 200 positions: with a length multiplier of -1e20 every far cell rounds to the same multiple of 1e20, so a
    row's maximum is tied across many column blocks and only the first-maximum rule of every merge picks the column"""
    return (np.asarray(length) > 200).astype(np.float64)


FUNCTIONS = dict(ro.FUNCTIONS, far=_far)
TIES = (0, -1e20, 'far')


def _spec(num, length, fn):
    return (length, FUNCTIONS[fn], num, _identity)


def _kwargs(num, length, fn):
    return dict(split_number_regularization=num, length_regularization=length,
                length_regularization_function=fn if length else 'none')


def _ns_from_prev(prev):
    ns = np.zeros(len(prev), dtype=np.int64)
    for j in range(1, len(prev)):
        ns[j] = ns[prev[j]] + 1 if prev[j] != 0 else 0
    return ns


@pytest.fixture
def eng():
    e = _native.engine()
    yield e
    e.set_tuning('reg_exact', BY_SIZE)


def _device(eng, counts, cands, ab, case, mode):
    """(score, splits, P, prev) of the device DP over cands (None: all positions), kernel chosen by mode"""
    eng.set_tuning('reg_exact', mode)
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts)
    eng.set_candidates(cands)
    m = len(counts) + 1 if cands is None else len(cands)
    return eng.square_split_regularized(*penalty_tables(_spec(*case), len(counts) + 1, m), want_arrays=True)


def _check(got, want, what):
    score, splits, P, prev = got
    o_score, o_splits, o_P, o_prev, o_ns = want
    assert np.array_equal(P, o_P) and np.array_equal(prev, o_prev), what
    assert np.array_equal(_ns_from_prev(prev), o_ns), what
    assert score == o_score and np.array_equal(splits, o_splits), what


def _data(n, seed):
    """0/1 data, a plateau (exact ties), and constant data, where column 0 wins every row (the refund matters)"""
    rs = np.random.RandomState(seed)
    plateau = (rs.random_sample(n) < 0.2).astype(np.int64)
    plateau[n // 4:n // 2] = 3
    return {'ties01': (rs.random_sample(n) < 0.3).astype(np.int64), 'plateau': plateau,
            'flat': np.full(n, 2, dtype=np.int64)}


# rows start at 1 in blocks of 128: 0, 1 and 2 worker CTAs, the first hand-over to a worker
@pytest.mark.parametrize('n', [2, 3, 33, 128, 129, 130, 257, 258, 385, 386])
@pytest.mark.parametrize('ab', [(1, 1.0), (2.5, 0.3)])
def test_k9_vs_c_oracle_at_block_seams(eng, n, ab):
    for name, base in _data(4 * n + 8, n).items():
        for cands_name in ['all', 'sparse']:
            if cands_name == 'all':
                counts, cands = base[:n - 1], None
                ocands = np.arange(n, dtype=np.int64)
            else:
                counts = base
                cands = synth.random_candidates(len(base), n, seed=n)
                ocands = cands
            for case in PENALTY_CASES + [TIES]:
                want = ro.FlatOracleReg(counts, ab[0], ab[1], _spec(*case)).square_split(ocands)
                _check(_device(eng, counts, cands, ab, case, K9), want, (name, cands_name, case))


@pytest.mark.parametrize('ab', [(1, 1.0), (2.5, 0.3)])
def test_k9_vs_c_oracle_many_blocks_per_worker(eng, ab):
    """N = 60 001 > 128 x (resident CTAs + 2): every worker owns several row blocks"""
    n = 60001
    counts = synth.dnase_like(n - 1, 11, hotspot_share=0.3)
    for case in [(0.75, 40.0, 'revlog'), (-1.5, 3.0, 'revlog'), TIES]:
        want = ro.FlatOracleReg(counts, ab[0], ab[1], _spec(*case), threads=THREADS).square_split(np.arange(n))
        _check(_device(eng, counts, None, ab, case, K9), want, case)
    long = synth.dnase_like(400000, 12, hotspot_share=0.3)
    cands = synth.random_candidates(len(long), n, seed=13)
    case = (3.0, 0, 'none')
    want = ro.FlatOracleReg(long, ab[0], ab[1], _spec(*case), threads=THREADS).square_split(cands)
    _check(_device(eng, long, cands, ab, case, K9), want, 'sparse')


@pytest.mark.parametrize('n', [20001, 100001])
def test_k9_equals_k6(eng, n):
    counts = synth.piecewise_poisson(n - 1, 21)
    cases = PENALTY_CASES[2:3] + PENALTY_CASES[5:] if n > 50000 else PENALTY_CASES[:3] + PENALTY_CASES[5:]
    for case in cases:
        a = _device(eng, counts, None, (1, 1.0), case, K6)
        b = _device(eng, counts, None, (1, 1.0), case, K9)
        assert a[0] == b[0] and all(np.array_equal(x, y) for x, y in zip(a[1:], b[1:])), case


def test_default_dispatch(eng):
    """reg_exact = 1 on both sides of the threshold: the oracle's results, N(N-1)/2 cells, none skipped, one launch"""
    counts = synth.dnase_like(3 * THRESHOLD, 5, hotspot_share=0.3)
    case = (0.75, 40.0, 'revlog')
    for n in [THRESHOLD - 1, THRESHOLD, 3 * THRESHOLD + 1]:
        c = counts[:n - 1]
        want = ro.FlatOracleReg(c, 1, 1.0, _spec(*case)).square_split(np.arange(n))
        eng.timing_reset(True)
        try:
            got = _device(eng, c, None, (1, 1.0), case, BY_SIZE)
            timing = eng.timing()
        finally:
            eng.timing_reset(False)
        _check(got, want, n)
        assert eng.round_stats() == (n * (n - 1) // 2, 0)
        assert timing['exact_dp'][1] == 1
        for mode in [K6, K9]:
            _check(_device(eng, c, None, (1, 1.0), case, mode), want, (n, mode))
            assert eng.round_stats() == (n * (n - 1) // 2, 0)


def _segments(counts, splitter):
    segs = list(pasio_b200.segments_with_scores(counts, splitter))
    splits = np.array([s.start for s in segs] + [segs[-1].stop])
    return splits, np.array([s.mean_count for s in segs]), np.array([s.log_marginal_likelyhood for s in segs])


def _check_segments(counts, got, splits, what):
    sc = po.Scorer(counts, splits, po.Tables(1, 1.0))
    assert np.array_equal(got[0], splits), what
    assert np.array_equal(got[1], sc.mean_counts()) and np.array_equal(got[2], sc.log_marginal_likelyhoods()), what


CLI_CASE = (2, 5, 'revlog')


def test_exact_route_100kb(eng):
    counts = synth.dnase_like(100000, 17, hotspot_share=0.3)
    fo = ro.FlatOracleReg(counts, 1, 1.0, _spec(*CLI_CASE), threads=THREADS)
    _, splits, _, _, _ = fo.square_split(np.arange(len(counts) + 1))
    got = _segments(counts, configure_splitter(algorithm='exact', **_kwargs(*CLI_CASE)))
    _check_segments(counts, got, splits, 'exact')


def test_slidingwindow_route_1mb(eng):
    counts = synth.piecewise_poisson(1000000, 18)           # about 2 500 survivors of the window step
    fo = ro.FlatOracleReg(counts, 1, 1.0, _spec(*CLI_CASE), threads=THREADS)
    survivors, _ = fo.round(np.arange(len(counts) + 1), 2500, 1250, 'constants')
    assert len(survivors) > THRESHOLD
    _, splits, _, _, _ = fo.square_split(survivors)
    got = _segments(counts, configure_splitter(algorithm='slidingwindow', **_kwargs(*CLI_CASE)))
    _check_segments(counts, got, splits, 'slidingwindow')


def test_length_table_grows_in_final_dp(eng):
    """slidingwindow over a zero run longer than the log table (2^20 entries): the final DP spans it, asks for longer
    tables (PASIO_E_TABLE_TOO_SHORT) and runs again"""
    counts = np.concatenate([synth.dnase_like(40000, 1), np.zeros(1200000, dtype=np.int64), synth.dnase_like(40000, 2)])
    case = (0.5, 5.0, 'revlog')
    fo = ro.FlatOracleReg(counts, 1, 1.0, _spec(*case), threads=THREADS)
    survivors, _ = fo.round(np.arange(len(counts) + 1), 2500, 1250, 'constants')
    assert len(survivors) > THRESHOLD
    _, splits, _, _, _ = fo.square_split(survivors)
    got = _segments(counts, configure_splitter(algorithm='slidingwindow', **_kwargs(*case)))
    _check_segments(counts, got, splits, 'table growth')
    assert survivors[-1] - survivors[0] > 1 << 20
    assert eng._tables[_native.TAB_LOG][1] > 1 << 20


def test_cli_exact_equals_one_cta(eng, tmp_path):
    """the CLI (default dispatch, one contig above the threshold) writes byte for byte what the one-CTA kernel gives"""
    lines = []
    for c, n in enumerate([30000, 1500, 29000, 800]):
        lines.extend(synth.to_bedgraph_lines('chr%d' % c, synth.dnase_like(n, seed=300 + c, hotspot_share=0.3)))
    text = ''.join(lines)
    path = tmp_path / 'in.bedgraph'
    path.write_text(text)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    got = subprocess.run([sys.executable, '-m', 'pasio_b200', str(path), '--algorithm', 'exact',
                          '--split-number-regularization', '2', '--length-regularization', '5',
                          '--length-regularization-function', 'revlog', '-o', '-'],
                         cwd=root, check=True, stdout=subprocess.PIPE).stdout.decode()
    eng.set_tuning('reg_exact', K6)
    out = io.StringIO()
    split_bedgraph_stream(io.StringIO(text), out, configure_splitter(algorithm='exact', **_kwargs(*CLI_CASE)))
    assert got == out.getvalue()
    assert got.count('\n') > 4
