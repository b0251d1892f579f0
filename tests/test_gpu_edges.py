"""The DP kernels at the edges of their exactness arguments, bit for bit against the C oracles:
- the far-column bound (K4 pruned rounds, K3 pruned exact DP) at the alpha where it is switched off (2^-10), at small,
  large real and large integer alpha, at extreme beta and at window totals around 10^7; the bound must really skip
  cells where it is on and skip none where it is off;
- the largest fused windows (8 192 candidates unregularised), the step to the object route one candidate later (and at
  7 169 regularised candidates), and windows of 2 and 3 candidates;
- the whole-list regularised DP (K6): P and prev at its 32-row block edges, with penalties whose rounding makes exact
  ties; the regularised window DP (K8) at beta != 1; the regularised `slidingwindow` graph."""
import os

import numpy as np
import pytest

import reg_oracle as ro
import pasio_b200
from oracle import c_oracle, pasio_oracle as po
from pasio_b200 import _native, configure_splitter, synth
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from pasio_b200.splitters import _fusion
from pasio_b200.splitters.square_splitter import _identity, penalty_tables

pytestmark = pytest.mark.gpu

THREADS = max(1, min(32, os.cpu_count() or 1))
ALPHA_BOUND_MIN = 0.0009765625          # 2^-10: below it K3 and K4 evaluate every cell (window_dp.cu, exact_dp.cu)


@pytest.fixture(scope='module')
def eng():
    return _native.engine()


def _spec(num, length, fn):
    return (length, ro.FUNCTIONS[fn], num, _identity)


def _kwargs(num, length, fn):
    return dict(split_number_regularization=num, length_regularization=length,
                length_regularization_function=fn if length else 'none')


def _explicit(n, share, seed):
    rs = np.random.RandomState(seed)
    return np.concatenate([[0], np.flatnonzero(rs.random_sample(n - 1) < share) + 1, [n]]).astype(np.int64)


def _segments(counts, splitter):
    segs = list(pasio_b200.segments_with_scores(counts, splitter))
    splits = np.array([s.start for s in segs] + [segs[-1].stop])
    return splits, np.array([s.mean_count for s in segs]), np.array([s.log_marginal_likelyhood for s in segs])


def _refuse(what):
    def refuse(*args, **kwargs):
        raise AssertionError(what)
    return refuse


# ---- A. the far-column bound at its parameter edges ----------------------------------------------------------------
# 2^-10 exactly (bound on) and just below (off); lgamma(u + alpha) decreasing in u (alpha < 1); large real and integer
# alpha; extreme beta
BOUND_AB = [(2 ** -10, 1.0), (2 ** -10, 1000.0), (0.0009, 1.0), (0.0009, 0.01), (0.3, 1.0), (0.3, 0.01), (40.5, 1.0),
            (1000, 1.0), (1, 0.01), (1, 1000.0)]


def _bound_data(kind, ab):
    """The bound cuts a far column block only if it lies below the row's lower bound, the value of a split at every
    candidate.  Where the data carry no segments (0/1 noise) or are far below the prior mean alpha / beta (0/1 data at
    alpha = 1000), a single segment wins by a wide margin, every far column stays close to the maximum and nothing can
    be cut.  So the 0/1 and DNase-like profiles have segments, and their values are scaled to the prior mean."""
    rs = np.random.RandomState(11)
    scale = max(1, int(round(ab[0] / ab[1])))
    if kind == 'ties01':                     # two values only: equal values everywhere, exact ties in the arg-max
        parts, n = [], 0
        while n < 60000:                     # blocks of 100 .. 600 positions, 1 % or 95 % of them non-zero
            length = rs.randint(100, 600)
            parts.append(rs.random_sample(length) < rs.choice([0.01, 0.95]))
            n += length
        return scale * np.concatenate(parts)[:60000].astype(np.int64)
    if kind == 'dnase':
        return scale * synth.dnase_like(60000, 12, hotspot_share=0.3)
    # deep: ~3 000 per position, a window of 2 500 candidates (70 % of the positions) holds ~10^7 counts
    return (np.repeat(rs.randint(1000, 5000, 24), 2500) + rs.poisson(40, 60000)).astype(np.int64)


@pytest.mark.parametrize('data', ['ties01', 'dnase', 'deep'])
@pytest.mark.parametrize('ab', BOUND_AB)
def test_window_bound_at_parameter_edges(eng, ab, data):
    """three rounds from an explicit list (the pipelined, pruned path from the first round) against the oracle, with the
    default kernels, with pruning but no window skipping (so the skipped count is the bound's alone) and with neither"""
    counts = _bound_data(data, ab)
    cands0 = _explicit(len(counts), 0.7, 12)
    fo = c_oracle.FlatOracle(counts, *ab, threads=THREADS)
    factory = ScorerFactory(*ab)
    try:
        for wsize, wshift in [(2500, 1250), (1000, 500)]:
            want = []
            cands = cands0
            for r in range(3):
                cands, cells = fo.round(cands, wsize, wshift, 'none')
                want.append((cands, cells))
            skipped = {}
            for prune, phases in [(1, 1), (1, 0), (0, 0)]:
                eng.set_tuning('window_prune', prune)
                eng.set_tuning('window_phases', phases)
                eng.use_scorer(factory)
                eng.load(counts)
                eng.set_candidates(cands0)
                skipped[prune, phases] = 0
                for r in range(3):
                    eng.round(wsize, wshift, 'none')
                    got = eng.candidates()
                    cells, sk = eng.round_stats()
                    assert np.array_equal(got, want[r][0]), (ab, data, wsize, prune, phases, r)
                    assert cells == want[r][1] and 0 <= sk <= cells
                    skipped[prune, phases] += sk
            assert skipped[0, 0] == 0
            if ab[0] >= ALPHA_BOUND_MIN:
                assert skipped[1, 0] > 0, (ab, data, wsize)         # the bound ran and cut cells
            else:
                assert skipped[1, 0] == 0, (ab, data, wsize)        # switched off
    finally:
        eng.set_tuning('window_prune', 1)
        eng.set_tuning('window_phases', 1)


EXACT_AB = [(2 ** -10, 1.0), (0.0009, 1.0), (0.3, 0.01), (40.5, 1.0), (1000, 1.0), (1, 1000.0)]


@pytest.mark.parametrize('data', ['ties01', 'dense'])
@pytest.mark.parametrize('ab', EXACT_AB)
def test_exact_bound_at_parameter_edges(eng, ab, data):
    """the whole-contig DP: P and prev equal the oracle's with the default kernel (lag 5), lag 3 and no pruning"""
    rs = np.random.RandomState(13)
    counts = (rs.random_sample(20000) < 0.3).astype(np.int64) if data == 'ties01' else synth.two_level_poisson(10000, seed=3)
    cands = np.arange(len(counts) + 1, dtype=np.int64)
    o_score, o_splits, o_P, o_prev = c_oracle.FlatOracle(counts, *ab, threads=THREADS).square_split(cands)
    factory = ScorerFactory(*ab)
    try:
        for prune, lag in [(1, 5), (1, 3), (0, 5)]:
            eng.set_tuning('exact_prune', prune)
            eng.set_tuning('exact_lag', lag)
            eng.use_scorer(factory)
            eng.load(counts)
            eng.set_candidates(None)
            score, splits, P, prev = eng.square_split(want_arrays=True)
            cells, skipped = eng.round_stats()
            assert np.array_equal(P, o_P) and np.array_equal(prev, o_prev), (ab, data, prune, lag)
            assert score == o_score and np.array_equal(splits, o_splits)
            assert cells == len(cands) * (len(cands) - 1) // 2
            if prune and ab[0] >= ALPHA_BOUND_MIN:
                assert 0 < skipped < cells, (ab, data, lag)
            else:
                assert skipped == 0, (ab, data, prune)
    finally:
        eng.set_tuning('exact_prune', 1)
        eng.set_tuning('exact_lag', 5)


# ---- B. window size limits -----------------------------------------------------------------------------------------
LARGEST = 8191                  # window_size of the largest fused window: 8 192 candidates (_fusion.MAX_FUSED_WINDOW_CANDIDATES)


def _rounds_vs_oracle(eng, fo, counts, cands, wsize, wshift, constraint, n_rounds, what):
    eng.load(counts)
    eng.set_candidates(None if len(cands) == len(counts) + 1 else cands)
    for r in range(n_rounds):
        want, cells = fo.round(cands, wsize, wshift, constraint)
        n_in, _, got_cells = eng.round(wsize, wshift, constraint)
        got = eng.candidates()
        assert n_in == len(cands) and np.array_equal(got, want), (what, r)
        assert got_cells == cells, (what, r)
        cands = want


@pytest.mark.parametrize('alpha', [1, 2.5])
def test_largest_fused_window(eng, monkeypatch, alpha):
    """8 192 candidates per window, one CTA each: plain steps from all positions, pruned pipelined steps from an
    explicit list, and the whole pipeline, which must run fused (no per-window device call)"""
    counts = synth.dnase_like(40000, 31, hotspot_share=0.4)
    fo = c_oracle.FlatOracle(counts, alpha, 1.0, threads=THREADS)
    eng.use_scorer(ScorerFactory(alpha, 1.0))
    _rounds_vs_oracle(eng, fo, counts, np.arange(len(counts) + 1), LARGEST, 4096, 'none', 2, 'all positions')
    _rounds_vs_oracle(eng, fo, counts, _explicit(len(counts), 0.7, 31), LARGEST, 4096, 'none', 2, 'explicit')
    monkeypatch.setattr(_native.Engine, 'square_split', _refuse('per-window exact DP: the largest window was not fused'))
    monkeypatch.setattr(_native.Engine, 'filter_candidates', _refuse('per-window filter in the fused rounds'))
    splitter = configure_splitter(alpha=alpha, window_size=LARGEST, window_shift=4096, split_constraints='none')
    splits, means, _ = _segments(counts, splitter)
    want, _, _ = fo.rounds(LARGEST, 4096, 'none')
    assert np.array_equal(splits, want)
    assert np.array_equal(means, po.Scorer(counts, want, po.Tables(po.normalise_alpha(alpha), 1.0)).mean_counts())


def test_one_past_the_largest_fused_window(monkeypatch):
    """8 193 candidates: the plans refuse the window, each window goes through the objects and the exact DP (K3)"""
    counts = synth.dnase_like(40000, 32, hotspot_share=0.4)
    splitter = configure_splitter(window_size=LARGEST + 1, window_shift=4096, split_constraints='none')
    assert _fusion.window_plan(splitter.reducers[0].base_reducer) is None
    monkeypatch.setattr(_native.Engine, 'round', _refuse('fused round for a window past the limit'))
    monkeypatch.setattr(_native.Engine, 'load_and_round', _refuse('fused round for a window past the limit'))
    splits, _, _ = _segments(counts, splitter)
    want, _, _ = c_oracle.FlatOracle(counts, 1, 1.0, threads=THREADS).rounds(LARGEST + 1, 4096, 'none')
    assert np.array_equal(splits, want)


def test_one_past_the_largest_fused_regularised_window(monkeypatch):
    """7 169 candidates with a regularised splitter: each window goes through the objects and K6"""
    size = _fusion.MAX_FUSED_REG_WINDOW_CANDIDATES
    counts = synth.dnase_like(30000, 33, hotspot_share=0.4)
    case = (2.0, 5.0, 'revlog')
    window = configure_splitter(window_size=size, window_shift=3584, split_constraints='none',
                                **_kwargs(*case)).reducers[0].base_reducer
    assert _fusion.window_plan(window) is None
    monkeypatch.setattr(_native.Engine, 'round', _refuse('fused round for a window past the limit'))
    fo = ro.FlatOracleReg(counts, 1, 1.0, _spec(*case), threads=THREADS)
    cands = np.arange(len(counts) + 1)
    for r in range(2):
        want, _ = fo.round(cands, size, 3584, 'none')
        got = window.reduce_candidate_list(counts, cands)
        assert np.array_equal(got, want), r
        cands = want


@pytest.mark.parametrize('wsize,wshift', [(1, 1), (1, 3), (2, 1), (2, 5)])
@pytest.mark.parametrize('case', [None, (2.0, 5.0, 'revlog'), (-1.5, 3.0, 'revlog')])
def test_smallest_windows(eng, wsize, wshift, case):
    """windows of 2 and 3 candidates, overlapping and with gaps between them (K4, and K8 when regularised)"""
    counts = synth.dnase_like(3000, 34, hotspot_share=0.4)
    if case is None:
        fo = c_oracle.FlatOracle(counts, 1, 1.0)
    else:
        fo = ro.FlatOracleReg(counts, 1, 1.0, _spec(*case))
    for constraint in ['constants', 'zeros', 'none']:
        eng.use_scorer(ScorerFactory(1, 1.0), None if case is None else _spec(*case))
        _rounds_vs_oracle(eng, fo, counts, np.arange(len(counts) + 1), wsize, wshift, constraint, 3,
                          (case, constraint, wsize, wshift))


# ---- C. regularised DP arrays and graphs ---------------------------------------------------------------------------
# a subset of test_gpu_regularized.PENALTY_CASES (the integer and the negative multiplier among them), and identity
# length penalties so large that the rounding of the cell values makes exact ties between distant columns
K6_CASES = [(3.0, 0, 'none'), (0.75, 40.0, 'revlog'), (2, 0, 'none'), (-1.5, 3.0, 'revlog'), (0, 1e12, 'none'),
            (0, 1e20, 'none')]


def _ns_from_prev(prev):
    ns = np.zeros(len(prev), dtype=np.int64)
    for j in range(1, len(prev)):
        ns[j] = ns[prev[j]] + 1 if prev[j] != 0 else 0
    return ns


@pytest.mark.parametrize('n', [2, 3, 32, 33, 34, 63, 64, 65, 66, 1024, 1025, 1057, 1058, 4100])
@pytest.mark.parametrize('ab', [(1, 1.0), (2.5, 3.0)])
def test_regularized_dp_arrays_at_block_edges(eng, n, ab):
    """K6 over n candidates (all positions): P, prev and the split numbers equal FlatOracleReg.square_split"""
    rs = np.random.RandomState(n)
    data = {'poisson': (rs.poisson(3, n - 1) * (rs.random_sample(n - 1) < 0.6)).astype(np.int64),
            'ties01': (rs.random_sample(n - 1) < 0.3).astype(np.int64)}
    cands = np.arange(n, dtype=np.int64)
    factory = ScorerFactory(*ab)
    for name, counts in data.items():
        for case in K6_CASES:
            o_score, o_splits, o_P, o_prev, o_ns = ro.FlatOracleReg(counts, ab[0], ab[1], _spec(*case)).square_split(cands)
            eng.use_scorer(factory)
            eng.load(counts)
            eng.set_candidates(None)
            tables = penalty_tables(_spec(*case), len(counts) + 1, n)
            score, splits, P, prev = eng.square_split_regularized(*tables, want_arrays=True)
            assert np.array_equal(P, o_P) and np.array_equal(prev, o_prev), (name, case)
            assert np.array_equal(_ns_from_prev(prev), o_ns)
            assert score == o_score and np.array_equal(splits, o_splits)


@pytest.mark.parametrize('case', [(3.0, 0, 'none'), (0, 1.5, 'revlog'), (0.75, 40.0, 'revlog'), (0, 0.001, 'none'),
                                  (2, 0, 'none'), (-1.5, 3.0, 'revlog')])
@pytest.mark.parametrize('ab', [(2.5, 0.3), (0.7, 20.0)])
def test_regularised_round_real_alpha_and_beta(eng, case, ab):
    """K8 with real alpha and beta != 1: a round from all positions and one from the explicit list it leaves"""
    sparse = np.zeros(20000, dtype=np.int64)
    sparse[::53] = 1
    sparse[6000:6400] = 4
    for name, counts in [('dnase', synth.dnase_like(20000, 35, hotspot_share=0.3)), ('sparse', sparse)]:
        fo = ro.FlatOracleReg(counts, ab[0], ab[1], _spec(*case), threads=THREADS)
        for wsize, constraint in [(159, 'constants'), (513, 'none'), (600, 'zeros'), (2500, 'none')]:
            eng.use_scorer(ScorerFactory(*ab), _spec(*case))
            _rounds_vs_oracle(eng, fo, counts, np.arange(len(counts) + 1), wsize, wsize // 2, constraint, 2,
                              (name, wsize, constraint))


@pytest.mark.parametrize('case', [(2.0, 5.0, 'revlog'), (-1.5, 3.0, 'revlog')])
def test_regularised_slidingwindow_graph(case):
    """--algorithm slidingwindow with penalties: one fused K8 window round, then K6 over the whole reduced list"""
    counts = synth.dnase_like(200000, 36, hotspot_share=0.3)
    splitter = configure_splitter(algorithm='slidingwindow', window_size=1000, window_shift=500, **_kwargs(*case))
    tables = po.Tables(1, 1.0)
    reduced = ro.sliding_window_round(counts, np.arange(len(counts) + 1), tables, 1000, 500, 'constants',
                                      **ro.penalty_kwargs(*case))
    o_score, o_splits, _, _, _ = ro.FlatOracleReg(counts, 1, 1.0, _spec(*case)).square_split(reduced)
    score, splits = splitter.split(counts, np.arange(len(counts) + 1))
    assert score == o_score and np.array_equal(splits, o_splits)
    got, means, lmm = _segments(counts, splitter)
    sc = po.Scorer(counts, o_splits, tables)
    assert np.array_equal(got, o_splits)
    assert np.array_equal(means, sc.mean_counts()) and np.array_equal(lmm, sc.log_marginal_likelyhoods())
