"""Regularised window splitters without a GPU: which graphs the fused device plans accept, and the flat C oracle of
the regularised round (tests/reg_oracle.c) against the object-faithful numpy composition, bit for bit."""
import pickle

import numpy as np
import pytest

import reg_oracle as ro
from oracle import pasio_oracle as po
from pasio_b200 import configure_splitter, synth
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from pasio_b200.splitters import _fusion
from pasio_b200.splitters.square_splitter import SquareSplitter, _identity, _revlog, penalty_tables
from pasio_b200.splitters.sliding_window_reducer import SlidingWindowReducer
from pasio_b200.splitters.round_reducer import RoundReducer
from pasio_b200.splitters.reducer_combiner import ReducerCombiner
from pasio_b200.splitters.nop_splitter import NopSplitter
from pasio_b200.dto.sliding_window import SlidingWindow

# (split-number multiplier, length multiplier, length function): the cases of test_regularized_dp_on_device_vs_oracle
# (an integer multiplier among them) and a negative multiplier
PENALTY_CASES = [(3.0, 0, 'none'), (0, 1.5, 'revlog'), (0.75, 40.0, 'revlog'), (0, 0.001, 'none'), (2, 0, 'none'),
                 (-1.5, 3.0, 'revlog')]


def _spec(num, length, fn):
    return (length, ro.FUNCTIONS[fn], num, _identity)


@pytest.mark.parametrize('constraint', ['constants', 'zeros', 'none'])
@pytest.mark.parametrize('fn', ['none', 'revlog'])
def test_device_plan_recognises_the_regularised_rounds_graph(constraint, fn):
    length = 3.0 if fn == 'revlog' else 0                     # the CLI takes a length multiplier only with revlog
    s = configure_splitter(split_constraints=constraint, split_number_regularization=2, length_regularization=length,
                           length_regularization_function=fn, window_size=1000, window_shift=400, num_rounds=4)
    assert _fusion.pipeline_plan(s) is None                    # the unregularised pipeline plan stays as it is
    plan = _fusion.device_plan(s)
    assert plan['final'] == 'nop' and len(plan['steps']) == 1
    step = plan['steps'][0]
    assert step[0] == 'rounds' and step[2:6] == (1000, 400, constraint, 4)
    assert step[6] == (length, ro.FUNCTIONS[fn], 2, _identity)
    again = pickle.loads(pickle.dumps(plan))
    assert again['steps'][0][6][1] is ro.FUNCTIONS[fn] and again['steps'][0][2:6] == step[2:6]
    # the slidingwindow graph: its window step is fused, its final regularised DP is not a whole-contig plan
    sw = configure_splitter(algorithm='slidingwindow', split_constraints=constraint, split_number_regularization=1)
    assert _fusion.device_plan(sw) is None
    assert _fusion.window_plan(sw.reducers[0])[4] == (0, _identity, 1, _identity)


def test_device_plan_keeps_unregularised_plans_and_refuses_the_rest():
    s = configure_splitter()
    assert _fusion.device_plan(s) == _fusion.pipeline_plan(s)
    assert _fusion.device_plan(s)['steps'][0][2:] == (2500, 1250, 'constants', None)
    factory = ScorerFactory(1, 1)

    def graph(base):
        win = SlidingWindowReducer(SlidingWindow(window_size=100, window_shift=50), base)
        return ReducerCombiner(RoundReducer(win), NopSplitter(factory))
    lam = SquareSplitter(factory, split_number_regularization_multiplier=2, split_number_regularization_function=lambda x: x)
    assert _fusion.device_plan(graph(lam)) is None

    class Sub(SquareSplitter):
        pass
    assert _fusion.device_plan(graph(Sub(factory, length_regularization_multiplier=1,
                                         length_regularization_function=_revlog))) is None
    ok = SquareSplitter(factory, length_regularization_multiplier=1, length_regularization_function=_revlog)
    assert _fusion.device_plan(graph(ok)) is not None
    big = SlidingWindowReducer(SlidingWindow(window_size=_fusion.MAX_FUSED_REG_WINDOW_CANDIDATES, window_shift=50), ok)
    assert _fusion.window_plan(big) is None
    assert _fusion.device_plan(ReducerCombiner(RoundReducer(big), NopSplitter(factory))) is None


def test_penalty_tables_are_the_reference_expressions():
    lp, sp, refund = penalty_tables((5.0, _revlog, 2, _identity), 100, 50)
    with np.errstate(divide='ignore'):
        assert np.array_equal(lp, 5.0 * (1 / np.log(np.arange(100) + 1)))
    assert np.array_equal(sp, 2 * (np.arange(50, dtype=np.float64) + 1)) and refund == 2.0
    assert penalty_tables((0, _identity, 0.5, _revlog), 10, 10)[0] is None


def _contigs():
    sparse = np.zeros(1500, dtype=np.int64)
    sparse[::97] = 1
    sparse[700:760] = 3                      # runs and equal values: ties
    return [('dnase', synth.dnase_like(2000, 5, hotspot_share=0.3)), ('poisson', synth.piecewise_poisson(1800, 11)),
            ('sparse', sparse)]


@pytest.mark.parametrize('case', PENALTY_CASES)
@pytest.mark.parametrize('constraint', ['constants', 'zeros', 'none'])
@pytest.mark.parametrize('alpha', [1, 2.5])
def test_c_round_equals_numpy_round(case, constraint, alpha):
    num, length, fn = case
    tables = po.Tables(po.normalise_alpha(alpha), 1.0)
    pen = ro.penalty_kwargs(num, length, fn)
    for name, counts in _contigs():
        cands = np.arange(len(counts) + 1)
        fo = ro.FlatOracleReg(counts, alpha, 1.0, _spec(*case))
        for _ in range(2):                                        # round 1 (all positions) and one explicit list
            want = ro.sliding_window_round(counts, cands, tables, 120, 50, constraint, **pen)
            got, _ = fo.round(cands, 120, 50, constraint)
            assert np.array_equal(got, want), (name, case, constraint, alpha)
            cands = want


@pytest.mark.parametrize('case', PENALTY_CASES)
@pytest.mark.parametrize('alpha', [1, 2.5])
def test_c_square_split_equals_numpy(case, alpha):
    """FlatOracleReg.square_split (the whole-list regularised DP of tests/reg_oracle.c): score and splits equal
    po.square_split_regularized, and every row of its P / prev / split numbers is the numpy row recomputed from the
    oracle's own earlier rows (so by induction the whole arrays are the numpy recurrence's)"""
    num, length, fn = case
    pen = ro.penalty_kwargs(num, length, fn)
    tables = po.Tables(po.normalise_alpha(alpha), 1.0)
    for name, counts in _contigs():
        counts = counts[:400]
        for cands in [np.arange(len(counts) + 1), np.concatenate([[0], np.arange(3, len(counts), 4), [len(counts)]])]:
            score, splits, P, prev, ns = ro.FlatOracleReg(counts, alpha, 1.0, _spec(*case)).square_split(cands)
            o_score, o_splits = po.square_split_regularized(counts, cands, tables, **pen)
            assert score == o_score and np.array_equal(splits, o_splits), (name, case, alpha)
            sc = po.Scorer(counts, cands, tables)
            assert P[0] == 0 and prev[0] == 0 and ns[0] == 0
            for j in range(1, len(cands)):
                t = sc.row(j)
                t += P[:j]
                if num != 0:
                    t -= pen['num_mult'] * pen['num_fn'](ns[:j].astype(np.float64) + 1)
                    t[0] += pen['num_mult'] * pen['num_fn'](1)
                if length != 0:
                    t -= (pen['len_mult'] * pen['len_fn'](cands[j] - cands[:j]))[:j]
                k = np.argmax(t)
                assert prev[j] == k and P[j] == t[k] + sc.pen and ns[j] == (ns[k] + 1 if k else 0), (name, case, alpha, j)


def test_c_rounds_multithreaded_and_pipeline_match_numpy():
    counts = synth.dnase_like(3000, 8, hotspot_share=0.3)
    spec = _spec(2.0, 5.0, 'revlog')
    want = ro.default_pipeline(counts, po.Tables(1, 1.0), 200, 90, 'constants', **ro.penalty_kwargs(2.0, 5.0, 'revlog'))
    for threads in (1, 4):
        got = ro.pipeline(counts, spec, window_size=200, window_shift=90, threads=threads)
        assert np.array_equal(got['splits'], want['splits']) and list(got['sizes']) == list(want['sizes'])
        assert got['score'] == want['score'] and np.array_equal(got['lmm'], want['lmm'])
    plain = po.default_pipeline(counts, po.Tables(1, 1.0), 200, 90, 'constants')
    assert len(plain['splits']) != len(want['splits'])           # the penalties change the segmentation
