"""Regularised window splitters on the GPU (csrc/window_dp_reg.cu): the fused rounds against the flat C oracle
(tests/reg_oracle.c) and against the object route through the exact regularised DP, bit for bit on splits, means and
LMM, 1e-9 on summed scores."""
import io
import os
import subprocess
import sys

import numpy as np
import pytest

import reg_oracle as ro
import pasio_b200
from pasio_b200 import _native, configure_splitter, synth
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from pasio_b200.process_bedgraph import split_bedgraph_stream
from pasio_b200.splitters.square_splitter import SquareSplitter, _identity, _revlog
from oracle import pasio_oracle as po

pytestmark = pytest.mark.gpu

THREADS = max(1, min(32, os.cpu_count() or 1))
# (split-number multiplier, length multiplier, length function); the cases of test_regularized_dp_on_device_vs_oracle
# and a negative multiplier
PENALTY_CASES = [(3.0, 0, 'none'), (0, 1.5, 'revlog'), (0.75, 40.0, 'revlog'), (0, 0.001, 'none'), (2, 0, 'none'),
                 (-1.5, 3.0, 'revlog')]


def _spec(num, length, fn):
    return (length, ro.FUNCTIONS[fn], num, _identity)


def _kwargs(num, length, fn):
    return dict(split_number_regularization=num, length_regularization=length,
                length_regularization_function=fn if length else 'none')


def _segments(counts, splitter):
    segs = list(pasio_b200.segments_with_scores(counts, splitter))
    splits = np.array([s.start for s in segs] + [segs[-1].stop])
    return splits, np.array([s.mean_count for s in segs]), np.array([s.log_marginal_likelyhood for s in segs])


def _round_contigs():
    sparse = np.zeros(30000, dtype=np.int64)
    sparse[::53] = 1
    sparse[::211] = 2
    sparse[9000:9400] = 4                                       # a plateau: equal values, ties in the DP
    return [('dnase', synth.dnase_like(30000, 3, hotspot_share=0.3)), ('sparse', sparse)]


@pytest.mark.parametrize('case', PENALTY_CASES)
@pytest.mark.parametrize('constraint', ['constants', 'zeros', 'none'])
@pytest.mark.parametrize('alpha', [1, 2.5])
def test_round_vs_c_oracle(case, constraint, alpha):
    """one round from all positions and one from an explicit list; with constraint `none` the windows have exactly
    160, 161, 512, 513, 514 and the largest fused number of candidates, so every kernel class runs"""
    eng = _native.engine()
    sizes = [159, 160, 511, 512, 513, 7167] if constraint == 'none' else [159, 600, 2500]
    for name, counts in _round_contigs():
        fo = ro.FlatOracleReg(counts, alpha, 1.0, _spec(*case), threads=THREADS)
        for ws in sizes:
            shift = max(1, ws // 2)
            eng.use_scorer(ScorerFactory(alpha, 1.0), _spec(*case))
            eng.load(counts)
            cands = np.arange(len(counts) + 1)
            eng.set_candidates(None)
            for r in range(2):
                want, cells = fo.round(cands, ws, shift, constraint)
                n_in, n_out, got_cells = eng.round(ws, shift, constraint)
                got = eng.candidates()
                assert n_in == len(cands) and np.array_equal(got, want), (name, case, constraint, alpha, ws, r)
                assert got_cells == cells
                cands = want


@pytest.mark.parametrize('num_rounds', [None, 2])
def test_segments_with_scores_5mb_vs_c_oracle(num_rounds):
    counts = synth.dnase_like(5000000, 21)
    case = (2.0, 5.0, 'revlog')
    splitter = configure_splitter(window_size=1000, window_shift=500, num_rounds=num_rounds, **_kwargs(*case))
    want = ro.pipeline(counts, _spec(*case), window_size=1000, window_shift=500, num_rounds=num_rounds, threads=THREADS)
    splits, means, lmm = _segments(counts, splitter)
    assert np.array_equal(splits, want['splits'])
    assert np.array_equal(means, want['mean_counts']) and np.array_equal(lmm, want['lmm'])
    eng = _native.engine()
    eng.use_scorer(ScorerFactory(1, 1.0), _spec(*case))
    eng.load(counts)
    eng.set_candidates(None)
    sizes, final, _ = eng.rounds(1000, 500, 'constants', num_rounds)
    assert sizes == list(want['sizes'][:len(sizes)]) and final == len(want['splits'])
    score = eng.segment_scores_sum()
    assert abs(score - want['score']) <= 1e-9 * abs(want['score'])


class _ObjectRoute(SquareSplitter):
    """a subclass: the plans refuse it, so every window goes through the objects and the exact regularised DP (K6)"""


def test_fused_route_equals_object_route():
    counts = synth.dnase_like(100000, 7, hotspot_share=0.3)
    for case in [(2.0, 5.0, 'revlog'), (-1.5, 3.0, 'revlog')]:
        fused = configure_splitter(window_size=1000, window_shift=500, **_kwargs(*case))
        obj = configure_splitter(window_size=1000, window_shift=500, **_kwargs(*case))
        sq = obj.reducers[0].base_reducer.base_reducer.reducers[1]
        sq.__class__ = _ObjectRoute
        a = _segments(counts, fused)
        b = _segments(counts, obj)
        for x, y in zip(a, b):
            assert np.array_equal(x, y), case


def test_no_per_window_work(monkeypatch):
    def refuse(*args, **kwargs):
        raise AssertionError('per-window device call in the fused regularised rounds')
    monkeypatch.setattr(_native.Engine, 'square_split_regularized', refuse)
    monkeypatch.setattr(_native.Engine, 'filter_candidates', refuse)
    counts = synth.dnase_like(300000, 9)
    case = (2.0, 5.0, 'revlog')
    splits, _, _ = _segments(counts, configure_splitter(**_kwargs(*case)))
    assert np.array_equal(splits, ro.pipeline(counts, _spec(*case), threads=THREADS)['splits'])


def _transcripts(n_contigs, seed):
    lines = []
    for c, n in enumerate(synth.transcript_lengths(n_contigs, seed=seed)):
        lines.extend(synth.to_bedgraph_lines('tx%05d' % c, synth.dnase_like(int(n), seed=5000 + c, hotspot_share=0.3)))
    return ''.join(lines)


def test_batches_pool_and_cli_vs_oracle(monkeypatch, tmp_path):
    from pasio_b200 import process_bedgraph
    text = _transcripts(60, 3)
    case = (2.0, 5.0, 'revlog')
    kw = dict(window_size=500, window_shift=250, **_kwargs(*case))
    outs = {}
    for mode in ['bedgraph', 'bed', 'bedgraph+length+LMM']:
        out = io.StringIO()
        split_bedgraph_stream(io.StringIO(text), out, configure_splitter(**kw), output_mode=mode)
        assert out.getvalue() == ro.split_bedgraph_text(text, _spec(*case), window_size=500, window_shift=250,
                                                        output_mode=mode, threads=THREADS), mode
        outs[mode] = out.getvalue()
    # batched (the default) == one contig per launch
    monkeypatch.setattr(process_bedgraph, 'BATCH_NT', 0)
    alone = io.StringIO()
    split_bedgraph_stream(io.StringIO(text), alone, configure_splitter(**kw), output_mode='bedgraph+length+LMM')
    assert alone.getvalue() == outs['bedgraph+length+LMM']
    monkeypatch.undo()
    # two worker processes
    monkeypatch.setenv('PASIO_B200_POOL_SAME_DEVICE', '1')
    multi = io.StringIO()
    split_bedgraph_stream(io.StringIO(text), multi, configure_splitter(**kw), output_mode='bedgraph+length+LMM', devices=2)
    assert multi.getvalue() == outs['bedgraph+length+LMM']
    # the CLI
    path = tmp_path / 'in.bedgraph'
    small = _transcripts(8, 4)
    path.write_text(small)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    got = subprocess.run([sys.executable, '-m', 'pasio_b200', str(path), '--split-number-regularization', '2',
                          '--length-regularization', '5', '--length-regularization-function', 'revlog', '-o', '-'],
                         cwd=root, check=True, stdout=subprocess.PIPE).stdout.decode()
    assert got == ro.split_bedgraph_text(small, (5.0, _revlog, 2.0, _identity), threads=THREADS)


def test_length_table_grows():
    """a zero run longer than the log table (2^20 entries): round 2 has a window spanning it, the round asks for longer
    tables (PASIO_E_TABLE_TOO_SHORT) and the length penalty table grows with the log table"""
    counts = np.concatenate([synth.dnase_like(40000, 1), np.zeros(1200000, dtype=np.int64), synth.dnase_like(40000, 2)])
    case = (0.5, 5.0, 'revlog')
    splits, means, lmm = _segments(counts, configure_splitter(**_kwargs(*case)))
    want = ro.pipeline(counts, _spec(*case), threads=THREADS)
    assert np.array_equal(splits, want['splits']) and np.array_equal(lmm, want['lmm'])
    assert max(np.diff(splits)) > 1 << 20
    eng = _native.engine()
    assert eng._penalty_spec is None and eng._tables[_native.TAB_LOG][1] > 1 << 20
    assert eng._penalties[1] > 1 << 20                                # the device's length table grew with the log table


def test_no_state_leak_into_unregularised_run(golden):
    counts = synth.dnase_like(50000, 4)
    _segments(counts, configure_splitter(window_size=600, window_shift=300, **_kwargs(2.0, 5.0, 'revlog')))
    g = golden('pipeline.npz')
    name = 'zeros100k'
    c = g[name + '.counts'].astype(np.int64)
    splitter = configure_splitter(split_constraints='zeros', window_size=600, window_shift=300)
    splits, means, lmm = _segments(c, splitter)
    want = np.concatenate([g[name + '.starts'], g[name + '.stops'][-1:]])
    score, _ = splitter.split(c, np.arange(len(c) + 1))
    g.check_splits(splits, want, score, g[name + '.score'], name)
    if g.bit_exact(name):
        assert np.array_equal(means, g[name + '.mean']) and np.array_equal(lmm, g[name + '.lmm'])
    plain = po.default_pipeline(c, po.Tables(1, 1.0), 600, 300, 'zeros')
    assert np.array_equal(splits, plain['splits'])
