"""The whole-list DP of `--algorithm exact` / `slidingwindow` over a batch of contigs (pasio_square_split_batch), against
per-contig oracles.

The reference segments contigs one by one (process_bedgraph.py:69), so the oracle runs SquareSplitter.split
(c_oracle.FlatOracle.square_split) on every contig's own slice of the candidates, shifts the splits by the contig's offset
and takes the union; everything is compared bit for bit.  Lists of at most CAP candidates run as whole-list windows of the
window DP, longer ones through the whole-chip DP one after another: the batches below have lists on both sides of that
seam, 1-, 2- and 3-nt contigs between them, a list long enough for the whole-chip DP to wrap its self-score ring, a deep
contig that makes the tables grow inside the call, and a batch whose summed count passes 2^31.  The CPU tests check how
process_bedgraph._batches groups contigs for exact plans."""
import io
import os

import numpy as np
import pytest

import test_gpu_batches as tgb
from oracle import c_oracle
from pasio_b200 import _native, configure_splitter, synth
from pasio_b200 import process_bedgraph as pb
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from pasio_b200.process_bedgraph import split_bedgraph_stream

THREADS = max(1, min(32, os.cpu_count() or 1))
CAP = 8192                                      # window_dp_max_candidates on a B200: the longest list of one K4 window
AB = [(1, 1.0), (2.5, 0.3), (0.0009, 1.0)]      # 0.0009 < 2^-10: unpruned whole-chip DP, window bound off
CONSTRAINTS = ['none', 'zeros', 'constants']


# ---- CPU: grouping of exact plans -------------------------------------------------------------------------------------
def _runs(counts):
    change = np.flatnonzero(counts[1:] != counts[:-1]) + 1
    starts = np.concatenate([[0], change])
    return np.diff(np.concatenate([starts, [len(counts)]])).astype(np.int64), counts[starts].astype(np.int64)


def _contig_stream(lens, deep=()):
    out = []
    for c, n in enumerate(lens):
        counts = np.full(n, 3 << 20, dtype=np.int64) if c in deep else (np.arange(n) % 3).astype(np.int64)
        run_len, run_val = _runs(counts)
        out.append(('c%d' % c, run_len, run_val, 0))
    return out


def _grouping(contigs, plan):
    return [[item[0] for item in batch] for batch in pb._batches(iter(contigs), plan)]


LENS = [5, 1, 2, 3, 4000, 70000, 12, 900, 1, 30000, 60000, 8]


@pytest.mark.parametrize('batch_nt,batch_contigs', [(pb.BATCH_NT, pb.BATCH_CONTIGS), (100000, 4), (0, 20000)])
def test_exact_plans_group_like_nop_plans(monkeypatch, batch_nt, batch_contigs):
    """unregularised exact plans (`exact`: no steps, `slidingwindow`: one window step) are grouped as 'nop' plans are"""
    monkeypatch.setattr(pb, 'BATCH_NT', batch_nt)
    monkeypatch.setattr(pb, 'BATCH_CONTIGS', batch_contigs)
    monkeypatch.setattr(pb, 'BATCH_ALONE', 50000)
    contigs = _contig_stream(LENS)
    nop = _grouping(contigs, _fusion_plan(configure_splitter()))
    for algorithm in ('exact', 'slidingwindow'):
        plan = _fusion_plan(configure_splitter(algorithm=algorithm))
        assert plan['final'] == 'exact'
        assert _grouping(contigs, plan) == nop, algorithm
    if batch_nt:
        assert max(len(g) for g in nop) > 1


def _fusion_plan(splitter):
    from pasio_b200.splitters import _fusion
    return _fusion.device_plan(splitter)


def test_contig_over_the_exact_count_limit_goes_alone():
    """a contig whose own total count reaches the exact DP's limit runs alone (and is refused there, as before); a 'nop'
    plan batches it"""
    contigs = _contig_stream([10, 20, 1000, 30, 40], deep={2})
    assert int(np.dot(contigs[2][1], contigs[2][2])) >= 2 ** 31
    exact = _grouping(contigs, _fusion_plan(configure_splitter(algorithm='exact')))
    assert exact == [['c0', 'c1'], ['c2'], ['c3', 'c4']]
    assert _grouping(contigs, _fusion_plan(configure_splitter())) == [['c0', 'c1', 'c2', 'c3', 'c4']]


def test_regularised_exact_plans_stay_one_contig_per_batch():
    """regularised `exact` / `slidingwindow` have no device plan: one contig per batch, as before"""
    contigs = _contig_stream([10, 20, 30])
    for algorithm in ('exact', 'slidingwindow'):
        splitter = configure_splitter(algorithm=algorithm, split_number_regularization=2.0)
        assert _fusion_plan(splitter) is None
        assert _grouping(contigs, None) == [['c0'], ['c1'], ['c2']]


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def eng():
    return _native.engine()


@pytest.fixture(scope='module')
def batch():
    return tgb.make_batch()


def _parts(counts, offsets):
    return [counts[a:b] for a, b in zip(offsets[:-1].tolist(), offsets[1:].tolist())]


def _local(cands, offsets, c):
    a, b = offsets[c], offsets[c + 1]
    return cands[(cands >= a) & (cands <= b)] - a


def batch_split(oracles, offsets, cands):
    """every contig's SquareSplitter.split over its own slice, shifted and united -> (splits, cells)"""
    out, cells = [], 0
    for c, fo in enumerate(oracles):
        local = _local(cands, offsets, c)
        out.append(fo.square_split(local)[1] + offsets[c])
        cells += len(local) * (len(local) - 1) // 2
    return np.unique(np.concatenate(out)), cells


def _list_lengths(cands, offsets):
    ranks = np.searchsorted(cands, offsets)
    return np.diff(ranks) + 1


def _check(eng, oracles, offsets, cands, what):
    want, want_cells = batch_split(oracles, offsets, cands)
    eng.square_split_batch()
    got = eng.candidates()
    if not np.array_equal(got, want):
        diff = np.setxor1d(got, want)[:10]
        raise AssertionError('%s: splits differ at %s (contigs %s)'
                             % (what, diff.tolist(), (np.searchsorted(offsets, diff, 'right') - 1).tolist()))
    cells, skipped = eng.round_stats()
    assert cells == want_cells and 0 <= skipped <= cells, (what, cells, want_cells, skipped)


def _oracles(parts, ab):
    return [c_oracle.FlatOracle(p, ab[0], ab[1], threads=THREADS) for p in parts]


@pytest.mark.gpu
@pytest.mark.parametrize('ab', AB)
def test_all_positions_of_the_batch(eng, batch, ab):
    """`exact`: every position of every contig of test_gpu_batches' layout is a candidate (lists on both sides of CAP)"""
    counts, offsets = batch
    lens = _list_lengths(np.arange(len(counts) + 1), offsets)
    assert lens.max() > CAP and np.any(lens <= 3) and len(lens) > 64
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts, offsets=offsets)
    eng.set_candidates(None)
    _check(eng, _oracles(_parts(counts, offsets), ab), offsets, np.arange(len(counts) + 1), ('all positions', ab))


@pytest.mark.gpu
@pytest.mark.parametrize('ab', AB[:2])
@pytest.mark.parametrize('constraint', CONSTRAINTS)
def test_reduced_lists_after_one_window_round(eng, batch, constraint, ab):
    """`slidingwindow`: the explicit list one window round leaves, per constraint"""
    counts, offsets = batch
    parts = _parts(counts, offsets)
    oracles = _oracles(parts, ab)
    cands, _ = tgb.batch_round(oracles, offsets, np.arange(len(counts) + 1), 2500, 1250, constraint)
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts, offsets=offsets)
    eng.set_candidates(None)
    eng.round(2500, 1250, constraint)
    assert np.array_equal(eng.candidates(), cands)
    _check(eng, oracles, offsets, cands, ('one round', constraint, ab))


def seam_batch():
    """all-positions lists of CAP - 1, CAP and CAP + 1 candidates, two longer ones (20 001 candidates and more: the
    whole-chip DP runs 157 row blocks and wraps its self-score ring), 1-, 2- and 3-nt contigs between them"""
    lens = [1, CAP - 2, 2, CAP - 1, 3, CAP, 1, 9000, 2, 20001, 3, 700, 1]
    parts = [synth.dnase_like(n, 300 + k, hotspot_share=0.4) if n > 3 else np.array([0, 4, 4][:n], dtype=np.int64)
             for k, n in enumerate(lens)]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    return np.concatenate(parts), offsets


@pytest.mark.gpu
@pytest.mark.parametrize('ab', AB)
def test_lists_at_the_class_seam(eng, ab):
    counts, offsets = seam_batch()
    lens = _list_lengths(np.arange(len(counts) + 1), offsets)
    assert {CAP - 1, CAP, CAP + 1} <= set(lens.tolist()) and lens.max() > 20000
    parts = _parts(counts, offsets)
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts, offsets=offsets)
    eng.set_candidates(None)
    _check(eng, _oracles(parts, ab), offsets, np.arange(len(counts) + 1), ('seam', ab))


@pytest.mark.gpu
def test_tables_grow_inside_the_call():
    """a deep contig (counts past 2^20) in a fresh context: the call asks for longer tables once, the retry finishes it"""
    counts, offsets = tgb.make_batch(seed=3)
    assert max(int(p.sum()) for p in _parts(counts, offsets)) > 1 << 20
    e = _native.Engine(_native.default_device())
    try:
        grown = []
        real = e._grow_tables
        e._grow_tables = lambda: (grown.append(1), real())
        e.use_scorer(ScorerFactory(1, 1.0))
        e.load(counts, offsets=offsets)
        e.set_candidates(None)
        _check(e, _oracles(_parts(counts, offsets), (1, 1.0)), offsets, np.arange(len(counts) + 1), 'deep')
        assert len(grown) >= 1
    finally:
        e.close()


@pytest.mark.gpu
def test_batch_count_past_2_31_and_one_contig_over_it(eng):
    """600 contigs of up to 2^24 counts each: the batch holds more than 2^31, every contig less -- it runs; a contig of 2^31 or
    more in a batch raises PasioDeviceError and leaves the candidates as they were"""
    rs = np.random.RandomState(11)
    lens = rs.randint(1, 60, 600)
    parts = [rs.randint(150000, 250000, n).astype(np.int64) for n in lens]
    counts = np.concatenate(parts)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    assert counts.sum() >= 2 ** 31 and max(int(p.sum()) for p in parts) < 2 ** 24
    fo = c_oracle.FlatOracle(counts, 1, 1.0, threads=THREADS)        # one oracle: its tables only reach one contig's total
    want = np.unique(np.concatenate([fo.square_split(np.arange(a, b + 1))[1]
                                     for a, b in zip(offsets[:-1].tolist(), offsets[1:].tolist())]))
    eng.use_scorer(ScorerFactory(1, 1.0))
    eng.load(counts, offsets=offsets)
    eng.set_candidates(None)
    eng.square_split_batch()
    assert np.array_equal(eng.candidates(), want)

    deep = [np.array([1, 2, 3], dtype=np.int64), np.full(1000, 3 << 20, dtype=np.int64), np.array([5, 0], dtype=np.int64)]
    offsets = np.concatenate([[0], np.cumsum([len(p) for p in deep])]).astype(np.int64)
    eng.load(np.concatenate(deep), offsets=offsets)
    eng.set_candidates(None)
    with pytest.raises(_native.PasioDeviceError, match='contig 1 of the batch'):
        eng.square_split_batch()
    assert eng.candidate_count() == offsets[-1] + 1


# ---- through the text route: batched against contig by contig -------------------------------------------------------
def _text(lens, seed, blocks=()):
    """bedgraph text of DNase-like and Poisson contigs; the contigs numbered in `blocks` are short constant blocks instead,
    whose boundaries a window round keeps (test_gpu_batches._blocks)"""
    rs = np.random.RandomState(seed)
    lines = []
    for c, n in enumerate(lens):
        if c in blocks:
            counts = tgb._blocks(int(n), seed + c)
        elif c % 3:
            counts = synth.dnase_like(int(n), seed + c, hotspot_share=0.4)
        else:
            counts = rs.poisson(4, int(n)).astype(np.int64)
        lines.extend(synth.to_bedgraph_lines('tx%04d' % c, counts, chrom_start=int(rs.randint(0, 100))))
    return ''.join(lines)


def _split_text(text, splitter, mode, **kw):
    out = io.StringIO()
    split_bedgraph_stream(io.StringIO(text), out, splitter, output_mode=mode, **kw)
    return out.getvalue()


SPLITTERS = {'exact': dict(algorithm='exact'),
             'slidingwindow': dict(algorithm='slidingwindow', window_size=1000, window_shift=500, split_constraints='none')}


@pytest.mark.gpu
@pytest.mark.parametrize('algorithm', sorted(SPLITTERS))
def test_text_route_batched_equals_contig_by_contig(monkeypatch, algorithm):
    """short and long lists (12 000 constant blocks keep more than CAP candidates after the window round), tiny contigs;
    all three output modes"""
    rs = np.random.RandomState(4)
    lens = np.concatenate([rs.randint(1, 400, 60), [1, 2, 3, 9000, 12000, 30000], rs.randint(1, 3000, 30)])
    text = _text(lens, 40, blocks={64})
    splitter = configure_splitter(**SPLITTERS[algorithm])
    batches = list(pb._batches(pb.contig_runs(text.encode()), _fusion_plan(splitter)))
    assert len(batches) == 1 and len(batches[0]) == len(lens)
    for mode in ['bedgraph', 'bed', 'bedgraph+length+LMM']:
        batched = _split_text(text, splitter, mode)
        monkeypatch.setattr(pb, 'BATCH_NT', 0)
        alone = _split_text(text, splitter, mode)
        monkeypatch.undo()
        assert batched == alone, (algorithm, mode)
        assert batched.count('\n') > len(lens)


@pytest.mark.gpu
@pytest.mark.parametrize('algorithm', sorted(SPLITTERS))
def test_config5_subsample_batched_pool_and_alone(monkeypatch, algorithm):
    """a config-5 sub-sample (transcripts of 1-50 kb): batched == contig by contig == two worker processes"""
    lens = synth.transcript_lengths(40, seed=8)
    text = _text(lens, 900)
    splitter = configure_splitter(**SPLITTERS[algorithm])
    mode = 'bedgraph+length+LMM'
    batched = _split_text(text, splitter, mode)
    monkeypatch.setattr(pb, 'BATCH_NT', 0)
    assert _split_text(text, splitter, mode) == batched
    monkeypatch.undo()
    import torch
    if torch.cuda.device_count() < 2:
        monkeypatch.setenv('PASIO_B200_POOL_SAME_DEVICE', '1')      # two workers on the one GPU
    assert _split_text(text, splitter, mode, devices=2) == batched
