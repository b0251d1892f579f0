"""The window check of the pruned window DP (certify_window in csrc/window_dp.cu, PASIO_TUNE_WINDOW_CERTIFY).

Before its block pipeline, the CTA kernel may check a whole window under the hypothesis "the first maximum of every row
j is column j-1".  If every row holds, every candidate survives; if row j* fails, the pipeline resumes at the block
that holds j*.  These tests check that results do not depend on the switch, and that the check's counters
(pasio_round_certify_stats) agree with what the oracle predicts for hand-built windows: failures in the first block,
at 32-row seams, in the last row, on an exact tie between t_{j-2,j} and t_{j-1,j}, and a failing window between
passing ones, whose done flag the phase-2 fast path reads."""
import os

import numpy as np
import pytest

from oracle import c_oracle, pasio_oracle as po
from pasio_b200 import _native, synth
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from test_gpu_batches import _explicit, make_batch

THREADS = max(1, min(32, os.cpu_count() or 1))
WS, SH = 2500, 1250
MEDIUM_MAX = 512          # larger windows go to the CTA kernel (WD_MEDIUM_MAX_CANDIDATES)
AB = [(1, 1.0), (2.5, 0.3), (0.0009, 1.0)]      # 0.0009 < 2^-10: no far bound, so no check


# ---- hand-built candidate lists ------------------------------------------------------------------------------------
def _fixed_point(o, n):
    c = np.arange(n + 1)
    while True:
        new, _ = o.round(c, WS, SH, 'none')
        if len(new) == len(c):
            return c
        c = new


def _insert(c, idx):
    """a spurious candidate halfway between c[i-1] and c[i] (i moved up to the next gap of two or more)"""
    i = idx
    while c[i] - c[i - 1] < 2:
        i += 1
    return np.insert(c, i, (c[i - 1] + c[i]) // 2)


def _first_bad(o, cands):
    """per window: (candidates, first row whose first maximum is not the row before, or None)"""
    out = []
    for st, en in po.window_ranges(len(cands), WS, SH):
        _, _, _, prev = o.square_split(cands[st:en])
        bad = np.flatnonzero(prev[1:] != np.arange(en - st - 1)) + 1
        out.append((en - st, int(bad[0]) if len(bad) else None))
    return out


def predicted_stats(o, cands):
    """(passed, fell back, rows proven before the resume) with every CTA-class window checked (window_phases 0)"""
    passed = fell = rows = 0
    for n, f in _first_bad(o, cands):
        if n <= MEDIUM_MAX:
            continue
        if f is None:
            passed += 1
        else:
            fell += 1
            kf = (f - 1) // 32
            rows += 32 * kf if kf >= 2 else 0
    return passed, fell, rows


_CASES = {}


def hand_built():
    """name -> (counts, candidates, oracle)"""
    if _CASES:
        return _CASES
    counts = synth.dnase_like(1_200_000, 7)
    o = c_oracle.FlatOracle(counts, 1, 1.0, threads=THREADS)
    fp = _fixed_point(o, len(counts))
    for name, idx in [('first_block', 11), ('seam_64', 63), ('seam_96', 96), ('last_row', 2499), ('pass_fail_pass', 3750)]:
        _CASES[name] = (counts, _insert(fp, idx), o)
    rs = np.random.RandomState(0)
    ties = (rs.random_sample(300_000) < 0.35).astype(np.int64)
    ot = c_oracle.FlatOracle(ties, 1, 1.0, threads=THREADS)
    c = np.arange(len(ties) + 1)
    for _ in range(3):
        c, _ = ot.round(c, WS, SH, 'none')
    _CASES['ties'] = (ties, c, ot)
    return _CASES


def _tie_windows(counts, cands, o):
    """CTA-class windows whose first failing row j has t_{prev,j} == t_{j-1,j} exactly (alpha 1, beta 1)"""
    tab = po.Tables(1, 1.0)
    cs = np.concatenate([[0], np.cumsum(counts)])
    found = 0
    for st, en in po.window_ranges(len(cands), WS, SH):
        w = cands[st:en]
        if len(w) <= MEDIUM_MAX:
            continue
        _, _, P, prev = o.square_split(w)
        bad = np.flatnonzero(prev[1:] != np.arange(len(w) - 1)) + 1
        if not len(bad):
            continue
        j = bad[0]

        def t(i):
            u = cs[w[j]] - cs[w[i]] + 1
            return (tab.lgam_tab[u] - float(u) * tab.log_tab[w[j] - w[i]]) + P[i]
        found += t(prev[j]) == t(j - 1)
    return found


def test_hand_built_windows_fail_where_intended():
    """the failures sit in the first block, at the 64/65 and 96/97 seams, in the last row, on exact ties, and one
    failing window (resuming after the first two blocks) lies between two passing phase-1 windows"""
    cases = hand_built()
    fb = {name: _first_bad(o, c) for name, (_, c, o) in cases.items()}
    assert 1 <= fb['first_block'][0][1] <= 32
    assert fb['seam_64'][0][1] in (64, 65)
    assert fb['seam_96'][0][1] in (96, 97)
    assert fb['last_row'][0] == (2501, 2500)
    w = fb['pass_fail_pass']
    assert w[0][1] is None and w[4][1] is None and w[2][1] > 64
    assert _tie_windows(*cases['ties']) > 0


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def eng():
    e = _native.engine()
    yield e
    e.set_tuning('window_certify', 1)
    e.set_tuning('window_phases', 1)


def _rounds(eng, cands, constraint, certify, max_rounds=64):
    """rounds until the fixed point: [(n_in, n_out, cells, candidates, certify stats)]"""
    eng.set_tuning('window_certify', certify)
    eng.set_candidates(cands)
    out = []
    for _ in range(max_rounds):
        n_in, n_out, cells = eng.round(WS, SH, constraint)
        out.append((n_in, n_out, cells, eng.candidates().copy(), eng.round_certify_stats()))
        if n_in == n_out:
            return out
    raise AssertionError('no fixed point')


def _same(a, b, what):
    assert len(a) == len(b), what
    for r, (x, y) in enumerate(zip(a, b)):
        assert x[:3] == y[:3] and np.array_equal(x[3], y[3]), (what, r)


def _check_switch(eng, cands, constraint, ab, what):
    off, dflt, always = (_rounds(eng, cands, constraint, v) for v in (0, 1, 2))
    _same(off, dflt, what)
    _same(off, always, what)
    assert all(r[4] == (0, 0, 0) for r in off)
    return [sum(r[4][k] for r in always) for k in range(3)]


@pytest.mark.gpu
@pytest.mark.parametrize('ab', AB)
def test_bench_contig_prefix_identical_with_and_without_check(eng, ab):
    """the first 30 Mb of the bench contig: every round equal with the check off, on by default and in every round"""
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(synth.dnase_like(30_000_000, 1000))
    passed, fell, rows = _check_switch(eng, None, 'constants', ab, ('30Mb', ab))
    if ab[0] >= 2 ** -10:
        assert passed > 0 and fell > 0 and rows > 0, (passed, fell, rows)
    else:
        assert (passed, fell, rows) == (0, 0, 0)


@pytest.mark.gpu
@pytest.mark.parametrize('ab', AB)
def test_batch_identical_with_and_without_check(eng, ab):
    """the 67-contig batch, from all positions and from per-contig 70 % lists"""
    counts, offsets = make_batch()
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts, offsets=offsets)
    for cands, constraint in [(None, 'constants'), (_explicit(offsets, 0.7, 5), 'none')]:
        stats = _check_switch(eng, cands, constraint, ab, ('batch', ab, constraint))
        if ab[0] < 2 ** -10:
            assert stats == [0, 0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['first_block', 'seam_64', 'seam_96', 'last_row', 'pass_fail_pass', 'ties'])
def test_hand_built_windows_round_by_round(eng, name):
    """every window through the CTA kernel (phases off): the counters are the oracle's prediction and every round
    equals the oracle; then again with phases on, where the phase-2 fast path reads the flags of checked windows"""
    counts, cands, o = hand_built()[name]
    eng.use_scorer(ScorerFactory(1, 1.0))
    eng.load(counts)
    eng.set_tuning('window_certify', 2)
    try:
        for phases in (0, 1):
            eng.set_tuning('window_phases', phases)
            eng.set_candidates(cands)
            c = cands
            for r in range(64):
                want, want_cells = o.round(c, WS, SH, 'none')
                expect = predicted_stats(o, c)
                n_in, n_out, cells = eng.round(WS, SH, 'none')
                got = eng.candidates()
                assert np.array_equal(got, want) and cells == want_cells, (name, phases, r)
                stats = eng.round_certify_stats()
                if phases == 0:
                    assert stats == expect, (name, r, stats, expect)
                    if r == 0:
                        assert stats[1] > 0, (name, stats)
                if len(want) == len(c):
                    break
                c = want
    finally:
        eng.set_tuning('window_phases', 1)
        eng.set_tuning('window_certify', 1)
