"""The window check of the pruned window DP (certify_window in csrc/window_dp.cu) at the edges of its structure.

The check works in groups of CT_RB = 16 row blocks (rows [1 + 512 g, 513 + 512 g)), each with its own P prefix, its own
level-1 list and its own early exit.  The windows below are built so that the first failing row (the first row j whose
first maximum is not column j - 1) lies where those groups meet: rows 511 .. 514, 1024 / 1025 and 2048 / 2049 of a
2 501-candidate window, the last group of windows of 513, 514, 1 025 and 1 026 candidates (the last two end in a group
of one row block, and 514 and 1 026 in a block of one row), and in the last row block (255) and at the seam of the last
group (row 7 681) of 8 192-candidate windows, whose level-1 entries carry the largest column blocks.  They run round by
round with the check forced (window_certify 2) and off, against the C oracle bit for bit: candidates, cells and the
check's counters (pasio_round_certify_stats), at alpha = beta = 1, at the far bound's parameter edges (2^-10, small,
large real and large integer alpha, extreme beta; real alpha runs the AI = false instantiation of the check) and in the
batched whole-list DP (pasio_square_split_batch), where every list of up to 8 192 candidates is one window.

Construction: constant blocks at alternating low and high levels (test_gpu_batches._blocks).  Their boundaries are a
list in which every row's first maximum is the row before, in every window.  One spurious candidate halfway through the
block that ends at candidate r - 1 makes row r skip it: row r is then the first failing row of every window that holds
rows r - 2 .. r.  Other windows fail first by an exact tie (TIE_CASES): there only the strict comparison against T_r
tells a failure from a pass.  The CPU tests check all of that with the oracle.  Every constructed failure lies in a near
column (r - 2, found exactly in step (c) of the check); the far levels (d) and (e) run as bounds over the rows before
it, in 8 192-candidate windows with level-1 entries of every column block."""
import os

import numpy as np
import pytest

import test_gpu_batches as tgb
import test_gpu_exact_batches as teb
from oracle import c_oracle, pasio_oracle as po
from pasio_b200 import _native
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from test_gpu_edges import _bound_data
from test_gpu_edges import _explicit as _explicit_positions

THREADS = max(1, min(32, os.cpu_count() or 1))
MEDIUM_MAX = 512          # larger windows go to the CTA kernel (WD_MEDIUM_MAX_CANDIDATES)
CAP = teb.CAP             # the largest fused window: 8 192 candidates
ALPHA_BOUND_MIN = 2 ** -10
NO_BOUND_AB = (0.0009, 1.0)     # 0.0009 < 2^-10: no far bound, so no check


# ---- hand-built candidate lists ------------------------------------------------------------------------------------
def _boundaries(counts):
    """both ends and every position where the value changes"""
    return np.concatenate([[0], np.flatnonzero(counts[1:] != counts[:-1]) + 1, [len(counts)]]).astype(np.int64)


def _spurious(cands, rows):
    """one spurious candidate per row r (indices of the returned list), halfway between the candidates that become
    r - 2 and r: row r's first maximum is then column r - 2"""
    c = cands
    for r in sorted(rows):
        assert c[r - 1] - c[r - 2] >= 2
        c = np.insert(c, r - 1, (c[r - 2] + c[r - 1]) // 2)
    return c


def first_bad(o, cands, ws, sh):
    """per window: (candidates, first row whose first maximum is not the row before, or None)"""
    out = []
    for st, en in po.window_ranges(len(cands), ws, sh):
        prev = o.square_split(cands[st:en])[3]
        bad = np.flatnonzero(prev[1:] != np.arange(en - st - 1)) + 1
        out.append((en - st, int(bad[0]) if len(bad) else None))
    return out


def expected_bad(m, ws, sh, rows):
    """first_bad as the construction intends it: the first row r of `rows` with r - 2 .. r inside the window"""
    out = []
    for st, en in po.window_ranges(m, ws, sh):
        inside = [r - st for r in sorted(rows) if st + 2 <= r < en]
        out.append((en - st, inside[0] if inside else None))
    return out


def stats_of(bad):
    """the counters for windows [(candidates, first failing row or None)] that all go through the check (window_phases
    0): CTA-class windows (more than 512 candidates) pass, or fall back with the rows of the blocks before the failing
    row's block proven (none when that block is one of the first two, where the pipeline starts anyway)"""
    passed = fell = rows = 0
    for n, f in bad:
        if n <= MEDIUM_MAX:
            continue
        if f is None:
            passed += 1
        else:
            fell += 1
            kf = (f - 1) // 32
            rows += 32 * kf if kf >= 2 else 0
    return passed, fell, rows


# seam cases: one 2 501-candidate window (size 2500, shift 1250), the first failure at row r of window 0; 2049 is the
# first row of the last group (rows 2049 .. 2500)
SEAM_ROWS = [511, 512, 513, 514, 1024, 1025, 2048, 2049]
# size cases: windows of n candidates (size = shift = n - 1): window 0 passes, window 1 fails at this row of its last
# group (for 514 and 1 026 the last row, alone in its row block and group)
SIZE_ROWS = {513: 512, 514: 513, 1025: 513, 1026: 1025}
# the largest fused window: size = shift = 8191; window 0 passes, window 1 fails in block 255, window 2 at row 7 681
# (first row of group 15)
BIG_ROWS = [8170, 7681]

# block levels scaled towards the prior mean alpha / beta (so that every block boundary is worth a split)
SCALE = {(1, 1.0): 1, (2 ** -10, 1.0): 1, (0.3, 0.01): 30, (40.5, 1.0): 40, (1000, 1.0): 25, (1, 0.01): 5,
         (2.5, 0.3): 1, NO_BOUND_AB: 1}


def _case(name, ab):
    """-> (counts, candidates, window size, shift, first failing rows)"""
    seed = sum(map(ord, name))
    if name.startswith('row'):
        r = int(name[3:])
        counts = SCALE[ab] * tgb._blocks(6000, seed)
        return counts, _spurious(_boundaries(counts), [r]), 2500, 1250, [r]
    if name.startswith('n'):
        n = int(name[1:])
        ws = n - 1
        counts = SCALE[ab] * tgb._blocks(2 * ws - 1, seed)
        r = ws + SIZE_ROWS[n]
        return counts, _spurious(_boundaries(counts), [r]), ws, ws, [r]
    assert name == 'big'
    ws = CAP - 1
    counts = SCALE[ab] * tgb._blocks(3 * ws - 2, seed)
    rows = [ws + BIG_ROWS[0], 2 * ws + BIG_ROWS[1]]
    return counts, _spurious(_boundaries(counts), rows), ws, ws, rows


SEAM_CASES = ['row%d' % r for r in SEAM_ROWS] + ['n%d' % n for n in SIZE_ROWS]


# ---- windows whose first failing row is an exact tie ----------------------------------------------------------------
# At alpha = beta = 1 (segment creation cost 0) a segment of 2 positions holding one count and a segment of 3 empty
# positions score exactly what the 5 positions score together: 0 - 2 log 3 - log 4 = -2 log 6, and in the tables
# 1 * log(4) == 2 * log(2) bit for bit.  Blocks A = [1, 0] and B = [0, 0, 0] between two high blocks, with candidates at
# their starts and at B's end (row r), make t_{r-2,r} = T_r in exact arithmetic; rounded, the two sums agree for some
# prefixes only, so the seed of the other blocks is searched until the oracle's first maximum of row r is column r - 2
# by an exact tie.  The check must then fail row r: only the strict `<` against T_r tells the tie from a pass.
# name -> (window size, shift, blocks, row r (index in the list), first candidate of the window that must fail at r)
TIE_CASES = {'tie512': (2500, 1250, 6000, 512, 0), 'tie513': (2500, 1250, 6000, 513, 0),
             'tie2049': (2500, 1250, 6000, 2049, 0),
             'tie_n1026': (1025, 1025, 3 * 1025, 2 * 1025, 1025),          # last row of the window, alone in its group
             'tie_big': (CAP - 1, CAP - 1, 2 * (CAP - 1), CAP - 1 + 7681, CAP - 1)}   # row 7 681 of an 8 192 window


def _tie_blocks(n_blocks, r, seed):
    """-> (counts, candidates): the starts of n_blocks blocks and the end; blocks r - 2 and r - 1 are A and B, the
    blocks on both sides of them high, the others alternating low / high"""
    rs = np.random.RandomState(seed)
    # lengths and high levels scaled by the seed: that moves |P| at row r across binades, which decides the rounding
    lens, lo = rs.randint(3, 10, n_blocks) * (1 + seed % 3), rs.randint(0, 3, n_blocks)
    hi = rs.randint(40, 80, n_blocks) * (1 + seed % 7)
    parts = []
    for k in range(n_blocks):
        if k == r - 2:
            parts.append(np.array([1, 0]))
        elif k == r - 1:
            parts.append(np.zeros(3, dtype=np.int64))
        else:
            high = (r - 3 - k) % 2 == 0 if k < r else (k - r) % 2 == 0
            parts.append(np.full(lens[k], hi[k] if high else lo[k]))
    return (np.concatenate(parts).astype(np.int64),
            np.concatenate([[0], np.cumsum([len(q) for q in parts])]).astype(np.int64))


def tie_row(o, counts, w):
    """(first failing row of window w, whether its first maximum ties exactly with column row - 1)"""
    _, _, P, prev = o.square_split(w)
    bad = np.flatnonzero(prev[1:] != np.arange(len(w) - 1)) + 1
    if not len(bad):
        return None, False
    j = int(bad[0])

    def t(i):                                   # alpha = 1: the integer-alpha tables, gammaln(u) and log(L + 1)
        u = o.Cg[w[j]] - o.Cg[w[i]] + 1
        return (o.g[u] - float(u) * o.lg[w[j] - w[i]]) + P[i]
    return j, bool(t(prev[j]) == t(j - 1))


def tie_list(n_blocks, r, st, en):
    """the first seed whose window [st, en) fails first at row r by an exact tie -> (counts, candidates, oracle)"""
    for seed in range(32):
        counts, cands = _tie_blocks(n_blocks, r, seed)
        o = c_oracle.FlatOracle(counts, 1, 1.0, threads=THREADS)
        if tie_row(o, counts, cands[st:en]) == (r - st, True):
            return counts, cands, o
    raise AssertionError('no exact tie at row %d' % r)
EDGE_AB = [(2 ** -10, 1.0), (0.3, 0.01), (40.5, 1.0), (1000, 1.0), (1, 0.01)]
# (1, 1000): with beta far above every segment length a segment's score hardly depends on its length, so neighbouring
# blocks merge and the block boundaries are no fixed point; that point runs the _bound_data profiles only
EDGE_AB_PROFILES_ONLY = [(1, 1000.0)]

_CACHE = {}


def hand_built(name, ab=(1, 1.0)):
    """-> (counts, candidates, window size, shift, oracle, first failing rows)"""
    key = (name, ab)
    if key not in _CACHE and name in TIE_CASES:
        assert ab == (1, 1.0)
        ws, sh, nb, r, st = TIE_CASES[name]
        counts, cands, o = tie_list(nb, r, st, st + ws + 1)
        _CACHE[key] = (counts, cands, ws, sh, o, [r])
    if key not in _CACHE:
        counts, cands, ws, sh, rows = _case(name, ab)
        _CACHE[key] = (counts, cands, ws, sh, c_oracle.FlatOracle(counts, *ab, threads=THREADS), rows)
    return _CACHE[key]


def _check_construction(name, ab):
    counts, cands, ws, sh, o, rows = hand_built(name, ab)
    got = first_bad(o, cands, ws, sh)
    assert got == expected_bad(len(cands), ws, sh, rows), (name, ab, got)
    # without the spurious candidates every window passes
    clean = np.delete(cands, [r - 1 for r in rows])
    assert all(f is None for _, f in first_bad(o, clean, ws, sh)), (name, ab)
    return got


def test_hand_built_windows_fail_where_intended():
    """(CPU) every construction fails exactly at the intended row of the intended window size, and passes without its
    spurious candidates"""
    for name in SEAM_CASES:
        got = _check_construction(name, (1, 1.0))
        if name.startswith('row'):
            assert got[0] == (2501, int(name[3:])), (name, got)
        else:
            n = int(name[1:])
            assert got[:2] == [(n, None), (n, SIZE_ROWS[n])], (name, got)
    got = _check_construction('big', (1, 1.0))
    assert got == [(CAP, None), (CAP, BIG_ROWS[0]), (CAP, BIG_ROWS[1])]
    assert (BIG_ROWS[0] - 1) // 32 == 255 and (BIG_ROWS[1] - 1) % 512 == 0


@pytest.mark.parametrize('ab', EDGE_AB)
def test_hand_built_windows_at_parameter_edges_fail_where_intended(ab):
    """(CPU) the same seam and size constructions at the far bound's parameter edges"""
    for name in SEAM_CASES:
        _check_construction(name, ab)


def test_tie_windows_fail_where_intended():
    """(CPU) the first failing row of the intended window is an exact tie at rows 512, 513 and 2049 of a 2 501-candidate
    window, at the last row of a 1 026-candidate window and at row 7 681 of an 8 192-candidate window"""
    for name, (ws, sh, nb, r, st) in TIE_CASES.items():
        counts, cands, _, _, o, _ = hand_built(name)
        w = [(a, b) for a, b in po.window_ranges(len(cands), ws, sh) if a == st][0]
        assert w[1] - w[0] == ws + 1 and tie_row(o, counts, cands[w[0]:w[1]]) == (r - st, True), name
    assert TIE_CASES['tie_n1026'][3] - TIE_CASES['tie_n1026'][4] == 1025


# ---- GPU: hand-built windows round by round --------------------------------------------------------------------------
@pytest.fixture(scope='module')
def eng():
    e = _native.engine()
    yield e
    _reset(e)


# the keys these tests set, and the defaults a context takes from the environment (api.cu)
TUNING_DEFAULTS = {key: int(os.environ.get(env, '1')) for key, env in
                   [('window_certify', 'PASIO_WD_CERTIFY'), ('window_phases', 'PASIO_WD_PHASES'),
                    ('window_speculate', 'PASIO_WD_SPECULATE')]}


def _reset(e):
    for key, value in TUNING_DEFAULTS.items():
        e.set_tuning(key, value)


def oracle_rounds(o, cands, ws, sh):
    """[(candidates in, candidates out, cells, counters with every window checked)] until the fixed point"""
    out, c = [], cands
    for _ in range(64):
        new, cells = o.round(c, ws, sh, 'none')
        out.append((c, new, cells, stats_of(first_bad(o, c, ws, sh))))
        if len(new) == len(c):
            return out
        c = new
    raise AssertionError('no fixed point')


def device_rounds(eng, want, ws, sh, certify, phases, speculate, what):
    """the device's rounds from want[0]'s list, each against the oracle's; the counters are the prediction whenever
    every window goes through the check (forced, phases off), zero with the check off.  -> counters per round"""
    eng.set_tuning('window_certify', certify)
    eng.set_tuning('window_phases', phases)
    eng.set_tuning('window_speculate', speculate)
    eng.set_candidates(want[0][0])
    out = []
    for r, (c, new, cells, predicted) in enumerate(want):
        n_in, n_out, got_cells = eng.round(ws, sh, 'none')
        got = eng.candidates()
        assert (n_in, n_out) == (len(c), len(new)), (what, certify, phases, speculate, r)
        if not np.array_equal(got, new):
            raise AssertionError('%s: round %d (certify %d, phases %d, speculate %d): candidates differ at %s'
                                 % (what, r, certify, phases, speculate, np.setxor1d(got, new)[:10].tolist()))
        assert got_cells == cells, (what, certify, phases, speculate, r, got_cells, cells)
        stats = eng.round_certify_stats()
        if certify == 0:
            assert stats == (0, 0, 0), (what, r, stats)
        elif phases == 0:
            assert stats == predicted, (what, r, phases, speculate, stats, predicted)
        out.append(stats)
    return out


def _run_hand_built(eng, name, ab, settings):
    counts, cands, ws, sh, o, rows = hand_built(name, ab)
    want = oracle_rounds(o, cands, ws, sh)
    assert want[0][3][1] >= 1, (name, ab, want[0][3])        # the first round has a failing CTA-class window
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts)
    try:
        for certify, phases, speculate in settings:
            stats = device_rounds(eng, want, ws, sh, certify, phases, speculate, (name, ab))
            if certify == 2 and phases == 0:
                assert sum(stats[0][:2]) > 0, (name, ab, stats)   # the forced check ran
    finally:
        _reset(eng)


# (window_certify, window_phases, window_speculate)
ALL_SETTINGS = [(2, 0, 1), (2, 0, 0), (2, 1, 1), (2, 1, 0), (0, 0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize('name', SEAM_CASES + ['big'] + sorted(TIE_CASES))
def test_hand_built_windows_round_by_round(eng, name):
    """alpha = beta = 1 (integer alpha): with every window checked (phases off) the counters are the oracle's prediction
    and every round equals the oracle, with speculation on and off; with phases on (the phase-2 fast path reads the
    flags of checked windows) and with the check off every round equals the oracle as well"""
    _run_hand_built(eng, name, (1, 1.0), ALL_SETTINGS)


# ---- GPU: parameter edges ------------------------------------------------------------------------------------------
def _run_profile(eng, ab, data):
    """test_gpu_edges' profile from a 70 % list to the fixed point (2500 / 1250) with the check forced (phases off:
    counters as predicted) and off: every round equals the oracle, and the forced check ran"""
    counts = _bound_data(data, ab)
    o = c_oracle.FlatOracle(counts, *ab, threads=THREADS)
    want = oracle_rounds(o, _explicit_positions(len(counts), 0.7, 12), 2500, 1250)
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts)
    try:
        forced = device_rounds(eng, want, 2500, 1250, 2, 0, 1, (data, ab))
        device_rounds(eng, want, 2500, 1250, 0, 0, 1, (data, ab))
    finally:
        _reset(eng)
    assert sum(s[0] + s[1] for s in forced) > 0, (ab, data, forced)


@pytest.mark.gpu
@pytest.mark.parametrize('ab', EDGE_AB)
def test_parameter_edges(eng, ab):
    """every seam and size case, and the 'ties01', 'dnase' and 'deep' profiles, with the check forced (phases off:
    counters as predicted) and off, against the oracle; 2^-10, 0.3 and 40.5 run the real-alpha instantiation"""
    for name in SEAM_CASES:
        _run_hand_built(eng, name, ab, [(2, 0, 1), (0, 0, 1)])
    for data in ('ties01', 'dnase', 'deep'):
        _run_profile(eng, ab, data)


@pytest.mark.gpu
@pytest.mark.parametrize('ab', EDGE_AB_PROFILES_ONLY)
def test_profiles_at_extreme_beta(eng, ab):
    """beta = 1000: the three profiles only (see EDGE_AB_PROFILES_ONLY)"""
    for data in ('ties01', 'dnase', 'deep'):
        _run_profile(eng, ab, data)


# ---- the check inside pasio_square_split_batch -----------------------------------------------------------------------
# (candidates of the contig's list, first failing row or None); tiny contigs (1 .. 3 nt, all positions) in between
BATCH_LISTS = [(300, None), (512, 300), (513, 512), (514, 513), (2501, None), (2501, 2049), (8191, 7681), (8192, 8170),
               (8192, None), (9000, 5000)]
BATCH_AB = [(1, 1.0), (2.5, 0.3)]
# at alpha = beta = 1 also lists whose first failing row is an exact tie (TIE_CASES)
BATCH_TIES = [(2501, 2049), (CAP, 7681)]


def _batch_lists(ab):
    return [(n, row, False) for n, row in BATCH_LISTS] + [(n, row, True) for n, row in BATCH_TIES if ab == (1, 1.0)]


def check_batch(ab=(1, 1.0)):
    """-> (counts, offsets, candidates, kinds): kinds = [(list length, first failing row or None, exact tie)] of the
    non-tiny contigs"""
    key = ('batch', ab)
    if key in _CACHE:
        return _CACHE[key]
    parts, lists, kinds = [], [], []
    tiny = iter([1, 2, 3] * 5)
    for k, (n, row, tie) in enumerate(_batch_lists(ab)):
        t = next(tiny)
        parts.append(np.array([0, 4, 4][:t], dtype=np.int64))
        lists.append(np.arange(t + 1))
        if tie:
            counts, cands, _ = tie_list(n - 1, row, 0, n)
        else:
            counts = SCALE[ab] * tgb._blocks(n - 1 - (row is not None), 700 + k)
            cands = _boundaries(counts)
            cands = cands if row is None else _spurious(cands, [row])
        lists.append(cands)
        parts.append(counts)
        kinds.append((n, row, tie))
    t = next(tiny)
    parts.append(np.array([0, 4, 4][:t], dtype=np.int64))
    lists.append(np.arange(t + 1))
    offsets = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.int64)
    cands = np.unique(np.concatenate([c + o for c, o in zip(lists, offsets[:-1])]))
    _CACHE[key] = (np.concatenate(parts), offsets, cands, kinds)
    return _CACHE[key]


def _batch_oracles(counts, offsets, ab):
    key = ('oracles', ab)
    if key not in _CACHE:
        _CACHE[key] = [c_oracle.FlatOracle(p, *ab, threads=THREADS) for p in teb._parts(counts, offsets)]
    return _CACHE[key]


def batch_stats(oracles, offsets, cands):
    """the counters of pasio_square_split_batch with the check on: a list of 513 .. CAP candidates is one CTA-class
    window over the whole list; shorter lists go to the warp kernels, longer ones to the whole-chip DP"""
    bad = []
    for c, o in enumerate(oracles):
        local = teb._local(cands, offsets, c)
        if MEDIUM_MAX < len(local) <= CAP:
            prev = o.square_split(local)[3]
            f = np.flatnonzero(prev[1:] != np.arange(len(local) - 1)) + 1
            bad.append((len(local), int(f[0]) if len(f) else None))
    return stats_of(bad)


def test_batch_lists_fail_where_intended():
    """(CPU) the batch's lists have the intended lengths and first failing rows; one window round (2500 / 1250,
    constraint none) removes exactly the spurious candidates, under 1 % of the list"""
    for ab in BATCH_AB:
        counts, offsets, cands, kinds = check_batch(ab)
        oracles = _batch_oracles(counts, offsets, ab)
        parts = teb._parts(counts, offsets)
        lens = teb._list_lengths(cands, offsets)
        assert sorted(n for n, _, _ in kinds) == sorted(int(x) for x in lens if x > 4)
        assert set(lens.tolist()) >= {2, 3, 4, 300, 512, 513, 514, 2501, CAP - 1, CAP} and lens.max() > CAP
        for c, o in enumerate(oracles):
            local = teb._local(cands, offsets, c)
            if len(local) <= 4:
                continue
            n, row, tie = kinds[c // 2]
            assert len(local) == n and tie_row(o, parts[c], local) == (row, tie), (ab, c, n, row, tie)
        failing = [row for n, row, _ in kinds if MEDIUM_MAX < n <= CAP and row is not None]
        rows = 32 * sum((f - 1) // 32 for f in failing)
        assert batch_stats(oracles, offsets, cands) == (2, len(failing), rows)
        assert len(failing) == (7 if ab == (1, 1.0) else 5)
        after, _ = tgb.batch_round(oracles, offsets, cands, 2500, 1250, 'none')
        before_lens, after_lens = lens[1::2], teb._list_lengths(after, offsets)[1::2]
        spurious = [not tie and row is not None for _, row, tie in kinds]
        assert np.array_equal((before_lens - after_lens)[spurious], np.ones(sum(spurious)))
        assert 100 * (len(cands) - len(after)) < len(cands)
        # the lists without a tie pass (512 + 1 candidates became 512: warp class); the round drops the tied candidate
        # of the 2 501-candidate list and keeps that of the 8 192-candidate one, whose whole list still fails at
        # row 7 681
        want = (6, 0, 0) if ab != (1, 1.0) else (7, 1, 32 * (7680 // 32))
        assert batch_stats(oracles, offsets, after) == want, ab


def _batch_switch(eng, ab, predicted):
    counts, offsets, cands, _ = check_batch(ab)
    oracles = _batch_oracles(counts, offsets, ab)
    eng.use_scorer(ScorerFactory(*ab))
    eng.load(counts, offsets=offsets)
    try:
        for certify in (0, 1, 2):
            eng.set_tuning('window_certify', certify)
            eng.set_candidates(cands)
            teb._check(eng, oracles, offsets, cands, ('batch', ab, certify))
            stats = eng.round_certify_stats()
            assert stats == (predicted if certify == 2 else (0, 0, 0)), (ab, certify, stats, predicted)
    finally:
        _reset(eng)


@pytest.mark.gpu
@pytest.mark.parametrize('ab', BATCH_AB)
def test_batch_whole_lists_with_and_without_check(eng, ab):
    """window_certify 0, 1 and 2 give the oracle's splits and cells; with 2 the counters are the per-contig prediction;
    with 0, and with 1 right after set_candidates (no round to go by), they are zero.  At alpha = 1 the same batch
    runs at alpha 0.0009 too, where the far bound and so the check are off: the counters stay zero"""
    counts, offsets, cands, _ = check_batch(ab)
    predicted = batch_stats(_batch_oracles(counts, offsets, ab), offsets, cands)
    assert predicted[0] > 0 and predicted[1] > 0
    _batch_switch(eng, ab, predicted)
    if ab == (1, 1.0):
        _batch_switch(eng, NO_BOUND_AB, (0, 0, 0))


@pytest.mark.gpu
def test_batch_default_rule_after_a_round(eng):
    """the default rule (window_certify 1) on the route `slidingwindow` takes: a window round that removes under 1 %
    turns the check on for the whole-list DP that follows; after load or set_candidates it stays off"""
    ab = (1, 1.0)
    counts, offsets, cands, _ = check_batch(ab)
    oracles = _batch_oracles(counts, offsets, ab)
    after, after_cells = tgb.batch_round(oracles, offsets, cands, 2500, 1250, 'none')
    eng.use_scorer(ScorerFactory(*ab))
    _reset(eng)
    eng.set_tuning('window_certify', 1)
    try:
        eng.load(counts, offsets=offsets)
        eng.set_candidates(cands)
        _, _, cells = eng.round(2500, 1250, 'none')
        assert np.array_equal(eng.candidates(), after) and cells == after_cells
        teb._check(eng, oracles, offsets, after, 'after a round')
        assert eng.round_certify_stats() == batch_stats(oracles, offsets, after) == (7, 1, 7680)

        eng.load(counts, offsets=offsets)
        eng.set_candidates(after)
        teb._check(eng, oracles, offsets, after, 'after set_candidates')
        assert eng.round_certify_stats() == (0, 0, 0)

        eng.set_candidates(cands)                      # the counters of a checked round ...
        eng.set_tuning('window_certify', 2)
        eng.round(2500, 1250, 'none')
        assert sum(eng.round_certify_stats()[:2]) > 0
        eng.set_tuning('window_certify', 1)
        eng.load(counts, offsets=offsets)              # ... do not survive into the whole-list DP after load
        eng.square_split_batch()
        assert eng.round_certify_stats() == (0, 0, 0)
    finally:
        _reset(eng)
