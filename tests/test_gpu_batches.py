"""Batched contigs through every kernel, round by round, against per-contig oracles.

Short contigs reach the device many at a time: one "super-contig" with forced boundaries (load with offsets,
process_bedgraph._batches).  The reference segments contigs one by one (process_bedgraph.py:69), so the oracle here runs
every contig on its own (c_oracle.FlatOracle, reg_oracle.FlatOracleReg, po.Scorer), shifts its result by the contig's
offset and takes the union.  Everything is compared bit for bit, except the parallel log-factorial scan
(logfac_exact = 0, 1e-9).

The batch (_layout) puts contig boundaries on bitmap-word seams (31, 32, 33 mod 32), scan-tile seams (4095, 4096,
4097 mod 4096) and a log-factorial tile seam (2048); it has contigs of 1, 2 and 3 nt at the start, in the middle and at
the end, contigs whose round-1 or tail windows hold exactly 160, 161, 512, 513 and 514 candidates, contigs with several
CTA-class windows, an all-zero and a constant contig next to dense ones, a deep contig whose window counts pass 2^20,
DNase-like and 0/1 contigs, and more than 64 contigs."""
import io
import os

import numpy as np
import pytest

import reg_oracle as ro
from oracle import c_oracle, pasio_oracle as po
from pasio_b200 import _native, configure_splitter, synth
from pasio_b200.log_marginal_likelyhood import ScorerFactory
from pasio_b200.splitters.square_splitter import _identity

THREADS = max(1, min(32, os.cpu_count() or 1))
CLASS_EDGES = [160, 161, 512, 513, 514]     # candidates per window around the warp / CTA class limits (common.cuh)
EDGE_GEOMS = [(2500, 1250), (512, 256), (1000, 333)]
CONSTRAINTS = ['none', 'zeros', 'constants']


# ---- the batch ---------------------------------------------------------------------------------------------------------
def _layout():
    """(offsets, kinds): the contig boundaries are chosen first, the contig lengths follow from them"""
    bounds, kinds = [0], []

    def add(length, kind):
        bounds.append(bounds[-1] + int(length))
        kinds.append(kind)

    def reach(mod, rem, kind, min_len=1):          # next boundary at a position = rem (mod mod), min_len or more further on
        p = bounds[-1] + min_len
        add(min_len + (rem - p) % mod, kind)

    for k in (1, 2, 3):                            # tiny contigs at the start
        add(k, 'dnase')
    reach(32, 31, 'dnase', 40)                     # bitmap-word seams: 31, 32, 33 (mod 32)
    add(1, 'ties')
    add(1, 'dnase')
    reach(32, 0, 'ties', 300)
    reach(32, 1, 'dnase', 700)
    reach(4096, 4095, 'dnase', 100)                # scan-tile seams: 4095, 4096, 4097 (mod 4096)
    add(1, 'dnase')
    add(1, 'ties')
    reach(4096, 4096 - 2048, 'ties', 100)          # a log-factorial tile seam (2048)
    reach(4096, 1, 'dnase', 2000)
    for wsize, wshift in EDGE_GEOMS:               # round-1 (constraint none) or tail windows at the class edges
        for c in CLASS_EDGES:
            if c - 1 <= wshift:
                add(wshift + c - 1, 'dnase')       # two windows, the tail one of c candidates
            elif c <= wsize + 1:
                add(c - 1, 'ties')                 # one window of c candidates
    add(12000, 'dnase')                            # several CTA-class windows at 2500 / 1250
    for k in (1, 2, 3):                            # tiny contigs in the middle
        add(k, 'ties')
    add(3000, 'dnase')
    add(2500, 'zero')                              # all-zero next to dense
    add(3000, 'dnase')
    add(1700, 'const')                             # constant next to dense
    add(2600, 'dense')
    add(6000, 'deep')                              # window counts above 2^20: the tables grow inside the round
    add(900, 'first')                              # the only count >= 2 at the first position
    add(900, 'last')                               # ... at the last
    for k in range(24):                            # many short contigs (more than 64 in all)
        add(5 + 17 * k, 'ties' if k % 3 == 0 else 'dnase')
    add(3000, 'dnase')
    add(1, 'dnase')                                # tiny contigs at the end; the last one has no log-factorial term
    add(2, 'dnase')
    add(3, 'ones')
    return np.array(bounds, dtype=np.int64), kinds


def _contig(kind, n, seed):
    rs = np.random.RandomState(seed)
    if kind == 'dnase':
        return synth.dnase_like(n, seed, hotspot_share=0.4)
    if kind == 'ties':                             # 0/1 only: exact ties, no log-factorial term
        return (rs.random_sample(n) < 0.35).astype(np.int64)
    if kind == 'zero':
        return np.zeros(n, dtype=np.int64)
    if kind == 'const':
        return np.full(n, 7, dtype=np.int64)
    if kind == 'dense':
        return synth.piecewise_poisson(n, seed)
    if kind == 'deep':                             # ~1 500 per position: 1 000 positions hold 1.5 * 10^6 counts
        return (np.repeat(rs.randint(800, 2200, n // 500 + 1), 500)[:n] + rs.poisson(30, n)).astype(np.int64)
    if kind == 'ones':
        return np.array([0, 1, 1][:n], dtype=np.int64)
    c = (rs.random_sample(n) < 0.3).astype(np.int64)
    c[0 if kind == 'first' else n - 1] = 5
    return c


def make_batch(seed=0):
    offsets, kinds = _layout()
    parts = [_contig(k, int(b - a), seed * 1000 + i) for i, (k, a, b) in enumerate(zip(kinds, offsets[:-1], offsets[1:]))]
    return np.concatenate(parts), offsets


def _parts(counts, offsets):
    return [counts[a:b] for a, b in zip(offsets[:-1].tolist(), offsets[1:].tolist())]


def _local(cands, offsets, c):
    a, b = offsets[c], offsets[c + 1]
    return cands[(cands >= a) & (cands <= b)] - a


def batch_round(oracles, offsets, cands, wsize, wshift, constraint):
    """The expected batch state after one round: every contig's oracle round on its own slice of the candidates, shifted
    by the contig's offset, united; cells summed over the contigs.  -> (candidates, cells)"""
    out, cells = [], 0
    for c, fo in enumerate(oracles):
        new, n_cells = fo.round(_local(cands, offsets, c), wsize, wshift, constraint)
        out.append(new + offsets[c])
        cells += n_cells
    return np.unique(np.concatenate(out)), cells


def _explicit(offsets, share, seed):
    """share of the positions of every contig, plus every contig boundary"""
    rs = np.random.RandomState(seed)
    n = int(offsets[-1])
    keep = rs.random_sample(n + 1) < share
    keep[offsets] = True
    return np.flatnonzero(keep).astype(np.int64)


def window_table(cands, offsets, wsize, wshift):
    """build_window_table (api.cu) on the host: [(first index, stop index, contig)] per window, in window-number order"""
    ranks = np.searchsorted(cands, offsets)
    out = []
    for c in range(len(offsets) - 1):
        b0, mc = int(ranks[c]), int(ranks[c + 1] - ranks[c] + 1)
        for st in range(0, mc - 1, wshift):
            out.append((b0 + st, b0 + min(st + wsize + 1, mc), c))
    return out


# ---- CPU: the batch oracle against the object-faithful reference round -------------------------------------------------
@pytest.mark.parametrize('wsize,wshift', [(40, 20), (7, 3), (2, 5), (1, 4)])
@pytest.mark.parametrize('constraint', CONSTRAINTS)
def test_batch_round_helper_vs_reference_round(wsize, wshift, constraint):
    """batch_round == po.sliding_window_round contig by contig; with shift > size both ends of every contig survive"""
    rs = np.random.RandomState(wsize * 10 + wshift)
    lens = [1, 2, 3, 90, 1, 57, 120, 2, 64, 3]
    parts = [synth.dnase_like(n, 50 + k, hotspot_share=0.5) if k % 2 else (rs.random_sample(n) < 0.4).astype(np.int64)
             for k, n in enumerate(lens)]
    parts[5][:] = 0
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    tables = po.Tables(1, 1.0)
    oracles = [c_oracle.FlatOracle(p, 1, 1.0) for p in parts]
    for cands in [np.arange(offsets[-1] + 1), _explicit(offsets, 0.6, 3)]:
        got, cells = batch_round(oracles, offsets, cands, wsize, wshift, constraint)
        want = np.unique(np.concatenate([
            po.sliding_window_round(p, _local(cands, offsets, c), tables, wsize, wshift, constraint) + offsets[c]
            for c, p in enumerate(parts)]))
        assert np.array_equal(got, want)
        assert cells >= 0
        assert np.all(np.isin(offsets, got))
        if wshift > wsize:                        # some contig's last candidate lies in no window
            assert any(len(_local(cands, offsets, c)) - 1 not in
                       [i for st, en, _ in window_table(_local(cands, offsets, c), offsets[c:c + 2] - offsets[c], wsize, wshift)
                        for i in range(st, en)] for c in range(len(parts)))


def test_batch_layout():
    """the batch has the seams, sizes and contig kinds the GPU tests rely on"""
    counts, offsets = make_batch()
    lens = np.diff(offsets)
    n_contigs = len(lens)
    assert n_contigs > 64
    for mod, rems in [(32, (31, 0, 1)), (4096, (4095, 0, 1)), (2048, (0,))]:
        for r in rems:
            assert np.any(offsets[1:-1] % mod == r), (mod, r)
    for where in (lens[:3], lens[n_contigs // 2 - 20:n_contigs // 2 + 20], lens[-3:]):
        assert {1, 2, 3} <= set(where.tolist())
    for wsize, wshift in EDGE_GEOMS:              # round 1, constraint none: every position is a candidate
        sizes = set(en - st for st, en, _ in window_table(np.arange(offsets[-1] + 1), offsets, wsize, wshift))
        want = [c for c in CLASS_EDGES if c - 1 <= wshift or c <= wsize + 1]
        assert set(want) <= sizes, (wsize, wshift)
    big = window_table(np.arange(offsets[-1] + 1), offsets, 2500, 1250)
    assert max(np.bincount([c for st, en, c in big if en - st > 512])) >= 5
    parts = _parts(counts, offsets)
    assert any(not p.any() for p in parts) and any(len(p) > 100 and np.all(p == p[0]) and p[0] > 0 for p in parts)
    assert max(int(np.sum(p[:1000])) for p in parts) > 1 << 20
    # (2, 5): the batch's last position lies in no window, so only the forced boundary keeps it
    last = window_table(np.arange(offsets[-1] + 1), offsets, 2, 5)[-1]
    assert last[1] - 1 < offsets[-1]
    assert not np.any(parts[-1] >= 2)                  # the last contig has no log-factorial term


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def eng():
    return _native.engine()


@pytest.fixture(scope='module')
def batch():
    return make_batch()


_ORACLES = {}


def _oracles(counts, offsets, ab, spec=None):
    key = (ab, spec, id(counts))
    if key not in _ORACLES:
        if spec is None:
            _ORACLES[key] = [c_oracle.FlatOracle(p, ab[0], ab[1], threads=THREADS) for p in _parts(counts, offsets)]
        else:
            _ORACLES[key] = [ro.FlatOracleReg(p, ab[0], ab[1], spec, threads=THREADS) for p in _parts(counts, offsets)]
    return _ORACLES[key]


def _rounds_vs_oracle(eng, oracles, offsets, cands, wsize, wshift, constraint, what, max_rounds=64):
    """device rounds from the loaded batch and its current candidates, each against batch_round, until the fixed point"""
    for r in range(max_rounds):
        want, want_cells = batch_round(oracles, offsets, cands, wsize, wshift, constraint)
        n_in, n_out, cells = eng.round(wsize, wshift, constraint)
        got = eng.candidates()
        assert n_in == len(cands) and n_out == len(want), (what, r, n_in, n_out, len(cands), len(want))
        if not np.array_equal(got, want):
            diff = np.setxor1d(got, want)[:10]
            raise AssertionError('%s round %d: candidates differ at %s (contigs %s)'
                                 % (what, r, diff.tolist(), (np.searchsorted(offsets, diff, 'right') - 1).tolist()))
        assert cells == want_cells, (what, r, cells, want_cells)
        if len(want) == len(cands):
            return r + 1
        cands = want
    raise AssertionError('%s: no fixed point after %d rounds' % (what, max_rounds))


AB = [(1, 1.0), (2.5, 0.3), (0.0009, 1.0)]      # 0.0009 < 2^-10: the far-column bound is off


@pytest.mark.gpu
@pytest.mark.parametrize('ab', AB)
@pytest.mark.parametrize('wsize,wshift', EDGE_GEOMS + [(300, 150), (1, 1), (2, 5), (200, 400)])
def test_rounds_from_all_positions(eng, batch, wsize, wshift, ab):
    """every round until the fixed point, all three constraints: n_in / n_out, the candidates and the cells"""
    counts, offsets = batch
    oracles = _oracles(counts, offsets, ab)
    for constraint in CONSTRAINTS:
        eng.use_scorer(ScorerFactory(*ab))
        eng.load(counts, offsets=offsets)
        eng.set_candidates(None)
        assert eng.info() == (len(counts), int(counts.sum()), len(offsets) - 1)
        _rounds_vs_oracle(eng, oracles, offsets, np.arange(len(counts) + 1), wsize, wshift, constraint,
                          (wsize, wshift, ab, constraint))


SWITCHES = [(1, 1), (1, 0), (0, 0)]             # (window_prune, window_phases)


def _with_switches(eng, prune, phases, speculate):
    eng.set_tuning('window_prune', prune)
    eng.set_tuning('window_phases', phases)
    eng.set_tuning('window_speculate', speculate)


def _reset_switches(eng):
    _with_switches(eng, 1, 1, 1)


@pytest.mark.gpu
@pytest.mark.parametrize('wsize,wshift', [(2500, 1250), (1000, 333)])
def test_explicit_lists_across_contig_boundaries(eng, batch, wsize, wshift):
    """per-contig explicit lists (70 %, every boundary): the pruned, two-phase rounds equal the oracle with every switch
    setting; with pruning and phases on cells are skipped, with both off none are"""
    counts, offsets = batch
    oracles = _oracles(counts, offsets, (1, 1.0))
    cands0 = _explicit(offsets, 0.7, wsize)
    want, cands = [], cands0
    for r in range(3):
        cands, cells = batch_round(oracles, offsets, cands, wsize, wshift, 'none')
        want.append((cands, cells))
    try:
        for prune, phases in SWITCHES:
            for speculate in (1, 0):
                _with_switches(eng, prune, phases, speculate)
                eng.use_scorer(ScorerFactory(1, 1.0))
                eng.load(counts, offsets=offsets)
                eng.set_candidates(cands0)
                skipped = 0
                for r in range(3):
                    eng.round(wsize, wshift, 'none')
                    got = eng.candidates()
                    cells, sk = eng.round_stats()
                    assert np.array_equal(got, want[r][0]), (wsize, prune, phases, speculate, r)
                    assert cells == want[r][1] and 0 <= sk <= cells
                    skipped += sk
                if (prune, phases) == (1, 1):
                    assert skipped > 0, (wsize, speculate)
                if (prune, phases) == (0, 0):
                    assert skipped == 0, (wsize, speculate)
    finally:
        _reset_switches(eng)


def _blocks(n_blocks, seed):
    """constant blocks of 3..9 positions at alternating low and high levels: the oracle's fixed point (constraint none)
    is the block boundaries, and a window over them keeps every one"""
    rs = np.random.RandomState(seed)
    vals = np.where(np.arange(n_blocks) % 2 == 0, rs.randint(0, 3, n_blocks), rs.randint(40, 80, n_blocks))
    return np.repeat(vals, rs.randint(3, 10, n_blocks)).astype(np.int64)


def cross_contig_layout(wsize, wshift):
    """A batch in which a phase-2 CTA-class window (C0, first window of contig C) has its phase-1 neighbour `lo` in an
    earlier contig A (A's last window) and `hi` in C, with stride - 2 one-window contigs between A and C (none at stride
    2).  The two neighbours together do not cover C0 (`lo` ends before `hi` starts): only that keeps the kernel from
    taking the covered-window fast path.  -> (counts, offsets, fixed-point candidates, (lo, C0, hi) window numbers)"""
    stride = wsize // wshift
    m_a = wshift + 513 if wshift >= 512 else None       # A's last window: more than 512 candidates
    assert m_a is not None
    a = _blocks(m_a - 1, 1)
    c = _blocks(wshift + 700, 2)
    tiny = [np.array([3, 0], dtype=np.int64)] * (stride - 2)
    # one-window contigs in front so that A's last window number is a multiple of the stride
    n_a = len(range(0, m_a - 1, wshift))
    lead = (-(n_a - 1)) % stride
    parts = [np.array([1], dtype=np.int64)] * lead + [a] + tiny + [c]
    offsets = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.int64)
    fixed = [c_oracle.FlatOracle(p, 1, 1.0).rounds(wsize, wshift, 'none')[0] + o for p, o in zip(parts, offsets)]
    cands = np.unique(np.concatenate(fixed))
    win = window_table(cands, offsets, wsize, wshift)
    lo = lead + n_a - 1
    w, hi = lo + stride - 1, lo + stride
    return np.concatenate(parts), offsets, cands, (lo, w, hi), win


@pytest.mark.parametrize('wsize,wshift', [(2500, 1250), (2048, 512)])
def test_cross_contig_layout(wsize, wshift):
    """(CPU) the layout really puts the fast-path decision on the coverage test: lo in contig A, C0 and hi in contig C,
    all three CTA-class, lo and hi keep every candidate (oracle DP over the window), lo ends before hi starts"""
    counts, offsets, cands, (lo, w, hi), win = cross_contig_layout(wsize, wshift)
    stride = wsize // wshift
    assert lo % stride == 0 and w % stride != 0 and hi % stride == 0
    (s1, e1, ca), (s0, e0, cw), (s2, e2, ch) = win[lo], win[w], win[hi]
    assert ca < cw == ch and cw - ca == stride - 1
    assert min(e1 - s1, e0 - s0, e2 - s2) > 512
    assert s1 <= s0 and e2 >= e0 and e1 < s2
    fo = c_oracle.FlatOracle(counts, 1, 1.0)
    for st, en, _ in (win[lo], win[hi]):
        assert len(fo.square_split(cands[st:en])[1]) == en - st          # keeps every candidate
    assert len(fo.square_split(cands[s0:e0])[1]) > 2                     # C0 keeps candidates only it covers


@pytest.mark.gpu
@pytest.mark.parametrize('wsize,wshift', [(2500, 1250), (2048, 512)])
def test_phase2_fast_path_across_contigs(eng, wsize, wshift):
    """a round from the oracle's fixed point (constraint none) in the layout above, with every switch setting"""
    counts, offsets, cands, _, _ = cross_contig_layout(wsize, wshift)
    oracles = [c_oracle.FlatOracle(p, 1, 1.0) for p in _parts(counts, offsets)]
    want, want_cells = batch_round(oracles, offsets, cands, wsize, wshift, 'none')
    assert np.array_equal(want, cands)
    try:
        for prune, phases in SWITCHES:
            for speculate in (1, 0):
                _with_switches(eng, prune, phases, speculate)
                eng.use_scorer(ScorerFactory(1, 1.0))
                eng.load(counts, offsets=offsets)
                eng.set_candidates(cands)
                _, _, cells = eng.round(wsize, wshift, 'none')
                assert np.array_equal(eng.candidates(), want), (prune, phases, speculate)
                assert cells == want_cells
    finally:
        _reset_switches(eng)


REG_CASES = [(2.0, 5.0, 'revlog'), (-1.5, 3.0, 'revlog'), (3.0, 0, 'none')]


def _spec(num, length, fn):
    return (length, ro.FUNCTIONS[fn], num, _identity)


@pytest.mark.gpu
@pytest.mark.parametrize('case', REG_CASES)
@pytest.mark.parametrize('wsize,wshift', [(513, 256), (2500, 1250), (2, 5)])
def test_regularised_batch_rounds(eng, batch, wsize, wshift, case):
    """K8 over the batch: rounds from all positions to the fixed point and two rounds from an explicit list"""
    counts, offsets = batch
    oracles = _oracles(counts, offsets, (1, 1.0), _spec(*case))
    for constraint in ('none', 'constants'):
        eng.use_scorer(ScorerFactory(1, 1.0), _spec(*case))
        eng.load(counts, offsets=offsets)
        eng.set_candidates(None)
        _rounds_vs_oracle(eng, oracles, offsets, np.arange(len(counts) + 1), wsize, wshift, constraint,
                          (wsize, case, constraint))
    cands = _explicit(offsets, 0.7, 5)
    eng.use_scorer(ScorerFactory(1, 1.0), _spec(*case))
    eng.load(counts, offsets=offsets)
    eng.set_candidates(cands)
    for r in range(2):
        want, want_cells = batch_round(oracles, offsets, cands, wsize, wshift, 'none')
        _, _, cells = eng.round(wsize, wshift, 'none')
        assert np.array_equal(eng.candidates(), want) and cells == want_cells, (wsize, case, r)
        cands = want


@pytest.mark.gpu
@pytest.mark.parametrize('ab', [(1, 1.0), (2.5, 0.3)])
def test_segment_outputs_and_logfac_sums(eng, batch, ab):
    """after the rounds: scores, counts, means per contig against po.Scorer; the LMM column bit for bit (logfac_exact 1)
    and to 1e-9 (0); the sequential total is the last contig's; the prefetch route gives the same arrays"""
    counts, offsets = batch
    parts = _parts(counts, offsets)
    tables = po.Tables(po.normalise_alpha(ab[0]), ab[1])
    oracles = _oracles(counts, offsets, ab)
    want = np.unique(np.concatenate([fo.rounds(2500, 1250, 'constants')[0] + o for fo, o in zip(oracles, offsets)]))
    scorers = [po.Scorer(p, _local(want, offsets, c), tables) for c, p in enumerate(parts)]
    w_scores = np.concatenate([s.scores() for s in scorers])
    w_counts = np.concatenate([np.diff(s.cumsum) for s in scorers])
    w_means = np.concatenate([s.mean_counts() for s in scorers])
    w_lmm = np.concatenate([s.log_marginal_likelyhoods() for s in scorers])
    w_total = scorers[-1].total_sum_logfac()
    assert w_total == 0.0 and any(s.total_sum_logfac() > 0 for s in scorers)
    try:
        for prefetch in (False, True):
            for exact in (1, 0):
                eng.set_tuning('logfac_exact', exact)
                eng.use_scorer(ScorerFactory(*ab))
                eng.load(counts, offsets=offsets)
                if prefetch:
                    eng.logfac_prefetch()                 # the sums run beside the rounds (process_bedgraph's route)
                eng.set_candidates(None)
                eng.rounds(2500, 1250, 'constants')
                assert np.array_equal(eng.candidates(), want)
                s, c, mu, _ = eng.segment_scores(scores=True, counts=True, means=True)
                assert np.array_equal(s, w_scores) and np.array_equal(c, w_counts) and np.array_equal(mu, w_means)
                lmm, total = eng.segment_lmm()
                if exact:
                    assert np.array_equal(lmm, w_lmm), prefetch
                    assert total == w_total, (prefetch, total)
                else:
                    # one scan over the whole batch: a segment's term is a difference of prefix sums as large as the
                    # batch's total, so the rounding is relative to that (still far below one term, >= log 2)
                    batch_total = sum(s.total_sum_logfac() for s in scorers)
                    assert np.allclose(lmm, w_lmm, rtol=1e-9, atol=1e-11 * batch_total), prefetch
                    assert abs(total - batch_total) <= 1e-9 * batch_total
    finally:
        eng.set_tuning('logfac_exact', 1)


def _rle(parts):
    """run-length form of a batch with every run ending at or before its contig's end (the product's route)"""
    starts, values, pos = [0], [], 0
    for p in parts:
        change = np.flatnonzero(p[1:] != p[:-1]) + 1
        s = np.concatenate([[0], change])
        e = np.concatenate([change, [len(p)]])
        starts.extend((e + pos).tolist())
        values.extend(p[s].tolist())
        pos += len(p)
    return np.array(starts, dtype=np.int64), np.array(values, dtype=np.int64)


def _load_state(eng, wsize=512, wshift=256):
    cum = eng.cumsum_at_candidates()
    eng.round(wsize, wshift, 'constants')
    return eng.info(), cum, eng.candidates().copy()


@pytest.mark.gpu
def test_load_paths_with_offsets(eng, batch):
    """load, load_rle and load_device with offsets: info, the prefix sums at every position and round-1 candidates"""
    import torch
    counts, offsets = batch
    oracles = _oracles(counts, offsets, (1, 1.0))
    want_cum = np.concatenate([[0], np.cumsum(counts)])
    want_r1, _ = batch_round(oracles, offsets, np.arange(len(counts) + 1), 512, 256, 'constants')
    eng.use_scorer(ScorerFactory(1, 1.0))
    starts, values = _rle(_parts(counts, offsets))
    assert np.any(np.diff(starts) > 8) and np.any(starts % 8 != 0)
    dev = torch.from_numpy(counts).cuda()
    for how in ('load', 'rle', 'device'):
        eng.invalidate()
        if how == 'load':
            eng.load(counts, offsets=offsets)
        elif how == 'rle':
            eng.load_rle(starts, values, offsets=offsets)
        else:
            eng.load_device(dev.data_ptr(), len(counts), owner=dev, offsets=offsets)
        eng.set_candidates(None)
        info, cum, r1 = _load_state(eng)
        assert info == (len(counts), int(counts.sum()), len(offsets) - 1), how
        assert np.array_equal(cum, want_cum), how
        assert np.array_equal(r1, want_r1), how


@pytest.mark.gpu
def test_narrowed_upload_of_a_batch(eng):
    """a batch past 2^24 positions goes up narrowed (upload_narrow 1, and 3 to mix narrowed and plain slices) with a
    boundary on a 2^19-element slice seam: the same state as the plain upload (0)"""
    slice_ = 1 << 19
    lens = [3 * slice_, 1, 2, 5 * slice_ - 3 - 1000, 1000, (1 << 24) + 5000 - 8 * slice_]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    assert np.any(offsets[1:-1] % slice_ == 0) and offsets[-1] >= 1 << 24
    counts = np.concatenate([synth.dnase_like(n, 90 + k, hotspot_share=0.3) for k, n in enumerate(lens)])
    counts[offsets[3]:offsets[3] + 200] = 70000                # a slice that cannot be narrowed to 3 bits
    eng.use_scorer(ScorerFactory(1, 1.0))
    states = {}
    try:
        for mode in (0, 1, 3):
            eng.set_tuning('upload_narrow', mode)
            eng.invalidate()
            eng.load(counts, offsets=offsets)
            eng.set_candidates(None)
            states[mode] = _load_state(eng, 2500, 1250)
            if mode:
                assert eng.upload_stats() < counts.nbytes, mode
    finally:
        eng.set_tuning('upload_narrow', 1)
    info, cum, r1 = states[0]
    assert info == (len(counts), int(counts.sum()), len(lens))
    assert np.array_equal(cum, np.concatenate([[0], np.cumsum(counts)]))
    for mode in (1, 3):
        assert states[mode][0] == info and np.array_equal(states[mode][1], cum) and np.array_equal(states[mode][2], r1)


@pytest.mark.gpu
def test_full_batch_of_contigs_through_the_text_route():
    """20 001 contigs: one launch holds BATCH_CONTIGS, the next one contig; bedgraph+length+LMM byte for byte"""
    from pasio_b200 import process_bedgraph as pb
    from pasio_b200.process_bedgraph import split_bedgraph_stream
    rs = np.random.RandomState(21)
    n_contigs = pb.BATCH_CONTIGS + 1
    lens = rs.randint(1, 401, n_contigs)
    lens[rs.choice(n_contigs, 6, replace=False)] = rs.randint(3000, 20001, 6)
    assert lens.sum() < pb.BATCH_NT and lens.max() < pb.BATCH_ALONE
    lines = []
    for c, n in enumerate(lens.tolist()):
        counts = synth.dnase_like(n, 9000 + c, hotspot_share=0.4) if c % 4 else (rs.random_sample(n) < 0.3).astype(np.int64)
        lines.extend(synth.to_bedgraph_lines('tx%05d' % c, counts, chrom_start=int(rs.randint(0, 100))))
    text = ''.join(lines)
    sizes = [len(b) for b in pb._batches(pb.contig_runs(text.encode()), {'final': 'nop'})]
    assert sizes == [pb.BATCH_CONTIGS, 1]
    out = io.StringIO()
    split_bedgraph_stream(io.StringIO(text), out, configure_splitter(), output_mode='bedgraph+length+LMM')
    want = po.split_bedgraph_text(text, po.Tables(1, 1.0), output_mode='bedgraph+length+LMM', threads=THREADS)
    assert out.getvalue() == want
