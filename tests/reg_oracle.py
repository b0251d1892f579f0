"""Oracles of the regularised sliding-window pipeline -- TEST INFRASTRUCTURE ONLY.

The numpy half composes oracle/pasio_oracle.py's restatements the way the reference composes its objects when the
window's base splitter is a regularised SquareSplitter: per window the constraint filter, then
square_split_regularized (square_splitter.py:29-65) on the window as a contig of its own
(sliding_window_reducer.py:10-29), rounds until a fixed point (round_reducer.py:10-31), NopSplitter scoring
(default_splitters.py:65-66, segmentation.py:5-20).  The C half (tests/reg_oracle.c) is the flat restatement of the
same round, fast enough for Mb-scale checks; tests/test_regularized_plans.py checks the two against each other bit for
bit.  oracle/ itself is left as it is: its restatements pin the golden vectors.
"""
import ctypes
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import c_oracle, pasio_oracle as po          # noqa: E402
from pasio_b200.splitters.square_splitter import _identity, _revlog, penalty_tables   # noqa: E402

FUNCTIONS = {'none': _identity, 'revlog': _revlog}


def penalty_kwargs(num_mult=0, len_mult=0, len_fn='none'):
    """keyword arguments of po.square_split_regularized for the CLI's flags (split-number function: identity)"""
    return dict(len_mult=len_mult, len_fn=FUNCTIONS[len_fn], num_mult=num_mult, num_fn=_identity)


# ---- numpy, object-faithful -------------------------------------------------------------------------------------
def base_reduce(counts, cands, tables, constraint, **pen):
    """default_splitters.py:52-59 with a regularised SquareSplitter: filter, then split_with_normalizations"""
    if constraint == 'constants':
        cands = po.not_constant(counts, cands)
    elif constraint == 'zeros':
        cands = po.not_zero(counts, cands)
    elif constraint != 'none':
        raise ValueError(constraint)
    return po.square_split_regularized(counts, cands, tables, **pen)[1]


def sliding_window_round(counts, cands, tables, window_size, window_shift, constraint, **pen):
    keep = set([0, len(counts)])
    for st, en in po.window_ranges(len(cands), window_size, window_shift):
        win = cands[st:en]
        a, b = win[0], win[-1]
        keep.update((base_reduce(counts[a:b], win - a, tables, constraint, **pen) + a).tolist())
    return np.array(sorted(keep))


def round_reduce(counts, cands, tables, window_size, window_shift, constraint, num_rounds=None, **pen):
    rounds = max(1, len(counts) if num_rounds is None else num_rounds)
    sizes = [len(cands)]
    for _ in range(rounds):
        new = sliding_window_round(counts, cands, tables, window_size, window_shift, constraint, **pen)
        if np.array_equal(new, cands):
            return new, sizes
        cands = new
        sizes.append(len(cands))
    return cands, sizes


def default_pipeline(counts, tables, window_size=2500, window_shift=1250, constraint='constants', num_rounds=None, **pen):
    counts = np.asarray(counts)
    cands, sizes = round_reduce(counts, np.arange(len(counts) + 1), tables, window_size, window_shift, constraint,
                                num_rounds, **pen)
    score, splits = po.nop_split(counts, cands, tables)
    sc = po.Scorer(counts, splits, tables)
    return dict(score=score, splits=splits, mean_counts=sc.mean_counts(), lmm=sc.log_marginal_likelyhoods(),
                sum_logfac=sc.total_sum_logfac(), sizes=np.array(sizes))


# ---- C, flat ----------------------------------------------------------------------------------------------------
_lib = None


def lib():
    """tests/reg_oracle.c, compiled once per source version into the temporary directory"""
    global _lib
    if _lib is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'reg_oracle.c')
        tag = hashlib.sha1(open(src, 'rb').read()).hexdigest()[:12]
        so = os.path.join(tempfile.gettempdir(), 'pasio_reg_oracle_%s_%d.so' % (tag, os.getuid()))
        if not os.path.exists(so):
            tmp = so + '.%d' % os.getpid()
            flags = ['-O2', '-ffp-contract=off', '-fno-fast-math', '-fPIC', '-shared', '-Wall']
            if subprocess.call(['gcc'] + flags + ['-fopenmp', '-o', tmp, src], stderr=subprocess.DEVNULL) != 0:
                subprocess.check_call(['gcc'] + flags + ['-o', tmp, src])
            os.replace(tmp, so)
        _lib = ctypes.CDLL(so)
        i64, i64p = ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)
        f64, f64p, u8p = ctypes.c_double, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint8)
        _lib.dp_oracle_reg.restype = ctypes.c_int
        _lib.dp_oracle_reg.argtypes = [i64p, i64p, i64, f64p, i64, f64p, i64, ctypes.c_int, f64, f64,
                                       f64p, i64, f64, f64p, i64, f64p, i64p, i64p]
        _lib.round_oracle_reg.restype = ctypes.c_int
        _lib.round_oracle_reg.argtypes = [i64p, u8p, i64, i64p, i64, i64, i64, ctypes.c_int, f64p, i64, f64p, i64,
                                          ctypes.c_int, f64, f64, f64p, i64, f64, f64p, i64, u8p, i64p, ctypes.c_int]
    return _lib


def _p(a, ct):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ct))


class FlatOracleReg(c_oracle.FlatOracle):
    """c_oracle.FlatOracle with the penalties of a regularised window splitter; spec as
    square_splitter.penalty_spec: (length multiplier, length function, split-number multiplier, its function)."""

    MAX_WINDOW = 1 << 13

    def __init__(self, counts, alpha, beta, spec, threads=1):
        super(FlatOracleReg, self).__init__(counts, alpha, beta, threads=threads)
        self.spec = spec

    def square_split(self, cands):
        """The regularised DP over one whole candidate list (dp_oracle_reg); returns (score, splits, P, prev, ns)."""
        cands = np.ascontiguousarray(cands, dtype=np.int64)
        C = np.ascontiguousarray(self.Cg[cands])
        N = len(cands)
        span = int(cands[-1] - cands[0])
        a_int = int(self.alpha) if self.int_alpha else 0
        self._ensure_tables(span + 1, int(C[-1] - C[0]) + a_int + 1)
        lr, nr, refund = penalty_tables(self.spec, span + 1, N)
        P = np.empty(N)
        prev = np.empty(N, dtype=np.int64)
        ns = np.empty(N, dtype=np.int64)
        rc = lib().dp_oracle_reg(
            _p(C, ctypes.c_int64), _p(cands, ctypes.c_int64), N, _p(self.g, ctypes.c_double), len(self.g),
            _p(self.lg, ctypes.c_double), len(self.lg), int(self.int_alpha), float(self.alpha), self.pen,
            _p(nr, ctypes.c_double), 0 if nr is None else len(nr), refund, _p(lr, ctypes.c_double),
            0 if lr is None else len(lr), _p(P, ctypes.c_double), _p(prev, ctypes.c_int64), _p(ns, ctypes.c_int64))
        assert rc == 0, rc
        return P[-1], cands[po.backtrace(prev)], P, prev, ns

    def round(self, cands, window_size, window_shift, constraint):
        cands = np.ascontiguousarray(cands, dtype=np.int64)
        m = len(cands)
        span = cnt = 0
        for st, en in po.window_ranges(m, window_size, window_shift):
            a, b = cands[st], cands[en - 1]
            span = max(span, int(b - a))
            cnt = max(cnt, int(self.Cg[b] - self.Cg[a]))
        a_int = int(self.alpha) if self.int_alpha else 0
        self._ensure_tables(span + 1, cnt + a_int + 1)
        lr, nr, refund = penalty_tables(self.spec, span + 1, min(window_size + 1, self.MAX_WINDOW))
        keep = np.zeros(self.n + 1, dtype=np.uint8)
        cells = ctypes.c_int64(0)
        rc = lib().round_oracle_reg(
            _p(self.Cg, ctypes.c_int64), _p(self.cp, ctypes.c_uint8), self.n, _p(cands, ctypes.c_int64), m,
            window_size, window_shift, c_oracle.CONSTRAINTS[constraint], _p(self.g, ctypes.c_double), len(self.g),
            _p(self.lg, ctypes.c_double), len(self.lg), int(self.int_alpha), float(self.alpha), self.pen,
            _p(nr, ctypes.c_double), 0 if nr is None else len(nr), refund, _p(lr, ctypes.c_double),
            0 if lr is None else len(lr), _p(keep, ctypes.c_uint8), ctypes.byref(cells), self.threads)
        assert rc == 0, rc
        return np.flatnonzero(keep).astype(np.int64), cells.value


def pipeline(counts, spec, alpha=1, beta=1.0, window_size=2500, window_shift=1250, constraint='constants',
             num_rounds=None, threads=1):
    """default pipeline with the flat C rounds: dict(score, splits, mean_counts, lmm, sizes)"""
    fo = FlatOracleReg(counts, alpha, beta, spec, threads=threads)
    splits, sizes, cells = fo.rounds(window_size, window_shift, constraint, num_rounds)
    tables = po.Tables(po.normalise_alpha(alpha), beta)
    score, _ = po.nop_split(np.asarray(counts), splits, tables)
    sc = po.Scorer(counts, splits, tables)
    return dict(score=score, splits=splits, mean_counts=sc.mean_counts(), lmm=sc.log_marginal_likelyhoods(),
                sizes=sizes, cells=cells)


def split_bedgraph_text(text, spec, alpha=1, beta=1.0, window_size=2500, window_shift=1250, constraint='constants',
                        num_rounds=None, split_at_gaps=False, output_mode='bedgraph', threads=1):
    """po.split_bedgraph_text with the regularised rounds"""
    out = []
    for chrom, counts, chrom_start in po.parse_bedgraph_text(text, split_at_gaps):
        r = pipeline(counts, spec, alpha, beta, window_size, window_shift, constraint, num_rounds, threads)
        splits, means, lmm = r['splits'], r['mean_counts'], r['lmm']
        for k in range(len(splits) - 1):
            a, b = splits[k] + chrom_start, splits[k + 1] + chrom_start
            if output_mode == 'bedgraph':
                out.append('%s\t%d\t%d\t%f\n' % (chrom, a, b, means[k]))
            elif output_mode == 'bed':
                out.append('%s\t%d\t%d\n' % (chrom, a, b))
            else:
                out.append('%s\t%d\t%d\t%f\t%d\t%f\n' % (chrom, a, b, means[k], splits[k + 1] - splits[k], lmm[k]))
    return ''.join(out)
