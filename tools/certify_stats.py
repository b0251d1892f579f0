"""Pass rate of the window DP's whole-window check (csrc/window_dp.cu, certify_window), on the CPU from the C oracle.

For a prefix of the bench contig (synth.dnase_like(nt, seed=1000)), every round of the default pipeline (constants,
2500 / 1250, alpha = beta = 1) until the fixed point.  From round 2 on, every window is put through
FlatOracle.square_split: a window passes when the first maximum of every row j is column j-1.  Per round: windows,
windows that pass, phase-1 windows (even window numbers) that pass, the median position of the first failing row as a
share of the window, and the median number of failing rows per failing window.

    python tools/certify_stats.py 10000000
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import c_oracle as co, pasio_oracle as po  # noqa: E402
from pasio_b200 import synth  # noqa: E402

WS, SH = 2500, 1250


def main(nt):
    counts = synth.dnase_like(nt, seed=1000)
    o = co.FlatOracle(counts, 1, 1.0, threads=max(1, min(32, os.cpu_count() or 1)))
    cands = np.arange(nt + 1, dtype=np.int64)
    print('# tools/certify_stats.py %d: synth.dnase_like(%d, seed=1000), constants, %d / %d, alpha = beta = 1' % (nt, nt, WS, SH))
    print('round | candidates in -> out | windows | pass | phase-1 windows that pass | first failing row (median share) '
          '| failing rows per failing window (median)')
    r = 0
    while True:
        r += 1
        new, _ = o.round(cands, WS, SH, 'constants')
        if r >= 2:
            wins = po.window_ranges(len(cands), WS, SH)
            keep, firsts, nbad = np.zeros(len(wins), bool), [], []
            for k, (st, en) in enumerate(wins):
                w = cands[st:en]                                   # the window's candidates after the constraint filter
                inner = w[1:-1]
                w = np.concatenate([w[:1], inner[counts[inner - 1] != counts[np.minimum(inner, nt - 1)]], w[-1:]])
                _, _, _, prev = o.square_split(w)
                bad = np.flatnonzero(prev[1:] != np.arange(len(w) - 1)) + 1
                keep[k] = not len(bad)
                if len(bad):
                    firsts.append(bad[0] / len(w))
                    nbad.append(len(bad))
            p1 = keep[0::2]
            print('%d | %d -> %d | %d | %d | %d / %d | %s | %s'
                  % (r, len(cands), len(new), len(wins), keep.sum(), p1.sum(), len(p1),
                     '%.2f' % np.median(firsts) if firsts else '-', '%g' % np.median(nbad) if nbad else '-'), flush=True)
        else:
            print('%d | %d -> %d | (all positions: not checked) | | | |' % (r, len(cands), len(new)), flush=True)
        if len(new) == len(cands):
            break
        cands = new


if __name__ == '__main__':
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000)
