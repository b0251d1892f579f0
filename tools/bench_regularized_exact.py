"""The regularised whole-list DP: one CTA (K6, csrc/regularized_dp.cu) against every SM (K9, csrc/regularized_exact.cu).

    python tools/bench_regularized_exact.py [--reps R] [--sizes N,N,...] [--k6-once-ms MS] [--no-e2e]

Prints JSON lines.  The first names the card, its power limit and top SM clock (nvidia-smi, read in the same run).  Then:
  - `kernel`: per size N and penalty setting, K6 and K9 forced through the reg_exact tuning key, alternating in one process
    after a warm-up call of each, a device synchronise around every call; ms of the device DP (the TF_EXACT_DP timing family:
    CUDA events around the kernel), N(N-1)/2 cells over that time, and whether P, prev and splits of the two kernels are
    equal in every repetition.  N = 100 001 is config 1's contig (synth.piecewise_poisson(100000, 0), all positions),
    N = 200 000 config 3's candidate list (synth.random_candidates(2000000, 200000, 1)); the other sizes are prefixes of
    config 1.  A K6 call slower than --k6-once-ms is not repeated.
  - `e2e`: segments_with_scores with configure_splitter(algorithm='exact') on configs 1 and 3's contigs cut to the same
    sizes, and with algorithm='slidingwindow' on a 10 Mb synth.dnase_like contig: seconds with the default dispatch and
    with reg_exact = 0 (always K6), and whether the segmentations are equal.
Writes nothing into the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np    # noqa: E402

# (name, split-number multiplier, length multiplier, length function)
SETTINGS = [('split_number', 2.0, 0, 'none'), ('length_revlog', 0, 5.0, 'revlog'), ('both_negative', -1.5, 3.0, 'revlog')]
SIZES = [257, 1025, 2501, 8193, 20001, 100001, 200000]


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=30, check=True).stdout.decode()
    name, limit, clock = [x.strip() for x in out.splitlines()[0].split(',')]
    return dict(gpu=name, power_limit=limit, max_sm_clock=clock)


def spec_of(num, length, fn):
    from pasio_b200.splitters.square_splitter import _identity, _revlog
    return (length, _revlog if fn == 'revlog' else _identity, num, _identity)


def kwargs_of(num, length, fn):
    return dict(split_number_regularization=num, length_regularization=length,
                length_regularization_function=fn if length else 'none')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--sizes', default=','.join(str(n) for n in SIZES))
    ap.add_argument('--k6-once-ms', type=float, default=10000.0)
    ap.add_argument('--no-e2e', action='store_true')
    args = ap.parse_args()

    from pasio_b200 import _native, configure_splitter, synth
    from pasio_b200.log_marginal_likelyhood import ScorerFactory
    from pasio_b200.segmentation import segments_with_scores
    from pasio_b200.splitters.square_splitter import penalty_tables

    info = card()
    print(json.dumps(info), flush=True)
    eng = _native.engine()
    config1 = synth.piecewise_poisson(100000, 0)
    config3 = synth.piecewise_poisson(2000000, 1)
    config3_cands = synth.random_candidates(2000000, 200000, 1)
    ok = True

    def data_for(n):
        if n == 200000:
            return config3, config3_cands
        return config1[:n - 1], None

    def call(counts, cands, spec, mode):
        eng.set_tuning('reg_exact', mode)
        eng.use_scorer(ScorerFactory(1, 1.0))
        eng.load(counts)
        eng.set_candidates(cands)
        m = len(counts) + 1 if cands is None else len(cands)
        tables = penalty_tables(spec, len(counts) + 1, m)
        eng.timing_reset(True)
        out = eng.square_split_regularized(*tables, want_arrays=True)
        ms = eng.timing()['exact_dp'][0]
        eng.timing_reset(False)
        return ms, out

    for n in [int(x) for x in args.sizes.split(',') if x]:
        counts, cands = data_for(n)
        for label, num, length, fn in SETTINGS:
            spec = spec_of(num, length, fn)
            times = {0: [], 2: []}
            first = {}
            same = True
            warm = {mode: call(counts, cands, spec, mode) for mode in (0, 2)}       # warm-up (and K6's first time)
            k6_once = warm[0][0] > args.k6_once_ms
            for rep in range(args.reps):
                for mode in (0, 2):
                    if mode == 0 and k6_once:
                        ms, out = warm[0]
                        if rep > 0:
                            continue
                    else:
                        ms, out = call(counts, cands, spec, mode)
                    times[mode].append(ms)
                    first.setdefault(mode, out)
                    ref = first[0] if 0 in first else warm[0][1]
                    same = same and out[0] == ref[0] and all(np.array_equal(x, y) for x, y in zip(out[1:], ref[1:]))
            ok = ok and same
            cells = n * (n - 1) // 2
            k6, k9 = min(times[0]), min(times[2])
            print(json.dumps(dict(setting='kernel', n=n, penalties=label, k6_ms=times[0], k9_ms=times[2],
                                  k6_cells_per_s=cells / (k6 * 1e-3), k9_cells_per_s=cells / (k9 * 1e-3),
                                  speedup=k6 / k9, equal_p_prev_splits=bool(same), k6_repeated=not k6_once, **info)),
                  flush=True)
    eng.set_tuning('reg_exact', 1)

    if not args.no_e2e:
        kw = kwargs_of(2.0, 5.0, 'revlog')
        runs = [(config1, 'exact'), (config3[:199999], 'exact'), (synth.dnase_like(10000000, 7), 'slidingwindow')]
        for counts, algorithm in runs:
            res = {}
            for mode in (1, 0):
                eng.set_tuning('reg_exact', mode)
                t0 = time.perf_counter()
                segs = list(segments_with_scores(counts, configure_splitter(algorithm=algorithm, **kw)))
                res[mode] = (time.perf_counter() - t0, np.array([s.start for s in segs] + [segs[-1].stop]))
            eng.set_tuning('reg_exact', 1)
            same = bool(np.array_equal(res[0][1], res[1][1]))
            ok = ok and same
            print(json.dumps(dict(setting='e2e', algorithm=algorithm, n=len(counts), penalties='split_number 2, revlog 5',
                                  default_s=round(res[1][0], 3), k6_only_s=round(res[0][0], 3),
                                  speedup=res[0][0] / res[1][0], segments=len(res[1][1]) - 1, same_segments=same,
                                  **info)), flush=True)
    return 0 if ok else 1


if __name__ == '__main__':
    sys.exit(main())
