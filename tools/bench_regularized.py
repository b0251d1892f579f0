"""Regularised segmentation (--split-number-regularization / --length-regularization) on the bench contig.

    python tools/bench_regularized.py [--steps K] [--warmup W] [--n NT] [--prefix NT] [--parity NT]

Prints one JSON line per setting (split-number only, revlog length only, both) for the chr1-sized bench contig
(synth.dnase_like(248956422, seed=1000), resident in HBM): ms/step from CUDA events for the rounds plus the segment
scores, rounds and candidates per round, DP cells (every cell is evaluated) and cells/s, and the share of the FP64 pipe
(4 FP64 operations per cell plus one per active penalty term, over pasio_fp64_peak), with the card name and power limit
read in the same run.  Then:
  - `before`: the object route (every window through the objects and the exact regularised DP, forced with a
    SquareSplitter subclass) and the fused route on a prefix of the same contig, alternating;
  - `parity`: the fused rounds against the flat C oracle (tests/reg_oracle.c) on a prefix; exit 1 on a mismatch;
  - `batched`: transcript-like contigs through split_bedgraph_stream, batches of short contigs in effect.
Writes nothing into the tree.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import numpy as np    # noqa: E402

# (name, split-number multiplier, length multiplier, length function): multipliers chosen so that every setting changes
# the chr1 segmentation visibly against the unregularised run (segments in the JSON lines)
SETTINGS = [('split_number', 2.0, 0, 'none'), ('length_revlog', 0, 5.0, 'revlog'), ('both', 2.0, 5.0, 'revlog')]
WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT = 2500, 1250, 'constants'


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=30).stdout.decode().strip()
        name, limit = out.splitlines()[0].split(', ')
        return name, limit
    except Exception:      # noqa: BLE001
        import torch
        return torch.cuda.get_device_name(0), 'unknown'


def spec_of(num, length, fn):
    from pasio_b200.splitters.square_splitter import _identity, _revlog
    return (length, _revlog if fn == 'revlog' else _identity, num, _identity)


def kwargs_of(num, length, fn):
    return dict(split_number_regularization=num, length_regularization=length,
                length_regularization_function=fn if length else 'none')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--n', type=int, default=248956422)
    ap.add_argument('--prefix', type=int, default=300000, help='length of the before/after prefix')
    ap.add_argument('--parity', type=int, default=2000000, help='length of the parity prefix')
    args = ap.parse_args()

    import torch
    from pasio_b200 import _native, configure_splitter, synth
    from pasio_b200.log_marginal_likelyhood import ScorerFactory
    from pasio_b200.segmentation import segments_with_scores
    from pasio_b200.splitters.square_splitter import SquareSplitter
    import reg_oracle as ro

    name, limit = card()
    counts = synth.dnase_like(args.n, seed=1000)
    eng = _native.engine()
    resident = torch.from_numpy(counts).to('cuda:0')
    stream = torch.cuda.ExternalStream(eng.stream_handle(), device='cuda:0')
    peak = eng.fp64_peak()                      # FP64 instructions/s of this card, measured (pasio_fp64_peak)
    factory = ScorerFactory(1, 1)

    def step(spec):
        eng.use_scorer(factory, spec)
        eng.load_device(resident.data_ptr(), len(counts), owner=resident)
        eng.set_candidates(None)
        sizes, final, cells = eng.rounds(WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
        eng.use_scorer(factory)
        eng.segment_scores(scores=True, means=True)
        return sizes, final, cells, float(eng.segment_scores_sum())

    plain = None
    for label, num, length, fn in [('none', 0, 0, 'none')] + SETTINGS:
        spec = None if label == 'none' else spec_of(num, length, fn)
        for _ in range(args.warmup):
            step(spec)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(args.steps):
            sizes, final, cells, score = step(spec)
        ev1.record(stream)
        ev1.synchronize()
        ms = ev0.elapsed_time(ev1) / args.steps
        terms = (num != 0) + (length != 0)
        fp64 = cells * (4 + terms) / (ms * 1e-3)
        row = dict(setting=label, split_number_regularization=num, length_regularization=length,
                   length_regularization_function=fn, n=len(counts), window_size=WINDOW_SIZE, window_shift=WINDOW_SHIFT,
                   ms_per_step=round(ms, 3), rounds=len(sizes), candidates_per_round=sizes, segments=final - 1,
                   score=score, cells=cells, cells_per_s=cells / (ms * 1e-3),
                   fp64_pipe_share=fp64 / peak if label != 'none' else None, fp64_peak_instr_per_s=peak,
                   gpu=name, power_limit=limit)
        if label == 'none':
            plain = final
        else:
            row['segments_unregularised'] = plain - 1
        print(json.dumps(row), flush=True)

    # before / after on a prefix: the object route (per-window objects and K6) against the fused route, alternating
    class ObjectRoute(SquareSplitter):
        pass
    prefix = counts[:args.prefix]
    num, length, fn = SETTINGS[2][1:]
    times = {'object': [], 'fused': []}
    results = {}
    for _ in range(2):
        for route in ('object', 'fused'):
            sp = configure_splitter(**kwargs_of(num, length, fn))
            if route == 'object':
                sp.reducers[0].base_reducer.base_reducer.reducers[1].__class__ = ObjectRoute
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            segs = list(segments_with_scores(prefix, sp))
            torch.cuda.synchronize()
            times[route].append(time.perf_counter() - t0)
            results[route] = np.array([s.start for s in segs] + [segs[-1].stop])
    same = np.array_equal(results['object'], results['fused'])
    print(json.dumps(dict(setting='before_after_prefix', n=len(prefix), object_route_s=times['object'],
                          fused_route_s=times['fused'], speedup=min(times['object']) / min(times['fused']),
                          same_splits=bool(same), gpu=name, power_limit=limit)), flush=True)

    # parity on a prefix: fused rounds == flat C oracle
    ok = same
    part = counts[:args.parity]
    for label, num, length, fn in SETTINGS:
        spec = spec_of(num, length, fn)
        eng.use_scorer(factory, spec)
        eng.load(part)
        eng.set_candidates(None)
        sizes, final, _ = eng.rounds(WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
        got = eng.candidates()
        want = ro.pipeline(part, spec, threads=max(1, min(32, os.cpu_count() or 1)))
        match = bool(np.array_equal(got, want['splits']) and sizes == list(want['sizes'][:len(sizes)]))
        ok = ok and match
        print(json.dumps(dict(setting='parity', penalties=label, n=len(part), parity=match, segments=len(got) - 1)),
              flush=True)
    eng.use_scorer(factory)

    # batched transcript-like contigs through the stream API
    from pasio_b200.process_bedgraph import split_bedgraph_stream
    lines = []
    for c, n in enumerate(synth.transcript_lengths(20000, seed=3)):
        lines.extend(synth.to_bedgraph_lines('tx%05d' % c, synth.dnase_like(int(n), seed=5000 + c, hotspot_share=0.3)))
    text = ''.join(lines)
    for devices_label, rounds in (('regularised', True), ('unregularised', False)):
        sp = configure_splitter(**kwargs_of(*SETTINGS[2][1:])) if rounds else configure_splitter()
        out = io.StringIO()
        split_bedgraph_stream(io.StringIO(text), io.StringIO(), sp)            # warm-up
        t0 = time.perf_counter()
        split_bedgraph_stream(io.StringIO(text), out, sp)
        s = time.perf_counter() - t0
        print(json.dumps(dict(setting='batched_transcripts', splitter=devices_label, contigs=20000,
                              nt=int(sum(synth.transcript_lengths(20000, seed=3))), seconds=round(s, 3),
                              segments=out.getvalue().count('\n'), gpu=name, power_limit=limit)), flush=True)
    return 0 if ok else 1


if __name__ == '__main__':
    sys.exit(main())
