"""`--algorithm exact` and `slidingwindow` on a config-5 sub-sample: short contigs batched (the default) against one contig
per launch (process_bedgraph.BATCH_NT = 0, the route before pasio_square_split_batch).

    python tools/bench_exact_batches.py [--transcripts N] [--reps R] [--seed S]

Prints JSON lines.  The first names the card, its power limit and top SM clock (nvidia-smi, read in the same run).  Then one
line per algorithm: seconds of split_bedgraph_stream over the same in-memory text (seeded synth.transcript_lengths, 1-50 kb,
DNase-like coverage), batched and alone alternating after a warm-up run of each, and whether the output bytes of every
run equal the first batched run's.  Writes nothing into the tree.
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

ALGORITHMS = {'exact': dict(algorithm='exact'),
              'slidingwindow': dict(algorithm='slidingwindow', window_size=2500, window_shift=1250)}


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=30, check=True).stdout.decode()
    name, limit, clock = [x.strip() for x in out.splitlines()[0].split(',')]
    return dict(gpu=name, power_limit=limit, max_sm_clock=clock)


def transcripts_text(n, seed):
    """-> (bedgraph text, total nt)"""
    from pasio_b200 import synth
    lines = []
    lens = synth.transcript_lengths(n, seed=seed)
    for c, length in enumerate(lens):
        lines.extend(synth.to_bedgraph_lines('tx%05d' % c, synth.dnase_like(int(length), seed=5000 + c, hotspot_share=0.3)))
    return ''.join(lines), int(lens.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--transcripts', type=int, default=2000)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--seed', type=int, default=5)
    args = ap.parse_args()
    print(json.dumps(card()), flush=True)
    from pasio_b200 import configure_splitter, _native
    from pasio_b200 import process_bedgraph as pb
    text, nt = transcripts_text(args.transcripts, args.seed)
    _native.engine()
    batch_nt = pb.BATCH_NT

    def run(splitter, batched):
        pb.BATCH_NT = batch_nt if batched else 0
        try:
            out = io.StringIO()
            t0 = time.perf_counter()
            pb.split_bedgraph_stream(io.StringIO(text), out, splitter)
            return time.perf_counter() - t0, out.getvalue()
        finally:
            pb.BATCH_NT = batch_nt

    for name, kw in ALGORITHMS.items():
        splitter = configure_splitter(**kw)
        _, ref = run(splitter, True)                       # warm-up of both routes (tables, modules)
        _, alone0 = run(splitter, False)
        times = {'batched': [], 'alone': []}
        equal = alone0 == ref
        for _ in range(args.reps):
            for batched in (True, False):
                secs, got = run(splitter, batched)
                times['batched' if batched else 'alone'].append(round(secs, 4))
                equal = equal and got == ref
        print(json.dumps(dict(algorithm=name, transcripts=args.transcripts, nt=nt,
                              seconds=times, best_speedup=round(min(times['alone']) / min(times['batched']), 3),
                              output_bytes=len(ref), outputs_equal=bool(equal))), flush=True)


if __name__ == '__main__':
    main()
