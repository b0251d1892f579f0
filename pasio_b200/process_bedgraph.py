"""Bedgraph in, segments out (reference: /root/reference/src/pasio/process_bedgraph.py:9-92).

Same functions and semantics as the reference: intervals are grouped per chromosome (consecutive lines),
gaps between intervals are zero-filled unless `split_at_gaps`, a contig starts at its first interval's
start, three output modes with the reference's %-formats.  What differs is where the time goes: the text
is parsed by one C++ pass (csrc/textio.cpp) instead of a per-line Python loop, contigs are handed to the
GPU as run-length intervals (pasio_contig_load_rle expands them on the device: the dense 8 B/nt profile
never exists on the host), and the output lines are formatted in C++.
"""
import os
import sys
import numpy as np

from . import _native
from .logging import logger
from .segmentation import segments_with_scores, run_loaded_pipeline
from .dto.intervals import BedgraphInterval
from .utils.gzip_utils import open_for_read, open_for_write
from .splitters import _fusion

OUTPUT_MODES = {'bedgraph': 0, 'bed': 1, 'bedgraph+length+LMM': 2}


def fill_interval_gaps(intervals):
    """Reference helper kept for API compatibility: yields the intervals with zero-coverage gap tuples."""
    previous_stop = None
    for interval in intervals:
        start = interval[1]
        if previous_stop and previous_stop != start:
            yield (interval[0], previous_stop, start, 0)
        yield interval
        previous_stop = interval[2]


def intervals_not_adjacent(interval_1, interval_2):
    return interval_1.stop != interval_2.start


def interval_groups(intervals, split_at_gaps):
    """Reference helper kept for API compatibility (groups of BedgraphInterval objects forming one contig)."""
    import itertools
    from .utils.slice_when import slice_when
    for _, chromosome_intervals in itertools.groupby(intervals, key=lambda interval: interval.chrom):
        if split_at_gaps:
            for group in slice_when(chromosome_intervals, condition=intervals_not_adjacent):
                yield group
        else:
            yield fill_interval_gaps(chromosome_intervals)


CHUNK_BYTES = 64 << 20        # the input is read in pieces of this size, cut at line starts


class _Reader(object):
    """read(n) -> bytes, plus readinto(buffer) -> n when the object underneath has it (files, BytesIO, gzip): the
    streaming reader then fills its one reusable buffer without intermediate bytes objects"""

    def __init__(self, read, readinto=None):
        self.read = read
        self.readinto = readinto

    def __call__(self, n):
        return self.read(n)


def _binary_reader(stream):
    """read(n) -> bytes over the input.  A text stream over a binary one (open(..., 'rt'), gzip.open(..., 'rt'),
    sys.stdin) is read through the binary object underneath instead of decoding gigabytes of ASCII to str and
    encoding them back.  If the caller already consumed part of a seekable text stream, the binary object is first
    moved to the text layer's position (its read-ahead would otherwise be lost); a NON-seekable text stream (a pipe)
    must not have been read from before: its read-ahead cannot be recovered."""
    raw = getattr(stream, 'buffer', None)
    if raw is not None and hasattr(raw, 'read'):
        try:
            if stream.seekable():
                pos = stream.tell()              # byte offset of the next character (plain cookie for ASCII / UTF-8)
                if 0 <= pos < (1 << 62):
                    raw.seek(pos)
                    return _Reader(raw.read, getattr(raw, 'readinto', None))
            else:
                return _Reader(raw.read, getattr(raw, 'readinto', None))
        except (OSError, ValueError, AttributeError):
            pass

    def read_text(n):
        data = stream.read(n)
        return data.encode() if isinstance(data, str) else bytes(data)
    return _Reader(read_text)


def _read_all(stream):
    read = _binary_reader(stream)
    pieces = []
    while True:
        piece = read(CHUNK_BYTES)
        if not piece:
            break
        pieces.append(piece)
    return b''.join(pieces)


def _contig_runs_chunked(read, split_at_gaps=False):
    """Generator over the contigs of a bedgraph stream read in bounded pieces: yields
    (chrom, run_lengths, run_values, chrom_start) as soon as a contig is complete (the reference also yields contig by
    contig, process_bedgraph.py:46-60).  Memory: one piece of text plus the parsed lines of the contig in progress.

    Restatement (csrc/textio.cpp: pasio_bedgraph_parse / pasio_bedgraph_runs) of BedgraphInterval.each_in_stream,
    interval_groups and the accumulation loop of parse_bedgraph_stream (reference process_bedgraph.py:26-60): consecutive
    lines of one chromosome form a group; with split_at_gaps a group also ends where an interval does not start at the
    previous stop; otherwise a zero run is inserted between non-adjacent intervals (when the previous stop is non-zero,
    as in the reference's `if previous_stop and ...`).  Runs of non-positive length contribute nothing."""
    # one reusable buffer: the unfinished last line of a piece is moved to its front, the next piece is read behind it and
    # parsed in place (no bytes object per piece, no concatenation, no slicing copies)
    data = bytearray(CHUNK_BYTES + (1 << 16))
    readinto = getattr(read, 'readinto', None)
    tail_len = 0
    pend = None          # lines of the last (possibly unfinished) group: (chrom, starts, stops, counts)
    while True:
        filled = tail_len
        eof = False
        while filled - tail_len < CHUNK_BYTES // 2:              # (gzip and pipes return short reads)
            room = min(len(data) - filled, CHUNK_BYTES - (filled - tail_len))
            if room <= 0:
                break
            if readinto is not None:
                with memoryview(data) as mv:
                    got = readinto(mv[filled:filled + room])
                got = 0 if got is None else got
            else:
                piece = read(room)
                got = len(piece)
                data[filled:filled + got] = piece
            if got == 0:
                eof = True
                break
            filled += got
        if eof:
            cut = filled
        else:
            cut = data.rfind(b'\n', 0, filled) + 1
            if cut == 0 and filled == len(data):                 # a line longer than the buffer: grow and keep reading
                data.extend(bytes(len(data)))
                tail_len = filled
                continue
        # the lines of the contig in progress (from the pieces before) go in front of this piece's lines, in place
        n_old = len(pend[1]) if pend is not None else 0
        rec = _native.parse_bedgraph_text(data, front=n_old, length=cut) if cut else None
        n_new = len(rec['starts']) - n_old if rec is not None else 0
        if rec is not None and rec['n_float']:
            logger.warning("Pasio cannot be used with floating point counts. %d count(s) were automatically converted "
                           "to integers as an approximation. Make sure these values were designed to actually be "
                           "integer counts." % rec['n_float'])
        if n_new == 0 and not eof:
            tail_len = filled - cut
            data[0:tail_len] = data[cut:filled]
            continue
        if pend is not None:
            if n_new:
                first = bytes(data[rec['name_off'][n_old]:rec['name_off'][n_old] + rec['name_len'][n_old]])
                rec['starts'][:n_old] = pend[1]
                rec['stops'][:n_old] = pend[2]
                rec['counts'][:n_old] = pend[3]
                rec['new_chrom'][:n_old] = 0
                rec['new_chrom'][0] = 1
                rec['new_chrom'][n_old] = first != pend[0]
                lines = rec
            else:
                new_chrom = np.zeros(n_old, dtype=np.uint8)
                new_chrom[0] = 1
                lines = dict(starts=pend[1], stops=pend[2], counts=pend[3], new_chrom=new_chrom)
        elif n_new:
            lines = rec
        else:
            return                                   # end of an empty input
        run_len, run_val, group_line, group_run = _native.bedgraph_runs(lines, split_at_gaps)
        first_line = group_line.tolist()
        bounds = group_run.tolist()
        n_groups = len(first_line)
        first_start = lines['starts'][group_line].tolist()

        def name_of(k):
            gl = first_line[k]
            if gl < n_old:
                return pend[0]
            off, ln = int(rec['name_off'][gl]), int(rec['name_len'][gl])
            return bytes(data[off:off + ln])
        done = n_groups if eof else n_groups - 1     # the last group may continue in the next piece
        for k in range(done):
            yield name_of(k).decode(), run_len[bounds[k]:bounds[k + 1]], run_val[bounds[k]:bounds[k + 1]], first_start[k]
        if eof:
            return
        gl = first_line[-1]
        pend = (bytes(name_of(n_groups - 1)), lines['starts'][gl:].copy(), lines['stops'][gl:].copy(),
                lines['counts'][gl:].copy())
        tail_len = filled - cut                      # the unfinished last line moves to the front (names were read above)
        data[0:tail_len] = data[cut:filled]


def contig_runs(data, split_at_gaps=False):
    """The contigs of a bedgraph text held in memory (bytes): (chrom, run_lengths, run_values, chrom_start) each."""
    view = memoryview(data)
    pos = [0]

    def read(n):
        piece = bytes(view[pos[0]:pos[0] + n])
        pos[0] += len(piece)
        return piece
    return _contig_runs_chunked(read, split_at_gaps)


def parse_bedgraph(filename, split_at_gaps=False):
    """yields (chrom, dense int profile, chromosome_start); like the reference, ignores split_at_gaps"""
    with open_for_read(filename) as stream:
        for item in parse_bedgraph_stream(stream):
            yield item


def parse_bedgraph_stream(input_stream, split_at_gaps=False):
    for chrom, run_len, run_val, chrom_start in _contig_runs_chunked(_binary_reader(input_stream), split_at_gaps):
        yield chrom, np.repeat(run_val.astype(int), run_len), chrom_start


def split_bedgraph(in_filename, out_filename, splitter, split_at_gaps=False, output_mode='bedgraph', devices=None):
    """devices (new, not in the reference): number of GPUs to shard the contigs over, one worker process per GPU
    (pasio_b200/device_pool.py); None / 1 = this process's GPU."""
    with open_for_write(out_filename) as output_stream:
        with open_for_read(in_filename) as input_stream:
            split_bedgraph_stream(input_stream, output_stream, splitter,
                                  split_at_gaps=split_at_gaps, output_mode=output_mode, devices=devices)


def _write(output_stream, payload):
    raw = getattr(output_stream, 'buffer', None)
    if raw is not None and not getattr(output_stream, 'closed', False):
        output_stream.flush()
        raw.write(payload)
    else:
        try:
            output_stream.write(payload.decode('ascii'))
        except TypeError:
            output_stream.write(payload)


# Short contigs (scaffolds, transcripts) are segmented many per launch: consecutive contigs are collected until the
# batch holds BATCH_NT positions or BATCH_CONTIGS contigs and go to the device as one "super-contig" with forced
# boundaries (pasio_contig_load_rle with offsets); contigs never interact (reference process_bedgraph.py:69 handles
# them one by one), so the output is the same, in input order.  A contig of BATCH_ALONE positions or more runs alone.
BATCH_NT = 1 << 27
BATCH_CONTIGS = 20000
BATCH_ALONE = 1 << 24


def _segment_runs_on_device(plan, contigs, want_lmm):
    """contigs: list of (run_len, run_val), segmented in one launch sequence.
    -> (splits, means, lmm or None, first_split, offsets): split positions of the concatenation (they contain every
    contig boundary), per-segment outputs, the index of each contig's first split point, the contig offsets"""
    eng = _native.engine()
    eng.use_scorer(plan['factory'])
    lengths = np.array([int(rl.sum()) for rl, _ in contigs], dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    if len(contigs) == 1:
        run_len, run_val = contigs[0]
        eng.load_rle(np.concatenate([[0], np.cumsum(run_len)]), run_val)
    else:
        starts = np.concatenate([[0], np.cumsum(np.concatenate([rl for rl, _ in contigs]))]).astype(np.int64)
        eng.load_rle(starts, np.concatenate([rv for _, rv in contigs]), offsets=offsets)
    if want_lmm:
        eng.logfac_prefetch()                     # the sequential log-factorial sums run beside the rounds
    _, splits, means, lmm, _ = run_loaded_pipeline(eng, plan, want_lmm=want_lmm)
    first_split = np.searchsorted(splits, offsets)           # every contig boundary is a split point
    assert np.array_equal(splits[first_split], offsets)
    return splits, means, lmm, first_split, offsets


def _batches(contigs, plan):
    """Group the contig stream into launches: lists of (chrom, chrom_start, run_len, run_val), in input order."""
    pending, pending_nt = [], 0
    for chrom, run_len, run_val, chrom_start in contigs:
        n = int(run_len.sum())
        logger.info('Starting chrom %s of length %d' % (chrom, n))
        item = (chrom, chrom_start, run_len, run_val)
        # the exact DP is a single-contig kernel; other splitter objects go contig by contig through their protocol
        if plan is None or n >= BATCH_ALONE or BATCH_NT <= 0 or plan['final'] != 'nop':
            if pending:
                yield pending
                pending, pending_nt = [], 0
            yield [item]
            continue
        if pending and (pending_nt + n > BATCH_NT or len(pending) >= BATCH_CONTIGS):
            yield pending
            pending, pending_nt = [], 0
        pending.append(item)
        pending_nt += n
    if pending:
        yield pending


def _segment_batch(splitter, plan, batch, mode):
    """One launch sequence -> the arrays the formatter needs."""
    if plan is not None:
        # canonical splitter graph: run-length intervals go straight to the device
        assert all(int(rl.sum()) > 0 for _, _, rl, _ in batch)
        splits, means, lmm, first_split, offsets = _segment_runs_on_device(
            plan, [(rl, rv) for _, _, rl, rv in batch], want_lmm=(mode == 2))
        shifts = np.array([cs for _, cs, _, _ in batch], dtype=np.int64) - offsets[:-1]
        return [c for c, _, _, _ in batch], shifts, first_split, splits, means, lmm
    (chrom, chrom_start, run_len, run_val), = batch
    counts = np.repeat(run_val.astype(int), run_len)
    segs = list(segments_with_scores(counts, splitter))
    splits = np.array([s.start for s in segs] + [segs[-1].stop], dtype=np.int64)
    means = np.array([s.mean_count for s in segs], dtype=np.float64)
    lmm = np.array([s.log_marginal_likelyhood for s in segs], dtype=np.float64)
    return [chrom], np.array([chrom_start], dtype=np.int64), np.array([0, len(splits) - 1], dtype=np.int64), splits, means, lmm


def _format_batch(result, mode):
    chroms, shifts, first_split, splits, means, lmm = result
    return _native.format_segments_batch(chroms, shifts, first_split, splits, means if mode != 1 else None,
                                         lmm if mode == 2 else None, mode)


def segment_and_format(splitter, plan, batch, mode):
    """bytes of the output lines of one batch (device_pool workers call this)"""
    return _format_batch(_segment_batch(splitter, plan, batch, mode), mode)


class _Stage(object):
    """A pipeline stage on its own thread: items from `source` (an iterator) go through fn into a bounded queue.  The
    C calls behind fn (parser, kernels, formatter) release the GIL, so the stages overlap."""
    _END = object()

    def __init__(self, source, fn, depth=2):
        import queue
        import threading
        self.q = queue.Queue(maxsize=depth)
        self.error = None
        self.stop = False

        def run():
            try:
                for item in source:
                    if self.stop:
                        break
                    self.q.put(fn(item))
            except BaseException as e:       # noqa: BLE001 -- re-raised in the consumer
                self.error = e
            finally:
                self.q.put(self._END)
        self.thread = threading.Thread(target=run, daemon=True)
        self.thread.start()

    def __iter__(self):
        while True:
            item = self.q.get()
            if item is self._END:
                if self.error is not None:
                    raise self.error
                return
            yield item

    def cancel(self):
        self.stop = True
        try:
            while True:
                self.q.get_nowait()
        except Exception:                    # noqa: BLE001 -- queue.Empty
            pass


def split_bedgraph_stream(input_stream, output_stream, splitter, split_at_gaps=False, output_mode='bedgraph',
                          devices=None):
    """Reference: process_bedgraph.py:67-92.  The input is read in bounded pieces and a contig (or a batch of short
    contigs) is segmented and written as soon as it is complete; reading + parsing of the next piece, the device work
    and the formatting + writing of the previous batch run on three threads.  devices > 1: the batches are sharded over
    that many GPUs by longest-processing-time-first, one worker process per GPU, the text gathered on the host in
    input order (device_pool.py)."""
    logger.info('Reading input file')
    plan = _fusion.device_plan(splitter)
    if output_mode not in OUTPUT_MODES:
        raise ValueError('Unknown output mode `%s`' % output_mode)
    mode = OUTPUT_MODES[output_mode]
    contigs = _contig_runs_chunked(_binary_reader(input_stream), split_at_gaps)
    if devices is not None and int(devices) > 1:
        from . import device_pool
        for payload, chroms in device_pool.run(list(_batches(contigs, plan)), splitter, mode, int(devices)):
            _write(output_stream, payload)
            for chrom in chroms:
                logger.info('Output of chromosome %s finished' % chrom)
        return
    import queue
    import threading
    busy = {'read': 0.0, 'device': 0.0, 'write': 0.0}               # seconds of work per stage (PASIO_B200_STAGE_TIMES=1 prints them)
    import time as _time

    def timed_batches():
        it = iter(_batches(contigs, plan))
        while True:
            t0 = _time.perf_counter()
            try:
                b = next(it)
            except StopIteration:
                return
            finally:
                busy['read'] += _time.perf_counter() - t0
            yield b
    parsed = _Stage(timed_batches(), lambda b: b)                  # thread 1: read + parse + group
    out_q = queue.Queue(maxsize=2)
    writer_error = []

    def writer():                                                  # thread 3: format + write, in input order
        try:
            while True:
                item = out_q.get()
                if item is None:
                    return
                batch, result = item
                t0 = _time.perf_counter()
                _write(output_stream, _format_batch(result, mode))
                busy['write'] += _time.perf_counter() - t0
                for chrom, _, _, _ in batch:
                    logger.info('Output of chromosome %s finished' % chrom)
        except BaseException as e:           # noqa: BLE001 -- re-raised below
            writer_error.append(e)
            while out_q.get() is not None:   # keep draining so the producer never blocks
                pass
    thread = threading.Thread(target=writer, daemon=True)
    thread.start()
    try:
        for batch in parsed:                                       # this thread: the device
            if writer_error:
                break
            t0 = _time.perf_counter()
            result = _segment_batch(splitter, plan, batch, mode)
            busy['device'] += _time.perf_counter() - t0
            out_q.put((batch, result))
    except BaseException:
        parsed.cancel()
        raise
    finally:
        out_q.put(None)
        thread.join()
    if os.environ.get('PASIO_B200_STAGE_TIMES'):
        sys.stderr.write('[pasio_b200 stages] read+parse %.3f s, device %.3f s, format+write %.3f s (busy time per thread)\n'
                         % (busy['read'], busy['device'], busy['write']))
    if writer_error:
        raise writer_error[0]
