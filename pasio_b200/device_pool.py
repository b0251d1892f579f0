"""split_bedgraph(..., devices=N): the contigs of one input sharded over N GPUs.

Contigs never interact (reference process_bedgraph.py:69 handles them one by one), so they are partitioned, not
exchanged: one worker PROCESS per GPU (its own CUDA context, tables and Engine), longest-processing-time-first
assignment of the batches (the ordering heuristic of the reference's per-chromosome script generator,
/root/reference/tests/pasio_parallel_wrapper.py:68-74), every worker writes the text of its batches to shard files,
the parent concatenates them in input order.  No collective, no NCCL: the run-length intervals reach the workers
through one shared-memory block, the results come back as files.
"""
import multiprocessing as mp
import os
import pickle
import shutil
import tempfile
from multiprocessing import shared_memory

import numpy as np

from . import sharding


def _attach(name, n_runs):
    shm = shared_memory.SharedMemory(name=name)
    arr = np.ndarray((2, n_runs), dtype=np.int64, buffer=shm.buf)
    return shm, arr


def _worker(device, jobs, shm_name, n_runs, splitter_blob, mode, tmpdir, done_q):
    try:
        # (PASIO_B200_POOL_SAME_DEVICE: tests on a one-GPU box run both workers on device 0)
        os.environ['PASIO_B200_DEVICE'] = '0' if os.environ.get('PASIO_B200_POOL_SAME_DEVICE') else str(device)
        from . import process_bedgraph
        from .splitters import _fusion
        splitter = pickle.loads(splitter_blob)
        plan = _fusion.device_plan(splitter)
        shm, runs = _attach(shm_name, n_runs)
        try:
            for index, contigs in jobs:
                batch = [(chrom, chrom_start, runs[0, a:b], runs[1, a:b]) for chrom, chrom_start, a, b in contigs]
                payload = process_bedgraph.segment_and_format(splitter, plan, batch, mode)
                path = os.path.join(tmpdir, 'part_%08d.tsv' % index)
                with open(path, 'wb') as f:
                    f.write(payload)
                done_q.put((index, path, None))
        finally:
            del runs
            shm.close()
    except BaseException as e:               # noqa: BLE001 -- reported to the parent
        import traceback
        done_q.put((-1, None, '%s\n%s' % (e, traceback.format_exc())))


def plan_shards(batch_nt, n_devices):
    """LPT over the batches: -> per device the batch indices, longest first."""
    rank_of = sharding.lpt_assign([sharding.contig_cost(n) for n in batch_nt], n_devices)
    order = sorted(range(len(batch_nt)), key=lambda i: (-batch_nt[i], i))
    return [[i for i in order if rank_of[i] == d] for d in range(n_devices)]


def run(batches, splitter, mode, n_devices):
    """batches: list of lists of (chrom, chrom_start, run_len, run_val).  Yields (payload bytes, chrom names) per batch
    in input order as soon as every earlier batch is finished."""
    if not batches:
        return
    batch_nt = [sum(int(rl.sum()) for _, _, rl, _ in b) for b in batches]
    shards = plan_shards(batch_nt, n_devices)
    n_runs = sum(len(rl) for b in batches for _, _, rl, _ in b)
    shm = shared_memory.SharedMemory(create=True, size=max(16, 2 * n_runs * 8))
    tmpdir = tempfile.mkdtemp(prefix='pasio_b200_shards_')
    procs = []
    try:
        runs = np.ndarray((2, n_runs), dtype=np.int64, buffer=shm.buf)
        meta, pos = [], 0
        for b in batches:
            rows = []
            for chrom, chrom_start, rl, rv in b:
                runs[0, pos:pos + len(rl)] = rl
                runs[1, pos:pos + len(rl)] = rv
                rows.append((chrom, int(chrom_start), pos, pos + len(rl)))
                pos += len(rl)
            meta.append(rows)
        del runs
        ctx = mp.get_context('spawn')                       # a forked child must not inherit a CUDA context
        done_q = ctx.Queue()
        blob = pickle.dumps(splitter)
        for d in range(n_devices):
            jobs = [(i, meta[i]) for i in shards[d]]
            if not jobs:
                continue
            p = ctx.Process(target=_worker, args=(d, jobs, shm.name, n_runs, blob, mode, tmpdir, done_q), daemon=True)
            p.start()
            procs.append(p)
        ready, nxt = {}, 0
        while nxt < len(batches):
            try:
                index, path, err = done_q.get(timeout=1.0)
            except Exception:                # noqa: BLE001 -- queue.Empty: is everybody still alive?
                dead = [p for p in procs if p.exitcode not in (None, 0)]
                if dead:
                    raise RuntimeError('pasio_b200 device worker exited with code %s' % dead[0].exitcode)
                continue
            if err is not None:
                raise RuntimeError('pasio_b200 device worker failed: %s' % err)
            ready[index] = path
            while nxt in ready:
                with open(ready.pop(nxt), 'rb') as f:
                    payload = f.read()
                yield payload, [c for c, _, _, _ in batches[nxt]]
                nxt += 1
        for p in procs:
            p.join()
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
        shm.close()
        shm.unlink()
        shutil.rmtree(tmpdir, ignore_errors=True)
