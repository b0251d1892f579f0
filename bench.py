#!/usr/bin/env python
"""bench.py -- throughput of the Pasio segmentation hot path on B200.

A "step" is one pass of the default pasio pipeline (NotConstantReducer + RoundReducer over
SlidingWindowReducer(2500, 1250) + SquareSplitter, then NopSplitter scoring) over one synthetic
hg38-chr1-sized DNase-like contig (BASELINE.json configs[1]).  With N GPUs every rank segments
the SAME chr1-sized contig (contigs are independent: no data-path collective; weak scaling, so
the N-GPU efficiency measures the machine, not the data).

  value : whole-job nt/s with the counts already resident in HBM when the timed region starts
  e2e   : the same through the public API (pasio_b200.segmentation.segment_on_device) from a
          PINNED HOST int64 buffer: H2D of the counts and D2H of splits / scores / means / logfac
          inside the timed region
  roofline : the dominant kernel (batched window DP), 4 FP64 ops per (i,j) cell (SURVEY 8d) against
          the FP64-pipe instruction rate; `frac` counts ALGORITHMIC cells (what the reference
          evaluates), `frac_evaluated` only the cells the kernel really evaluated (the rest is
          proved irrelevant by the exact bound), `pipe_fp64_pct` is ncu's pipe utilisation
  cpu_baseline : oracle/ (numpy port of the reference) on a bounded prefix of the same contig
  parity : the GPU's splits / score on that prefix against the oracle's, bit for bit; the line is
          REFUSED (exit 1) if they differ
  exact_dp : BASELINE configs[0] and configs[2] -- the whole-contig SquareSplitter DP (K3): kernel
          time, ns per row of the dependent chain, FP64-roofline fractions (algorithmic / evaluated)
  genome : BASELINE configs[3] -- the hg38 contig-size profile (195 contigs, 3.10e9 nt) partitioned
          over the N ranks by longest-processing-time-first (pasio_b200.sharding), STRONG scaling:
          resident and from-host throughput, per-rank ms / nt / rounds / segments

`--impl reference` times the reference's CPU algorithm (oracle port; the reference is pure Python
and /root/reference does not exist on the GPU box) on all host cores, same metric and config.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CHR1 = 248956422
WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT = 2500, 1250, 'constants'
FP64_OPS_PER_CELL = 4            # DMUL s*Lg, DADD G-.., DADD +P_i, compare (SURVEY 8d)
BIG_CONTIG = 16 << 20            # genome leg: shorter contigs share one batched launch sequence
DUMP_MAX_SEGMENTS = 1 << 20      # --dump-outputs: five float64 arrays of at most this length, 40 MB in all


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        return json.load(open(path)), 'measured'
    return {'hbm_gbs': 6650.0, 'sm_max_mhz': 1965.0}, 'fallback'


class ClockSampler(object):
    """SM clock and throttle reasons sampled DURING the timed region: NVML in a thread of this process (a sample every
    few ms: the timed region of a short run is ~0.1 s, less than nvidia-smi needs to start on an 8-GPU box), with the
    nvidia-smi loop of the profiling recipe as the fallback when the NVML binding is missing."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    REASON_BITS = [(0x8, 'hw_slowdown'), (0x40, 'hw_thermal_slowdown'), (0x20, 'sw_thermal_slowdown'), (0x4, 'sw_power_cap')]

    def __init__(self, index, uuid=None):
        self.index = index
        self.uuid = uuid
        self.proc = None
        self.path = None
        self.thread = None
        self.stop_flag = threading.Event()
        self.sm, self.reasons, self.mx = [], set(), None

    def _nvml_loop(self, nv, handle):
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(handle)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                for bit, name in self.REASON_BITS:
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                break
            self.stop_flag.wait(0.004)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            handle = None
            if self.uuid:
                for cand in (self.uuid, 'GPU-' + self.uuid):
                    try:
                        handle = nv.nvmlDeviceGetHandleByUUID(cand.encode() if hasattr(cand, 'encode') else cand)
                        break
                    except Exception:
                        handle = None
            if handle is None:
                handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        fd, self.path = tempfile.mkstemp(suffix='.csv')
        os.close(fd)
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            if self.sm:
                out.update(sm_mhz=float(np.median(self.sm)), sm_max_mhz=self.mx, reasons=sorted(self.reasons),
                           samples=len(self.sm), source='nvml')
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in open(self.path):
            f = [x.strip() for x in line.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       source='nvidia-smi')
        return out


def dist_setup(n_gpus):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend='nccl', device_id=torch.device('cuda', local))
    return rank, world, local, dist


def gather_rows(row, dist, device, world):
    """every rank's list of floats -> list of lists on all ranks (timing control plane only)"""
    if dist is None:
        return [list(row)]
    import torch
    t = torch.tensor(row, dtype=torch.float64, device=device)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [o.tolist() for o in out]


def barrier(dist, torch):
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


# ---- config 4: the genome profile, generated per rank before CUDA starts ------------------------
_GEN = {}


def _gen_one(job):
    index, length, offset = job
    from pasio_b200 import synth
    arr = np.frombuffer(_GEN['raw'], dtype=np.int64)
    arr[offset:offset + length] = synth.dnase_like(length, seed=index)      # SURVEY 8d: config-2 generator, seed = contig index
    return index


def genome_generate(args):
    """This rank's LPT share of the hg38 contig-size profile, as one int64 buffer: contigs of BIG_CONTIG positions or
    more first (longest first), then the short ones contiguously (they go to the device as one batch)."""
    if args.genome_scale <= 0:
        return None
    import multiprocessing as mp
    from pasio_b200 import synth, sharding
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    sizes = synth.genome_profile(scale=args.genome_scale)
    costs = [sharding.contig_cost(n) for _, n in sizes]
    rank_of = sharding.lpt_assign(costs, world)
    mine = [i for i in range(len(sizes)) if rank_of[i] == rank]
    big = sorted([i for i in mine if sizes[i][1] >= BIG_CONTIG], key=lambda i: -sizes[i][1])
    small = [i for i in mine if sizes[i][1] < BIG_CONTIG]
    order = big + small
    offsets, pos = {}, 0
    for i in order:
        if i in big or (small and i == small[0]):
            pos += pos & 1                       # device pointers handed to pasio_contig_load_device are 16-byte aligned
        offsets[i] = pos
        pos += sizes[i][1]
    raw = mp.RawArray('q', max(1, pos))
    _GEN['raw'] = raw
    procs = max(1, min(len(order), (os.cpu_count() or 1) // max(1, min(world, 8))))
    t0 = time.perf_counter()
    if order:
        with mp.get_context('fork').Pool(procs) as pool:
            pool.map(_gen_one, [(i, sizes[i][1], offsets[i]) for i in order], chunksize=1)
    loads = [sum(costs[i] for i in range(len(sizes)) if rank_of[i] == r) for r in range(world)]
    return dict(sizes=sizes, big=big, small=small, offsets=offsets, nt=pos, host=np.frombuffer(raw, dtype=np.int64)[:pos],
                gen_s=time.perf_counter() - t0, lpt_max_over_mean=max(loads) / (sum(loads) / world),
                total_nt=sum(n for _, n in sizes))


def genome_leg(args, g, eng, plan, torch, dist, device, world):
    """config 4, strong scaling: every rank segments its LPT share; the step time is the max over ranks."""
    from pasio_b200.segmentation import segment_on_device
    sizes, big, small, offs = g['sizes'], g['big'], g['small'], g['offsets']
    resident = torch.from_numpy(g['host']).to(device) if g['nt'] else None
    small_nt = sum(sizes[i][1] for i in small)
    small_off = offs[small[0]] if small else 0
    small_bounds = np.concatenate([[0], np.cumsum([sizes[i][1] for i in small])]).astype(np.int64) if small else None
    stream = torch.cuda.ExternalStream(eng.stream_handle(), device=device)
    stat = {}

    def finish():
        eng.segment_scores(scores=True, means=True)
        return eng.candidate_count() - 1, float(eng.segment_scores_sum())

    def step_resident():
        nseg, rounds, cells = 0, 0, 0
        for i in big:
            eng.use_scorer(plan['factory'])
            eng.load_device(resident.data_ptr() + 8 * offs[i], sizes[i][1], owner=resident)
            eng.set_candidates(None)
            sz, _, c = eng.rounds(WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
            rounds += len(sz)
            cells += c
            nseg += finish()[0]
        if small:
            eng.use_scorer(plan['factory'])
            eng.load_device(resident.data_ptr() + 8 * small_off, small_nt, owner=resident, offsets=small_bounds)
            eng.set_candidates(None)
            sz, _, c = eng.rounds(WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
            rounds += len(sz)
            cells += c
            nseg += finish()[0]
        stat.update(segments=nseg, rounds=rounds, cells=cells)

    def step_e2e():
        nseg = 0
        for i in big:
            eng.invalidate()
            _, splits, means, _, _ = segment_on_device(g['host'][offs[i]:offs[i] + sizes[i][1]], plan, want_lmm=False)
            nseg += len(splits) - 1
        if small:
            eng.invalidate()
            eng.use_scorer(plan['factory'])
            eng.load(g['host'][small_off:small_off + small_nt], offsets=small_bounds)
            eng.set_candidates(None)
            eng.rounds(WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
            eng.candidates()
            nseg += finish()[0]
        return nseg

    steps = max(1, args.genome_steps)
    step_resident()
    barrier(dist, torch)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        step_resident()
    ev1.record(stream)
    ev1.synchronize()
    my_ms = ev0.elapsed_time(ev1) / steps
    barrier(dist, torch)
    step_e2e()
    barrier(dist, torch)
    t0 = time.perf_counter()
    nseg_e2e = step_e2e()
    my_e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier(dist, torch)
    assert nseg_e2e == stat['segments']
    rows = gather_rows([my_ms, my_e2e_ms, float(g['nt']), float(len(big) + len(small)), float(stat['rounds']),
                        float(stat['cells']), float(stat['segments'])], dist, device, world)
    ms = max(r[0] for r in rows)
    e2e_ms = max(r[1] for r in rows)
    total_nt = g['total_nt']
    return {
        'workload': 'BASELINE configs[3]: hg38 contig-size profile (scale %g): %d contigs, %d nt, default pipeline, '
                    'partitioned over %d GPU(s) by longest-processing-time-first; contigs under %d nt of a rank share one '
                    'batched launch sequence' % (args.genome_scale, len(sizes), total_nt, world, BIG_CONTIG),
        'scaling': 'strong', 'n_gpus': world, 'nt': total_nt, 'steps': steps,
        'value': total_nt / (ms * 1e-3), 'unit': 'nt/s', 'ms_per_step': ms,
        'e2e': {'value': total_nt / (e2e_ms * 1e-3), 'unit': 'nt/s', 'ms_per_step': e2e_ms,
                'h2d_bytes_per_step': int(total_nt * 8), 'source': 'pageable host numpy arrays (staged upload)',
                'note': 'per-rank results on the host; the ordered gather of the text is host-side (shard files, '
                        'pasio_b200/device_pool.py) and not part of this number'},
        'lpt_max_over_mean': g['lpt_max_over_mean'],
        'per_rank': {'ms': [r[0] for r in rows], 'e2e_ms': [r[1] for r in rows], 'nt': [int(r[2]) for r in rows],
                     'contigs': [int(r[3]) for r in rows], 'rounds': [int(r[4]) for r in rows],
                     'cells': [int(r[5]) for r in rows], 'segments': [int(r[6]) for r in rows]},
        'segments': int(sum(r[6] for r in rows)), 'dp_cells': int(sum(r[5] for r in rows)),
        'host_generation_s': g['gen_s'],
    }


# ---- configs 1 and 3: the whole-contig exact DP --------------------------------------------------
def exact_leg(eng, peak_nominal):
    from pasio_b200 import synth
    from pasio_b200.log_marginal_likelyhood import ScorerFactory
    out = {}
    eng.use_scorer(ScorerFactory(1.0, 1.0))
    for name, counts, cands in [('config1', synth.piecewise_poisson(100000, 0), None),
                                ('config3', synth.piecewise_poisson(2000000, 1), synth.random_candidates(2000000, 200000, 1))]:
        N = len(counts) + 1 if cands is None else len(cands)
        eng.invalidate()
        eng.load(counts)
        best = None
        for rep in range(4):
            eng.set_candidates(cands)
            eng._cands_obj = None
            eng.timing_reset(True)
            score, splits = eng.square_split()
            ms = eng.timing()['exact_dp'][0]
            if rep > 0 and (best is None or ms < best):
                best = ms
        eng.timing_reset(False)
        cells, skipped = eng.round_stats()
        out[name] = {
            'workload': 'BASELINE configs[%d]: exact SquareSplitter, N = %d candidates' % (0 if name == 'config1' else 2, N),
            'cells': cells, 'cells_evaluated': cells - skipped, 'evaluated_frac': (cells - skipped) / cells,
            'kernel_ms': best, 'cells_per_s': cells / (best * 1e-3), 'ns_per_row': best * 1e6 / N,
            'roofline': {'bound': 'fp64 (algorithmic cells) / dependent chain of N rows', 'peak': peak_nominal / 1e12,
                         'unit': 'TFLOP/s', 'achieved': cells * FP64_OPS_PER_CELL / (best * 1e-3) / 1e12,
                         'frac': cells * FP64_OPS_PER_CELL / (best * 1e-3) / peak_nominal,
                         'frac_evaluated': (cells - skipped) * FP64_OPS_PER_CELL / (best * 1e-3) / peak_nominal},
            'splits': len(splits), 'score': float(score),
        }
    return out


def dump_outputs(out_dir, splits, scores, means, total_score):
    """The segmentation of the last timed step as float64 .npy files under out_dir, for comparing two builds output for
    output: per segment its index, start, stop, score and mean count, for every segment when there are at most
    DUMP_MAX_SEGMENTS of them and otherwise for a fixed seeded sample of that many; plus the total score and the number
    of segments.  float64 holds every position and index exactly."""
    nseg = len(splits) - 1
    idx = np.arange(nseg)
    if nseg > DUMP_MAX_SEGMENTS:
        idx = np.sort(np.random.RandomState(0).choice(nseg, DUMP_MAX_SEGMENTS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'segment_index': idx, 'segment_start': splits[idx], 'segment_stop': splits[idx + 1],
              'segment_score': scores[idx], 'segment_mean': means[idx],
              'total_score': [total_score], 'n_segments': [nseg]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.asarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
def run_b200(args):
    genome_host = genome_generate(args)          # host data of this rank's LPT share, before CUDA starts (fork pool)
    import torch
    from pasio_b200 import synth, _native
    from pasio_b200.splitters import configure_splitter, _fusion
    from pasio_b200.segmentation import segment_on_device, _run_device_pipeline

    rank, world, local, dist = dist_setup(args.gpus)
    os.environ.setdefault('PASIO_B200_DEVICE', str(local))
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    n = args.nt
    peaks, peak_kind = measured_peaks()

    # synthetic input, generated straight into pinned host memory (the same chr1-sized contig on every rank)
    host = torch.empty(n, dtype=torch.int64, pin_memory=True)
    counts = host.numpy()
    counts[:] = synth.dnase_like(n, seed=1000)
    resident = host.to(device, non_blocking=False)          # the HBM-resident copy for `value`
    torch.cuda.synchronize()

    eng = _native.engine()
    splitter = configure_splitter(window_size=WINDOW_SIZE, window_shift=WINDOW_SHIFT, split_constraints=CONSTRAINT)
    plan = _fusion.pipeline_plan(splitter)
    assert plan is not None
    stream = torch.cuda.ExternalStream(eng.stream_handle(), device=device)

    def step_resident():
        eng.use_scorer(plan['factory'])
        eng.load_device(resident.data_ptr(), n, owner=resident)
        eng.set_candidates(None)
        _run_device_pipeline(eng, plan)
        scores, _, means, _ = eng.segment_scores(scores=True, means=True)
        return eng.candidate_count(), float(eng.segment_scores_sum()), scores, means

    def step_e2e():
        eng.invalidate()                                     # force the H2D copy every step
        score, splits, means, lmm, _ = segment_on_device(counts, plan, want_lmm=True)
        return len(splits), float(score)

    # ---- device-resident throughput ------------------------------------------------------------
    for _ in range(args.warmup):
        m_final, score = step_resident()[:2]
    fp64_peak_measured = eng.fp64_peak() if rank == 0 else 0.0
    eng.timing_reset(True)
    sampler = ClockSampler(local, str(getattr(torch.cuda.get_device_properties(local), 'uuid', '') or ''))
    barrier(dist, torch)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = None              # frees the previous step's pinned result buffers for this step to reuse
        last = step_resident()
    ev1.record(stream)
    ev1.synchronize()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    barrier(dist, torch)
    dev_ms = ev0.elapsed_time(ev1)
    timing = eng.timing()
    eng.timing_reset(False)
    m_final, score = last[:2]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng.candidates(), last[2], last[3], score)
    del last
    rank_rows = gather_rows([dev_ms / args.steps], dist, device, world)
    step_ms = max(r[0] for r in rank_rows)
    total_nt = float(n) * world
    value = total_nt / (step_ms * 1e-3)

    # cells of one step (same every step): one extra instrumented pass, round by round
    eng.use_scorer(plan['factory'])
    eng.load_device(resident.data_ptr(), n, owner=resident)
    eng.set_candidates(None)
    sizes, cells, cells_skipped = [], 0, 0
    while True:
        n_in, n_out, c = eng.round(WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
        sizes.append(n_in)
        cells += c
        cells_skipped += eng.round_stats()[1]
        if n_in == n_out:
            break
    final = eng.candidate_count()

    # ---- end to end from pinned host memory ----------------------------------------------------
    for _ in range(min(args.warmup, 2)):
        step_e2e()
    barrier(dist, torch)
    eng.timing_reset(True)
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    e2e_each = []
    for _ in range(e2e_steps):
        t1 = time.perf_counter()
        m_e2e, score_e2e = step_e2e()
        e2e_each.append((time.perf_counter() - t1) * 1e3)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    e2e_timing = eng.timing()
    e2e_wire_bytes = int(eng.upload_stats())
    eng.timing_reset(False)
    e2e_rows = gather_rows([e2e_s * 1e3], dist, device, world)
    e2e_s = max(r[0] for r in e2e_rows) * 1e-3
    e2e_value = total_nt / e2e_s
    assert m_e2e == m_final and abs(score_e2e - score) <= 1e-9 * abs(score)

    # ---- parity gate: the GPU against the oracle on the cpu_baseline prefix (rank 0) -------------
    cpu, parity = None, None
    if rank == 0:
        cpu, oracle_out = cpu_baseline_port(counts, args.cpu_sample_nt)
        prefix = np.ascontiguousarray(counts[:args.cpu_sample_nt])
        eng.invalidate()
        g_score, g_splits, g_means, _, _ = segment_on_device(prefix, plan, want_lmm=False)
        equal = bool(np.array_equal(np.asarray(g_splits), oracle_out['splits']))
        rel = abs(float(g_score) - float(oracle_out['score'])) / max(1e-300, abs(float(oracle_out['score'])))
        parity = {'prefix_nt': int(len(prefix)), 'splits_equal': equal, 'n_splits': int(len(oracle_out['splits'])),
                  'means_equal': bool(np.array_equal(np.asarray(g_means), oracle_out['mean_counts'])),
                  'score_rel': rel, 'oracle': 'oracle/pasio_oracle.default_pipeline (numpy restatement of the reference)'}

    # ---- the other configs ------------------------------------------------------------------------
    fp64_peak_nominal = 148 * 64 * peaks.get('sm_max_mhz', 1965.0) * 1e6
    exact = exact_leg(eng, fp64_peak_nominal) if rank == 0 and not args.skip_exact else None
    del resident, host, counts
    torch.cuda.empty_cache()
    barrier(dist, torch)
    genome = genome_leg(args, genome_host, eng, plan, torch, dist, device, world) if genome_host is not None else None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if not (parity['splits_equal'] and parity['means_equal'] and parity['score_rel'] <= 1e-9):
        print(json.dumps({'error': 'PARITY FAILED: the GPU path disagrees with the oracle on the cpu_baseline prefix; '
                                   'no throughput is reported', 'parity': parity}))
        sys.exit(1)

    # ---- roofline of the dominant kernel -------------------------------------------------------
    wd_ms, wd_launches = timing['window_dp']
    scan_ms, scan_launches = timing['scan']
    cells_per_launch = cells / max(1, len(sizes))
    # one timed span per round: the CTA-per-window kernel and the two warp-per-window kernels of a round overlap
    # (side stream), so the per-round span is the unit; wd_launches counts the kernels themselves
    wd_rounds = max(1, len(sizes) * args.steps)
    wd_avg_s = (wd_ms / wd_rounds) * 1e-3
    achieved = cells_per_launch * FP64_OPS_PER_CELL / wd_avg_s
    evaluated = cells - cells_skipped
    traffic, pipe = None, None
    prof = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
    if os.path.exists(prof):
        pj = json.load(open(prof))
        traffic = pj.get('window_dp_dram_bytes_per_launch')
        pipe = pj.get('window_dp_pipe_fp64_pct')
    roofline = {
        'kernel': 'window DP of one round: window_dp_kernel (CTA per window) + small_window_dp_kernel x2 (warp per window, '
                  'side stream), timed as one span per round',
        'bound': 'fp64', 'achieved': achieved / 1e12, 'peak': fp64_peak_nominal / 1e12, 'unit': 'TFLOP/s',
        'frac': achieved / fp64_peak_nominal, 'traffic': traffic,
        'cells_algorithmic': cells, 'cells_evaluated': evaluated, 'evaluated_frac': evaluated / max(1, cells),
        'frac_evaluated': (evaluated / max(1, len(sizes))) * FP64_OPS_PER_CELL / wd_avg_s / fp64_peak_nominal,
        'pipe_fp64_pct': pipe,
        'note': '`frac` counts the cells the reference evaluates (N(N-1)/2 per window); the kernel proves most of them '
                'irrelevant with an exact bound and evaluates `cells_evaluated`; pipe_fp64_pct is ncu '
                'sm__inst_executed_pipe_fp64 of window_dp_kernel (profiles/)',
        'peak_source': '148 SM x 64 FP64 lanes x sm_max_mhz (%s MEASURED_PEAKS.json has no FP64 entry); '
                       'DFMA micro-benchmark on this box: %.3g instr/s' % (peak_kind, fp64_peak_measured),
        'algorithmic_ops_per_cell': FP64_OPS_PER_CELL, 'cells_per_launch': cells_per_launch,
        'avg_launch_ms': wd_avg_s * 1e3, 'launches': wd_rounds, 'kernels_launched': wd_launches,
        'share_of_step': wd_ms / (dev_ms if dev_ms > 0 else 1.0),
        'scan_kernel': {'bound': 'hbm', 'achieved': 16.0 * n / ((scan_ms / max(1, scan_launches)) * 1e-3) / 1e9,
                        'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                        'frac': 16.0 * n / ((scan_ms / max(1, scan_launches)) * 1e-3) / 1e9 / peaks['hbm_gbs'],
                        'peak_source': peak_kind},
    }

    gpu_launches = int(sum(timing[k][1] for k in ['scan', 'window_dp', 'compact', 'exact_dp', 'score']))
    line = {
        'metric': 'whole-contig segmentation throughput, default pasio pipeline (nt/s); DP cell updates/s in dp_cells_per_s',
        'value': value, 'unit': 'nt/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': step_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'BASELINE configs[1]: default pasio pipeline (constants + rounds over sliding window '
                               '2500/1250 + SquareSplitter, alpha=beta=1) on one synthetic chr1-sized (%d nt) DNase-like '
                               'contig per GPU (the same contig on every GPU)' % n,
                   'nt_per_gpu': n, 'window_size': WINDOW_SIZE, 'window_shift': WINDOW_SHIFT,
                   'split_constraints': CONSTRAINT, 'rounds': len(sizes), 'candidates_per_round': sizes,
                   'segments': final - 1, 'l2_policy': 'inputs larger than L2 (2 GB counts + 2 GB prefix sums per step)',
                   'parallelism': 'one replica of the contig per GPU (%d), no collective; the LPT partition of a whole '
                                  'genome over the GPUs is the `genome` key' % world},
        'per_rank_ms_per_step': [r[0] for r in rank_rows],
        'dp_cells_per_step': cells, 'dp_cells_per_s': cells * world / (step_ms * 1e-3),
        'window_dp_cells_per_s_kernel_only': cells / (wd_ms / args.steps * 1e-3),
        'e2e': {'value': e2e_value, 'unit': 'nt/s', 'h2d_bytes_per_step': int(n * 8),
                'h2d_wire_bytes_per_step': e2e_wire_bytes,
                'h2d_note': 'h2d_bytes_per_step = the int64 counts tensor handed to the API (pinned host memory); the library packs '
                            'counts that fit 31 bits to int32 on host threads before the DMA and widens them on the device, '
                            'h2d_wire_bytes_per_step is what crossed PCIe',
                'd2h_bytes_per_step': int(final * 8 * 4), 'ms_per_step': e2e_s * 1e3,
                'api': 'pasio_b200.segmentation.segment_on_device(counts_pinned_host, plan)',
                'device_ms_per_step': {k: e2e_timing[k][0] / e2e_steps for k in e2e_timing},
                'ms_each_step': e2e_each, 'per_rank_ms_per_step': [r[0] for r in e2e_rows]},
        'gpu_launches': gpu_launches,
        'kernel_ms_per_step': {k: timing[k][0] / args.steps for k in timing},
        'wall_ms_per_step': wall / args.steps * 1e3,
        'clocks': {'sm_mhz': clocks['sm_mhz'], 'sm_max_mhz': clocks['sm_max_mhz'], 'reasons': clocks['reasons'],
                   'samples': clocks['samples'], 'source': clocks.get('source')},
        'roofline': roofline, 'cpu_baseline': cpu, 'parity': parity, 'exact_dp': exact, 'genome': genome,
    }
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
def cpu_baseline_port(counts, sample_nt):
    """oracle/pasio_oracle.py (numpy restatement, one core) on the first sample_nt nt -> (cpu_baseline, oracle output)."""
    from oracle import pasio_oracle as po
    sample = np.ascontiguousarray(counts[:sample_nt])
    tables = po.Tables(1, 1.0)
    t0 = time.perf_counter()
    out = po.default_pipeline(sample, tables, WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
    dt = time.perf_counter() - t0
    return {'value': len(sample) / dt, 'unit': 'nt/s', 'cores': 1, 'kind': 'port',
            'sample': 'first %d nt of the rank-0 workload contig through oracle/pasio_oracle.default_pipeline '
                      '(numpy port of the reference, %d segments, %.1f s)' % (len(sample), len(out['splits']) - 1, dt)}, out


_REF_COUNTS = None      # set in the parent before the pool forks


def _ref_worker(job):
    lo, hi = job
    from oracle import pasio_oracle as po
    counts = _REF_COUNTS[lo:hi]
    tables = po.Tables(1, 1.0)
    t0 = time.perf_counter()
    out = po.default_pipeline(np.ascontiguousarray(counts), tables, WINDOW_SIZE, WINDOW_SHIFT, CONSTRAINT)
    return hi - lo, time.perf_counter() - t0, len(out['splits']) - 1


def run_reference(args):
    """The reference's CPU algorithm (oracle port) on every host core: one slice of the workload contig
    per core per step, the process-per-contig model of tests/pasio_parallel_wrapper.py."""
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    slice_nt = args.ref_slice_nt
    head = min(args.nt, cores * slice_nt * (args.steps + args.warmup))
    jobs_per_step = cores
    global _REF_COUNTS
    from pasio_b200 import synth
    _REF_COUNTS = synth.dnase_like(head, seed=1000)
    pool = mp.get_context('fork').Pool(cores)
    step_times, nt_per_step = [], jobs_per_step * slice_nt
    k = 0
    for step in range(args.warmup + args.steps):
        jobs = []
        for c in range(jobs_per_step):
            lo = (k * slice_nt) % max(slice_nt, head - slice_nt + 1)
            jobs.append((lo, lo + slice_nt))
            k += 1
        t0 = time.perf_counter()
        pool.map(_ref_worker, jobs)
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            step_times.append(dt)
    pool.close()
    ms = float(np.mean(step_times)) * 1e3
    value = nt_per_step / (ms * 1e-3)
    sample = ('%d slices of %d nt of the workload contig per step, one per host core, each through '
              'oracle/pasio_oracle.default_pipeline (numpy port of the reference; the reference itself is pure '
              'Python under /root/reference, which does not exist on the GPU box)' % (jobs_per_step, slice_nt))
    line = {
        'impl': 'reference',
        'metric': 'whole-contig segmentation throughput, default pasio pipeline (nt/s); DP cell updates/s in dp_cells_per_s',
        'value': value, 'unit': 'nt/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': {'workload': 'BASELINE configs[1]: default pasio pipeline on synthetic chr1-sized DNase-like contig '
                               '(bounded sample per step)', 'window_size': WINDOW_SIZE, 'window_shift': WINDOW_SHIFT,
                   'split_constraints': CONSTRAINT},
        'cpu_baseline': {'value': value, 'unit': 'nt/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'nt/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--nt', type=int, default=CHR1, help='contig length per GPU (default: hg38 chr1)')
    ap.add_argument('--cpu-sample-nt', type=int, default=2000000)
    ap.add_argument('--ref-slice-nt', type=int, default=500000)
    ap.add_argument('--genome-scale', type=float, default=1.0,
                    help='scale of the hg38 contig-size profile of the `genome` leg (configs[3]); 0 skips the leg')
    ap.add_argument('--genome-steps', type=int, default=2)
    ap.add_argument('--skip-exact', action='store_true', help='skip the `exact_dp` leg (configs[0], configs[2])')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the segments of the last one as DIR/<name>.npy (float64)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what the GPU path computed; --impl reference has no such output')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
