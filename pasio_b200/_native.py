"""ctypes binding of libpasio_b200.so (include/pasio_b200.h) and the per-process Engine.

The library is built in-tree (pasio_b200/libpasio_b200.so) by `__graft_entry__.build()` or
`make -C pasio_b200/csrc`.  There is NO CPU fallback: if the library is missing, or no
sm_100 device is visible, every LogML code path raises RuntimeError.
"""
import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('PASIO_B200_LIB') or os.path.join(_HERE, 'libpasio_b200.so')   # override: kernel experiments

OK = 0
E_CUDA, E_ARG, E_COUNTS, E_CANDIDATES, E_TABLE_TOO_SHORT, E_STATE, E_TOO_LARGE, E_NOMEM = range(-1, -9, -1)
TAB_LOG, TAB_LGAMMA, TAB_LGAMMA_ALPHA = 0, 1, 2
CONSTRAINTS = {'none': 0, 'zeros': 1, 'constants': 2}
TUNE = {'window_prune': 0, 'window_phases': 1, 'exact_prune': 2, 'exact_lag': 3, 'exact_ring': 4, 'logfac_exact': 5,
        'window_speculate': 6, 'upload_narrow': 7,
        'logfac_eager': 8, 'exact_nblock': 9, 'window_certify': 10, 'reg_exact': 11}
TIMING_FAMILIES = ['scan', 'window_dp', 'compact', 'exact_dp', 'score', 'h2d', 'd2h']

_i64 = ctypes.c_int64
_i64p = ctypes.POINTER(ctypes.c_int64)
_f64p = ctypes.POINTER(ctypes.c_double)
_vp = ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/pasio_b200.h declares
SIGNATURES = {
    'pasio_ctx_create': (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(_vp)]),
    'pasio_ctx_destroy': (ctypes.c_int, [_vp]),
    'pasio_last_error': (ctypes.c_char_p, [_vp]),
    'pasio_abi_version': (ctypes.c_int, []),
    'pasio_set_params': (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double]),
    'pasio_table_upload': (ctypes.c_int, [_vp, ctypes.c_int, _f64p, _i64]),
    'pasio_table_need': (ctypes.c_int, [_vp, _i64p, _i64p, _i64p]),
    'pasio_contig_load': (ctypes.c_int, [_vp, _i64p, _i64, _i64p, _i64]),
    'pasio_contig_load_round': (ctypes.c_int, [_vp, _i64p, _i64, _i64, _i64, ctypes.c_int, _i64p, _i64p, _i64p]),
    'pasio_contig_load_rle': (ctypes.c_int, [_vp, _i64p, _i64p, _i64, _i64p, _i64]),
    'pasio_contig_load_device': (ctypes.c_int, [_vp, _vp, _i64, _i64p, _i64]),
    'pasio_contig_info': (ctypes.c_int, [_vp, _i64p, _i64p, _i64p]),
    'pasio_cumsum_at': (ctypes.c_int, [_vp, _i64p, _i64, _i64p]),
    'pasio_candidates_set': (ctypes.c_int, [_vp, _i64p, _i64]),
    'pasio_candidates_count': (ctypes.c_int, [_vp, _i64p]),
    'pasio_candidates_download': (ctypes.c_int, [_vp, _i64p, _i64, _i64p]),
    'pasio_filter_candidates': (ctypes.c_int, [_vp, ctypes.c_int, _i64p, _i64p]),
    'pasio_round': (ctypes.c_int, [_vp, _i64, _i64, ctypes.c_int, _i64p, _i64p, _i64p]),
    'pasio_round_stats': (ctypes.c_int, [_vp, _i64p, _i64p]),
    'pasio_round_certify_stats': (ctypes.c_int, [_vp, _i64p, _i64p, _i64p]),
    'pasio_exact_task_plan': (ctypes.c_int, [_i64, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int32), _i64, _i64p]),
    'pasio_upload_stats': (ctypes.c_int, [_vp, _i64p]),
    'pasio_set_tuning': (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int]),
    'pasio_rounds': (ctypes.c_int, [_vp, _i64, _i64, ctypes.c_int, _i64, _i64p, _i64p, _i64p, _i64p, _i64]),
    'pasio_set_penalties': (ctypes.c_int, [_vp, _f64p, _i64, ctypes.c_double, _f64p, _i64]),
    'pasio_square_split': (ctypes.c_int, [_vp, _i64p, _i64, _i64p, _f64p, _f64p, _i64p]),
    'pasio_square_split_batch': (ctypes.c_int, [_vp, _i64p, _i64p, _i64p]),
    'pasio_square_split_regularized': (ctypes.c_int, [_vp, _f64p, _i64, _f64p, _i64, ctypes.c_double, _i64p, _i64, _i64p, _f64p,
                                                     _f64p, _i64p]),
    'pasio_suffix_scores': (ctypes.c_int, [_vp, _i64, _f64p]),
    'pasio_segment_scores': (ctypes.c_int, [_vp, _f64p, _i64p, _f64p, _f64p, _i64, _i64p]),
    'pasio_segment_scores_sum': (ctypes.c_int, [_vp, _f64p]),
    'pasio_segment_lmm': (ctypes.c_int, [_vp, _f64p, _i64, _f64p]),
    'pasio_logfac_prefetch': (ctypes.c_int, [_vp]),
    'pasio_host_alloc': (ctypes.c_int, [_i64, ctypes.POINTER(_vp)]),
    'pasio_host_free': (ctypes.c_int, [_vp]),
    'pasio_bedgraph_count_lines': (_i64, [ctypes.c_void_p, _i64]),
    'pasio_bedgraph_parse': (ctypes.c_int, [ctypes.c_void_p, _i64, _i64, _i64p, _i64p, _i64p, _i64p,
                                            ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_uint8), _i64p, _i64p]),
    'pasio_bedgraph_runs': (_i64, [_i64p, _i64p, _i64p, ctypes.POINTER(ctypes.c_uint8), _i64, ctypes.c_int, _i64p, _i64p, _i64p,
                                   _i64p, _i64p]),
    'pasio_format_segments': (_i64, [ctypes.c_char_p, _i64, _i64p, _i64, _f64p, _f64p, ctypes.c_int,
                                     ctypes.c_char_p, _i64]),
    'pasio_format_segments_batch': (_i64, [ctypes.c_char_p, _i64p, _i64p, _i64p, _i64, _i64p, _f64p, _f64p, ctypes.c_int,
                                           ctypes.c_char_p, _i64]),
    'pasio_timing_reset': (ctypes.c_int, [_vp, ctypes.c_int]),
    'pasio_timing_get': (ctypes.c_int, [_vp, ctypes.c_int, _f64p, _i64p]),
    'pasio_stream': (_vp, [_vp]),
    'pasio_fp64_peak': (ctypes.c_int, [_vp, _f64p]),
}

_lib = None
_lib_lock = threading.Lock()


def load_library():
    """dlopen the in-tree shared library and set every prototype.  Raises RuntimeError if absent."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError('pasio_b200: %s is missing -- build it with `python -c "import __graft_entry__ as g; '
                                   'g.build()"` or `make -C pasio_b200/csrc`; there is no CPU fallback' % LIB_PATH)
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def _ptr(arr, ct):
    return arr.ctypes.data_as(ctypes.POINTER(ct))


class PasioDeviceError(RuntimeError):
    pass


def exact_total_fits(total, alpha):
    """whether the whole-list DP can take a contig of this total count: it indexes the lgamma table with count + alpha in
    32 bits"""
    return total + alpha < 2 ** 31 - 2


class _PinnedPool(object):
    """Result arrays live in page-locked buffers so device->host copies run at PCIe rate and touch no
    fresh pages.  Every call still hands out an array nobody else references (the reference returns new
    arrays); a buffer goes back to the pool when its array is garbage collected."""

    def __init__(self, lib):
        self.lib = lib
        self.free = {}            # capacity -> [pointer, ...]
        self.lock = threading.Lock()
        self.total = 0

    @staticmethod
    def _capacity(nbytes):
        cap = 1 << 16
        while cap < nbytes:
            cap <<= 1
        return cap

    def empty(self, n, dtype):
        import weakref
        dtype = np.dtype(dtype)
        nbytes = max(1, int(n) * dtype.itemsize)
        cap = self._capacity(nbytes)
        with self.lock:
            bucket = self.free.get(cap)
            ptr = bucket.pop() if bucket else None
        if ptr is None:
            if self.total + cap > (8 << 30):          # do not pin without bound; fall back to pageable memory
                return np.empty(int(n), dtype=dtype)
            out = _vp()
            if self.lib.pasio_host_alloc(cap, ctypes.byref(out)) != OK:
                return np.empty(int(n), dtype=dtype)
            ptr = out.value
            self.total += cap
        buf = (ctypes.c_char * cap).from_address(ptr)
        arr = np.frombuffer(buf, dtype=dtype, count=int(n))
        weakref.finalize(buf, self._give_back, cap, ptr)
        return arr

    def _give_back(self, cap, ptr):
        with self.lock:
            self.free.setdefault(cap, []).append(ptr)


class Engine(object):
    """One CUDA context + stream of this process: tables, one loaded contig batch, candidates."""

    def __init__(self, device=0):
        self.lib = load_library()
        handle = _vp()
        rc = self.lib.pasio_ctx_create(int(device), ctypes.byref(handle))
        if rc != OK:
            raise PasioDeviceError('pasio_b200: cannot create a device context (%s); the LogML path has no CPU '
                                   'fallback' % self.lib.pasio_last_error(None).decode())
        self.ctx = handle
        self.device = device
        self._params = None          # (alpha_is_int, alpha, beta, pen)
        self._tables = {}            # table id -> (computer object, uploaded length)
        self._scorer_source = None   # object providing the three computers
        self._penalty_spec = None    # penalty spec of the last use_scorer: what the next round applies
        self._penalties = None       # (penalty spec, length of the length table) set on the device, or None
        self._penalty_host = None    # (the same key, the host tables built for it): setting them again is an upload only
        self._loaded = None          # strong ref to the loaded counts array (identity cache)
        self._loaded_print = None    # its sampled content fingerprint
        self._cands_print = None
        self._loaded_offsets = None
        self._cands_obj = None       # array object the device candidates correspond to (identity cache)
        self._pool = _PinnedPool(self.lib)

    def close(self):
        if self.ctx:
            self.lib.pasio_ctx_destroy(self.ctx)
            self.ctx = None

    # -- errors ------------------------------------------------------------------------------
    def _check(self, rc):
        if rc == OK:
            return
        msg = self.lib.pasio_last_error(self.ctx).decode()
        if rc in (E_COUNTS, E_CANDIDATES):
            raise AssertionError(msg)         # the reference asserts (log_marginal_likelyhood.py:30-40)
        if rc == E_ARG:
            raise ValueError(msg)
        if rc == E_NOMEM:
            raise MemoryError(msg)
        raise PasioDeviceError('pasio_b200 error %d: %s' % (rc, msg))

    # -- scorer parameters and tables --------------------------------------------------------
    def use_scorer(self, source, penalties=None):
        """source has .alpha (int or float), .beta, .log_computer, .log_gamma_computer,
        .log_gamma_alpha_computer, .segment_creation_cost (ScorerFactory or a scorer).
        penalties: the penalty_spec (splitters/square_splitter.py) of a regularised window splitter, which the rounds
        then apply, or None; set or cleared on every call, so no later call inherits them.  Only the rounds read the
        penalties, so the device follows this setting when the next round starts (_sync_penalties): switching them off
        for scoring and on again for the next contig uploads nothing."""
        alpha = source.alpha
        is_int = isinstance(alpha, (int, np.integer)) and not isinstance(alpha, bool)
        params = (int(is_int), float(alpha), float(source.log_computer.shift), float(source.segment_creation_cost))
        if params != self._params:
            self._check(self.lib.pasio_set_params(self.ctx, *params))
            self._params = params
        comps = {TAB_LOG: source.log_computer, TAB_LGAMMA: source.log_gamma_computer,
                 TAB_LGAMMA_ALPHA: source.log_gamma_alpha_computer}
        for tid, comp in comps.items():
            have = self._tables.get(tid)
            if have is None or have[0] is not comp:
                self._upload_table(tid, comp, comp.cache_size)
        self._scorer_source = source
        self._penalty_spec = penalties

    def _sync_penalties(self):
        """Before a round: the device's penalty tables (pasio_set_penalties) are those of the last use_scorer.  The
        split-number table covers the largest fused window, the length table is as long as the log table (both are
        indexed by span)."""
        spec = self._penalty_spec
        want = None if spec is None else (spec, self._tables[TAB_LOG][1])
        if want == self._penalties:
            return
        self._penalties = None       # pasio_set_penalties switches both terms off first: so does this record
        if spec is None:
            self._check(self.lib.pasio_set_penalties(self.ctx, None, 0, 0.0, None, 0))
        else:
            from .splitters.square_splitter import penalty_tables
            from .splitters._fusion import MAX_FUSED_WINDOW_CANDIDATES
            if self._penalty_host is None or self._penalty_host[0] != want:      # (a long length table costs seconds to build)
                self._penalty_host = (want, penalty_tables(spec, want[1], MAX_FUSED_WINDOW_CANDIDATES))
            lp, sp, refund = self._penalty_host[1]
            self._check(self.lib.pasio_set_penalties(
                self.ctx, None if sp is None else _ptr(sp, ctypes.c_double), 0 if sp is None else len(sp), refund,
                None if lp is None else _ptr(lp, ctypes.c_double), 0 if lp is None else len(lp)))
        self._penalties = want

    def _upload_table(self, tid, comp, n):
        tab = comp.table(n)
        self._check(self.lib.pasio_table_upload(self.ctx, tid, _ptr(tab, ctypes.c_double), len(tab)))
        self._tables[tid] = (comp, len(tab))

    def _grow_tables(self):
        need = [_i64(0), _i64(0), _i64(0)]
        self._check(self.lib.pasio_table_need(self.ctx, *[ctypes.byref(x) for x in need]))
        for tid in (TAB_LOG, TAB_LGAMMA, TAB_LGAMMA_ALPHA):
            comp, have = self._tables[tid]
            if need[tid].value > have:
                self._upload_table(tid, comp, max(need[tid].value, int(have * 1.5)))
        if self._penalty_spec is not None:
            self._sync_penalties()                      # the length table follows the log table

    def _retry(self, fn):
        """Call fn() until it stops asking for longer tables."""
        while True:
            rc = fn()
            if rc != E_TABLE_TOO_SHORT:
                self._check(rc)
                return
            self._grow_tables()

    # -- contig ------------------------------------------------------------------------------
    @staticmethod
    def _fingerprint(arr):
        """cheap content check behind the identity caches: length, both ends and a strided sample of <= 4096 elements.
        (The reference recomputes from the array on every call; an array mutated in place between calls is re-uploaded
        if the sample sees the change -- callers that mutate loaded arrays should call invalidate().)"""
        n = len(arr)
        if n == 0:
            return (0,)
        step = max(1, n // 4096)
        return (n, int(arr[0]), int(arr[-1]), int(np.asarray(arr[::step]).sum()))

    def load(self, counts, offsets=None):
        """H2D + prefix scan + change-point bitmap; cached by array identity (+ a sampled content fingerprint)."""
        if (self._loaded is counts and offsets is None and self._loaded_offsets is None
                and self._loaded_print == self._fingerprint(counts)):
            return
        assert isinstance(counts, np.ndarray)
        assert counts.dtype == int
        assert len(counts) > 0
        c = np.ascontiguousarray(counts)
        self._loaded = None
        self._cands_obj = None
        if offsets is None:
            rc = self.lib.pasio_contig_load(self.ctx, _ptr(c, ctypes.c_int64), len(c), None, 1)
        else:
            off = np.ascontiguousarray(offsets, dtype=np.int64)
            rc = self.lib.pasio_contig_load(self.ctx, _ptr(c, ctypes.c_int64), len(c), _ptr(off, ctypes.c_int64),
                                            len(off) - 1)
        self._check(rc)
        self._loaded = counts
        self._loaded_print = self._fingerprint(counts)
        self._loaded_offsets = None if offsets is None else np.array(offsets, dtype=np.int64)

    def load_and_round(self, counts, window_size, window_shift, constraint, want_logfac=False):
        """load(counts) fused with the first round(): the upload overlaps the scan and the round (pasio_contig_load_round).
        want_logfac: the sequential log-factorial sums (LMM column) will be asked for -- they then follow the chunks of
        the upload on a side stream.  Returns (n_in, n_out, cells) of that round."""
        assert isinstance(counts, np.ndarray)
        assert counts.dtype == int
        assert len(counts) > 0
        c = np.ascontiguousarray(counts)
        self._loaded = None
        self._cands_obj = None
        n_in, n_out, cells = _i64(0), _i64(0), _i64(0)
        self.set_tuning('logfac_eager', 1 if want_logfac else 0)
        self._sync_penalties()
        try:
            rc = self.lib.pasio_contig_load_round(self.ctx, _ptr(c, ctypes.c_int64), len(c), window_size, window_shift,
                                                  CONSTRAINTS[constraint], ctypes.byref(n_in), ctypes.byref(n_out),
                                                  ctypes.byref(cells))
        finally:
            if want_logfac:
                self.set_tuning('logfac_eager', 0)
        if rc != E_TABLE_TOO_SHORT:
            self._check(rc)
        self._loaded = counts
        self._loaded_print = self._fingerprint(counts)
        self._loaded_offsets = None
        if rc == E_TABLE_TOO_SHORT:          # the contig is loaded; longer tables, then the round on its own
            self._grow_tables()
            return self.round(window_size, window_shift, constraint)
        return n_in.value, n_out.value, cells.value

    def load_device(self, device_ptr, n, owner=None, offsets=None):
        """counts already in HBM (int64[n] at device_ptr, e.g. a torch tensor's data_ptr()); no copy."""
        self._loaded = None
        self._cands_obj = None
        if offsets is None:
            rc = self.lib.pasio_contig_load_device(self.ctx, _vp(device_ptr), n, None, 1)
        else:
            off = np.ascontiguousarray(offsets, dtype=np.int64)
            rc = self.lib.pasio_contig_load_device(self.ctx, _vp(device_ptr), n, _ptr(off, ctypes.c_int64), len(off) - 1)
        self._check(rc)
        self._loaded = owner if owner is not None else object()   # keeps the device buffer alive
        self._loaded_offsets = None if offsets is None else np.array(offsets, dtype=np.int64)

    def invalidate(self):
        """Forget the identity caches (the next load / set_candidates re-uploads)."""
        self._loaded = None
        self._cands_obj = None

    def stream_handle(self):
        return self.lib.pasio_stream(self.ctx)

    def fp64_peak(self):
        v = ctypes.c_double(0)
        self._check(self.lib.pasio_fp64_peak(self.ctx, ctypes.byref(v)))
        return v.value

    def load_rle(self, starts, values, offsets=None):
        starts = np.ascontiguousarray(starts, dtype=np.int64)
        values = np.ascontiguousarray(values, dtype=np.int64)
        self._loaded = None
        self._cands_obj = None
        if offsets is None:
            rc = self.lib.pasio_contig_load_rle(self.ctx, _ptr(starts, ctypes.c_int64), _ptr(values, ctypes.c_int64),
                                                len(values), None, 1)
        else:
            off = np.ascontiguousarray(offsets, dtype=np.int64)
            rc = self.lib.pasio_contig_load_rle(self.ctx, _ptr(starts, ctypes.c_int64), _ptr(values, ctypes.c_int64),
                                                len(values), _ptr(off, ctypes.c_int64), len(off) - 1)
        self._check(rc)
        self._loaded = object()      # no host array corresponds to this load
        self._loaded_offsets = None if offsets is None else np.array(offsets, dtype=np.int64)

    def info(self):
        n, total, k = _i64(0), _i64(0), _i64(0)
        self._check(self.lib.pasio_contig_info(self.ctx, ctypes.byref(n), ctypes.byref(total), ctypes.byref(k)))
        return n.value, total.value, k.value

    # -- candidates --------------------------------------------------------------------------
    def set_candidates(self, cands):
        """cands: None (all positions) or an int64 array; cached by array identity."""
        if cands is None:
            self._check(self.lib.pasio_candidates_set(self.ctx, None, 0))
            self._cands_obj = None
            return
        if self._cands_obj is cands and self._cands_print == self._fingerprint(cands):
            return
        c = np.ascontiguousarray(cands, dtype=np.int64)
        self._cands_obj = None
        self._check(self.lib.pasio_candidates_set(self.ctx, _ptr(c, ctypes.c_int64), len(c)))
        self._cands_obj = cands
        self._cands_print = self._fingerprint(cands)

    def candidates(self):
        m = _i64(0)
        self._check(self.lib.pasio_candidates_count(self.ctx, ctypes.byref(m)))
        out = self._pool.empty(m.value, np.int64)
        self._check(self.lib.pasio_candidates_download(self.ctx, _ptr(out, ctypes.c_int64), len(out), None))
        self._cands_obj = out
        self._cands_print = self._fingerprint(out)
        return out

    def candidate_count(self):
        m = _i64(0)
        self._check(self.lib.pasio_candidates_count(self.ctx, ctypes.byref(m)))
        return m.value

    # -- kernels -----------------------------------------------------------------------------
    def filter_candidates(self, constraint):
        """NotZero / NotConstant reducer over the whole loaded contig; returns (n_in, n_out)"""
        a, b = _i64(0), _i64(0)
        self._cands_obj = None
        self._check(self.lib.pasio_filter_candidates(self.ctx, CONSTRAINTS[constraint], ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def round(self, window_size, window_shift, constraint):
        n_in, n_out, cells = _i64(0), _i64(0), _i64(0)
        self._cands_obj = None
        self._sync_penalties()
        self._retry(lambda: self.lib.pasio_round(self.ctx, window_size, window_shift, CONSTRAINTS[constraint],
                                                 ctypes.byref(n_in), ctypes.byref(n_out), ctypes.byref(cells)))
        return n_in.value, n_out.value, cells.value

    def set_tuning(self, key, value):
        """kernel variant switches (TUNE); results never depend on them"""
        self._check(self.lib.pasio_set_tuning(self.ctx, TUNE[key], int(value)))

    def upload_stats(self):
        """bytes the last load_and_round put on the PCIe link (half of counts.nbytes when the counts went up as int32)"""
        b = _i64(0)
        self._check(self.lib.pasio_upload_stats(self.ctx, ctypes.byref(b)))
        return b.value

    def round_stats(self):
        """(algorithmic cells, cells skipped by the exact bound) of the most recent round"""
        a, b = _i64(0), _i64(0)
        self._check(self.lib.pasio_round_stats(self.ctx, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def round_certify_stats(self):
        """(windows proven to keep every candidate, windows whose check failed, rows those checks still proved)
        of the most recent round"""
        a, b, c = _i64(0), _i64(0), _i64(0)
        self._check(self.lib.pasio_round_certify_stats(self.ctx, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return a.value, b.value, c.value

    def rounds(self, window_size, window_shift, constraint, num_rounds=None, first=None):
        """RoundReducer loop on the device.  Returns (sizes before each round run, final count, cells).
        first: (n_in, n_out, cells) of a first round that load_and_round already ran."""
        n, _, _ = self.info()
        limit = max(1, n if num_rounds is None else num_rounds)   # round_reducer.py:11-15
        self._cands_obj = None
        sizes, cells_total = [], 0
        if first is not None:
            sizes.append(first[0])
            cells_total += first[2]
            limit -= 1
            if first[0] == first[1] or limit == 0:
                return sizes, self.candidate_count(), cells_total
        while limit > 0:
            done, n_out, cells = _i64(0), _i64(0), _i64(0)
            buf = np.zeros(64, dtype=np.int64)
            step = min(limit, 64)
            self._sync_penalties()
            rc = self.lib.pasio_rounds(self.ctx, window_size, window_shift, CONSTRAINTS[constraint], step,
                                       ctypes.byref(done), ctypes.byref(n_out), ctypes.byref(cells),
                                       _ptr(buf, ctypes.c_int64), len(buf))
            sizes.extend(buf[:done.value].tolist())
            cells_total += cells.value
            limit -= done.value
            if rc == E_TABLE_TOO_SHORT:
                self._grow_tables()
                continue
            self._check(rc)
            if done.value < step or (done.value > 0 and sizes[-1] == n_out.value):
                break       # fixed point reached inside the library
        return sizes, self.candidate_count(), cells_total

    def _check_exact_limits(self):
        """The whole-contig DP indexes the lgamma table with the contig's TOTAL count (+ alpha) in 32 bits and needs the
        table up to there: refuse clearly before any multi-GB table is built.  (The default rounds pipeline has no such
        limit: its tables only reach the largest count inside one window.)"""
        n, total, _ = self.info()
        if not exact_total_fits(total, self._params[1] if self._params else 0):
            raise PasioDeviceError('pasio_b200: the exact SquareSplitter DP over a whole contig needs the total count (%d) below '
                                   '2^31; use the default `rounds` algorithm for deep-coverage contigs' % total)

    def square_split(self, want_arrays=False):
        """Exact DP over the current candidates; they are replaced by the splits."""
        self._check_exact_limits()
        m = self.candidate_count()
        splits = np.empty(m, dtype=np.int64)
        n_splits, score = _i64(0), ctypes.c_double(0.0)
        P = np.empty(m) if want_arrays else None
        prev = np.empty(m, dtype=np.int64) if want_arrays else None
        self._cands_obj = None
        self._retry(lambda: self.lib.pasio_square_split(
            self.ctx, _ptr(splits, ctypes.c_int64), m, ctypes.byref(n_splits), ctypes.byref(score),
            _ptr(P, ctypes.c_double) if want_arrays else None,
            _ptr(prev, ctypes.c_int64) if want_arrays else None))
        out = splits[:n_splits.value].copy()
        self._cands_obj = out
        self._cands_print = self._fingerprint(out)
        if want_arrays:
            return np.float64(score.value), out, P, prev
        return np.float64(score.value), out

    def square_split_batch(self):
        """square_split of every contig of the loaded batch over its own slice of the current candidates; they are
        replaced by the union of the splits.  A contig whose own total count is too large raises PasioDeviceError."""
        n_out, cells, skipped = _i64(0), _i64(0), _i64(0)
        self._cands_obj = None
        self._retry(lambda: self.lib.pasio_square_split_batch(self.ctx, ctypes.byref(n_out), ctypes.byref(cells),
                                                              ctypes.byref(skipped)))

    def square_split_regularized(self, length_penalty=None, split_number_penalty=None, first_column_refund=0.0,
                                 want_arrays=False):
        """split_with_normalizations over the current candidates on the device; penalty tables as in include/pasio_b200.h.
        want_arrays: also return the prefix scores P and the arg-maxes prev, as square_split does."""
        self._check_exact_limits()
        m = self.candidate_count()
        splits = np.empty(m, dtype=np.int64)
        n_splits, score = _i64(0), ctypes.c_double(0.0)
        lp = None if length_penalty is None else np.ascontiguousarray(length_penalty, dtype=np.float64)
        sp = None if split_number_penalty is None else np.ascontiguousarray(split_number_penalty, dtype=np.float64)
        P = np.empty(m) if want_arrays else None
        prev = np.empty(m, dtype=np.int64) if want_arrays else None
        self._cands_obj = None
        self._retry(lambda: self.lib.pasio_square_split_regularized(
            self.ctx, None if lp is None else _ptr(lp, ctypes.c_double), 0 if lp is None else len(lp),
            None if sp is None else _ptr(sp, ctypes.c_double), 0 if sp is None else len(sp), float(first_column_refund),
            _ptr(splits, ctypes.c_int64), m, ctypes.byref(n_splits), ctypes.byref(score),
            _ptr(P, ctypes.c_double) if want_arrays else None,
            _ptr(prev, ctypes.c_int64) if want_arrays else None))
        out = splits[:n_splits.value].copy()
        self._cands_obj = out
        self._cands_print = self._fingerprint(out)
        if want_arrays:
            return np.float64(score.value), out, P, prev
        return np.float64(score.value), out

    def suffix_scores(self, stop):
        out = np.empty(stop)
        if stop > 0:
            self._retry(lambda: self.lib.pasio_suffix_scores(self.ctx, stop, _ptr(out, ctypes.c_double)))
        return out

    def cumsum_at_candidates(self):
        m = self.candidate_count()
        out = np.empty(m, dtype=np.int64)
        self._check(self.lib.pasio_cumsum_at(self.ctx, None, m, _ptr(out, ctypes.c_int64)))
        return out

    def segment_scores(self, scores=True, counts=False, means=False, logfac=False):
        m = self.candidate_count()
        nseg = m - 1
        s = self._pool.empty(nseg, np.float64) if scores else None
        c = self._pool.empty(nseg, np.int64) if counts else None
        mu = self._pool.empty(nseg, np.float64) if means else None
        lf = self._pool.empty(m, np.float64) if logfac else None
        nout = _i64(0)
        self._retry(lambda: self.lib.pasio_segment_scores(
            self.ctx, _ptr(s, ctypes.c_double) if scores else None, _ptr(c, ctypes.c_int64) if counts else None,
            _ptr(mu, ctypes.c_double) if means else None, _ptr(lf, ctypes.c_double) if logfac else None,
            max(nseg, m if logfac else 0), ctypes.byref(nout)))
        return s, c, mu, lf

    def segment_scores_sum(self):
        """np.sum(scores) of the current segments, on the device in numpy's pairwise order (same float64 result)"""
        total = ctypes.c_double(0.0)
        self._retry(lambda: self.lib.pasio_segment_scores_sum(self.ctx, ctypes.byref(total)))
        return np.float64(total.value)

    def logfac_prefetch(self):
        """start the sequential log-factorial sums of the loaded batch beside whatever runs next (segment_lmm uses them)"""
        self._check(self.lib.pasio_logfac_prefetch(self.ctx))

    def segment_lmm(self):
        """(log_marginal_likelyhoods per segment, total_sum_logfac), formed on the device"""
        nseg = self.candidate_count() - 1
        out = self._pool.empty(nseg, np.float64)
        total = ctypes.c_double(0.0)
        self._retry(lambda: self.lib.pasio_segment_lmm(self.ctx, _ptr(out, ctypes.c_double), nseg, ctypes.byref(total)))
        return out, total.value

    # -- timing ------------------------------------------------------------------------------
    def timing_reset(self, enable=True):
        self._check(self.lib.pasio_timing_reset(self.ctx, int(enable)))

    def timing(self):
        out = {}
        for k, name in enumerate(TIMING_FAMILIES):
            ms, n = ctypes.c_double(0), _i64(0)
            self._check(self.lib.pasio_timing_get(self.ctx, k, ctypes.byref(ms), ctypes.byref(n)))
            out[name] = (ms.value, n.value)
        return out


def parse_bedgraph_text(data, front=0, length=None):
    """data: bytes of a bedgraph file (or a bytearray, of which the first `length` bytes are parsed in place).  Returns dict of arrays: starts, stops, counts (int64), name_off, name_len,
    new_chrom, plus n_float (counts that needed int(float(x))).  front: leave that many unfilled slots before the parsed
    lines in every array (the streaming reader puts the lines of a contig that began in the previous piece there, instead of
    concatenating whole arrays piece after piece); name_off / name_len / new_chrom of those slots are the caller's too."""
    lib = load_library()
    nbytes = len(data) if length is None else int(length)
    if isinstance(data, bytearray):
        data = (ctypes.c_char * len(data)).from_buffer(data) if len(data) else None
    cap = lib.pasio_bedgraph_count_lines(data, nbytes)
    starts = np.empty(front + cap, dtype=np.int64)
    stops = np.empty(front + cap, dtype=np.int64)
    counts = np.empty(front + cap, dtype=np.int64)
    name_off = np.empty(front + cap, dtype=np.int64)
    name_len = np.empty(front + cap, dtype=np.int32)
    new_chrom = np.empty(front + cap, dtype=np.uint8)
    n, nfloat = _i64(0), _i64(0)
    rc = lib.pasio_bedgraph_parse(data, nbytes, cap, _ptr(starts[front:], ctypes.c_int64), _ptr(stops[front:], ctypes.c_int64),
                                  _ptr(counts[front:], ctypes.c_int64), _ptr(name_off[front:], ctypes.c_int64),
                                  _ptr(name_len[front:], ctypes.c_int32), _ptr(new_chrom[front:], ctypes.c_uint8),
                                  ctypes.byref(n), ctypes.byref(nfloat))
    if rc != OK:
        raise ValueError('malformed bedgraph line %d (need: chrom start stop count)' % (n.value + 1))
    k = front + n.value
    return dict(starts=starts[:k], stops=stops[:k], counts=counts[:k], name_off=name_off[:k], name_len=name_len[:k],
                new_chrom=new_chrom[:k], n_float=nfloat.value)


def bedgraph_runs(rec, split_at_gaps):
    """parsed intervals (parse_bedgraph_text) -> (run_len, run_val, group_line, group_run): contigs as run lengths"""
    lib = load_library()
    n = len(rec['starts'])
    run_len = np.empty(2 * n, dtype=np.int64)
    run_val = np.empty(2 * n, dtype=np.int64)
    group_line = np.empty(n + 1, dtype=np.int64)
    group_run = np.empty(n + 1, dtype=np.int64)
    n_runs = _i64(0)
    g = lib.pasio_bedgraph_runs(_ptr(rec['starts'], ctypes.c_int64), _ptr(rec['stops'], ctypes.c_int64),
                                _ptr(rec['counts'], ctypes.c_int64), _ptr(rec['new_chrom'], ctypes.c_uint8), n,
                                int(bool(split_at_gaps)), _ptr(run_len, ctypes.c_int64), _ptr(run_val, ctypes.c_int64),
                                _ptr(group_line, ctypes.c_int64), _ptr(group_run, ctypes.c_int64), ctypes.byref(n_runs))
    return run_len[:n_runs.value], run_val[:n_runs.value], group_line[:g], group_run[:g + 1]


def format_segments(chrom, offset, splits, means, lmm, mode):
    """bytes of the output lines of one contig (mode 0 bedgraph, 1 bed, 2 bedgraph+length+LMM)"""
    lib = load_library()
    splits = np.ascontiguousarray(splits, dtype=np.int64)
    name = chrom.encode()
    pieces = []
    step = 1 << 22
    for lo in range(0, len(splits) - 1, step):
        hi = min(lo + step, len(splits) - 1)
        sub = splits[lo:hi + 1]
        m = np.ascontiguousarray(means[lo:hi]) if means is not None else None
        l = np.ascontiguousarray(lmm[lo:hi]) if lmm is not None else None
        cap = (hi - lo) * (len(name) + 56) + 1024
        while True:
            buf = np.empty(cap, dtype=np.uint8)                # not zero-filled
            w = lib.pasio_format_segments(name, int(offset), _ptr(sub, ctypes.c_int64), len(sub),
                                          _ptr(m, ctypes.c_double) if m is not None else None,
                                          _ptr(l, ctypes.c_double) if l is not None else None, mode,
                                          buf.ctypes.data_as(ctypes.c_char_p), cap)
            if w >= 0:
                pieces.append(buf[:w].tobytes())
                break
            cap = -w
    return b''.join(pieces)


def format_segments_batch(chroms, shifts, first_split, splits, means, lmm, mode):
    """format_segments for a batch segmented as one super-contig: chroms[c], shifts[c] (added to the positions) and
    first_split[c] (index of the contig's first split point; len(chroms) + 1 entries) per contig"""
    lib = load_library()
    names = [c.encode() for c in chroms]
    blob = b''.join(names)
    name_off = np.concatenate([[0], np.cumsum([len(x) for x in names])]).astype(np.int64)
    shifts = np.ascontiguousarray(shifts, dtype=np.int64)
    first_split = np.ascontiguousarray(first_split, dtype=np.int64)
    splits = np.ascontiguousarray(splits, dtype=np.int64)
    m = np.ascontiguousarray(means) if means is not None else None
    l = np.ascontiguousarray(lmm) if lmm is not None else None
    nseg = int(first_split[-1] - first_split[0])
    cap = nseg * (max(len(x) for x in names) + 56) + 1024
    while True:
        buf = np.empty(cap, dtype=np.uint8)
        w = lib.pasio_format_segments_batch(blob, _ptr(name_off, ctypes.c_int64), _ptr(shifts, ctypes.c_int64),
                                            _ptr(first_split, ctypes.c_int64), len(names), _ptr(splits, ctypes.c_int64),
                                            _ptr(m, ctypes.c_double) if m is not None else None,
                                            _ptr(l, ctypes.c_double) if l is not None else None, mode,
                                            buf.ctypes.data_as(ctypes.c_char_p), cap)
        if w >= 0:
            return buf[:w].tobytes()
        cap = -w


_engine = None
_engine_lock = threading.Lock()


def default_device():
    if 'PASIO_B200_DEVICE' in os.environ:
        return int(os.environ['PASIO_B200_DEVICE'])
    if 'LOCAL_RANK' in os.environ:
        return int(os.environ['LOCAL_RANK'])
    return 0


def engine():
    """The process-wide Engine (one process per GPU).  Raises if there is no usable device."""
    global _engine
    with _engine_lock:
        if _engine is None:
            _engine = Engine(default_device())
    return _engine


def reset_engine():
    global _engine
    with _engine_lock:
        if _engine is not None:
            _engine.close()
        _engine = None
