"""SlidingWindowReducer: one round of window-wise candidate reduction.

Interface of /root/reference/src/pasio/splitters/sliding_window_reducer.py:5-29.  When the base
reducer is one of the canonical graphs (_fusion.window_plan) the whole round is ONE launch with
one CTA per window (pasio_round, csrc/window_dp.cu); otherwise each window goes through the
base reducer object exactly as in the reference.
"""
import numpy as np

from .. import _native
from ..logging import logger, logging_filter
from . import _fusion


class SlidingWindowReducer(object):
    def __init__(self, sliding_window, base_reducer):
        self.sliding_window = sliding_window
        self.base_reducer = base_reducer

    def reduce_candidates_in_window(self, counts, candidates_in_window):
        start, stop = candidates_in_window[0], candidates_in_window[-1]
        logging_filter.put_to_context('window', '[%d, %d)' % (start, stop))
        # the base reducer sees the window as a contig of its own: sliced counts, re-based candidates
        local = self.base_reducer.reduce_candidate_list(counts[start:stop], candidates_in_window - start)
        return local + start

    def reduce_candidate_list(self, counts, split_candidates):
        plan = _fusion.window_plan(self)
        # (a candidate list without both ends is legal in the reference -- 0 and len(counts) are simply added to the
        # result -- but not for the fused device loop: those lists take the object route below)
        if plan is not None and isinstance(counts, np.ndarray) and _has_both_ends(split_candidates, counts):
            factory, size, shift, constraint = plan[:4]
            eng = _native.engine()
            eng.use_scorer(factory, plan[4] if len(plan) > 4 else None)
            eng.load(counts)
            _set_candidates(eng, counts, split_candidates)
            n_in, n_out, _ = eng.round(size, shift, constraint)
            logger.info('Sliding: %d --> %d split-points' % (n_in, n_out))
            return eng.candidates()
        survivors = set([0, len(counts)])
        for (candidates_in_window, completion) in self.sliding_window.windows(split_candidates):
            reduced = self.reduce_candidates_in_window(counts, candidates_in_window)
            survivors.update(reduced)
            logger.info('Sliding (completion: %.2f %%): %d --> %d split-points' % (
                100 * completion, len(candidates_in_window), len(reduced)))
        logging_filter.remove_from_context('window')
        return np.array(sorted(survivors))


def _has_both_ends(split_candidates, counts):
    return len(split_candidates) >= 2 and split_candidates[0] == 0 and split_candidates[-1] == len(counts)


def _set_candidates(eng, counts, split_candidates):
    from ..log_marginal_likelyhood import assert_correct_split_candidates, _is_all_positions
    assert_correct_split_candidates(split_candidates, counts)
    if _is_all_positions(split_candidates, len(counts)):
        eng.set_candidates(None)
    else:
        eng.set_candidates(split_candidates)
