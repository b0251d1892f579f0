"""RoundReducer: repeat a reducer until no candidate is removed.

Interface of /root/reference/src/pasio/splitters/round_reducer.py:5-31.  With a fusable
SlidingWindowReducer underneath, the loop runs on the device (pasio_rounds): candidates stay in
HBM between rounds and only two scalars per round cross PCIe.
"""
import numpy as np

from .. import _native
from ..logging import logger, logging_filter
from . import _fusion
from .sliding_window_reducer import _set_candidates, _has_both_ends


class RoundReducer(object):
    def __init__(self, base_reducer, num_rounds=None):
        self.base_reducer = base_reducer
        self.num_rounds = num_rounds

    def reduce_candidate_list(self, counts, split_candidates):
        plan = _fusion.rounds_plan(self)
        # (a candidate list without both ends is legal in the reference -- 0 and len(counts) are simply added to the
        # result -- but not for the fused device loop: those lists take the object route below)
        if plan is not None and isinstance(counts, np.ndarray) and _has_both_ends(split_candidates, counts):
            factory, size, shift, constraint, num_rounds = plan[:5]
            eng = _native.engine()
            eng.use_scorer(factory, plan[5] if len(plan) > 5 else None)
            eng.load(counts)
            _set_candidates(eng, counts, split_candidates)
            sizes, final, _ = eng.rounds(size, shift, constraint, num_rounds)
            _log_rounds(sizes, final)
            return eng.candidates()

        num_rounds = len(counts) if self.num_rounds is None else self.num_rounds
        num_rounds = max(1, num_rounds)
        for round_ in range(1, num_rounds + 1):
            logging_filter.put_to_context('round', round_)
            logger.info('Starting round, num_candidates %d' % len(split_candidates))
            new_split_candidates = self.base_reducer.reduce_candidate_list(counts, split_candidates)
            if np.array_equal(new_split_candidates, split_candidates):
                logger.info('No split points removed. Finishing round')
                logging_filter.remove_from_context('round')
                return new_split_candidates
            assert len(new_split_candidates) < len(split_candidates)
            logger.info('Finishing round, num_candidates %d' % len(new_split_candidates))
            split_candidates = new_split_candidates
        logging_filter.remove_from_context('round')
        logger.info('Splitting finished in %d rounds. Number of split points %d' % (round_, len(new_split_candidates)))
        return new_split_candidates


def _log_rounds(sizes, final):
    after = sizes[1:] + [final]
    for k, (a, b) in enumerate(zip(sizes, after), start=1):
        logging_filter.put_to_context('round', k)
        logger.info('Starting round, num_candidates %d' % a)
        if a == b:
            logger.info('No split points removed. Finishing round')
        else:
            logger.info('Finishing round, num_candidates %d' % b)
    logging_filter.remove_from_context('round')
