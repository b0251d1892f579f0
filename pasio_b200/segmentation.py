"""Per-contig driver (reference: /root/reference/src/pasio/segmentation.py:5-20).

For the canonical splitter graphs the whole contig stays on the device: counts are uploaded
once, candidates start as the implicit "all positions" list (the reference materialises
np.arange(n+1), 2 GB for chr1), rounds / exact DP run back to back, and only the final splits
and per-segment outputs are copied back.  Any other splitter object is driven through the
reference's own protocol.
"""
import os

import numpy as np

from . import _native
from .logging import logger
from .dto.intervals import ScoredInterval
from .splitters import _fusion


def _step_penalties(step):
    """the penalty spec a regularised 'rounds' / 'window' step carries after its arguments (_fusion), or None"""
    n = 6 if step[0] == 'rounds' else 5
    return step[n] if len(step) > n else None


def _run_device_pipeline(eng, plan, first=None):
    """Run the device steps of a pipeline plan on the loaded batch.  Returns (score or None, splits).
    first: result of the first step's first round when the load already ran it (Engine.load_and_round)."""
    score = None
    for k, step in enumerate(plan['steps']):
        if k == 0 and first is not None and step[0] == 'window':
            continue
        if step[0] == 'rounds':
            _, factory, size, shift, constraint, num_rounds = step[:6]
            eng.use_scorer(factory, _step_penalties(step))
            sizes, final, _ = eng.rounds(size, shift, constraint, num_rounds, first=first if k == 0 else None)
            from .splitters.round_reducer import _log_rounds
            _log_rounds(sizes, final)
        else:
            _, factory, size, shift, constraint = step[:5]
            eng.use_scorer(factory, _step_penalties(step))
            eng.round(size, shift, constraint)
    eng.use_scorer(plan['factory'])
    if plan['final'] == 'exact':
        score, _ = eng.square_split()
    return score


def run_loaded_pipeline(eng, plan, want_lmm=True, first=None):
    """The device pipeline over whatever contig the engine has loaded (dense, RLE or device-resident).
    -> (score, splits, mean_counts, log_marginal_likelyhoods or None, sum_logfac or None)"""
    if first is None:
        eng.set_candidates(None)                  # split_candidates = all positions (reference :8)
    score = _run_device_pipeline(eng, plan, first)
    splits = eng.candidates()
    scores, _, means, _ = eng.segment_scores(scores=True, means=True)
    if plan['final'] == 'nop':
        score = eng.segment_scores_sum()          # NopSplitter.split (nop_splitter.py:15-18): np.sum(scores), numpy's order
    lmm, sum_logfac = eng.segment_lmm() if want_lmm else (None, None)
    return score, splits, means, lmm, sum_logfac


def segment_on_device(counts, plan, want_lmm=True):
    """-> (score, splits, mean_counts, log_marginal_likelyhoods or None, sum_logfac or None)"""
    eng = _native.engine()
    steps = plan['steps']
    if (steps and steps[0][0] in ('rounds', 'window') and isinstance(counts, np.ndarray)
            and not os.environ.get('PASIO_B200_NO_FUSED_LOAD')):      # (switch for A/B measurements)
        # the first round always starts from all positions: run it while the counts are still going up
        _, factory, size, shift, constraint = steps[0][:5]
        eng.use_scorer(factory, _step_penalties(steps[0]))
        first = eng.load_and_round(counts, size, shift, constraint, want_logfac=want_lmm)
        if want_lmm:
            eng.logfac_prefetch()                 # the sequential log-factorial sums run beside the remaining rounds
        return run_loaded_pipeline(eng, plan, want_lmm, first=first)
    eng.use_scorer(plan['factory'])
    eng.load(counts)
    if want_lmm:
        eng.logfac_prefetch()
    return run_loaded_pipeline(eng, plan, want_lmm)


def segments_with_scores(profile, splitter):
    logger.info('Starting splitting profile of length %d' % len(profile))
    counts = np.array(profile)
    plan = _fusion.device_plan(splitter)
    if plan is not None:
        score, splits, means, lmm, sum_logfac = segment_on_device(counts, plan)
    else:
        split_candidates = np.arange(len(counts) + 1)
        score, splits = splitter.split(counts, split_candidates)
        scorer = splitter.scorer(counts, splits)
        sum_logfac = scorer.total_sum_logfac()
        means = scorer.mean_counts()
        lmm = scorer.log_marginal_likelyhoods()
    logger.info('Splitting finished, score %f, number of splits %d. '
                'Log likelyhood: %f.' % (score, len(splits), score - sum_logfac))
    logger.info('Scores calculated')
    for (start, stop, mean_count, log_marginal_likelyhood) in zip(splits[:-1], splits[1:], means, lmm):
        yield ScoredInterval(start, stop, mean_count, log_marginal_likelyhood)
