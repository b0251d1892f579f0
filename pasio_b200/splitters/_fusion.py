"""Recognise the canonical splitter graphs that run fused on the device (SURVEY 8b).

    base   := SquareSplitter(ScorerFactory, no regularisation or the CLI's penalty functions)
            | ReducerCombiner(NotConstantReducer | NotZeroReducer, SquareSplitter(...))
    window := SlidingWindowReducer(SlidingWindow, base)
    rounds := RoundReducer(window, num_rounds)

Only exact types match (a user subclass may override anything), and only factories that are
pasio_b200 ScorerFactory instances (a lambda factory could return anything per call; those go
window by window through the objects and still reach the GPU inside SquareSplitter.split).
A regularised base (penalty functions identity / revlog, square_splitter.penalty_spec) runs in the
regularised window kernels (csrc/window_dp_reg.cu); its plans carry the penalty spec as one more
element at the end of the tuple, so the tuples of unregularised plans are unchanged.
"""
from ..log_marginal_likelyhood import ScorerFactory

# one window is one CTA: its candidates must fit shared memory (csrc/window_dp.cu, window_dp_max_candidates).
# Larger windows are not fused: they go window by window through the objects, i.e. through the exact-DP kernel.
MAX_FUSED_WINDOW_CANDIDATES = 8192
# the same for the regularised window kernel (csrc/window_dp_reg.cu, RW_MAX_CANDIDATES): per candidate it also keeps
# the split number and its penalty
MAX_FUSED_REG_WINDOW_CANDIDATES = 7168


def base_plan(reducer):
    """-> (factory, constraint) or, regularised, (factory, constraint, penalty spec); or None"""
    from .square_splitter import SquareSplitter, penalty_spec
    from .constants_reducer import NotConstantReducer, NotZeroReducer
    from .reducer_combiner import ReducerCombiner
    constraint = 'none'
    if type(reducer) is ReducerCombiner and len(reducer.reducers) == 2:
        head, reducer = reducer.reducers
        if type(head) is NotConstantReducer:
            constraint = 'constants'
        elif type(head) is NotZeroReducer:
            constraint = 'zeros'
        else:
            return None
    if type(reducer) is not SquareSplitter or type(reducer.scorer_factory) is not ScorerFactory:
        return None
    if not reducer.is_regularized:
        return reducer.scorer_factory, constraint
    spec = penalty_spec(reducer)
    if spec is None:
        return None
    return reducer.scorer_factory, constraint, spec


def window_plan(reducer):
    """-> (factory, window_size, window_shift, constraint[, penalty spec]) or None"""
    from .sliding_window_reducer import SlidingWindowReducer
    from ..dto.sliding_window import SlidingWindow
    if type(reducer) is not SlidingWindowReducer or type(reducer.sliding_window) is not SlidingWindow:
        return None
    base = base_plan(reducer.base_reducer)
    if base is None:
        return None
    size, shift = reducer.sliding_window.window_size, reducer.sliding_window.window_shift
    if not (isinstance(size, int) and isinstance(shift, int) and size >= 1 and shift >= 1):
        return None
    if size + 1 > (MAX_FUSED_WINDOW_CANDIDATES if len(base) == 2 else MAX_FUSED_REG_WINDOW_CANDIDATES):
        return None
    return (base[0], size, shift, base[1]) + base[2:]


def rounds_plan(reducer):
    """-> (factory, window_size, window_shift, constraint, num_rounds[, penalty spec]) or None"""
    from .round_reducer import RoundReducer
    if type(reducer) is not RoundReducer:
        return None
    win = window_plan(reducer.base_reducer)
    if win is None:
        return None
    return win[:4] + (reducer.num_rounds,) + win[4:]



def pipeline_plan(splitter):
    """Whole-contig plans used by segments_with_scores: list of device steps + the final factory.

    -> dict(steps=[('rounds'|'window'|'exact', args...)], factory=ScorerFactory, final='nop'|'exact') or None"""
    from .square_splitter import SquareSplitter
    from .nop_splitter import NopSplitter
    from .reducer_combiner import ReducerCombiner
    if type(splitter) is SquareSplitter:
        if splitter.is_regularized or type(splitter.scorer_factory) is not ScorerFactory:
            return None
        return dict(steps=[], factory=splitter.scorer_factory, final='exact')
    if type(splitter) is not ReducerCombiner or len(splitter.reducers) < 1:
        return None
    steps = []
    for reducer in splitter.reducers[:-1]:
        plan = rounds_plan(reducer)
        if plan is not None and len(plan) == 5:
            steps.append(('rounds',) + plan)
            continue
        plan = window_plan(reducer)
        if plan is not None and len(plan) == 4:
            steps.append(('window',) + plan)
            continue
        return None
    last = splitter.reducers[-1]
    if type(last) is NopSplitter and type(last.scorer_factory) is ScorerFactory:
        return dict(steps=steps, factory=last.scorer_factory, final='nop')
    if type(last) is SquareSplitter and not last.is_regularized and type(last.scorer_factory) is ScorerFactory:
        return dict(steps=steps, factory=last.scorer_factory, final='exact')
    return None


def device_plan(splitter):
    """pipeline_plan(splitter), or for the `rounds` graph with a regularised window splitter
    (ReducerCombiner(RoundReducer(...), NopSplitter)) the same kind of whole-contig plan whose rounds step carries the
    penalty spec; None for everything else."""
    plan = pipeline_plan(splitter)
    if plan is not None:
        return plan
    from .nop_splitter import NopSplitter
    from .reducer_combiner import ReducerCombiner
    if type(splitter) is not ReducerCombiner or len(splitter.reducers) != 2:
        return None
    head, last = splitter.reducers
    rounds = rounds_plan(head)
    if rounds is None or type(last) is not NopSplitter or type(last.scorer_factory) is not ScorerFactory:
        return None
    return dict(steps=[('rounds',) + rounds], factory=last.scorer_factory, final='nop')
