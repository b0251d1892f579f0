"""SquareSplitter: exact optimal-partition DP over split candidates.

Interface of the reference's /root/reference/src/pasio/splitters/square_splitter.py:4-109
(constructor, `scorer`, `reduce_candidate_list`, `split`, `split_with_normalizations`,
`split_without_normalizations`, static `collect_split_points`).

Dispatch is on the scorer OBJECT the factory returns (the reference's tests pass lambda
factories): a pasio_b200 LogMarginalLikelyhoodComputer without regularisation runs the whole DP
on the GPU (pasio_square_split, kernels in csrc/exact_dp.cu).  Any other scorer is a
user-supplied Python object whose `all_suffixes_self_score` cannot run on a device; for those,
and for regularisation callables, the DP recurrence is driven from the host, row by row,
through the scorer protocol (this is API compatibility for foreign scorers, not a fallback of
the LogML path).
"""
import numpy as np

from ..log_marginal_likelyhood import LogMarginalLikelyhoodComputer


def _identity(x):
    return x


def _revlog(x):
    """the `revlog` length penalty of the CLI: 1 / log(1 + l) (reference default_splitters.py:38, cli.py:49-53)"""
    return 1 / np.log(x + 1)


def penalty_spec(splitter):
    """(length multiplier, length function, split-number multiplier, split-number function) of a regularised
    SquareSplitter whose penalty functions are the two the reference's CLI offers (identity and 1/log(1+l),
    default_splitters.py:36-39) -- those are element-wise, so their values can be tabulated; None otherwise (an
    arbitrary callable keeps the host route)."""
    builtin = (_identity, _revlog)
    if not splitter.is_regularized:
        return None
    if splitter.length_regularization_function not in builtin or splitter.split_number_regularization_function not in builtin:
        return None
    return (splitter.length_regularization_multiplier, splitter.length_regularization_function,
            splitter.split_number_regularization_multiplier, splitter.split_number_regularization_function)


def penalty_tables(spec, n_length, n_split_number):
    """Tables of the device DPs for a penalty_spec, evaluated with the reference's own expressions
    (square_splitter.py:46-54), element by element the doubles the reference subtracts:
    length_penalty[len] = multiplier * function(len) for len < n_length, split_number_penalty[k] = multiplier *
    function(k + 1) for k < n_split_number (num_splits is a float array, :40), first_column_refund = multiplier * function(1).
    -> (length_penalty or None, split_number_penalty or None, first_column_refund)"""
    len_mult, len_fn, num_mult, num_fn = spec
    length_penalty = split_number_penalty = None
    refund = 0.0
    with np.errstate(all='ignore'):
        if len_mult != 0:
            length_penalty = np.asarray(len_mult * len_fn(np.arange(n_length)), dtype=np.float64)
        if num_mult != 0:
            num_splits = np.arange(n_split_number, dtype=np.float64)
            split_number_penalty = np.asarray(num_mult * num_fn(num_splits + 1), dtype=np.float64)
            refund = float(num_mult * num_fn(1))
    return length_penalty, split_number_penalty, refund


class SquareSplitter(object):
    def __init__(self, scorer_factory,
                 length_regularization_multiplier=0,
                 length_regularization_function=_identity,
                 split_number_regularization_multiplier=0,
                 split_number_regularization_function=_identity):
        self.scorer_factory = scorer_factory
        self.length_regularization_multiplier = length_regularization_multiplier
        self.split_number_regularization_multiplier = split_number_regularization_multiplier
        self.length_regularization_function = length_regularization_function
        self.split_number_regularization_function = split_number_regularization_function

    @property
    def is_regularized(self):
        return not (self.split_number_regularization_multiplier == 0 and self.length_regularization_multiplier == 0)

    def scorer(self, counts, split_candidates):
        return self.scorer_factory(counts, split_candidates)

    def reduce_candidate_list(self, counts, split_candidates):
        return self.split(counts, split_candidates)[1]

    def split(self, counts, split_candidates):
        if self.is_regularized:
            return self.split_with_normalizations(counts, split_candidates)
        return self.split_without_normalizations(counts, split_candidates)

    def split_without_normalizations(self, counts, split_candidates):
        score_computer = self.scorer(counts, split_candidates)
        if isinstance(score_computer, LogMarginalLikelyhoodComputer):
            return score_computer._square_split()                      # device DP
        return self._scorer_protocol_dp(score_computer, split_candidates, regularized=False)

    def split_with_normalizations(self, counts, split_candidates):
        score_computer = self.scorer(counts, split_candidates)
        tables = self._device_penalty_tables(score_computer, counts, split_candidates)
        if tables is not None:
            return score_computer._square_split_regularized(*tables)       # device DP (csrc/regularized_dp.cu)
        return self._scorer_protocol_dp(score_computer, split_candidates, regularized=True)

    def _device_penalty_tables(self, score_computer, counts, split_candidates):
        """Penalty tables for the device version of the regularised DP, or None when it does not apply: the scorer must be
        a pasio_b200 LogML computer and the penalty functions the two the reference's CLI offers (penalty_spec)."""
        spec = penalty_spec(self)
        if spec is None or not isinstance(score_computer, LogMarginalLikelyhoodComputer):
            return None
        # split_candidates[j] - split_candidates[:j] takes the values 0 .. len(counts); num_splits < len(split_candidates)
        return penalty_tables(spec, len(counts) + 1, len(split_candidates))

    def _scorer_protocol_dp(self, score_computer, split_candidates, regularized):
        """Row-by-row recurrence through an arbitrary scorer object.

        P[0] = 0;  P[j] = max_i(row_j[i] + P[i] - penalties) + creation cost;  arg-max = first maximum.
        Penalties (reference square_splitter.py:45-53): lambda_n * f(#splits(i) + 1), waived for i = 0,
        and lambda_L * g(L_j - L_i)."""
        n = len(split_candidates)
        best = np.empty(n)
        back = np.empty(n, dtype=int)
        best[0] = 0
        back[0] = 0
        use_num = regularized and self.split_number_regularization_multiplier != 0
        use_len = regularized and self.length_regularization_multiplier != 0
        pieces = np.zeros(n)          # number of splits in the best segmentation of each prefix
        for j in range(1, n):
            row = score_computer.all_suffixes_self_score(j)
            row += best[:j]
            if use_num:
                row -= self.split_number_regularization_multiplier * self.split_number_regularization_function(pieces[:j] + 1)
                row[0] += self.split_number_regularization_multiplier * self.split_number_regularization_function(1)
            if use_len:
                lengths = split_candidates[j] - split_candidates[:j]
                row -= (self.length_regularization_multiplier * self.length_regularization_function(lengths))[:j]
            k = np.argmax(row)
            back[j] = k
            if regularized and k != 0:
                pieces[j] = pieces[k] + 1
            best[j] = row[k] + score_computer.segment_creation_cost
        indices = SquareSplitter.collect_split_points(back)
        return best[-1], split_candidates[indices]

    @staticmethod
    def collect_split_points(previous_splits):
        """Follow previous_splits from the last candidate back to 0; ascending list of indices."""
        k = len(previous_splits) - 1
        path = [k]
        while k != 0:
            k = previous_splits[k]
            path.append(k)
        path.reverse()
        return path
