"""Per-round algorithmic cells vs cells skipped by the exact far-column bound."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pasio_b200 import synth, _native
from pasio_b200.log_marginal_likelyhood import ScorerFactory
nt = int(sys.argv[1]) if len(sys.argv) > 1 else 100000000
eng = _native.engine(); eng.use_scorer(ScorerFactory(1.0, 1.0))
eng.load(synth.dnase_like(nt, seed=1000)); eng.set_candidates(None)
for r in range(12):
    eng.timing_reset(True)
    n_in, n_out, cells = eng.round(2500, 1250, 'constants')
    ms = eng.timing()['window_dp'][0]
    c, sk = eng.round_stats()
    passed, fell, rows = eng.round_certify_stats()
    print('round %d: %d -> %d cands, cells %.4g, skipped %.4g (%.1f%%), window_dp %.2f ms, checked windows passed %d fell back %d '
          '(rows proven before the resume %d)' % (r + 1, n_in, n_out, c, sk, 100.0 * sk / max(c, 1), ms, passed, fell, rows), flush=True)
    if n_in == n_out: break
