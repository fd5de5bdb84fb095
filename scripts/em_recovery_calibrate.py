"""Calibrates the bar of the EM recovery test (tests/test_gpu_em.py) on the CPU with the reference computation
(tests/em_oracle.c): the problem of tests/test_em.py's RECOVERY, EM driven by em_oracle's expected counts and
engine.m_step.  Prints one JSON line per iteration (log-likelihood, skipped cases, mean |CPT - generating CPT|).
No GPU needed.  The E-step is cut into contiguous case ranges, one process each (the same serial reference per
range; the counts are summed).

    python scripts/em_recovery_calibrate.py [--procs 8]
"""
import argparse
import json
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

_problem = None


def _estep(args):
    lo, hi, cpt = args
    global _problem
    import em_oracle
    import test_em
    if _problem is None:
        _problem = test_em.recovery_problem()
    net, ev, _ = _problem
    counts, _, _, _, le = em_oracle.run(test_em.with_cpt(net, cpt), ev.slice(lo, hi), eps=1e-6, max_sweeps=200)
    return counts, le


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--procs", type=int, default=os.cpu_count() or 4)
    a = ap.parse_args()
    import test_em
    from bayesiannetwork_b200.engine import m_step
    net, ev, cpt = test_em.recovery_problem()
    n = ev.n_cases
    cuts = np.linspace(0, n, a.procs + 1).astype(int)
    print(json.dumps({"start_mae": float(np.abs(cpt - net.cpt).mean()), **test_em.RECOVERY}), flush=True)
    with ProcessPoolExecutor(a.procs) as pool:
        for it in range(test_em.RECOVERY["iterations"]):
            t = time.time()
            parts = list(pool.map(_estep, [(int(cuts[i]), int(cuts[i + 1]), cpt) for i in range(a.procs)]))
            counts = sum(p[0] for p in parts)
            le = np.concatenate([p[1] for p in parts])
            ok = np.isfinite(le)
            cpt = m_step(net, counts)
            print(json.dumps({"iteration": it, "log_likelihood": float(le[ok].sum()), "skipped": int((~ok).sum()),
                              "mae_after": float(np.abs(cpt - net.cpt).mean()), "seconds": round(time.time() - t, 1)}),
                  flush=True)


if __name__ == "__main__":
    main()
