"""Cost of per-case log-evidence (bnbp_run_batch_log_evidence, DESIGN section 10) on alarm37, 1M hard-evidence cases,
20 fixed sweeps, fp64 and fp32, and its loopy-network cross-check against likelihood weighting.  Prints one JSON
line per measurement, the GPU's name and power limit first.

    log_evidence_kernel   device time of the scoring kernel alone (torch.profiler, its own run)
    device call           bnbp_run_batch_device with and without log-evidence (CUDA events): without it AUTO takes
                          the on-chip kernel, with it the specialised streaming sweeps
    host call             bnbp_run_batch with every marginal against log-evidence with marginals=False (wall clock)
    vs LW                 |log Z_B - ln(LW weight sum / n)| on 4 096 cases x 65 536 samples (loopy BP run to 1e-9)"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.engine import BeliefPropagation

N, SWEEPS, REPS = 1 << 20, 20, 5


def emit(row):
    print(json.dumps(row), flush=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def time_device(bp, d, out, le):
    """median ms of REPS device-path calls (CUDA events on the stream the calls are enqueued on: a stream of its own,
    since a NULL stream hands the call the handle's stream), after one warm-up call of the same shape"""
    st = torch.cuda.Stream()

    def call():
        bp.run_device(N, d["ev_off"], d["ev_node"], d["ev_state"], out, epsilon=0.0, max_sweeps=SWEEPS,
                      out_log_evidence=le, stream=st.cuda_stream)
    call()
    torch.cuda.synchronize()
    ts = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        call()
        b.record(st)
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), bp.stats()


def time_host(fn):
    fn()
    ts = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trace-dir", default=None, help="where torch.profiler writes its trace (default: none kept)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    emit(gpu_info())
    net = synth.alarm37()
    ev = synth.make_evidence(net, N, exact_k=4, seed=41)
    d = {k: torch.from_numpy(np.ascontiguousarray(getattr(ev, k))).cuda() for k in ("ev_off", "ev_node", "ev_state")}
    for precision in ("fp64", "fp32"):
        bp = BeliefPropagation(net, precision)
        dt = torch.float64 if precision == "fp64" else torch.float32
        out = torch.empty((N, net.belief_values), dtype=dt, device="cuda")
        le = torch.empty(N, dtype=torch.float64, device="cuda")
        ms_plain, st_plain = time_device(bp, d, out, None)
        ms_le, st_le = time_device(bp, d, out, le)
        ms_le_only, _ = time_device(bp, d, None, le)
        # the scoring kernel alone, in a profiled run of its own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            bp.run_device(N, d["ev_off"], d["ev_node"], d["ev_state"], out, epsilon=0.0, max_sweeps=SWEEPS,
                          out_log_evidence=le)
            torch.cuda.synchronize()
        if args.trace_dir:
            os.makedirs(args.trace_dir, exist_ok=True)
            prof.export_chrome_trace(os.path.join(args.trace_dir, f"log_evidence_{precision}.pt.trace.json"))
        k_us = [e.device_time_total for e in prof.key_averages() if "log_evidence_kernel" in e.key]
        sweep_us = sum(e.device_time_total for e in prof.key_averages() if "sweep" in e.key.lower())
        emit({"row": "device call", "precision": precision, "cases": N, "sweeps": SWEEPS,
              "log_evidence_kernel_ms": (sum(k_us) / 1e3) if k_us else None,
              "sweep_kernels_ms_same_run": sweep_us / 1e3,
              "call_ms_marginals_only": ms_plain, "family_marginals_only": {"onchip": st_plain["last_onchip"],
                                                                          "specialised": st_plain["last_specialised"]},
              "call_ms_marginals_and_log_evidence": ms_le, "family_log_evidence": {"onchip": st_le["last_onchip"],
                                                                                  "specialised": st_le["last_specialised"],
                                                                                  "fused": st_le["last_fused"]},
              "call_ms_log_evidence_only": ms_le_only})
        host_full = time_host(lambda: bp(ev, 0.0, max_sweeps=SWEEPS))
        host_le_full = time_host(lambda: bp(ev, 0.0, max_sweeps=SWEEPS, log_evidence=True))
        host_le_only = time_host(lambda: bp(ev, 0.0, max_sweeps=SWEEPS, log_evidence=True, marginals=False))
        emit({"row": "host call", "precision": precision, "cases": N, "sweeps": SWEEPS,
              "ms_marginals": host_full, "ms_marginals_and_log_evidence": host_le_full,
              "ms_log_evidence_only": host_le_only})
        del bp, out, le
        torch.cuda.empty_cache()
    # loopy cross-check: BP's Bethe estimate against the likelihood-weighting estimate of P(e)
    n_lw, samples = 4096, 65536
    ev_s = ev.slice(0, n_lw)
    bp = BeliefPropagation(net, "fp64")
    res = bp(ev_s, 1e-9, max_sweeps=200, log_evidence=True)
    _, wsum = bp.likelihood_weighting(ev_s, samples, seed=7, return_weight=True)
    diff = np.abs(res.log_evidence - np.log(wsum / samples))
    emit({"row": "vs LW", "cases": n_lw, "samples": samples, "bp_converged": int(res.converged.sum()),
          "median_abs_diff": float(np.median(diff)), "max_abs_diff": float(diff.max()),
          "median_abs_log_evidence": float(np.median(np.abs(res.log_evidence)))})


if __name__ == "__main__":
    main()
