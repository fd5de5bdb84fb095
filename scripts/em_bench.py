"""Cost of the EM E-step (expected family counts, bnbp_run_batch_expected_counts, DESIGN section 10) on alarm37,
1M cases of synth.make_evidence's defaults, 20 fixed sweeps, fp64 and fp32.  Prints one JSON line per measurement,
the GPU's name and power limit first.

    kernel       device time of log_evidence_kernel with the count pass (<T, true>) and without it (<T, false>),
                 each from a torch.profiler run of its own
    device call  bnbp_run_batch_device_expected_counts (counts only) against bnbp_run_batch_device_log_evidence
                 (log-evidence only), CUDA events, median of 5 after a warm-up
    host call    bnbp_run_batch_expected_counts, counts only (wall clock, median of 5)
    EM iteration E-step + m_step + refresh_cpt, as BeliefPropagation.em runs them (wall clock, median of 5)"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.engine import BeliefPropagation, m_step

N, SWEEPS, REPS = 1 << 20, 20, 5


def emit(row):
    print(json.dumps(row), flush=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def median_ms(fn, sync_stream=None):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(REPS):
        if sync_stream is not None:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(sync_stream)
            fn()
            b.record(sync_stream)
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        else:
            t0 = time.perf_counter()
            fn()
            ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts))


def kernel_ms(fn, flag):
    """device time of log_evidence_kernel<T, flag> in a profiled run of fn alone"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us = [e.device_time_total for e in prof.key_averages()
          if "log_evidence_kernel" in e.key and (", true>" in e.key) == flag]
    return (sum(us) / 1e3) if us else None


def main():
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    emit(gpu_info())
    net = synth.alarm37()
    ev = synth.make_evidence(net, N)
    nv = int(net.cpt_off[-1])
    d = {k: torch.from_numpy(np.ascontiguousarray(getattr(ev, k))).cuda() for k in ("ev_off", "ev_node", "ev_state")}
    for precision in ("fp64", "fp32"):
        bp = BeliefPropagation(net, precision)
        le = torch.empty(N, dtype=torch.float64, device="cuda")
        cnt = torch.zeros(nv, dtype=torch.float64, device="cuda")
        st = torch.cuda.Stream()

        def dev_logev():
            bp.run_device(N, d["ev_off"], d["ev_node"], d["ev_state"], None, epsilon=0.0, max_sweeps=SWEEPS,
                          out_log_evidence=le, stream=st.cuda_stream)

        def dev_counts():
            bp.run_device(N, d["ev_off"], d["ev_node"], d["ev_state"], None, epsilon=0.0, max_sweeps=SWEEPS,
                          out_counts=cnt, stream=st.cuda_stream)
        ms_logev = median_ms(dev_logev, st)
        st_logev = bp.stats()
        ms_counts = median_ms(dev_counts, st)
        st_counts = bp.stats()
        k_off = kernel_ms(dev_logev, False)
        k_on = kernel_ms(dev_counts, True)
        emit({"row": "device call", "precision": precision, "cases": N, "sweeps": SWEEPS, "cpt_values": nv,
              "kernel_ms_log_evidence_only": k_off, "kernel_ms_with_counts": k_on,
              "call_ms_log_evidence_only": ms_logev, "call_ms_counts_only": ms_counts,
              "family_counts": {"onchip": st_counts["last_onchip"], "specialised": st_counts["last_specialised"],
                                "fused": st_counts["last_fused"]},
              "family_log_evidence": {"onchip": st_logev["last_onchip"], "specialised": st_logev["last_specialised"]}})
        counts = np.zeros(nv)

        def host_counts():
            counts[:] = 0.0
            bp(ev, 0.0, max_sweeps=SWEEPS, expected_counts=True, marginals=False, counts_out=counts)
        ms_host = median_ms(host_counts)
        host_counts()
        t0 = time.perf_counter()
        cpt = m_step(net, counts)
        ms_m = 1e3 * (time.perf_counter() - t0)
        t0 = time.perf_counter()
        bp.refresh_cpt(cpt)
        ms_refresh = 1e3 * (time.perf_counter() - t0)
        bp.refresh_cpt(net.cpt)

        def iteration():
            counts[:] = 0.0
            r = bp(ev, 0.0, max_sweeps=SWEEPS, expected_counts=True, log_evidence=True, marginals=False, counts_out=counts)
            float(r.log_evidence[np.isfinite(r.log_evidence)].sum())
            bp.refresh_cpt(m_step(net, counts))
        ms_iter = median_ms(iteration)
        emit({"row": "host call", "precision": precision, "cases": N, "sweeps": SWEEPS,
              "ms_counts_only": ms_host, "ms_m_step": ms_m, "ms_refresh_cpt": ms_refresh, "ms_em_iteration": ms_iter,
              "spec_compile_ms_total": bp.stats()["spec_compile_ms"]})
        del bp, le, cnt
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
