#!/usr/bin/env python
"""bench.py -- evidence-case BP sweeps/sec of the batched loopy-BP path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload alarm37] [--precision fp64]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own CPU implementation, same metric
    python bench.py ... --dump-outputs DIR    # also write the outputs of the last timed step (rank 0's shard) to DIR/<name>.npy

One "step" = one pass of the hot path over one batch of synthetic evidence cases: init (K0),
`sweeps` synchronous sweeps (K1), beliefs (K4) -- belief_propagation.hpp:31-159 for every case.
`value` = case-sweeps/s with the evidence already resident in HBM (bnbp_run_batch_device);
`e2e`   = the same metric through the host-buffer C-ABI call (bnbp_run_batch) with pinned host
          evidence in and host marginals out, copies inside the timed region.
Multi-GPU: one process per GPU, cases sharded by contiguous ranges (weak scaling: every rank runs
the full per-GPU batch), no data-path collective; NCCL only all-reduces the sweep / convergence
summary each step; a second timed pass gathers the marginals inside the library (config.multi_gpu.with_gather).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bayesiannetwork_b200 import synth  # noqa: E402
from bayesiannetwork_b200.flat import EvidenceBatch  # noqa: E402

METRIC = "evidence-case BP sweeps/sec"
UNIT = "case-sweeps/s"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def fatal(msg: str, world: int = 1):
    """Stop the bench with a message.  In a multi-rank run the process leaves WITHOUT unwinding: raising SystemExit drops the
    frames first, the handle's destructor then waits in NCCL for the peers, and the message is never printed (r02c / r02e: a
    rank sat in bnbp_destroy while the other waited at a barrier until the launcher's timeout)."""
    sys.stderr.write("bench.py: " + msg + "\n")
    sys.stderr.flush()
    if world > 1:
        os._exit(1)
    raise SystemExit(1)


def kernel_source_hash() -> str:
    """Hash of the CUDA sources of the sweep kernels: a traffic figure measured under ncu is only quoted for the
    kernel text it was measured on (profiles/update_traffic.py writes it, bench.py refuses a stale one)."""
    import hashlib
    h = hashlib.sha1()
    for name in ("bnbp_spec.cuh", "bnbp_onchip.cuh", "bnbp_sweep.cuh", "bnbp_kernels.cuh"):
        with open(os.path.join(ROOT, "bayesiannetwork_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def measured_traffic(key: str):
    """(bytes per sweep | None, note) from profiles/traffic.json."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None, "profiles/traffic.json missing"
    ent = tj.get("entries", {}).get(key)
    if not ent:
        return None, f"no ncu capture recorded for {key}"
    if ent.get("source_hash") != kernel_source_hash():
        return None, f"stale: {ent.get('from')} was captured on other kernel sources (hash {ent.get('source_hash')})"
    return float(ent["dram_bytes_per_sweep"]), f"ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per sweep, {ent.get('from')}"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.thr = [], None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._pump, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def wait_first(self, timeout: float = 3.0) -> None:
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def mark(self) -> None:
        """Samples before this point (warm-up) are not part of the report."""
        self.first = len(self.rows)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        rows = self.rows[getattr(self, "first", 0):] or self.rows[-1:]
        for row in rows:
            f = [x.strip() for x in row.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(self.NAMES, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def build_workload(name: str, n_cases: int | None, rank: int, network_file: str | None = None):
    if network_file:
        # a network file (BIF / DSC through bnbp_netfile_*): evidence on each node with p = 0.10, 20 sweeps
        from bayesiannetwork_b200 import netfile
        net = netfile.load(network_file).net
        n = n_cases or (1 << 18)
        return net, synth.make_evidence(net, n, case_offset=rank * n, p=0.10), 20
    factory, default_cases, evkw, sweeps = synth.WORKLOADS[name]
    net = factory()
    n = n_cases or default_cases
    ev = synth.make_evidence(net, n, case_offset=rank * n, **evkw)
    return net, ev, sweeps


# ---------------------------------------------------------------------------------------------------
# CPU legs (the only places that touch oracle/): cpu_baseline of the main line, and --impl reference.
def _ref_worker(args):
    net, ev, sweeps = args
    from oracle import oracle
    t0 = time.perf_counter()
    oracle.run_reference(net, ev, eps=0.0, max_sweeps=sweeps)
    return time.perf_counter() - t0


def cpu_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def time_port(net, ev_sample, sweeps, threads):
    from oracle import oracle
    if not oracle.have_port():
        oracle.build()
    t0 = time.perf_counter()
    oracle.run_port(net, ev_sample, eps=0.0, max_sweeps=sweeps, threads=threads)
    dt = time.perf_counter() - t0
    return ev_sample.n_cases * sweeps / dt, dt


def run_reference_arm(args, rank: int, world: int):
    """The reference's own CPU implementation of the path (oracle/_ref = its unmodified headers
    compiled in place), one PROCESS per host core (its shared_ptr graph is not thread-friendly),
    each step a bounded sample of the same workload."""
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import oracle
    net, _, sweeps = build_workload(args.workload, 8, 0)
    sweeps = args.sweeps or sweeps
    cores = cpu_cores()
    use_ref = oracle.have_reference()
    # size the per-step sample for ~1 s: probe one core
    probe = synth.make_evidence(net, 2, case_offset=0, **synth.WORKLOADS[args.workload][2])
    if use_ref:
        t = _ref_worker((net, probe, sweeps)) / 2
    else:
        t = time_port(net, probe, sweeps, 1)[1] / 2
    per_core = max(1, min(4096, int(1.0 / max(t, 1e-6))))
    evkw = synth.WORKLOADS[args.workload][2]
    shards = [synth.make_evidence(net, per_core, case_offset=i * per_core, **evkw) for i in range(cores)]
    total_cases = per_core * cores

    def one_step():
        if use_ref:
            with mp.get_context("fork").Pool(cores) as pool:
                t0 = time.perf_counter()
                pool.map(_ref_worker, [(net, s, sweeps) for s in shards])
                return time.perf_counter() - t0
        big = synth.make_evidence(net, total_cases, **evkw)
        return time_port(net, big, sweeps, cores)[1]

    for _ in range(args.warmup):
        one_step()
    times = [one_step() for _ in range(args.steps)]
    dt = sum(times)
    value = total_cases * sweeps * args.steps / dt
    kind = "reference" if use_ref else "port"
    configs = None if args.no_configs else reference_scaled_configs(cores, use_ref)
    sample = (f"{total_cases} cases x {sweeps} sweeps per step ({per_core} per core), "
              f"{'oracle/_ref: unmodified reference headers' if use_ref else 'oracle C port (reference not compiled here)'}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "nodes": net.n_nodes, "edges": net.n_edges, "sweeps": sweeps,
                   "cases_per_step": total_cases},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "configs": configs,
    }
    print(json.dumps(line), flush=True)


def _ref_scaled_worker(args):
    net, ev, sweeps = args
    from oracle import oracle
    return oracle.run_reference(net, ev, eps=0.0, max_sweeps=sweeps)[3]     # seconds inside operator()


def reference_scaled_configs(cores: int, use_ref: bool):
    """BASELINE.md section 3(1): the UNMODIFIED reference on scaled instances of configs 3-5 (its cost grows
    ~N^3 with the node count, so the full sizes cannot be run: 100x100 grid = ~2.5e4 s per sweep per case), one
    process per core, one case each; full-size figures only as labelled extrapolations."""
    import multiprocessing as mp
    if not use_ref:
        return None
    scaled = [
        ("cfg3'", "grid 20x20 (cfg 3 is 100x100)", synth.grid(20), 2,
         (10000 / 400) ** 3, "N^3 (topology queries dominate: graph.hpp:378-413,466-481)"),
        ("cfg4'", "random DAG 200 nodes, <= 4 parents, card 2-8 (cfg 4 has 2000)", synth.random_dag(200), 2,
         (2000 / 200) ** 3, "N^3"),
        ("cfg5'", "64 nodes, 3 parents, card 8 (cfg 5 has card 32)", synth.high_card(64, card=8, n_parents=3), 3,
         (32 / 8) ** 4, "CPT entries (x256: same topology, hash-map CPT lookups dominate)"),
    ]
    out = []
    for key, what, net, sweeps, factor, law in scaled:
        shards = [synth.make_evidence(net, 1, case_offset=i, p=0.10) for i in range(cores)]
        with mp.get_context("fork").Pool(cores) as pool:
            t0 = time.perf_counter()
            secs = pool.map(_ref_scaled_worker, [(net, s, sweeps) for s in shards])
            wall = time.perf_counter() - t0
        per_core = sweeps / (sum(secs) / len(secs))
        out.append({"config": key, "instance": what, "nodes": net.n_nodes, "edges": net.n_edges, "cpt_entries": int(net.cpt.size),
                    "kind": "reference", "cores": cores, "sample": f"1 case x {sweeps} sweeps per core, {wall:.1f} s",
                    "case_sweeps_per_s_per_core": per_core, "value": per_core * cores, "unit": UNIT,
                    "full_size_extrapolation": {"value": per_core * cores / factor, "unit": UNIT, "factor": factor, "law": law,
                                                "note": "EXTRAPOLATED, not measured: the full-size instance cannot be run"}})
    return out


# ---------------------------------------------------------------------------------------------------
# BASELINE.json configs 3-5 as short measured entries of the same JSON line ("configs"): value, the roofline
# that BINDS the config (BASELINE.md section 4: HBM / FMA pipe / tensor pipe), a parity sample against the
# oracle port and the port's own rate on that sample (the cpu_baseline of the entry).
#   key, workload, BASELINE total cases, GPUs the config is defined on, precisions, parity sample (N=1, N>1), binding roofline
EXTRA_CONFIGS = [
    ("cfg3", "grid100", 1 << 16, 1, ["fp64"], (16, 16), "hbm"),
    ("cfg4", "dag2000", 1 << 18, 8, ["fp64"], (48, 128), "fma"),
    ("cfg5", "card32", 1 << 17, 8, ["fp32", "fp64"], (12, 24), "tensor"),
]
TOLERANCE = {"fp64": (1e-9, 1e-12), "fp32": (1e-5, 1e-7)}
FMA_PEAK_TFLOPS = {"fp64": 37.2, "fp32": 74.4}     # nominal: 2 x 148 SMs x 1.965 GHz x (64 | 128) lanes
FP64_TENSOR_PEAK_TFLOPS = 40.0                     # nominal B200 fp64 tensor (DMMA) rate


DUMP_BYTES = 60 << 20          # --dump-outputs: bound of the files written (a seeded sample of cases beyond it)


def dump_outputs(dirname: str, marginals, sweeps, converged, torch) -> None:
    """The outputs of the last timed step as DIR/<name>.npy, so that two builds run with the same arguments can be
    compared output for output: marginals [k, sum r_X] in the handle's precision, the sweeps each case ran and its
    converged flag (both as float64), and case_index, the cases (rows of the batch) the k rows are.  Every case when
    that fits DUMP_BYTES, else a fixed sample drawn with a fixed seed."""
    n, V = marginals.shape
    row_bytes = V * marginals.element_size() + 3 * 8
    k = min(n, DUMP_BYTES // row_bytes)
    rows = np.arange(n) if k == n else np.sort(np.random.default_rng(20240).choice(n, k, replace=False))
    idx = torch.from_numpy(rows).to(marginals.device)
    out = {"marginals": marginals[idx].cpu().numpy(), "sweeps": sweeps[idx].cpu().numpy().astype(np.float64),
           "converged": converged[idx].cpu().numpy().astype(np.float64), "case_index": rows.astype(np.float64)}
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def walk_flops(net) -> float:
    """F = sum_X (2k+2) r_X Q_X: one fused CPT pass for pi_X and all k lambda-messages (SURVEY.md 8d)."""
    k = np.diff(net.parent_off).astype(np.float64)
    size = np.diff(net.cpt_off).astype(np.float64)
    return float(((2 * k + 2) * size)[k > 0].sum())


def measure_config(key, workload, total_cases, base_gpus, precision, parity_cases, binding, *, torch, dist, dev,
                   local_rank, rank, world, with_cpu, hostpg=None):
    from bayesiannetwork_b200.engine import BeliefPropagation
    from bayesiannetwork_b200.flat import EvidenceBatch
    factory, _, evkw, sweeps = synth.WORKLOADS[workload]
    net = factory()
    # N = 1: the share one GPU holds when the config runs on the GPU count BASELINE.json names; N > 1: strong
    # scaling, the BASELINE total sharded N ways
    n = total_cases // (world if world > 1 else base_gpus)
    tdtype = torch.float64 if precision == "fp64" else torch.float32
    tsize = 8 if precision == "fp64" else 4
    V, S = net.belief_values, net.state_values
    t_gen = time.perf_counter()
    d_off, d_node, d_state = synth.make_evidence_torch(net, n, case_offset=rank * n, device=dev, **evkw)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    bp = BeliefPropagation(net, precision, device=local_rank)
    d_out = torch.empty((n, V), dtype=tdtype, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        bp.run_device(n, d_off, d_node, d_state, d_out, epsilon=0.0, max_sweeps=sweeps, stream=stream)

    def barrier():                                       # host-side (gloo): see main()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=hostpg)

    t0 = time.perf_counter()
    step()                                               # warm-up (allocates the state arena)
    barrier()
    warm_s = time.perf_counter() - t0
    if world > 1:                                        # every rank must take the same number of steps
        t = torch.tensor([warm_s], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=hostpg)
        warm_s = float(t[0])
    steps = 2 if warm_s < 5.0 else 1
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    st = bp.stats()
    dense_ms = max(0.0, st["last_dense_ms"]) if st["dense_nodes"] else 0.0
    sweep_ms = (st["last_sweep_ms"] - dense_ms) / max(1, st["last_sweep_launches"])
    dense_ms_per_sweep = dense_ms / max(1, st["last_sweep_launches"])
    if world > 1:
        t = torch.tensor([ms, sweep_ms, dense_ms_per_sweep, float(steps)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=hostpg)
        ms, sweep_ms, dense_ms_per_sweep = (float(x) for x in t[:3])
    value = world * n * sweeps * steps / (ms * 1e-3)
    per_gpu = value / world
    peak, peak_src = measured_peaks()
    hbm = {"bound": "hbm", "achieved": per_gpu * 2 * S * tsize / 1e9, "peak": peak, "unit": "GB/s", "peak_source": peak_src,
           "algorithmic_bytes_per_case_sweep": 2 * S * tsize,
           "note": "whole step (sweep kernel + dense products + init + beliefs) against the HBM copy peak"}
    hbm["frac"] = hbm["achieved"] / peak
    kern = {"sweep_kernel_ms_per_sweep": sweep_ms, "dense_ms_per_sweep": dense_ms_per_sweep,
            "sweep_kernel_hbm_frac": (2.0 * S * tsize * min(n, st["resident_cases"]) / (sweep_ms * 1e-3) / 1e9 / peak) if sweep_ms > 0 else None,
            "resident_cases": int(st["resident_cases"]), "dense_nodes": int(st["dense_nodes"]),
            "kernel_launches_per_step": int(st["last_kernel_launches"]),
            "sweep_kernel": (f"bnbp_spec_sweep, class-looped: one unrolled body per node shape class ({int(st['spec_class_count'])} classes "
                             f"for {net.n_nodes} nodes), NVRTC sm_100a" if st.get("spec_class_count", 0)
                             else "bnbp_spec_sweep (network-specialised, NVRTC sm_100a)" if st["last_specialised"] else "sweep_kernel (generic)"),
            "spec_compile_ms": st["spec_compile_ms"]}
    if binding == "hbm":
        roof = hbm
    elif binding == "fma":
        F = walk_flops(net)
        tf = per_gpu * F / 1e12
        roof = {"bound": "fma", "achieved": tf, "peak": FMA_PEAK_TFLOPS[precision], "unit": "TFLOP/s",
                "frac": tf / FMA_PEAK_TFLOPS[precision], "flops_per_case_sweep": F,
                "peak_source": "nominal CUDA-core FMA peak at 1965 MHz (fp64 64, fp32 128 lanes per SM)",
                "note": "algorithmic flops F = sum (2k+2) r Q (SURVEY 8d) x case-sweeps/s of the whole step; nodes on the dense "
                        "path spend 4|CPT| instead of (2k+2)|CPT|, so the executed flops are lower", "hbm_frac": hbm["frac"]}
    else:
        dense_flops = st["dense_flops_per_case_sweep"]
        if precision == "fp32" and st.get("dense_tensor_jobs", 0) and dense_ms_per_sweep > 0:
            mp = {}
            try:
                mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            except Exception:
                pass
            tpk = 0.5 * mp["bf16_tflops"] if mp.get("bf16_tflops") else 1100.0
            issued = 3.0 * st["dense_tensor_flops_per_case_sweep"]
            ttf = issued * min(n, st["resident_cases"]) / (dense_ms_per_sweep * 1e-3) / 1e12
            roof = {"bound": "tensor", "achieved": ttf, "peak": tpk, "unit": "TFLOP/s", "frac": ttf / tpk, "kernel": "dense_tc_kernel",
                    "issued_flops_per_case_sweep": issued, "algorithmic_flops_per_case_sweep": dense_flops,
                    "note": "tcgen05 kind::tf32, 3xTF32 (hi*hi + hi*lo + lo*hi): issued tf32 flops = 3 x algorithmic, over the time "
                            "of the dense launches of one sweep",
                    "peak_source": ("0.5 x measured bf16 (MEASURED_PEAKS.json bf16_tflops)" if mp.get("bf16_tflops")
                                    else "nominal tf32 dense 1.1 PFLOP/s"), "hbm_frac": hbm["frac"]}
        else:
            ttf = dense_flops * min(n, st["resident_cases"]) / max(dense_ms_per_sweep * 1e-3, 1e-12) / 1e12
            roof = {"bound": "tensor", "achieved": ttf, "peak": FP64_TENSOR_PEAK_TFLOPS, "unit": "TFLOP/s",
                    "frac": ttf / FP64_TENSOR_PEAK_TFLOPS, "kernel": "dense_gemm_kernel (fp64 mma.sync m8n8k4, DMMA)",
                    "algorithmic_flops_per_case_sweep": dense_flops, "peak_source": "nominal B200 fp64 tensor rate (40 TFLOP/s)",
                    "note": "no tensor-core format holds the 1e-9 bound, so the fp64 products run as DMMA", "hbm_frac": hbm["frac"]}
    entry = {"config": key, "workload": workload, "dtype": "f64" if precision == "fp64" else "f32", "value": value, "unit": UNIT,
             "n_gpus": world, "scaling": "strong" if world > 1 else f"1/{base_gpus} share of the BASELINE total" if base_gpus > 1 else "full size",
             "total_cases": n * world, "cases_per_gpu": n, "baseline_total_cases": total_cases, "sweeps": sweeps, "steps": steps,
             "ms_per_step": ms / steps, "nodes": net.n_nodes, "edges": net.n_edges, "state_values_per_case": S,
             "roofline": roof, "kernels": kern, "evidence_generation_s": t_gen}
    # parity (rank 0): evenly spaced cases of this rank's shard against the oracle port, same sweeps
    if rank == 0:
        k = min(parity_cases, n)
        idx = np.unique(np.linspace(0, n - 1, k).astype(np.int64))
        offs = d_off.cpu().numpy()
        rows = d_out[torch.from_numpy(idx).to(dev)].double().cpu().numpy()
        cases = []
        for c in idx:
            a, b = int(offs[c]), int(offs[c + 1])
            cases.append(dict(zip(d_node[a:b].cpu().numpy().tolist(), d_state[a:b].cpu().numpy().tolist())))
        sample = EvidenceBatch.from_cases(net, cases)
        cores = cpu_cores()
        from oracle import oracle
        if not oracle.have_port():
            oracle.build()
        t0 = time.perf_counter()
        om, _, _ = oracle.run_port(net, sample, eps=0.0, max_sweeps=sweeps, threads=cores)
        dt = time.perf_counter() - t0
        rtol, atol = TOLERANCE[precision]
        err = np.abs(rows - om)
        bound = rtol * np.maximum(np.abs(rows), np.abs(om)) + atol
        ratio = float(np.nanmax(err / bound))
        ok = bool(np.array_equal(np.isnan(rows), np.isnan(om)) and ratio <= 1.0)
        entry["parity"] = {"cases": int(len(idx)), "checker": "oracle/bp_oracle.c", "rtol": rtol, "atol": atol,
                           "max_err_over_bound": ratio, "ok": ok}
        if with_cpu:
            entry["cpu_baseline"] = {"value": len(idx) * sweeps / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                     "sample": f"{len(idx)} cases of the workload x {sweeps} sweeps, oracle/bp_oracle.c (OpenMP, {cores} threads), {dt:.1f} s"}
        if not ok:
            fatal(f"{key} {precision}: parity sample off (max err/bound {ratio:.3g})", world)
    bp.close()
    del d_out, d_off, d_node, d_state
    torch.cuda.empty_cache()
    return entry


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline measurement (the e2e leg times min(K, 10) calls, the N > 1 gather pass max(3, K // 2) steps, each `configs` entry 1 or 2 steps of its own)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="bnbp", choices=["bnbp", "reference"])
    ap.add_argument("--workload", default="alarm37", choices=sorted(synth.WORKLOADS))
    ap.add_argument("--network", default="", help="a .bif / .dsc network file instead of a synthetic workload")
    ap.add_argument("--cases", type=int, default=0, help="cases per GPU (default: the workload's)")
    ap.add_argument("--sweeps", type=int, default=0, help="fixed sweeps per step (default: the workload's)")
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"])
    ap.add_argument("--specialize", default="auto", choices=["auto", "always", "never"],
                    help="sweep-kernel family: network-specialised (NVRTC) or generic")
    ap.add_argument("--epsilon", type=float, default=0.0,
                    help="> 0: time-to-solution mode (reference stopping rule, delta < epsilon per case, "
                         "--sweeps = cap, default 200); value counts the sweeps actually executed")
    ap.add_argument("--dense-min", type=int, default=0,
                    help="CPT entries from which a node takes the dense contraction path (0 = library default, -1 = never)")
    ap.add_argument("--dense-tensor", type=int, default=0,
                    help="fp32: dense products on the tensor cores (0 = library default, 1 = every product, -1 = never)")
    ap.add_argument("--no-gather", action="store_true",
                    help="N > 1: skip the second timed pass in which every rank ends a step with ALL marginals "
                         "(exchanged over NCCL inside bnbp_run_batch_device) and the N-rank = 1-rank check that uses it")
    ap.add_argument("--onchip", default="auto", choices=["auto", "always", "never"],
                    help="the on-chip multi-sweep kernel (state in shared memory for all sweeps)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true",
                    help="skip the short measured entries for BASELINE configs 3-5 (the `configs` array of the line)")
    ap.add_argument("--only-configs", default="", help="comma-separated subset of cfg3,cfg4,cfg5")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the marginals, sweeps and converged flags of the last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path: it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "bnbp" else args.warmup

    if os.environ.get("BNBP_BENCH_WATCHDOG"):
        # debugging aid for multi-rank runs: every N seconds each rank prints where its Python threads are
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["BNBP_BENCH_WATCHDOG"]), repeat=True, exit=False)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from bayesiannetwork_b200.engine import BeliefPropagation

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the bnbp path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    hostpg = None
    saved_stdout = None
    if world > 1:
        # stdout carries ONE JSON line: NCCL prints its version banner there when its first communicator starts working,
        # so until that line is printed, file descriptor 1 points at stderr
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        # Barriers and the max-over-ranks of the timings go over a HOST group (gloo).  An NCCL barrier is a kernel that
        # spins on the GPU until every rank has joined, and once peer access is on, a cudaMalloc on rank A (pinned / staging
        # buffers of the e2e leg, a new handle per `configs` entry) waits for rank B's device -- which is spinning in the
        # barrier waiting for A.  r02c: rank 0 does 200 ms of extra work (the N-rank = 1-rank check), rank 1 reached the next
        # barrier first, and the run sat there until the NCCL watchdog fired.  The NCCL traffic of this bench is the
        # library's own (gather + summary inside the timed step, no allocation anywhere near it).
        hostpg = dist.new_group(backend="gloo")

    net, ev, sweeps = build_workload(args.workload, args.cases or None, rank, args.network or None)
    if args.network:
        args.workload = "file:" + os.path.basename(args.network)
    sweeps = args.sweeps or (200 if args.epsilon > 0 else sweeps)
    n, V = ev.n_cases, net.belief_values
    tdtype = torch.float64 if args.precision == "fp64" else torch.float32
    tsize = 8 if args.precision == "fp64" else 4
    bp = BeliefPropagation(net, args.precision, device=local_rank, specialize=args.specialize,
                           dense_min_cpt=args.dense_min, dense_tensor=args.dense_tensor, onchip=args.onchip)
    gather = world > 1 and not args.no_gather
    if world > 1:
        # the communicator lives in libbnbp: rank 0 draws the id, torch.distributed only ships its 128 bytes
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(BeliefPropagation.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0, group=hostpg)
        bp.comm_init(world, rank, bytes(uid.numpy().tobytes()))

    # ---- device-resident inputs --------------------------------------------------------------------
    d_off = torch.from_numpy(ev.ev_off).to(dev)
    d_node = torch.from_numpy(ev.ev_node).to(dev)
    d_state = torch.from_numpy(ev.ev_state).to(dev)
    # with the gather every rank holds [world * n, V]; its own kernels write rows [rank * n, (rank + 1) * n) in place
    gathered = torch.empty((world * n, V), dtype=tdtype, device=dev) if gather else None
    d_out = torch.empty((n, V), dtype=tdtype, device=dev)
    d_sw = torch.empty(n, dtype=torch.int32, device=dev)
    d_cv = torch.empty(n, dtype=torch.uint8, device=dev)
    summaries = []
    # a dedicated (non-default) stream: the library enqueues on it and the CUDA events below see it
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream

    def step(with_gather=False):
        # The collectives of the path live in libbnbp (NCCL).  Every step ends with the all-reduce of the convergence summary;
        # the marginals stay sharded on the GPU that computed them (SURVEY section 5: "leave marginals sharded and gather on
        # demand") in the headline steps, and a second timed pass below runs the same step WITH the gather inside
        # bnbp_run_batch_device, so the line carries both numbers.
        g = with_gather and gather
        bp.run_device(n, d_off, d_node, d_state, gathered if g else d_out, epsilon=args.epsilon, max_sweeps=sweeps,
                      out_sweeps=d_sw, out_converged=d_cv, stream=stream, gather=g)
        if world > 1:
            summaries.append(bp.comm_summary(d_sw, d_cv, n, stream=stream))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=hostpg)

    def reduce_host(values, op):
        """max / sum over the ranks of a few host numbers (gloo)."""
        if world == 1:
            return list(values)
        t = torch.tensor(list(values), dtype=torch.float64)
        dist.all_reduce(t, op=op, group=hostpg)
        return [float(x) for x in t]

    # nvidia-smi is started BEFORE the warm-up: its NVML initialisation takes driver locks and, started
    # right in front of the timed region, stalled the first timed launches by 7-70 ms (r01l); only the
    # samples taken after mark() are reported
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.wait_first()
    if world > 1:
        # first call without the exchange: whatever the handle allocates on first use is allocated on every rank before
        # any rank can sit in a collective (a cudaMalloc next to a peer's spinning NCCL kernel deadlocks, see hostpg above)
        bp.run_device(n, d_off, d_node, d_state, d_out, epsilon=args.epsilon, max_sweeps=sweeps,
                      out_sweeps=d_sw, out_converged=d_cv, stream=stream)
        barrier()
    for _ in range(args.warmup):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.mark()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    st = bp.stats()
    if args.dump_outputs:
        if rank == 0:
            dump_outputs(args.dump_outputs, d_out, d_sw, d_cv, torch)
        barrier()                                    # rank 0 allocates for the copy: no peer may sit in a collective meanwhile
    gather_pass = None
    if gather:
        # the same step with the gather of the marginals inside the call (every rank ends it with ALL marginals)
        g_steps = max(3, args.steps // 2)
        for _ in range(2):
            step(with_gather=True)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(g_steps):
            step(with_gather=True)
        g1.record()
        barrier()
        g_ms = reduce_host([g0.elapsed_time(g1)], dist.ReduceOp.MAX)[0]
        gather_pass = {"steps": g_steps, "ms_per_step": g_ms / g_steps,
                       "value": (None if args.epsilon > 0 else world * n * sweeps * g_steps / (g_ms * 1e-3)), "unit": UNIT,
                       "gathered_bytes_per_step_per_rank": int(world * n * V * tsize),
                       "received_bytes_per_step_per_rank": int((world - 1) * n * V * tsize)}
    launches_per_step = int(st["last_kernel_launches"])
    # the library's own CUDA events: around all sweeps of the last step, and around the dense
    # contraction launches inside them (nodes with large CPTs; 0 for the other workloads)
    dense_ms = max(0.0, st["last_dense_ms"]) if st["dense_nodes"] else 0.0
    sweep_ms_per_launch = (st["last_sweep_ms"] - dense_ms) / max(1, st["last_sweep_launches"])
    dense_ms_per_sweep = dense_ms / max(1, st["last_sweep_launches"])
    if world > 1:
        ms, sweep_ms_per_launch, dense_ms_per_sweep = reduce_host([ms, sweep_ms_per_launch, dense_ms_per_sweep], dist.ReduceOp.MAX)
    clocks = sampler.stop() if sampler else None
    multi_gpu = None
    if world > 1:
        # the N-rank sharded run equals a 1-rank run: rank 0 recomputes, on its own GPU, the first cases of EVERY rank's
        # shard (evidence is a function of the case index) and compares them with the rows the gather delivered
        multi_gpu = {"summary_all_reduce": summaries[-1] if summaries else None,
                     "collectives": "every step: ncclAllReduce of the convergence summary; gather pass: grouped ncclBroadcast per rank and "
                                    "chunk, all issued by libbnbp (the timed headline steps keep the marginals sharded)",
                     "with_gather": gather_pass}
        if gather_pass:
            gather_pass["cost_ms_per_step"] = gather_pass["ms_per_step"] - ms / args.steps
        if gather and rank == 0 and not args.network:
            # 4096 cases per rank: the recomputation takes the same kernel family as the batch (the on-chip kernel from
            # 4096 cases up; 256 cases would run the generic kernel, whose rounding differs in the last bits)
            k = min(4096, n)
            evkw = synth.WORKLOADS[args.workload][2]
            worst, same = 0.0, True
            chk = torch.empty((k, V), dtype=tdtype, device=dev)
            for r in range(world):
                e_r = synth.make_evidence(net, k, case_offset=r * n, **evkw)
                bp.run_device(k, torch.from_numpy(e_r.ev_off).to(dev), torch.from_numpy(e_r.ev_node).to(dev),
                              torch.from_numpy(e_r.ev_state).to(dev), chk, epsilon=args.epsilon, max_sweeps=sweeps, stream=stream)
                torch.cuda.synchronize()
                got = gathered[r * n:r * n + k]
                same = same and bool(torch.equal(got, chk))
                worst = max(worst, float((got - chk).abs().max()))
            multi_gpu["n_rank_equals_1_rank"] = {"cases_per_rank_checked": k, "bitwise_equal": same, "max_abs_diff": worst}
            if not (same or worst <= 1e-9):
                fatal(f"gathered marginals differ from a 1-rank run (max abs diff {worst:g})", world)
    eps_info = None
    if args.epsilon > 0:
        # time-to-solution mode: count the sweeps each case actually executed (same every step)
        tot = torch.stack([d_sw.sum(dtype=torch.int64), (d_cv != 0).sum(dtype=torch.int64),
                           d_sw.max().to(torch.int64)])
        tot = [float(x) for x in tot.tolist()]
        if world > 1:
            mx = reduce_host(tot[2:], dist.ReduceOp.MAX)
            tot = reduce_host(tot, dist.ReduceOp.SUM)
            tot[2] = mx[0]
        case_sweeps, n_conv, max_sw = (int(x) for x in tot)
        value = case_sweeps * args.steps / (ms * 1e-3)
        eps_info = {"epsilon": args.epsilon, "max_sweeps": sweeps, "case_sweeps_per_step": case_sweeps,
                    "mean_sweeps_per_case": case_sweeps / (world * n), "max_sweeps_seen": max_sw,
                    "converged_fraction": n_conv / (world * n), "sweep_launches_per_step": int(st["last_sweep_launches"])}
    else:
        value = world * n * sweeps * args.steps / (ms * 1e-3)

    # ---- roofline of the dominant kernel (sweep_kernel) ----------------------------------------------
    S = net.state_values
    peak, peak_src = measured_peaks()
    bytes_per_launch = 2.0 * S * tsize * n           # every state value read once and written once
    if eps_info:                                     # frozen cases move no data: average over the launches
        bytes_per_launch = 2.0 * S * tsize * eps_info["case_sweeps_per_step"] / world / max(1, st["last_sweep_launches"])
    achieved = bytes_per_launch / (sweep_ms_per_launch * 1e-3) / 1e9
    onchip = bool(st.get("last_onchip", 0))
    kernel = "bnbp_onchip_run" if onchip else ("bnbp_spec_sweep" if st["last_specialised"] else "sweep_kernel")
    traffic, traffic_note = measured_traffic(f"{args.workload}:{args.precision}:{kernel}")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_note": traffic_note, "kernel": kernel,
                "peak_source": peak_src,
                "algorithmic_bytes_per_case_sweep": 2 * S * tsize, "ms_per_launch": sweep_ms_per_launch,
                "launch_unit": "one sweep over the resident batch (achieved = 2*S*sizeof(T)*cases / ms_per_launch; traffic is "
                               "per sweep too). A fixed-count run of a specialised network may put its middle sweeps into ONE "
                               "looping launch (short grids / whole waves): ms_per_launch is then that launch's time / its sweeps",
                "sweeps_per_step": int(st["last_sweep_launches"]), "kernel_launches_per_step": launches_per_step,
                "fused_first_last": bool(st.get("last_fused", 0)), "compactions_per_step": int(st.get("last_compactions", 0))}
    if onchip:
        # the state of a case stays in shared memory for all its sweeps: the ALGORITHMIC bytes (2*S*sizeof(T) per
        # case-sweep, SURVEY 8d) never cross HBM, so `achieved` may exceed the HBM peak (SURVEY 8d / BASELINE.md 4 say to
        # report it as such); what binds the kernel is instruction issue / the fp64 pipe
        F = walk_flops(net)
        fpk = FMA_PEAK_TFLOPS[args.precision]
        rate = value / world
        roofline.update({
            "state_on_chip": True,
            "note": "on-chip kernel: frac is against the STREAMING roofline (what a kernel that moves the state through HBM every "
                    "sweep can reach at most); > 1 means faster than any streaming kernel. One launch runs init, every sweep and the "
                    "beliefs of the whole batch; ms_per_launch = launch time / sweeps",
            "hbm_bytes_moved_per_case": int(ev.nbytes() / max(1, n) + V * tsize + 5),
            "fma": {"bound": "fma", "achieved": rate * F / 1e12, "peak": fpk, "unit": "TFLOP/s", "frac": rate * F / 1e12 / fpk,
                    "flops_per_case_sweep": F, "note": "algorithmic flops F = sum (2k+2) r Q (SURVEY 8d) against the nominal CUDA-core FMA peak"},
            "groups_per_sm": int(st.get("onchip_blocks_per_sm", 0)), "warps_per_group": int(st.get("onchip_roles", 0)),
            "shared_memory_per_group": int(st.get("onchip_smem_bytes", 0)), "role_imbalance": st.get("onchip_role_imbalance")})

    dense = None
    if st["dense_nodes"] and dense_ms_per_sweep > 0 and not eps_info:
        # CUDA-core contraction (fp64 parity needs fp64 products): nominal B200 vector peaks
        # 2 x 148 SMs x 1.965 GHz x (64 fp64 | 128 fp32) lanes
        # fp64 products run as DMMA (tensor pipe); fp32 products without the tcgen05 path are CUDA-core FMAs
        pk = FP64_TENSOR_PEAK_TFLOPS if args.precision == "fp64" else FMA_PEAK_TFLOPS["fp32"]
        tf = st["dense_flops_per_case_sweep"] * n / (dense_ms_per_sweep * 1e-3) / 1e12
        dense = {"kernel": "dense_gemm_kernel", "nodes": int(st["dense_nodes"]),
                 "flops_per_case_sweep": st["dense_flops_per_case_sweep"], "ms_per_sweep": dense_ms_per_sweep,
                 "achieved": tf, "peak": pk, "unit": "TFLOP/s", "frac": tf / pk,
                 "peak_source": ("nominal B200 fp64 tensor rate (DMMA)" if args.precision == "fp64"
                                 else "nominal CUDA-core FMA peak at 1965 MHz (128 fp32 lanes per SM)"),
                 "table_values_per_case": int(st["dense_values_per_case"]),
                 "launches_per_sweep": int(st["last_dense_launches"]) // max(1, int(st["last_sweep_launches"])),
                 "share_of_sweep_time": dense_ms_per_sweep / (dense_ms_per_sweep + sweep_ms_per_launch)}
        if st.get("dense_tensor_jobs", 0):
            # tensor-core products (dense_tc_kernel, tcgen05 kind::tf32): every algorithmic multiply-add is
            # issued three times (hi*hi + hi*lo + lo*hi); the tensor-pipe rate is measured against half the
            # measured bf16 throughput (tf32 runs at half the bf16 rate), else the nominal 1.1 PFLOP/s
            mp = {}
            try:
                mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            except Exception:
                pass
            tpk = 0.5 * mp["bf16_tflops"] if mp.get("bf16_tflops") else 1100.0
            ttf = 3.0 * st["dense_tensor_flops_per_case_sweep"] * n / (dense_ms_per_sweep * 1e-3) / 1e12
            all_tc = int(st["dense_tensor_jobs"]) == 2 * int(st["dense_nodes"])
            for kdrop in ("achieved", "peak", "frac", "peak_source"):      # a tensor job has no CUDA-core roofline
                dense.pop(kdrop, None)
            dense.update({"kernel": "dense_tc_kernel" if all_tc else "dense_tc_kernel + dense_gemm_kernel",
                          "tensor_jobs": int(st["dense_tensor_jobs"]),
                          "tensor": {"bound": "tensor", "achieved": ttf, "peak": tpk, "unit": "TFLOP/s", "frac": ttf / tpk,
                                     "issued_flops_per_case_sweep": 3.0 * st["dense_tensor_flops_per_case_sweep"],
                                     "note": "3xTF32: issued tf32 flops = 3 x algorithmic; time includes any CUDA-core products of the same sweep",
                                     "peak_source": ("0.5 x measured bf16 (MEASURED_PEAKS.json bf16_tflops)"
                                                     if mp.get("bf16_tflops") else "nominal tf32 dense 1.1 PFLOP/s")}})

    # ---- end to end through the host-buffer C ABI (pinned host memory both ways) ----------------------
    e2e = None
    if not args.no_e2e:
        def pin(a):
            t = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
            t.numpy()[...] = a
            return t
        p_off, p_node, p_state = pin(ev.ev_off), pin(ev.ev_node), pin(ev.ev_state)
        p_out = torch.empty((n, V), dtype=torch.float64, pin_memory=True)
        ev_pinned = EvidenceBatch(n, p_off.numpy(), p_node.numpy(), p_state.numpy())
        out_np = p_out.numpy()
        # caller-owned count buffers too: a fresh 4 MB + 1 MB numpy array per call is an mmap / munmap pair on
        # the calling thread, and with gigabytes of pinned memory registered the unmap stalls the process for
        # 30-120 ms on bursts of calls (r01chk: 40 calls with reused buffers 27.96-29.20 ms, with fresh ones up to 130 ms)
        p_sw = torch.empty(n, dtype=torch.int32, pin_memory=True)
        p_cv = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        sw_np, cv_np = p_sw.numpy(), p_cv.numpy()
        e2e_steps = max(1, min(args.steps, 10))
        for _ in range(2):                                               # warm-up (staging buffers, pinned pages)
            bp(ev_pinned, args.epsilon, max_sweeps=sweeps, out=out_np, out_sweeps=sw_np, out_converged=cv_np)
        barrier()
        per_call, per_call_dev, per_call_lib = [], [], []
        # no garbage collection inside the timed calls (benchmark hygiene as in timeit; it is NOT what makes
        # bursts of calls take 30-120 ms of wall time at a constant 27 ms of device time on this pool's boxes,
        # r01y/r01z -- those stalls are host-side and outside the library: see ms_per_call_min_median_max)
        gc.collect()
        gc.disable()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            t1 = time.perf_counter()
            bp(ev_pinned, args.epsilon, max_sweeps=sweeps, out=out_np, out_sweeps=sw_np, out_converged=cv_np)
            per_call.append(1e3 * (time.perf_counter() - t1))
            st_call = bp.stats()                                         # the call has returned: no extra wait
            per_call_dev.append(st_call["last_total_ms"])
            per_call_lib.append((st_call["last_host_ms"], st_call["last_host_wait_ms"]))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        gc.enable()
        dt = reduce_host([dt], dist.ReduceOp.MAX)[0]
        # context for the number: what the host link moves when it does nothing else (the marginals
        # are 8*V bytes per case; on PCIe this copy, not the kernels, bounds the host-buffer call)
        probe = torch.empty(n * V, dtype=torch.float64, device=dev)
        p_out.view(-1).copy_(probe, non_blocking=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p_out.view(-1).copy_(probe, non_blocking=True)
        torch.cuda.synchronize()
        d2h_gbs = n * V * 8 / (time.perf_counter() - t0) / 1e9
        del probe
        units_per_step = eps_info["case_sweeps_per_step"] if eps_info else world * n * sweeps
        e2e = {"value": units_per_step * e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(ev.nbytes()), "d2h_bytes_per_step": int(n * V * 8 + n * 5),
               "steps": e2e_steps, "ms_per_step": 1e3 * dt / e2e_steps,
               "ms_per_call_min_median_max": [min(per_call), sorted(per_call)[len(per_call) // 2], max(per_call)],
               "device_ms_per_call_min_median_max": [min(per_call_dev), sorted(per_call_dev)[len(per_call_dev) // 2], max(per_call_dev)],
               "slowest_call": {"wall_ms": max(per_call), "device_ms": per_call_dev[per_call.index(max(per_call))],
                                "inside_bnbp_run_batch_ms": per_call_lib[per_call.index(max(per_call))][0],
                                "of_which_final_stream_waits_ms": per_call_lib[per_call.index(max(per_call))][1]},
               "note": "no nvidia-smi sampling during this leg: its NVML queries showed up as 100 ms outlier calls (r01chk2)",
               "d2h_link_gbs_measured": d2h_gbs, "d2h_floor_ms_per_step": 1e3 * n * V * 8 / (d2h_gbs * 1e9),
               "pipeline": "three streams: evidence H2D of chunk i+1 and marginal D2H of chunk i-1 overlap the kernels "
                           "of chunk i; chunks cut in whole waves of the sweep grid (BNBP_TRACE=1 prints the plan)"}

    # ---- e2e variants: the host link bounds the call, so what matters is what has to cross it ---------------
    if e2e is not None and not eps_info:
        def timed_calls(handle, calls, **kw):
            for _ in range(2):
                handle(ev_pinned, args.epsilon, max_sweeps=sweeps, out_sweeps=sw_np, out_converged=cv_np, **kw)
            barrier()
            gc.disable()
            t0 = time.perf_counter()
            for _ in range(calls):
                handle(ev_pinned, args.epsilon, max_sweeps=sweeps, out_sweeps=sw_np, out_converged=cv_np, **kw)
            dtv = time.perf_counter() - t0
            gc.enable()
            return reduce_host([dtv], dist.ReduceOp.MAX)[0]
        variants = []
        calls = 5
        q = np.unique(np.linspace(0, net.n_nodes - 1, min(8, net.n_nodes)).astype(np.int32))
        Vq = int(net.card[q].sum())
        p_q = torch.empty((n, Vq), dtype=torch.float64, pin_memory=True)
        dtv = timed_calls(bp, calls, out=p_q.numpy(), query_nodes=q)
        variants.append({"what": f"{len(q)} query nodes of {net.n_nodes} (bnbp_run_params.query_nodes): only their marginals leave the device",
                         "dtype": "f64" if args.precision == "fp64" else "f32", "value": world * n * sweeps * calls / dtv, "unit": UNIT,
                         "ms_per_step": 1e3 * dtv / calls, "d2h_bytes_per_step": int(n * Vq * 8 + n * 5)})
        del p_q
        bp32 = bp if args.precision == "fp32" else BeliefPropagation(net, "fp32", device=local_rank, specialize=args.specialize, onchip=args.onchip)
        p_f = torch.empty((n, V), dtype=torch.float32, pin_memory=True)
        dtv = timed_calls(bp32, calls, out=p_f.numpy(), out_dtype=np.float32)
        variants.append({"what": "fp32 handle, float marginals (bnbp_run_params.out_precision = BNBP_OUT_FP32): half the device-to-host copy",
                         "dtype": "f32", "value": world * n * sweeps * calls / dtv, "unit": UNIT, "ms_per_step": 1e3 * dtv / calls,
                         "d2h_bytes_per_step": int(n * V * 4 + n * 5)})
        del p_f
        if bp32 is not bp:
            bp32.close()
        e2e["variants"] = variants

    # ---- the same boundary from C++: bn::inference::belief_propagation::run_flat (tests/cpp/e2e_timing.cpp) -----
    if e2e is not None and not eps_info and rank == 0 and world == 1:
        exe = os.path.join(ROOT, "tests", "cpp", "_build", "e2e_timing")
        if os.path.exists(exe):
            import tempfile
            with tempfile.NamedTemporaryFile(suffix=".bnbp", delete=False) as f:
                np.array([net.n_nodes, net.n_edges, net.cpt.size, n, ev.nnz, sweeps], dtype=np.int64).tofile(f)
                for arr in (net.card, net.parent_off, net.parents, net.cpt_off, net.cpt, ev.ev_off, ev.ev_node, ev.ev_state):
                    arr.tofile(f)
                path = f.name
            try:
                r = subprocess.run([exe, path, "5", "2", args.precision, "0", "0"], capture_output=True, text=True, timeout=600)
                e2e["e2e_cxx"] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": r.stderr[-500:]}
            except Exception as ex:      # the C++ leg is a report, not the measurement: never fail the bench line on it
                e2e["e2e_cxx"] = {"error": str(ex)}
            finally:
                os.unlink(path)
        else:
            e2e["e2e_cxx"] = {"error": "tests/cpp/_build/e2e_timing not built"}

    # ---- CPU baseline beside it (rank 0, N == 1 only): the oracle port on all host cores ---------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and not eps_info:
        cores = cpu_cores()
        sample_cases = 256
        rate, dt = time_port(net, ev.slice(0, sample_cases), sweeps, cores)
        while dt < 5.0 and sample_cases < n and sample_cases < (1 << 18):
            sample_cases = min(n, sample_cases * max(2, int(10.0 / max(dt, 1e-3))))
            rate, dt = time_port(net, ev.slice(0, sample_cases), sweeps, cores)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {sample_cases} cases of the workload x {sweeps} sweeps, oracle/bp_oracle.c "
                         f"(OpenMP, {cores} threads), {dt:.1f} s"}

    # ---- BASELINE configs 3-5: short measured entries (every rank takes part; rank 0 checks parity) -----
    configs = None
    main_workload = args.workload == "alarm37" and not args.network and not args.cases and not eps_info
    if main_workload and not args.no_configs:
        bp.close()
        del d_out, d_off, d_node, d_state, d_sw, d_cv
        gathered = None
        if e2e is not None:
            del p_out, p_off, p_node, p_state, p_sw, p_cv, out_np, sw_np, cv_np, ev_pinned
        gc.collect()
        torch.cuda.empty_cache()
        only = [x for x in args.only_configs.split(",") if x]
        configs = []
        for key, workload, total, base_gpus, precisions, samples, binding in EXTRA_CONFIGS:
            if only and key not in only:
                continue
            for precision in precisions:
                try:
                    configs.append(measure_config(key, workload, total, base_gpus, precision, samples[1 if world > 1 else 0], binding,
                                                  torch=torch, dist=dist, dev=dev, local_rank=local_rank, rank=rank, world=world,
                                                  with_cpu=not args.no_cpu, hostpg=hostpg))
                except Exception as e:            # (a parity sample that is off ends the run inside measure_config: fatal())
                    if world > 1:                 # the ranks meet at barriers inside the entry: one of them cannot skip it alone
                        raise
                    # one GPU: an entry that cannot run here (e.g. no room for its state arena beside another tenant of the
                    # box) is reported as such; the headline measurement above stands on its own
                    configs.append({"config": key, "workload": workload, "dtype": "f64" if precision == "fp64" else "f32",
                                    "value": None, "unit": UNIT, "error": repr(e)[:600]})
                    gc.collect()
                    torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64" if args.precision == "fp64" else "f32",
            "data": "synthetic",
            "config": {"workload": args.workload, "nodes": net.n_nodes, "edges": net.n_edges,
                       "max_card": int(net.card.max()), "cases_per_gpu": n, "sweeps": sweeps,
                       "state_values_per_case": S,
                       "schedule": ("synchronous, stop per case at delta < epsilon (reference rule)" if eps_info
                                    else "synchronous, fixed sweeps, no damping"), "eps_mode": eps_info,
                       "sharding": f"cases x{world}", "gather": gather, "multi_gpu": multi_gpu,
                       "kernel_family": ("on-chip multi-sweep (NVRTC sm_100a, state in shared memory)" if onchip else
                                         f"network-specialised, class-looped walk over {int(st['spec_class_count'])} node shape classes (NVRTC sm_100a)"
                                         if st["last_specialised"] and st.get("spec_class_count", 0) else
                                         "network-specialised (NVRTC sm_100a)" if st["last_specialised"] else "generic"),
                       "cases_per_tile": int(st["cases_per_tile"]),
                       "spec_compile_ms": st["spec_compile_ms"],     # NVRTC time this handle paid (0: every kernel came from the cubin cache)
                       "l2": (f"on-chip kernel: no state in HBM; evidence in + marginals out = {(ev.nbytes() + n * V * tsize) / 1e9:.2f} GB per step vs 126 MB of L2"
                              if onchip else
                              f"inputs larger than L2: {st['resident_cases'] * (S + net.msg_values) * tsize / 1e9:.2f} GB "
                              f"of per-case state per GPU vs 126 MB")},
            "roofline": roofline, "dense": dense, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps, "clocks": clocks, "configs": configs,
        }
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
