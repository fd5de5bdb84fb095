"""Host-side checks of bench.py's contract that need no GPU: the measured-traffic figure quoted in `roofline.traffic`
belongs to the CURRENT kernel sources (profiles/traffic.json is stamped with their hash and bench.py drops a stale
entry -- this test makes a kernel edit without a fresh ncu capture visible here instead of on the GPU box), and the
workload table / extra configs name what BASELINE.json names; --dump-outputs, on the host and (-m gpu) end to end."""
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_traffic_entry_of_the_headline_kernel_is_current():
    import bench
    traffic, note = bench.measured_traffic("alarm37:fp64:bnbp_onchip_run")
    assert traffic is not None, note
    # the on-chip kernel moves evidence in and marginals out only: tens of MB per sweep of 1M cases, not the 7.4 GB of a streaming sweep
    assert 1e7 < traffic < 2e8
    src = note.split("profiles/")[1].split(" ")[0]
    assert os.path.exists(os.path.join(ROOT, "profiles", src)), "the capture the figure comes from must be committed under profiles/"


def test_bench_configs_match_baseline_json():
    import bench
    from bayesiannetwork_b200 import synth
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5
    keys = [c[0] for c in bench.EXTRA_CONFIGS]
    assert keys == ["cfg3", "cfg4", "cfg5"]
    for key, workload, total, gpus, precisions, parity, binding in bench.EXTRA_CONFIGS:
        assert workload in synth.WORKLOADS and binding in ("hbm", "fma", "tensor")
        assert total >= 1 << 16 and gpus in (1, 8)
    assert synth.WORKLOADS["alarm37"][1] == 1 << 20 and synth.WORKLOADS["alarm37"][3] == 20



def test_dump_outputs_is_a_bounded_seeded_sample_of_the_step(tmp_path, monkeypatch):
    """--dump-outputs: float arrays only, within DUMP_BYTES (itself under 64 MB), the same cases on every run, each row its
    case's.  A small DUMP_BYTES exercises the same sampling as a full-size batch."""
    import numpy as np
    import torch
    import bench
    assert bench.DUMP_BYTES + 4096 <= 64 * 10 ** 6
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    for n, V, dtype in ((20_000, 105, torch.float64), (20_000, 105, torch.float32), (1000, 7, torch.float64)):
        marg = torch.arange(n, dtype=dtype)[:, None].expand(n, V)          # row c holds c
        sweeps = torch.arange(n, dtype=torch.int32) % 20
        conv = (torch.arange(n) % 3 == 0).to(torch.uint8)
        dirs = [tmp_path / f"{n}_{V}_{dtype}_{i}" for i in range(2)]
        for d in dirs:
            bench.dump_outputs(str(d), marg, sweeps, conv, torch)
        runs = [{f.stem: np.load(f) for f in sorted(d.iterdir())} for d in dirs]
        assert sorted(runs[0]) == ["case_index", "converged", "marginals", "sweeps"]
        assert sum(f.stat().st_size for f in dirs[0].iterdir()) <= bench.DUMP_BYTES + 4096     # + the four .npy headers
        a = runs[0]
        assert all(x.dtype in (np.float32, np.float64) for x in a.values())
        assert a["marginals"].dtype == (np.float64 if dtype == torch.float64 else np.float32)
        assert all(np.array_equal(a[k], runs[1][k]) for k in a)
        rows = a["case_index"].astype(np.int64)
        assert len(rows) == n if n == 1000 else 0 < len(rows) < n
        assert np.all(np.diff(rows) > 0) and a["marginals"].shape == (len(rows), V)
        assert np.array_equal(a["marginals"][:, -1], rows.astype(a["marginals"].dtype))
        assert np.array_equal(a["sweeps"], rows % 20) and np.array_equal(a["converged"], (rows % 3 == 0).astype(np.float64))


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_steps_computed(tmp_path, oracle_mod):
    """bench.py --dump-outputs end to end: the same files from runs with different --steps (every step recomputes the same
    batch), and the marginals those of the oracle for the workload's cases (4096 cases: the on-chip kernel, as at full size)."""
    import subprocess
    import numpy as np
    from bayesiannetwork_b200 import synth
    from bayesiannetwork_b200.flat import EvidenceBatch
    dumps = []
    for steps in (1, 2):
        d = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--cases", "4096", "--steps", str(steps), "--warmup", "0",
                            "--no-e2e", "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({k: np.load(d / f"{k}.npy") for k in ("marginals", "sweeps", "converged", "case_index")})
    assert all(np.array_equal(dumps[0][k], dumps[1][k]) for k in dumps[0])
    out = dumps[0]
    assert np.array_equal(out["case_index"], np.arange(4096)) and np.all(out["sweeps"] == 20)
    net = synth.alarm37()
    _, _, evkw, sweeps = synth.WORKLOADS["alarm37"]
    ev = synth.make_evidence(net, 4096, **evkw)
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=sweeps, threads=0)
    from helpers import assert_close
    assert_close(out["marginals"], want, rtol=1e-9, atol=1e-12, what="bench.py --dump-outputs vs oracle")
