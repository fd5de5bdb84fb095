"""Per-case log-evidence (bnbp_run_batch_log_evidence / _device_log_evidence, include/bnbp.h) on the GPU against its
reference computation (tests/logev_oracle.c over the oracle's BP restatement) -- needs a B200 (-m gpu).

Bars: fp64 1e-9 * max(1, |L|) + 1e-12; fp32 1e-4 * max(1, |L|) (DESIGN section 10 records the largest fp32 error seen).
Every run asserts the kernel family it ran through (stats): log-evidence never takes the on-chip kernel or the fused
first / last sweeps."""
import os
import subprocess

import numpy as np
import pytest

from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.flat import EvidenceBatch
from helpers import assert_close

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MTOL = {"fp64": dict(rtol=1e-9, atol=1e-12), "fp32": dict(rtol=1e-5, atol=1e-6)}


def le_bar(precision, ref):
    a = np.where(np.isfinite(ref), np.maximum(1.0, np.abs(ref)), 1.0)
    return 1e-9 * a + 1e-12 if precision == "fp64" else 1e-4 * a


def assert_le(got, ref, precision, what=""):
    same_special = (np.isnan(got) & np.isnan(ref)) | (np.isinf(got) & (got == ref))
    assert np.array_equal(np.isfinite(got), np.isfinite(ref)) and same_special[~np.isfinite(ref)].all(), what
    f = np.isfinite(ref)
    err = np.abs(got[f] - ref[f])
    bad = err > le_bar(precision, ref[f])
    assert not bad.any(), (what, int(bad.sum()), float(err.max()))
    return float(err.max()) if err.size else 0.0


def check(bp, net, ev, precision, eps, cap, what, spec=None, **kw):
    """One log-evidence run against the oracle; asserts the family from stats().  Returns (result, stats, max error)."""
    import logev_oracle
    res = bp(ev, eps, max_sweeps=cap, log_evidence=True, **kw)
    st = bp.stats()
    assert st["last_onchip"] == 0 and st["last_fused"] == 0, (what, st["last_onchip"], st["last_fused"])
    if spec is not None:
        assert st["last_specialised"] == spec, (what, st["last_specialised"])
    om, osw, ocv, ole = logev_oracle.run(net, ev, eps=eps, max_sweeps=cap, damping=kw.get("damping", 0.0),
                                         check_interval=kw.get("check_interval", 1))
    if precision == "fp64":
        assert np.array_equal(res.sweeps, osw), what
        assert np.array_equal(res.converged, ocv), what
    if res.marginals.shape[1]:
        assert_close(res.marginals, om, what=what, **MTOL[precision])
    return res, st, assert_le(res.log_evidence, ole, precision, what)


def BP(*a, **k):
    from bayesiannetwork_b200.engine import BeliefPropagation
    return BeliefPropagation(*a, **k)


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("specialize", ["never", "always"])
def test_alarm37_settings(precision, specialize):
    net = synth.alarm37()
    ev = synth.make_evidence(net, 3000, exact_k=4, seed=21)
    bp = BP(net, precision, specialize=specialize)
    spec = 1 if specialize == "always" else 0
    worst = 0.0
    for T in (1, 2, 3, 20):
        worst = max(worst, check(bp, net, ev, precision, 0.0, T, f"fixed {T}", spec)[2])
    if precision == "fp64":
        for interval in (1, 3):
            check(bp, net, ev, precision, 1e-7, 200, f"eps interval {interval}", spec, check_interval=interval)
        check(bp, net, ev, precision, 1e-7, 300, "eps damping", spec, damping=0.2)
    check(bp, net, ev, precision, 0.0, 20, "fixed damping", spec, damping=0.2)
    print(f"alarm37 {precision} {specialize}: max |log-evidence error| at fixed sweeps {worst:.3g}")


def test_alarm37_compaction_and_chunks():
    net = synth.alarm37()
    ev = synth.make_evidence(net, 24000, exact_k=4, seed=22)
    for spec in ("never", "always"):
        bp = BP(net, "fp64", specialize=spec)
        _, st, _ = check(bp, net, ev, "fp64", 1e-7, 200, f"eps {spec} compaction")
        assert st["last_compactions"] >= 1, spec
    bp = BP(net, "fp64", max_resident_cases=5120)
    _, st, _ = check(bp, net, ev, "fp64", 1e-7, 200, "eps chunks")
    _, st, _ = check(bp, net, ev, "fp64", 0.0, 20, "fixed chunks")


def test_alarm37_auto_streams_and_marginals_off():
    net = synth.alarm37()
    ev = synth.make_evidence(net, 4608, exact_k=4, seed=23)
    bp = BP(net, "fp64")
    res, st, _ = check(bp, net, ev, "fp64", 0.0, 20, "AUTO", spec=1)
    plain = bp(ev, 0.0, max_sweeps=20)
    assert bp.stats()["last_onchip"] == 1                       # the same call without log-evidence keeps the on-chip kernel
    assert np.array_equal(plain.marginals, res.marginals) or np.allclose(plain.marginals, res.marginals, rtol=1e-9, atol=1e-12)
    only = bp(ev, 0.0, max_sweeps=20, log_evidence=True, marginals=False)
    assert only.marginals.shape == (ev.n_cases, 0)
    assert np.array_equal(only.log_evidence, res.log_evidence)
    assert np.array_equal(only.sweeps, res.sweeps) and np.array_equal(only.converged, res.converged)
    q = bp(ev, 0.0, max_sweeps=20, log_evidence=True, query_nodes=[5, 1, 30])
    assert np.array_equal(q.log_evidence, res.log_evidence)
    off = net.belief_off
    assert np.array_equal(q.marginals, np.concatenate([res.marginals[:, off[x]:off[x + 1]] for x in (5, 1, 30)], axis=1))
    for eps in (1e-7, 0.0):                                     # epsilon mode: cases retire at their own sweeps
        a = bp(ev, eps, max_sweeps=100, log_evidence=True)
        b = bp(ev, eps, max_sweeps=100, log_evidence=True, marginals=False)
        assert np.array_equal(a.log_evidence, b.log_evidence) and np.array_equal(a.sweeps, b.sweeps)


def test_polytree_matches_enumeration():
    from test_log_evidence import brute_log_p, cases_of
    net = synth.random_polytree(10, card_hi=4, max_parents=3, seed=7)
    cases = [{}] + cases_of(synth.make_evidence(net, 500, p=0.3, seed=8))
    ev = EvidenceBatch.from_cases(net, cases)
    want = np.array([brute_log_p(net, c) for c in cases])
    for spec in ("never", "always"):
        for precision in ("fp64", "fp32"):
            bp = BP(net, precision, specialize=spec)
            res, _, _ = check(bp, net, ev, precision, 0.0, 40, f"polytree {spec} {precision}", 1 if spec == "always" else 0)
            assert_le(res.log_evidence, want, precision, "polytree vs enumeration")


def test_grid_class_looped(monkeypatch):
    monkeypatch.setenv("BNBP_CLASSLOOP", "2")
    net = synth.grid(20)
    ev = synth.make_evidence(net, 2048, p=0.1, seed=24)
    for precision in ("fp64", "fp32"):
        bp = BP(net, precision, specialize="always")
        _, st, _ = check(bp, net, ev, precision, 0.0, 20, f"grid20 {precision}", 1)
        assert st["spec_class_count"] > 0
    bp = BP(net, "fp64", specialize="always")
    _, st, _ = check(bp, net, ev, "fp64", 1e-7, 200, "grid20 eps", 1)
    assert st["spec_class_count"] > 0


def test_card100_generic():
    net = synth._assemble([100, 100, 3, 100, 7], [[], [0], [], [1, 2], [3]], 31, "card100")
    ev = synth.make_evidence(net, 1500, p=0.3, seed=25)
    for precision in ("fp64", "fp32"):
        bp = BP(net, precision, dense_min_cpt=-1)
        check(bp, net, ev, precision, 0.0, 5, f"card100 {precision}", 0)
    bp = BP(net, "fp64", dense_min_cpt=-1)
    check(bp, net, ev, "fp64", 1e-7, 100, "card100 eps", 0)


def test_device_path_bit_identical():
    import torch
    net = synth.alarm37()
    ev = synth.make_evidence(net, 6000, exact_k=4, seed=26)
    bp = BP(net, "fp64")
    for eps in (0.0, 1e-7):
        host = bp(ev, eps, max_sweeps=50, log_evidence=True)
        dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(ev, k))).cuda() for k in ("ev_off", "ev_node", "ev_state")}
        le = torch.empty(ev.n_cases, dtype=torch.float64, device="cuda")
        out = torch.empty((ev.n_cases, net.belief_values), dtype=torch.float64, device="cuda")
        sw = torch.empty(ev.n_cases, dtype=torch.int32, device="cuda")
        bp.run_device(ev.n_cases, dev["ev_off"], dev["ev_node"], dev["ev_state"], out, epsilon=eps, max_sweeps=50,
                      out_sweeps=sw, out_log_evidence=le)
        torch.cuda.synchronize()
        assert np.array_equal(le.cpu().numpy(), host.log_evidence), eps
        assert np.array_equal(out.cpu().numpy(), host.marginals) and np.array_equal(sw.cpu().numpy(), host.sweeps)
        le2 = torch.full((ev.n_cases,), 7.0, dtype=torch.float64, device="cuda")
        bp.run_device(ev.n_cases, dev["ev_off"], dev["ev_node"], dev["ev_state"], None, epsilon=eps, max_sweeps=50,
                      out_log_evidence=le2)
        torch.cuda.synchronize()
        assert np.array_equal(le2.cpu().numpy(), host.log_evidence), eps


def test_refusals_name_their_reason():
    from bayesiannetwork_b200.engine import BnbpError
    net = synth.alarm37()
    ev = synth.make_evidence(net, 64, exact_k=4, seed=27)
    bp = BP(net, "fp64")
    soft = EvidenceBatch.from_cases(net, [{0: [0.5] * int(net.card[0])}])
    with pytest.raises(BnbpError, match="hard evidence"):
        bp(soft, 0.0, max_sweeps=5, log_evidence=True)
    with pytest.raises(BnbpError, match="MAX_PRODUCT"):
        bp(ev, 0.0, max_sweeps=5, log_evidence=True, semiring="max")
    with pytest.raises(BnbpError, match="onchip=ALWAYS"):
        BP(net, "fp64", onchip="always")(ev, 0.0, max_sweeps=5, log_evidence=True)
    dense = BP(synth._assemble([8, 8, 8, 8], [[], [], [], [0, 1, 2]], 32, "dense"), "fp64", dense_min_cpt=16)
    with pytest.raises(BnbpError, match="dense_min_cpt = -1"):
        dense(synth.make_evidence(dense.net, 8, p=0.3, seed=1), 0.0, max_sweeps=5, log_evidence=True)
    import torch
    d = {k: torch.from_numpy(np.ascontiguousarray(getattr(ev, k))).cuda() for k in ("ev_off", "ev_node", "ev_state")}
    with pytest.raises(BnbpError, match="gather"):
        bp.run_device(ev.n_cases, d["ev_off"], d["ev_node"], d["ev_state"], None, max_sweeps=5, gather=True,
                      out_log_evidence=torch.empty(ev.n_cases, dtype=torch.float64, device="cuda"))
    # the handle still works, with and without log-evidence
    check(bp, net, ev, "fp64", 0.0, 5, "after refusals")
    r = bp(ev, 0.0, max_sweeps=5)
    assert r.log_evidence is None and np.isfinite(r.marginals).all()


def test_group_handle_bit_identical():
    from bayesiannetwork_b200.engine import device_count
    if device_count() < 2:
        pytest.skip("needs 2 devices")
    net = synth.alarm37()
    ev = synth.make_evidence(net, 10000, exact_k=4, seed=28)
    one = BP(net, "fp64")(ev, 1e-7, max_sweeps=100, log_evidence=True)
    two = BP(net, "fp64", devices=[0, 1])(ev, 1e-7, max_sweeps=100, log_evidence=True)
    assert np.array_equal(one.log_evidence, two.log_evidence) and np.array_equal(one.marginals, two.marginals)
    three = BP(net, "fp64", devices=[0, 1])(ev, 1e-7, max_sweeps=100, log_evidence=True, marginals=False)
    assert np.array_equal(one.log_evidence, three.log_evidence)


def test_cpp_dropin_log_evidence(tmp_path):
    exe = tmp_path / "logev"
    subprocess.run(["g++", "-std=c++11", "-Wall", "-Wextra", "-Werror", "-O2", "-I" + os.path.join(ROOT, "include"),
                    "-I" + os.path.join(ROOT, "tests", "cpp"), "-o", str(exe),
                    os.path.join(ROOT, "tests", "cpp", "test_dropin_logev.cpp"),
                    "-L" + os.path.join(ROOT, "bayesiannetwork_b200", "lib"), "-lbnbp",
                    "-Wl,-rpath," + os.path.join(ROOT, "bayesiannetwork_b200", "lib")], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    cpp = np.array([float(v) for v in out[1::2]])
    net = synth.resume_network()
    ev = EvidenceBatch.from_cases(net, [{3: 0}, {3: 1}, {3: 2}, {0: 1, 2: 0}, {}])
    py = BP(net, "fp64")(ev, 0.0, max_sweeps=20, log_evidence=True)
    assert np.array_equal(cpp, py.log_evidence), (cpp, py.log_evidence)
    from test_log_evidence import brute_log_p
    want = np.array([brute_log_p(net, c) for c in ({3: 0}, {3: 1}, {3: 2}, {0: 1, 2: 0}, {})])
    assert_le(cpp, want, "fp64", "chain vs enumeration")
