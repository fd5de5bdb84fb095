"""Expected family counts (bnbp_run_batch_expected_counts / _device_expected_counts, include/bnbp.h) and EM
(BeliefPropagation.em) on the GPU against the reference computation (tests/em_oracle.c over the oracle's BP
restatement) -- needs a B200 (-m gpu).

Bars on counts: fp64 |d| <= 1e-9 * max(1, |c|); fp32 <= 1e-4 * max(1, |c|).  The counts are summed with atomics, so
they are compared with tolerances, never bit for bit.  Log-evidence, sweeps and flags are checked as
tests/test_gpu_log_evidence.py checks them.  Every run asserts from stats() that it ran the streaming kernels:
no on-chip kernel, no fused first / last sweep."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.flat import EvidenceBatch
from test_gpu_log_evidence import assert_le

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CTOL = {"fp64": 1e-9, "fp32": 1e-4}

# Mean |CPT - generating CPT| after the 30 EM iterations of the recovery problem (test_em.RECOVERY), calibrated on the
# CPU with the reference computation (scripts/em_recovery_calibrate.py, profiles/r03c_em_recovery_calibration.jsonl):
# 0.1616 at the start, 0.00695 after 30 iterations, the log-likelihood rising at every one.  The bar leaves 1.4x that.
RECOVERY_BAR = 0.01


def BP(*a, **k):
    from bayesiannetwork_b200.engine import BeliefPropagation
    return BeliefPropagation(*a, **k)


def assert_counts(got, ref, precision, what=""):
    err = np.abs(got - ref)
    bad = err > CTOL[precision] * np.maximum(1.0, np.abs(ref))
    assert not bad.any(), (what, int(bad.sum()), float(err.max()))
    return float(err.max())


def assert_streaming(bp, what, spec=None):
    st = bp.stats()
    assert st["last_onchip"] == 0 and st["last_fused"] == 0, (what, st["last_onchip"], st["last_fused"])
    if spec is not None:
        assert st["last_specialised"] == spec, (what, st["last_specialised"])
    return st


def totals(net, counts):
    return np.array([counts[net.cpt_off[x]:net.cpt_off[x + 1]].sum() for x in range(net.n_nodes)])


def check(bp, net, ev, precision, eps, cap, what, spec=None, weights=None, **kw):
    """One expected-counts run against the reference; returns (result, stats)."""
    import em_oracle
    res = bp(ev, eps, max_sweeps=cap, expected_counts=True, log_evidence=True, weights=weights, **kw)
    st = assert_streaming(bp, what, spec)
    ref, om, osw, ocv, ole = em_oracle.run(net, ev, eps=eps, max_sweeps=cap, damping=kw.get("damping", 0.0),
                                           check_interval=kw.get("check_interval", 1), weights=weights)
    if precision == "fp64":
        assert np.array_equal(res.sweeps, osw), what
        assert np.array_equal(res.converged, ocv), what
    assert_le(res.log_evidence, ole, precision, what)
    assert_counts(res.expected_counts, ref, precision, what)
    return res, st


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("specialize", ["never", "always"])
def test_alarm37_settings(precision, specialize):
    net = synth.alarm37()
    ev = synth.make_evidence(net, 3000, exact_k=4, seed=51)
    w = np.random.default_rng(52).uniform(0.0, 2.0, ev.n_cases)
    bp = BP(net, precision, specialize=specialize)
    spec = 1 if specialize == "always" else 0
    for T in (1, 2, 20):
        check(bp, net, ev, precision, 0.0, T, f"fixed {T}", spec)
    check(bp, net, ev, precision, 0.0, 20, "fixed 20 weighted", spec, weights=w)
    check(bp, net, ev, precision, 0.0, 20, "fixed damping", spec, damping=0.2)
    if precision == "fp64":                    # fp32 does not reach delta < 1e-7 where the fp64 reference does
        for interval in (1, 3):
            check(bp, net, ev, precision, 1e-7, 200, f"eps interval {interval}", spec, check_interval=interval)
        check(bp, net, ev, precision, 1e-7, 300, "eps damping", spec, damping=0.2, weights=w)


def test_calls_without_counts_keep_their_kernels():
    net = synth.alarm37()
    ev = synth.make_evidence(net, 4608, exact_k=4, seed=53)
    bp = BP(net, "fp64")
    res = bp(ev, 0.0, max_sweeps=20, expected_counts=True, marginals=False)
    assert_streaming(bp, "AUTO with counts", spec=1)
    assert res.marginals.shape == (ev.n_cases, 0) and res.log_evidence is None
    plain = bp(ev, 0.0, max_sweeps=20)
    assert bp.stats()["last_onchip"] == 1                      # the same call without counts keeps the on-chip kernel
    assert np.allclose(totals(net, res.expected_counts), ev.n_cases, rtol=1e-12)
    full = bp(ev, 0.0, max_sweeps=20, expected_counts=True)    # invariant 1 against this call's own marginals
    off = net.belief_off
    for x in range(net.n_nodes):
        per_x = full.expected_counts[net.cpt_off[x]:net.cpt_off[x + 1]].reshape(-1, int(net.card[x])).sum(axis=0)
        assert np.allclose(per_x, full.marginals[:, off[x]:off[x + 1]].sum(axis=0), rtol=1e-10, atol=1e-9), x
    assert np.allclose(plain.marginals, full.marginals, rtol=1e-9, atol=1e-12)


def test_alarm37_compaction_and_chunks():
    net = synth.alarm37()
    ev = synth.make_evidence(net, 24000, exact_k=4, seed=54)
    for spec in ("never", "always"):
        bp = BP(net, "fp64", specialize=spec)
        res = bp(ev, 1e-7, max_sweeps=200, expected_counts=True, log_evidence=True, marginals=False)
        st = assert_streaming(bp, f"eps {spec} compaction")
        assert st["last_compactions"] >= 1, spec
        assert np.allclose(totals(net, res.expected_counts), ev.n_cases, rtol=1e-10), spec   # nobody twice or missed
    bp = BP(net, "fp64", max_resident_cases=5120)
    check(bp, net, ev, "fp64", 1e-7, 200, "eps chunks")
    for eps in (1e-7, 0.0):
        res = bp(ev, eps, max_sweeps=50, expected_counts=True, marginals=False)
        assert_streaming(bp, f"chunks {eps}")
        assert np.allclose(totals(net, res.expected_counts), ev.n_cases, rtol=1e-10), eps


def test_polytree_matches_enumeration():
    from test_em import brute_family_counts
    from test_log_evidence import cases_of
    net = synth.random_polytree(8, card_hi=4, max_parents=3, seed=9)
    cases = [{}] + cases_of(synth.make_evidence(net, 150, p=0.3, seed=10))
    ev = EvidenceBatch.from_cases(net, cases)
    want = brute_family_counts(net, cases)
    for spec in ("never", "always"):
        for precision in ("fp64", "fp32"):
            bp = BP(net, precision, specialize=spec)
            res, _ = check(bp, net, ev, precision, 0.0, 3 * net.n_nodes + 3, f"polytree {spec} {precision}",
                           1 if spec == "always" else 0)
            assert_counts(res.expected_counts, want, precision, "polytree vs enumeration")


def test_grid_class_looped(monkeypatch):
    monkeypatch.setenv("BNBP_CLASSLOOP", "2")
    net = synth.grid(20)
    ev = synth.make_evidence(net, 2048, p=0.1, seed=55)
    for precision in ("fp64", "fp32"):
        bp = BP(net, precision, specialize="always")
        _, st = check(bp, net, ev, precision, 0.0, 20, f"grid20 {precision}", 1)
        assert st["spec_class_count"] > 0


def test_card100_generic():
    net = synth._assemble([100, 100, 3, 100, 7], [[], [0], [], [1, 2], [3]], 31, "card100")
    ev = synth.make_evidence(net, 1500, p=0.3, seed=56)
    for precision in ("fp64", "fp32"):
        bp = BP(net, precision, dense_min_cpt=-1)
        check(bp, net, ev, precision, 0.0, 5, f"card100 {precision}", 0)
    bp = BP(net, "fp64", dense_min_cpt=-1)
    check(bp, net, ev, "fp64", 1e-7, 100, "card100 eps", 0)


def test_device_call_adds_into_and_weights():
    import torch
    net = synth.alarm37()
    ev = synth.make_evidence(net, 6000, exact_k=4, seed=57)
    w = np.random.default_rng(58).uniform(0.0, 2.0, ev.n_cases)
    bp = BP(net, "fp64")
    nv = int(net.cpt_off[-1])
    for eps in (0.0, 1e-7):
        host = bp(ev, eps, max_sweeps=50, expected_counts=True, log_evidence=True, weights=w)
        dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(ev, k))).cuda() for k in ("ev_off", "ev_node", "ev_state")}
        wd = torch.from_numpy(w).cuda()
        cnt = torch.full((nv,), 1.5, dtype=torch.float64, device="cuda")       # adds into what is there
        le = torch.empty(ev.n_cases, dtype=torch.float64, device="cuda")
        sw = torch.empty(ev.n_cases, dtype=torch.int32, device="cuda")
        bp.run_device(ev.n_cases, dev["ev_off"], dev["ev_node"], dev["ev_state"], None, epsilon=eps, max_sweeps=50,
                      out_sweeps=sw, out_log_evidence=le, out_counts=cnt, case_weights=wd)
        torch.cuda.synchronize()
        assert_streaming(bp, f"device {eps}")
        assert_counts(cnt.cpu().numpy() - 1.5, host.expected_counts, "fp64", f"device vs host {eps}")
        assert np.array_equal(le.cpu().numpy(), host.log_evidence) and np.array_equal(sw.cpu().numpy(), host.sweeps)
    # host call: two halves into one array = one call; weight 2 = the case twice, weight 0 = the case left out
    h = ev.n_cases // 2
    acc = np.zeros(nv)
    bp(ev.slice(0, h), 0.0, max_sweeps=20, expected_counts=True, marginals=False, weights=w[:h], counts_out=acc)
    r = bp(ev.slice(h, ev.n_cases), 0.0, max_sweeps=20, expected_counts=True, marginals=False, weights=w[h:], counts_out=acc)
    assert r.expected_counts is acc
    one = bp(ev, 0.0, max_sweeps=20, expected_counts=True, marginals=False, weights=w)
    assert_counts(acc, one.expected_counts, "fp64", "two halves")
    w2 = np.ones(ev.n_cases)
    w2[:100] = 2.0
    w2[100:200] = 0.0
    a = bp(ev, 0.0, max_sweeps=20, expected_counts=True, marginals=False, weights=w2).expected_counts
    acc = np.zeros(nv)
    for lo, hi in ((0, 100), (0, 100), (200, ev.n_cases)):      # cases 0-99 twice, 100-199 not at all
        bp(ev.slice(lo, hi), 0.0, max_sweeps=20, expected_counts=True, marginals=False, counts_out=acc)
    assert_counts(a, acc, "fp64", "weights 2 and 0")


def test_refusals_name_their_reason():
    from bayesiannetwork_b200 import _capi
    from bayesiannetwork_b200.engine import BnbpError
    net = synth.alarm37()
    ev = synth.make_evidence(net, 64, exact_k=4, seed=59)
    bp = BP(net, "fp64")
    soft = EvidenceBatch.from_cases(net, [{0: [0.5] * int(net.card[0])}])
    with pytest.raises(BnbpError, match="hard evidence"):
        bp(soft, 0.0, max_sweeps=5, expected_counts=True)
    with pytest.raises(BnbpError, match="MAX_PRODUCT"):
        bp(ev, 0.0, max_sweeps=5, expected_counts=True, semiring="max")
    with pytest.raises(BnbpError, match="onchip=ALWAYS"):
        BP(net, "fp64", onchip="always")(ev, 0.0, max_sweeps=5, expected_counts=True)
    dense = BP(synth._assemble([8, 8, 8, 8], [[], [], [], [0, 1, 2]], 32, "dense"), "fp64", dense_min_cpt=16)
    with pytest.raises(BnbpError, match="dense_min_cpt = -1"):
        dense(synth.make_evidence(dense.net, 8, p=0.3, seed=1), 0.0, max_sweeps=5, expected_counts=True)
    bad_w = np.ones(ev.n_cases)
    bad_w[5] = -1.0
    with pytest.raises(BnbpError, match="case_weights"):
        bp(ev, 0.0, max_sweeps=5, expected_counts=True, weights=bad_w)
    bad_w[5] = np.nan
    with pytest.raises(BnbpError, match="case_weights"):
        bp(ev, 0.0, max_sweeps=5, expected_counts=True, weights=bad_w)
    evc = _capi.EvidenceC(ev.n_cases, ev.ev_off.ctypes.data, ev.ev_node.ctypes.data, ev.ev_state.ctypes.data, None, None)
    prm = _capi.RunParamsC(0.0, 5, 0.0, 1, 0, 0, 0, None, 0)
    with pytest.raises(BnbpError, match="counts is NULL"):
        _capi.check(bp._lib.bnbp_run_batch_expected_counts(bp._h, C.byref(evc), C.byref(prm), None, None, None, None,
                                                           None, None))
    import torch
    d = {k: torch.from_numpy(np.ascontiguousarray(getattr(ev, k))).cuda() for k in ("ev_off", "ev_node", "ev_state")}
    with pytest.raises(BnbpError, match="gather"):
        bp.run_device(ev.n_cases, d["ev_off"], d["ev_node"], d["ev_state"], None, max_sweeps=5, gather=True,
                      out_counts=torch.zeros(int(net.cpt_off[-1]), dtype=torch.float64, device="cuda"))
    with pytest.raises(BnbpError, match="counts is NULL"):
        _capi.check(bp._lib.bnbp_run_batch_device_expected_counts(bp._h, C.byref(evc), C.byref(prm), None, None, None,
                                                                  None, None, None, None))
    # the handle still works, with and without counts
    check(bp, net, ev, "fp64", 0.0, 5, "after refusals")
    r = bp(ev, 0.0, max_sweeps=5)
    assert r.expected_counts is None and np.isfinite(r.marginals).all()


def test_group_handle_matches_one_device():
    from bayesiannetwork_b200.engine import device_count
    if device_count() < 2:
        pytest.skip("needs 2 devices")
    net = synth.alarm37()
    ev = synth.make_evidence(net, 10000, exact_k=4, seed=60)
    w = np.random.default_rng(61).uniform(0.0, 2.0, ev.n_cases)
    one = BP(net, "fp64")(ev, 1e-7, max_sweeps=100, expected_counts=True, log_evidence=True, weights=w)
    two = BP(net, "fp64", devices=[0, 1])(ev, 1e-7, max_sweeps=100, expected_counts=True, log_evidence=True, weights=w)
    assert np.array_equal(one.log_evidence, two.log_evidence) and np.array_equal(one.marginals, two.marginals)
    assert_counts(two.expected_counts, one.expected_counts, "fp64", "group")
    acc = np.full(int(net.cpt_off[-1]), 2.0)
    BP(net, "fp64", devices=[0, 1])(ev, 1e-7, max_sweeps=100, expected_counts=True, marginals=False, weights=w,
                                    counts_out=acc)
    assert_counts(acc - 2.0, one.expected_counts, "fp64", "group adds into")


def test_em_on_a_specialised_handle_compiles_once():
    import em_oracle
    from bayesiannetwork_b200.engine import m_step
    from test_em import random_rows, with_cpt
    net = synth.alarm37()
    ev = synth.make_evidence(net, 4096, exact_k=6, seed=62)
    bp = BP(net, "fp64", specialize="always")
    cur = random_rows(net, seed=63)
    bp.refresh_cpt(cur)
    compile_ms = []
    for it in range(4):
        res = bp(ev, 1e-6, max_sweeps=200, expected_counts=True, log_evidence=True, marginals=False)
        st = assert_streaming(bp, f"iteration {it}", spec=1)
        compile_ms.append(st["spec_compile_ms"])
        ref, _, osw, _, ole = em_oracle.run(with_cpt(net, cur), ev, eps=1e-6, max_sweeps=200)
        assert np.array_equal(res.sweeps, osw), it
        assert_le(res.log_evidence, ole, "fp64", f"iteration {it}")
        assert_counts(res.expected_counts, ref, "fp64", f"iteration {it}")
        cur = m_step(net, res.expected_counts)
        bp.refresh_cpt(cur)
    assert all(c == compile_ms[0] for c in compile_ms[1:]), compile_ms
    r = bp.em(ev, iterations=5, tol=0.0)
    assert bp.stats()["spec_compile_ms"] == compile_ms[0]
    assert r.iterations >= 2 and r.skipped.sum() == 0 and r.log_likelihood.shape == (r.iterations,)
    assert not np.shares_memory(r.cpt, net.cpt) and np.array_equal(net.cpt, synth.alarm37().cpt)   # net untouched


def test_em_recovers_the_generating_cpt():
    import test_em
    net, ev, start = test_em.recovery_problem()
    for precision in ("fp64", "fp32"):
        bp = BP(net, precision)
        r = bp.em(ev, iterations=test_em.RECOVERY["iterations"], tol=-np.inf, cpt=start)
        assert r.iterations == test_em.RECOVERY["iterations"]
        assert_streaming(bp, f"recovery {precision}")
        ll = r.log_likelihood
        assert (np.diff(ll[:6]) > 0).all(), (precision, ll[:6])
        mae = float(np.abs(r.cpt - net.cpt).mean())
        print(f"recovery {precision}: {r.iterations} iterations, L {ll[0]:.6g} -> {ll[-1]:.6g}, "
              f"mean |CPT error| {np.abs(start - net.cpt).mean():.4g} -> {mae:.4g} (bar {RECOVERY_BAR})")
        assert mae < RECOVERY_BAR, (precision, mae)
        # the handle holds the returned CPT
        again = bp(ev.slice(0, 4096), 1e-6, max_sweeps=200, log_evidence=True, marginals=False)
        bp2 = BP(net, precision)
        bp2.refresh_cpt(r.cpt)
        assert_le(again.log_evidence, bp2(ev.slice(0, 4096), 1e-6, max_sweeps=200, log_evidence=True,
                                          marginals=False).log_evidence, precision, "handle holds the EM result")


def test_cpp_dropin_em(tmp_path):
    exe = tmp_path / "em"
    subprocess.run(["g++", "-std=c++11", "-Wall", "-Wextra", "-Werror", "-O2", "-I" + os.path.join(ROOT, "include"),
                    "-I" + os.path.join(ROOT, "tests", "cpp"), "-o", str(exe),
                    os.path.join(ROOT, "tests", "cpp", "test_dropin_em.cpp"),
                    "-L" + os.path.join(ROOT, "bayesiannetwork_b200", "lib"), "-lbnbp",
                    "-Wl,-rpath," + os.path.join(ROOT, "bayesiannetwork_b200", "lib")], check=True)
    lines = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    cpp_ll = np.array([float(l.split()[1]) for l in lines if l.startswith("L ")])
    cpp_cpt = np.array([float(v) for v in lines[-1].split()[1:]])
    net = synth.resume_network()
    cases = [{3: 0}, {3: 1}, {3: 2}, {0: 1, 2: 0}, {}, {0: 0, 1: 2}, {1: 1, 3: 2}, {0: 2, 2: 1, 3: 0}]
    ev = EvidenceBatch.from_cases(net, cases)
    py = BP(net, "fp64").em(ev, iterations=3, tol=-np.inf, epsilon=0.0, max_sweeps=20)
    assert py.iterations == 3
    assert np.allclose(cpp_ll, py.log_likelihood, rtol=1e-12, atol=1e-12), (cpp_ll, py.log_likelihood)
    assert np.allclose(cpp_cpt, py.cpt, rtol=1e-9, atol=1e-12), (cpp_cpt, py.cpt)
