"""Log-evidence (the Bethe estimate log Z_B of ln P(e), include/bnbp.h) in its reference computation
(tests/logev_oracle.c, over the oracle's BP restatement), against closed forms and exact enumeration of ln P(e) on
polytrees, where BP run to its fixed point makes it exact.  No GPU needed; the GPU side is
tests/test_gpu_log_evidence.py."""
import math

import numpy as np
import pytest

import edge_networks as E
import logev_oracle
from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.flat import EvidenceBatch, FlatNetwork


def brute_log_p(net: FlatNetwork, case: dict) -> float:
    """ln P(e) by summing the joint distribution over every unobserved state."""
    n = net.n_nodes
    shape = [int(c) for c in net.card]
    joint = np.ones(shape)
    for x in range(n):
        axes = [int(u) for u in net.parents[net.parent_off[x]:net.parent_off[x + 1]]] + [x]
        f = net.cpt[net.cpt_off[x]:net.cpt_off[x + 1]].reshape([shape[a] for a in axes])
        f = f.transpose(np.argsort(axes))
        bshape = [1] * n
        for a in axes:
            bshape[a] = shape[a]
        joint = joint * f.reshape(bshape)
    total = joint[tuple(case.get(i, slice(None)) for i in range(n))].sum()
    with np.errstate(divide="ignore"):
        return float(np.log(total))


def cases_of(ev: EvidenceBatch):
    return [{int(ev.ev_node[e]): int(ev.ev_state[e]) for e in range(ev.ev_off[c], ev.ev_off[c + 1])}
            for c in range(ev.n_cases)]


def oracle_logev(net, cases, **kw):
    """Default: a fixed 3n + 3 sweeps, past the polytree's exact fixed point.  The reference's stopping rule looks at the
    messages only, and on a polytree they can stand still for one sweep while a pi / lambda row further out is still
    changing (random_polytree seed 6, evidence 5 = 2: delta 0 at sweep 7, node 4's marginal 8e-6 off, settled at 9)."""
    ev = EvidenceBatch.from_cases(net, cases)
    kw.setdefault("eps", 0.0)
    kw.setdefault("max_sweeps", 3 * net.n_nodes + 3)
    return logev_oracle.run(net, ev, **kw)


def bar(L):
    return 1e-10 * max(1.0, abs(L))


def test_two_nodes_closed_form():
    # A -> B, evidence B = s: family B gives ln P(s) - sum_a P(a|s) ln P(a), family A sum_a P(a|s) ln P(a)
    pa = [0.3, 0.7]
    pba = [[0.9, 0.1], [0.2, 0.8]]
    net = FlatNetwork.from_lists(card=[2, 2], parents=[[], [0]], cpts=[pa, sum(pba, [])], name="ab")
    for s in (0, 1):
        ps = sum(pa[a] * pba[a][s] for a in range(2))
        post = [pa[a] * pba[a][s] / ps for a in range(2)]
        fam_b = math.log(ps) - sum(post[a] * math.log(pa[a]) for a in range(2))
        fam_a = sum(post[a] * math.log(pa[a]) for a in range(2))
        _, _, conv, le = oracle_logev(net, [{1: s}], eps=1e-14, max_sweeps=100)
        assert conv[0] == 1
        assert abs(fam_a + fam_b - math.log(ps)) < 1e-15
        assert abs(le[0] - math.log(ps)) <= bar(le[0]), (s, le[0], math.log(ps))
    # no evidence: ln 1
    _, _, _, le = oracle_logev(net, [{}])
    assert abs(le[0]) < 1e-14


def test_chain_closed_form():
    # A -> B -> C: P(C = c) and P(A = a, C = c) by hand
    pa = np.array([0.25, 0.75])
    pba = np.array([[0.6, 0.3, 0.1], [0.2, 0.2, 0.6]])
    pcb = np.array([[0.5, 0.5], [0.9, 0.1], [0.15, 0.85]])
    net = FlatNetwork.from_lists(card=[2, 3, 2], parents=[[], [0], [1]],
                                 cpts=[pa.tolist(), pba.ravel().tolist(), pcb.ravel().tolist()], name="chain3")
    for c in (0, 1):
        want = math.log(float(pa @ pba @ pcb[:, c]))
        _, _, _, le = oracle_logev(net, [{2: c}])
        assert abs(le[0] - want) <= bar(want)
        for a in (0, 1):
            want = math.log(float(pa[a] * (pba[a] @ pcb[:, c])))
            _, _, _, le = oracle_logev(net, [{0: a, 2: c}])
            assert abs(le[0] - want) <= bar(want)


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6])
def test_polytree_against_enumeration(seed):
    net = synth.random_polytree(8 + seed % 3, card_hi=4, max_parents=3, seed=seed)
    assert E.is_polytree(net)
    cases = [{}] + cases_of(synth.make_evidence(net, 24, p=0.3, seed=seed + 100))
    _, _, _, le = oracle_logev(net, cases)
    for c, case in enumerate(cases):
        want = brute_log_p(net, case)
        assert abs(le[c] - want) <= bar(want), (seed, case, le[c], want)


def test_determ_contradiction_is_minus_inf():
    net = E.catalogue()["determ"]
    # polytree component 5 -> 6 -> 7: 6 copies 5 exactly, 7 = NOT 6 up to 1e-12
    cases = [{5: 0, 6: 1}, {5: 1, 6: 0}, {6: 0, 7: 0}, {5: 1, 7: 0}, {7: 1}]
    _, _, _, le = oracle_logev(net, cases)
    for c, case in enumerate(cases):
        want = brute_log_p(net, case)
        if math.isinf(want):
            assert le[c] == -math.inf, (case, le[c])
        else:
            assert abs(le[c] - want) <= bar(want), (case, le[c], want)
    assert le[0] == -math.inf and le[1] == -math.inf and np.isfinite(le[2:]).all()


def test_damping_and_check_interval_keep_the_fixed_point():
    net = synth.random_polytree(9, card_hi=4, max_parents=3, seed=11)
    cases = [{}] + cases_of(synth.make_evidence(net, 16, p=0.3, seed=12))
    _, _, _, base = oracle_logev(net, cases)
    _, _, conv_d, damped = oracle_logev(net, cases, eps=1e-14, damping=0.2, max_sweeps=5000)
    _, _, conv_i, every3 = oracle_logev(net, cases, eps=1e-14, check_interval=3, max_sweeps=500)
    assert conv_d.all() and conv_i.all()
    for c, case in enumerate(cases):
        want = brute_log_p(net, case)
        for got in (base[c], damped[c], every3[c]):
            assert abs(got - want) <= bar(want), (case, got, want)


def test_reference_runs_the_pinned_oracle_bp(oracle_mod):
    # the log-evidence reference scores the very state the pinned restatement ends with
    net = synth.alarm37()
    ev = synth.make_evidence(net, 64, exact_k=4, seed=3)
    m0, s0, c0 = oracle_mod.run_port(net, ev, eps=1e-6, max_sweeps=100, threads=0)
    m1, s1, c1, le = logev_oracle.run(net, ev, eps=1e-6, max_sweeps=100)
    assert np.array_equal(m0, m1) and np.array_equal(s0, s1) and np.array_equal(c0, c1)
    assert np.isfinite(le).all() and (le < 0).all()
