"""Expected family counts (the E-step of EM, bnbp_run_batch_expected_counts in include/bnbp.h) in their reference
computation (tests/em_oracle.c, over the oracle's BP restatement), and the host M-step ``engine.m_step``: against exact
enumeration of P(x, u | e) on polytrees, the invariants every sweep count keeps, make_cpt on complete data, and an EM
loop whose likelihood must not fall.  No GPU needed; the GPU side is tests/test_gpu_em.py."""
import dataclasses

import numpy as np
import pytest

import edge_networks as E
import em_oracle
from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.engine import m_step
from bayesiannetwork_b200.flat import EvidenceBatch, FlatNetwork
from test_log_evidence import cases_of


def with_cpt(net: FlatNetwork, cpt) -> FlatNetwork:
    return dataclasses.replace(net, cpt=np.ascontiguousarray(cpt, dtype=np.float64))


def brute_family_counts(net: FlatNetwork, cases, weights=None) -> np.ndarray:
    """sum_c w_c P(x, u | e_c) in the CPT-arena layout, by conditioning the full joint distribution."""
    n = net.n_nodes
    shape = [int(c) for c in net.card]
    joint = np.ones(shape)
    for x in range(n):
        axes = [int(u) for u in net.parents[net.parent_off[x]:net.parent_off[x + 1]]] + [x]
        f = net.cpt[net.cpt_off[x]:net.cpt_off[x + 1]].reshape([shape[a] for a in axes])
        bshape = [1] * n
        for a in axes:
            bshape[a] = shape[a]
        joint = joint * f.transpose(np.argsort(axes)).reshape(bshape)
    out = np.zeros(int(net.cpt_off[-1]))
    for c, case in enumerate(cases):
        mask = np.zeros(shape, dtype=bool)
        mask[tuple(case.get(i, slice(None)) for i in range(n))] = True
        post = np.where(mask, joint, 0.0)
        tot = post.sum()
        if tot == 0.0:
            continue
        post /= tot
        w = 1.0 if weights is None else float(weights[c])
        for x in range(n):
            axes = [int(u) for u in net.parents[net.parent_off[x]:net.parent_off[x + 1]]] + [x]
            fam = post.sum(axis=tuple(a for a in range(n) if a not in axes))   # axes in increasing node order
            fam = np.transpose(fam, np.argsort(np.argsort(axes)))               # -> (parents..., x)
            out[net.cpt_off[x]:net.cpt_off[x + 1]] += w * fam.ravel()
    return out


def ancestral_sample(net: FlatNetwork, n: int, seed: int) -> np.ndarray:
    """n complete cases [n, N] int32 drawn from the network by seeded ancestral sampling (parents before children)."""
    rng = np.random.default_rng(seed)
    N = net.n_nodes
    out = np.zeros((n, N), dtype=np.int32)
    done = np.zeros(N, dtype=bool)
    while not done.all():
        for x in range(N):
            par = [int(u) for u in net.parents[net.parent_off[x]:net.parent_off[x + 1]]]
            if done[x] or not all(done[u] for u in par):
                continue
            r = int(net.card[x])
            q = np.zeros(n, dtype=np.int64)
            for u in par:
                q = q * int(net.card[u]) + out[:, u]
            rows = net.cpt[net.cpt_off[x]:net.cpt_off[x + 1]].reshape(-1, r)[q]
            cdf = np.cumsum(rows, axis=1)
            cdf[:, -1] = np.inf
            out[:, x] = (rng.random(n)[:, None] >= cdf).sum(axis=1)
            done[x] = True
    return out


def complete_evidence(net: FlatNetwork, samples: np.ndarray) -> EvidenceBatch:
    n, N = samples.shape
    return EvidenceBatch(n, np.arange(n + 1, dtype=np.int64) * N, np.tile(np.arange(N, dtype=np.int32), n),
                         np.ascontiguousarray(samples.ravel(), dtype=np.int32))


def hide_values(samples: np.ndarray, frac: float, seed: int) -> EvidenceBatch:
    """Complete cases with each value hidden independently with probability ``frac`` (seeded)."""
    keep = np.random.default_rng(seed).random(samples.shape) >= frac
    ev_off = np.concatenate([[0], np.cumsum(keep.sum(axis=1))]).astype(np.int64)
    return EvidenceBatch(samples.shape[0], ev_off, np.nonzero(keep)[1].astype(np.int32),
                         np.ascontiguousarray(samples[keep], dtype=np.int32))


def random_rows(net: FlatNetwork, seed: int) -> np.ndarray:
    """A CPT arena of seeded random rows, entries uniform in [0.2, 1) before normalisation (no zeros)."""
    rng = np.random.default_rng(seed)
    cpt = np.empty_like(net.cpt)
    for x in range(net.n_nodes):
        blk = rng.uniform(0.2, 1.0, int(net.cpt_off[x + 1] - net.cpt_off[x])).reshape(-1, int(net.card[x]))
        cpt[net.cpt_off[x]:net.cpt_off[x + 1]] = (blk / blk.sum(axis=1, keepdims=True)).ravel()
    return cpt


# EM recovery problem (tests/test_gpu_em.py, scripts/em_recovery_calibrate.py): 200 000 complete cases of alarm37 by
# seeded ancestral sampling, 40 % of the values hidden, 30 iterations from seeded random rows with the EM defaults
# (epsilon 1e-6, max_sweeps 200).
RECOVERY = dict(n=200_000, hide=0.4, iterations=30, sample_seed=41, hide_seed=42, start_seed=43)


def recovery_problem():
    """(generating network, evidence, starting CPT) of the recovery problem."""
    net = synth.alarm37()
    samples = ancestral_sample(net, RECOVERY["n"], seed=RECOVERY["sample_seed"])
    return net, hide_values(samples, RECOVERY["hide"], RECOVERY["hide_seed"]), random_rows(net, RECOVERY["start_seed"])


def node_sums(net, counts):
    """Per node: sum over parent configurations [r_X] and the grand total."""
    per_x, tot = [], []
    for x in range(net.n_nodes):
        blk = counts[net.cpt_off[x]:net.cpt_off[x + 1]].reshape(-1, int(net.card[x]))
        per_x.append(blk.sum(axis=0))
        tot.append(blk.sum())
    return per_x, np.array(tot)


def exact_run(net, cases, **kw):
    ev = EvidenceBatch.from_cases(net, cases)
    kw.setdefault("eps", 0.0)
    kw.setdefault("max_sweeps", 3 * net.n_nodes + 3)
    return em_oracle.run(net, ev, **kw)


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_polytree_counts_match_enumeration(seed):
    net = synth.random_polytree(8 + seed % 3, card_hi=4, max_parents=3, seed=seed)
    assert E.is_polytree(net)
    cases = [{}] + cases_of(synth.make_evidence(net, 24, p=0.3, seed=seed + 100))
    w = np.random.default_rng(seed).uniform(0.0, 3.0, len(cases))
    for weights in (None, w):
        counts, *_ = exact_run(net, cases, weights=weights)
        want = brute_family_counts(net, cases, weights)
        assert np.abs(counts - want).max() <= 1e-10 * max(1.0, np.abs(want).max()), seed


@pytest.mark.parametrize("mode", ["T1", "T2", "T20", "eps_damped"])
def test_invariants_on_loopy_alarm37(mode):
    net = synth.alarm37()
    ev = synth.make_evidence(net, 300, exact_k=4, seed=31)
    kw = {"T1": dict(eps=0.0, max_sweeps=1), "T2": dict(eps=0.0, max_sweeps=2), "T20": dict(eps=0.0, max_sweeps=20),
          "eps_damped": dict(eps=1e-7, max_sweeps=300, damping=0.2)}[mode]
    w = np.random.default_rng(5).uniform(0.0, 2.0, ev.n_cases)
    counts, marg, sweeps, conv, le = em_oracle.run(net, ev, weights=w, **kw)
    assert np.isfinite(le).all()
    per_x, tot = node_sums(net, counts)
    off = net.belief_off
    for x in range(net.n_nodes):                          # invariant 1: the family marginal over x is the node marginal
        want = (w[:, None] * marg[:, off[x]:off[x + 1]]).sum(axis=0)
        assert np.allclose(per_x[x], want, rtol=1e-12, atol=1e-12), (mode, x)
    assert np.allclose(tot, w.sum(), rtol=1e-12), mode    # invariant 2: every node's counts total sum_c w_c
    if mode == "eps_damped":
        assert conv.all()


def test_fully_observed_counts_are_make_cpt_counts():
    net = synth.alarm37()
    samples = ancestral_sample(net, 500, seed=7)
    uniq, mult = np.unique(samples, axis=0, return_counts=True)
    ev = complete_evidence(net, uniq)
    counts, *_ = em_oracle.run(net, ev, eps=0.0, max_sweeps=2, weights=mult.astype(np.float64))
    assert np.abs(counts - np.round(counts)).max() <= 1e-12
    direct = np.zeros_like(counts)
    for s, m in zip(uniq, mult):
        for x in range(net.n_nodes):
            q = 0
            for u in net.parents[net.parent_off[x]:net.parent_off[x + 1]]:
                q = q * int(net.card[u]) + int(s[u])
            direct[net.cpt_off[x] + q * net.card[x] + s[x]] += m
    assert np.array_equal(np.round(counts), direct)
    from oracle import oracle
    want = oracle.port_make_cpt(net, uniq, mult)
    assert np.abs(m_step(net, counts) - want).max() <= 1e-12
    # T = 1 reads the all-ones time-0 pi-messages: the family of an observed child still sees its parents' one-hot
    # lambda rows, but not through the messages, so the counts are not make_cpt's
    c1, *_ = em_oracle.run(net, ev, eps=0.0, max_sweeps=1, weights=mult.astype(np.float64))
    assert np.abs(c1 - direct).max() > 1e-3


def test_weight_two_is_a_duplicate_and_weight_zero_adds_nothing():
    net = synth.alarm37()
    cases = cases_of(synth.make_evidence(net, 40, exact_k=4, seed=32))
    kw = dict(eps=0.0, max_sweeps=20)
    w = np.ones(len(cases))
    w[3], w[10] = 2.0, 0.0
    got, *_ = em_oracle.run(net, EvidenceBatch.from_cases(net, cases), weights=w, **kw)
    dup = cases + [cases[3]]
    dup = [c for i, c in enumerate(dup) if i != 10]
    want, *_ = em_oracle.run(net, EvidenceBatch.from_cases(net, dup), **kw)
    assert np.allclose(got, want, rtol=1e-12, atol=1e-12)


def test_impossible_evidence_is_skipped():
    net = E.catalogue()["determ"]
    bad = [{5: 0, 6: 1}, {5: 1, 6: 0}]                  # 6 copies 5 exactly: these have probability 0
    good = [{6: 0, 7: 0}, {7: 1}, {}]
    counts, _, sweeps, _, le = exact_run(net, bad + good)
    assert (le[:2] == -np.inf).all() and np.isfinite(le[2:]).all()
    want, *_ = exact_run(net, good)
    assert np.allclose(counts, want, rtol=1e-14, atol=1e-14)
    assert (sweeps > 0).all()
    _, tot = node_sums(net, counts)
    assert np.allclose(tot, len(good))


def test_m_step_pseudo_count_and_zero_rows():
    net = FlatNetwork.from_lists(card=[2, 3], parents=[[], [0]], cpts=[[0.5, 0.5], [1 / 3] * 6], name="ab")
    counts = np.array([3.0, 1.0, 2.0, 0.0, 6.0, 0.0, 0.0, 0.0])
    got = m_step(net, counts)
    assert np.allclose(got, [0.75, 0.25, 0.25, 0.0, 0.75, 1 / 3, 1 / 3, 1 / 3], rtol=0, atol=1e-15)
    got = m_step(net, counts, pseudo_count=1.0)
    assert np.allclose(got, [4 / 6, 2 / 6, 3 / 11, 1 / 11, 7 / 11, 1 / 3, 1 / 3, 1 / 3], rtol=0, atol=1e-15)
    assert np.allclose(m_step(net, np.zeros(8)), [0.5, 0.5] + [1 / 3] * 6)
    with pytest.raises(ValueError):
        m_step(net, counts[:-1])


def test_exact_em_on_a_polytree_never_lowers_the_likelihood():
    true = synth.random_polytree(9, card_hi=3, max_parents=3, seed=13)
    assert E.is_polytree(true)
    ev = hide_values(ancestral_sample(true, 400, seed=14), 0.4, seed=15)
    cpt = random_rows(true, seed=16)
    lls = []
    for _ in range(12):
        net = with_cpt(true, cpt)
        counts, _, _, _, le = em_oracle.run(net, ev, eps=0.0, max_sweeps=3 * net.n_nodes + 3)
        assert np.isfinite(le).all()
        lls.append(float(le.sum()))
        cpt = m_step(net, counts)
    lls = np.array(lls)
    assert (np.diff(lls) >= -1e-9 * np.abs(lls[1:])).all(), lls
    assert lls[-1] > lls[0] + 1.0, lls
