"""The shape-boundary networks of tests/edge_networks.py through every kernel family that accepts them, against the
oracle -- needs a B200 (-m gpu).

    K1a  unrolled streaming sweeps (specialize="always"): fixed sweeps (first / last sweep fused with K0 / K4 on hard
         evidence: variants 5, 6, 7) and epsilon mode
    K1d  class-looped streaming sweeps (BNBP_CLASSLOOP=2), also a small batch that takes node slices
    K1c  the on-chip kernel (onchip="always")
    K1b  the generic kernel (specialize="never"), also max-product
    K2   dense contraction (dense_min_cpt low enough for the 16-state and in-degree-6 nodes), fp64 and fp32 tensor cores

Every run asserts the family it ran through (stats), so that a run cannot silently take another one.  Bars: fp64
1e-9 / 1e-12 with equal sweep counts and flags in epsilon mode, fp32 1e-5 / 1e-7 at fixed sweep counts.  The host
emulation of the same generated kernels is tests/test_edge_shapes_emul.py.

NVRTC: build() leaves every kernel this file asks for in the cubin cache (scripts/precompile_tests.py), so the run
itself compiles nothing; with them, the whole build() took 6.5 minutes wall on an 8-core build box.  The slowest of
them are the 65- and 66-node hubs, whose unrolled walks AUTO takes from the cache only.  The file's GPU run: 2.5
minutes for the whole GPU suite including it (profiles/r03a_pytest_gpu.log, one B200)."""
import numpy as np
import pytest

import edge_networks as E
from helpers import assert_close

pytestmark = pytest.mark.gpu
TOL = {"fp64": dict(rtol=1e-9, atol=1e-12), "fp32": dict(rtol=1e-5, atol=1e-7)}
NETS = E.catalogue()
N_CASES = 777                                   # ragged: not a multiple of any tile or case group
DENSE = {"indeg5_6": 200, "card16": 200}        # dense_min_cpt that sends the in-degree-5/6 and 16-state nodes dense


@pytest.fixture(scope="module")
def BP():
    from bayesiannetwork_b200.engine import BeliefPropagation
    return BeliefPropagation


def _check(bp, oracle_mod, net, ev, precision, eps, cap, what, **kw):
    res = bp(ev, eps, max_sweeps=cap, **kw)
    om, osw, ocv = oracle_mod.run_port(net, ev, eps=eps, max_sweeps=cap, threads=0, semiring=1 if kw.get("semiring") == "max" else 0)
    assert np.array_equal(res.sweeps, osw), (what, np.nonzero(res.sweeps != osw)[0][:5])
    assert np.array_equal(res.converged, ocv), what
    assert_close(res.marginals, om, what=what, **TOL[precision])
    return res, bp.stats()


def _runs(bp, oracle_mod, net, ev, precision, what, **kw):
    """A fixed-count run in the handle's precision, and an epsilon-mode run in fp64; the stats of both."""
    sts = [_check(bp, oracle_mod, net, ev, precision, 0.0, 9, f"{what} {precision} fixed", **kw)[1]]
    if precision == "fp64":
        sts.append(_check(bp, oracle_mod, net, ev, precision, 1e-7, 300, f"{what} eps", **kw)[1])
    return sts


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("name", E.NAMES)
def test_unrolled_streaming_k1a(BP, oracle_mod, monkeypatch, name, precision):
    monkeypatch.setenv("BNBP_CLASSLOOP", "0")
    net = NETS[name]
    ev = E.evidence(net, N_CASES, seed=17)
    bp = BP(net, precision, specialize="always")
    fixed, *eps = _runs(bp, oracle_mod, net, ev, precision, f"{name} K1a")
    assert fixed["last_specialised"] == 1 and fixed["spec_class_count"] == 0 and fixed["last_onchip"] == 0
    assert fixed["last_fused"] == 1                                  # hard evidence, fixed count: variants 5 and 6 / 7
    for st in eps:
        assert st["last_specialised"] == 1 and st["spec_class_count"] == 0 and st["last_onchip"] == 0


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("name", [n for n in E.NAMES if n not in E.CLASSLOOP_REFUSED])
def test_class_looped_streaming_k1d(BP, oracle_mod, monkeypatch, name, precision):
    monkeypatch.setenv("BNBP_CLASSLOOP", "2")
    net = NETS[name]
    ev = E.evidence(net, N_CASES, seed=17)
    bp = BP(net, precision, specialize="always")
    for st in _runs(bp, oracle_mod, net, ev, precision, f"{name} K1d"):
        assert st["last_specialised"] == 1 and st["spec_class_count"] > 0 and st["last_onchip"] == 0
    # one tile of cases: the plain variants split the classes into node slices (grid.y); sliced == unsliced
    small = E.evidence(net, 100, seed=4)
    a, _ = _check(bp, oracle_mod, net, small, precision, 0.0, 5, f"{name} K1d small batch")
    monkeypatch.setenv("BNBP_NO_NODE_SLICES", "1")
    b = bp(small, 0.0, max_sweeps=5)
    assert np.array_equal(a.marginals, b.marginals, equal_nan=True)


@pytest.mark.parametrize("name", E.NAMES)
def test_class_looped_refusals(BP, monkeypatch, name):
    """A network the class-looped walk refuses runs unrolled under BNBP_CLASSLOOP=2."""
    monkeypatch.setenv("BNBP_CLASSLOOP", "2")
    bp = BP(NETS[name], "fp64", specialize="always")
    bp(E.evidence(NETS[name], 40), 0.0, max_sweeps=2)
    assert bp.stats()["last_specialised"] == 1
    assert (bp.stats()["spec_class_count"] == 0) == (name in E.CLASSLOOP_REFUSED)


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("name", E.NAMES)
def test_onchip_k1c(BP, oracle_mod, monkeypatch, name, precision):
    from bayesiannetwork_b200.engine import BnbpError
    monkeypatch.setenv("BNBP_CLASSLOOP", "0")
    net = NETS[name]
    ev = E.evidence(net, N_CASES, seed=17)
    bp = BP(net, precision, onchip="always")
    if name in E.ONCHIP_REFUSED:
        assert bp.stats()["onchip_roles"] == 0
        with pytest.raises(BnbpError, match=E.ONCHIP_REFUSED[name]):
            bp(ev, 0.0, max_sweeps=3)
        return
    for st in _runs(bp, oracle_mod, net, ev, precision, f"{name} K1c"):
        assert st["last_onchip"] == 1 and st["onchip_blocks_per_sm"] >= 1


@pytest.mark.parametrize("name", E.NAMES)
def test_generic_k1b(BP, oracle_mod, name):
    net = NETS[name]
    ev = E.evidence(net, N_CASES, seed=17)
    for precision in ("fp64", "fp32"):
        bp = BP(net, precision, specialize="never")
        for st in _runs(bp, oracle_mod, net, ev, precision, f"{name} K1b"):
            assert st["last_specialised"] == 0 and st["last_onchip"] == 0
    bp = BP(net, "fp64", specialize="never", dense_min_cpt=-1)
    _, st = _check(bp, oracle_mod, net, ev, "fp64", 0.0, 9, f"{name} K1b max-product", semiring="max")
    assert st["last_specialised"] == 0 and st["last_dense_launches"] == 0


@pytest.mark.parametrize("name", list(DENSE))
def test_dense_k2(BP, oracle_mod, name):
    net = NETS[name]
    ev = E.evidence(net, N_CASES, seed=17)
    for precision, kw in (("fp64", {}), ("fp32", dict(dense_tensor=1))):
        bp = BP(net, precision, dense_min_cpt=DENSE[name], **kw)
        assert bp.stats()["dense_nodes"] >= 2
        for st in _runs(bp, oracle_mod, net, ev, precision, f"{name} K2"):
            assert st["last_dense_launches"] > 0 and st["last_specialised"] == 0
            if precision == "fp32":
                assert st["last_dense_tensor_launches"] > 0


FAMILIES = {"K1a": (dict(specialize="always"), {"BNBP_CLASSLOOP": "0"}),
            "K1d": (dict(specialize="always"), {"BNBP_CLASSLOOP": "2"}),
            "K1c": (dict(onchip="always"), {"BNBP_CLASSLOOP": "0"}),
            "K1b": (dict(specialize="never"), {})}


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("name", ["card1", "card16"])
def test_device_call_and_query_nodes(BP, oracle_mod, monkeypatch, name, family):
    import torch
    if name in E.CLASSLOOP_REFUSED and family == "K1d":
        pytest.skip("the class-looped walk refuses this network")
    opts, env = FAMILIES[family]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    net = NETS[name]
    ev = E.evidence(net, N_CASES, seed=19)
    om, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=9, threads=0)
    bp = BP(net, "fp64", **opts)

    def family_ran():
        st = bp.stats()
        assert st["last_onchip"] == (family == "K1c")
        assert st["last_specialised"] == (family != "K1b")            # the on-chip kernel is network-specialised too
        assert (st["spec_class_count"] > 0) == (family == "K1d")

    dev = torch.device("cuda", 0)
    out = torch.full((N_CASES, net.belief_values), -7.0, dtype=torch.float64, device=dev)
    sw = torch.zeros(N_CASES, dtype=torch.int32, device=dev)
    bp.run_device(N_CASES, *(torch.from_numpy(a).to(dev) for a in (ev.ev_off, ev.ev_node, ev.ev_state)), out,
                  epsilon=0.0, max_sweeps=9, out_sweeps=sw)
    torch.cuda.synchronize()
    bp.check_errors()
    family_ran()
    assert int(sw.min()) == 9 == int(sw.max())
    assert_close(out.cpu().numpy(), om, what=f"{name} {family} device call", **TOL["fp64"])
    query = [x for x in range(net.n_nodes) if int(net.card[x]) in (1, 16)]
    query += [x for x in (net.n_nodes - 1, 1) if x not in query]
    res = bp(ev, 0.0, max_sweeps=9, query_nodes=query)
    family_ran()
    cols = np.concatenate([np.arange(net.belief_off[x], net.belief_off[x + 1]) for x in query])
    assert_close(res.marginals, om[:, cols], what=f"{name} {family} query {query}", **TOL["fp64"])


def test_auto_does_not_take_the_onchip_kernel_for_a_hub_of_65_children(BP, oracle_mod):
    """With its kernels in the cubin cache, AUTO takes the on-chip kernel for a 66-node network and a batch of >= 4096
    hard-evidence cases -- but the hub's 65 children's lambda-messages cannot all be read before the sweep barrier: the
    on-chip kernel is refused, AUTO runs the streaming kernels, and they match the oracle."""
    from bayesiannetwork_b200 import engine
    net = NETS["hub65"]
    engine.precompile(net, "fp64", 0b11111111)
    with pytest.raises(engine.BnbpError, match=E.ONCHIP_REFUSED["hub65"]):
        engine.precompile(net, "fp64", (1 << 8) | (1 << 10))
    ev = E.evidence(net, 4096 + 77, seed=23)
    bp = BP(net, "fp64")
    assert bp.stats()["onchip_roles"] == 0
    for eps, cap in ((0.0, 2), (0.0, 9), (1e-7, 300)):
        _, st = _check(bp, oracle_mod, net, ev, "fp64", eps, cap, f"hub65 AUTO eps {eps} cap {cap}")
        assert st["last_onchip"] == 0 and st["last_specialised"] == 1
