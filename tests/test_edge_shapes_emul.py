"""The generated kernels on the shape boundaries of the network compiler (tests/edge_networks.py), emulated on the host
and compared with the oracle -- WITHOUT a GPU.

Every catalogue network goes through the unrolled streaming walk (variants 3 / 0 / 4 at 1, 2 and 9 sweeps, variant 5
from NaN arenas, variants 6 / 7 with guard rows behind a ragged batch, the epsilon loop over variants 1 / 2), the
class-looped walk (variants 0-4, bit for bit equal to the unrolled arenas) and the on-chip kernel (variants 8 / 9, fp64
and fp32, the default role count and one role).  Shapes a generator refuses are asserted refused, with their reason.
Bars: fp64 1e-9 / 1e-12, fp32 1e-5 / 1e-7 at fixed sweep counts; the NaN pattern equals the oracle's.  The GPU runs of
the same networks are tests/test_gpu_edge_shapes.py (-m gpu).
"""
import ctypes as C
import os
import re
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import edge_networks as E
from helpers import assert_close
from test_netcompiler_emul import HERE, Emulated, beliefs, generated_source as _source, initial_state, run_eps, run_fixed
from test_onchip_emul import OnchipEmulated

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")
NETS = E.catalogue()
TOL = {"fp64": (1e-9, 1e-12), "fp32": (1e-5, 1e-7)}


@pytest.fixture(scope="module")
def engine():
    from bayesiannetwork_b200 import _build, engine
    _build.build()
    return engine


# The unrolled walk, also for networks of more than 64 nodes (whose unrolled kernels AUTO takes from the cubin cache only)
UNROLLED = {"BNBP_CLASSLOOP": "0"}


def _parallel(makers):
    """Build several emulated kernels at once (each is a g++ run)."""
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        futs = [ex.submit(m) for m in makers]
        return [f.result() for f in futs]


def _register_plan(k):
    n = 4 * k.lib.emul_pl() + 64                     # more than nodes (or classes) in any network
    ch, cp = np.zeros(n, np.int32), np.zeros(n, np.int32)
    cnt = k.lib.emul_register_plan(ch.ctypes.data_as(C.c_void_p), cp.ctypes.data_as(C.c_void_p))
    return ch[:cnt].tolist(), cp[:cnt].tolist()


def _shapes(net):
    """(R, K, M, parent cardinalities, CPT entries) per node."""
    m = np.bincount(net.parents, minlength=net.n_nodes) if net.n_edges else np.zeros(net.n_nodes, int)
    out = []
    for x in range(net.n_nodes):
        ru = tuple(int(net.card[u]) for u in net.parents[net.parent_off[x]:net.parent_off[x + 1]])
        out.append((int(net.card[x]), len(ru), int(m[x]), ru, int(net.cpt_off[x + 1] - net.cpt_off[x])))
    return out


def _expected_plan(net, classloop):
    """What the generator budgets registers for (bnbp_jit.cu class_inputs): the lambda-messages of at most 4 children
    (streaming MREG) and, in a class-looped walk, a CPT of at most 32 entries (CPT_REG_MAX)."""
    shapes = _shapes(net)
    if classloop:                                    # classes in order of first appearance
        seen = []
        for s in shapes:
            if s[:4] not in [t[:4] for t in seen]:
                seen.append(s)
        shapes = seen
    return ([s[2] if 0 < s[2] <= 4 else 0 for s in shapes],
            [s[4] if classloop and s[4] <= 32 else 0 for s in shapes])


def _evst(net, ev, tbc, tiles):
    evst = np.zeros((tiles, net.n_nodes, tbc), np.uint8)
    for c in range(ev.n_cases):
        for e in range(int(ev.ev_off[c]), int(ev.ev_off[c + 1])):
            evst[c // tbc, int(ev.ev_node[e]), c % tbc] = int(ev.ev_state[e]) + 1
    return evst


@pytest.mark.parametrize("name", E.NAMES)
def test_streaming_walks_match_the_oracle(engine, oracle_mod, tmp_path, name):
    net = NETS[name]
    ev = E.evidence(net, 150)                                       # two tiles of 128, the second one ragged
    with_classes = name not in E.CLASSLOOP_REFUSED
    specs = [(v, False) for v in (0, 1, 2, 3, 4, 5)] + ([(v, True) for v in (0, 1, 2, 3, 4)] if with_classes else [])
    ks = dict(zip(specs, _parallel([lambda v=v, cl=cl: Emulated(engine, net, "fp64", v, cl, str(tmp_path)) for v, cl in specs])))
    if not with_classes:                                            # BNBP_CLASSLOOP=2 falls back to the unrolled walk
        assert "#define BNBP_CLASSLOOP 1" not in _source(engine, net, "fp64", 0, {"BNBP_CLASSLOOP": "2"})
    modes = [False, True] if with_classes else [False]
    for cl in modes:
        assert _register_plan(ks[(0, cl)]) == _expected_plan(net, cl), ("register plan", cl)
    for sweeps in (1, 2, 9):
        want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=sweeps)
        res = {}
        for cl in modes:
            st, cur = run_fixed({v: ks[(v, cl)] for v in (0, 3, 4)}, net, ev, sweeps)
            assert_close(beliefs(net, st, ev.n_cases), want, *TOL["fp64"], f"{name} {'class-looped' if cl else 'unrolled'} {sweeps} sweeps")
            res[cl] = (st["pl"], cur)
        if with_classes:
            assert np.array_equal(res[True][0], res[False][0], equal_nan=True), f"{name} {sweeps}: pi / lambda differ"
            assert np.array_equal(res[True][1], res[False][1], equal_nan=True), f"{name} {sweeps}: messages differ"
    # epsilon mode, tested every 3rd sweep: untested sweeps run the freeze variant (1), tested ones freeze + check (2)
    want, osw, ocv = oracle_mod.run_port(net, ev, eps=1e-7, max_sweeps=300, check_interval=3)
    res = {}
    for cl in modes:
        st, sw, conv = run_eps(ks[(2, cl)], net, ev, 1e-7, 300, interval=3, k_unchecked=ks[(1, cl)])
        assert np.array_equal(sw, osw), (name, cl, np.nonzero(sw != osw)[0][:8])
        assert np.array_equal(conv, ocv.astype(bool)), (name, cl)
        assert_close(beliefs(net, st, ev.n_cases), want, *TOL["fp64"], f"{name} eps mode {'class-looped' if cl else 'unrolled'}")
        res[cl] = st["pl"]
    if with_classes:
        assert np.array_equal(res[True], res[False], equal_nan=True)
    # variant 5: the first sweep fused with the initialisation; nothing of time 0 is read, the arenas hold NaN
    k0 = ks[(0, False)]
    st = initial_state(net, ev, k0)
    evst = _evst(net, ev, k0.TBC, st["tiles"])
    st["pl"][:] = np.nan
    cur, nxt = st["msg"]
    cur[:] = np.nan
    ks[(5, False)].launch(st, cur, nxt, evst=evst)
    for _ in range(4):
        cur, nxt = nxt, cur
        k0.launch(st, cur, nxt)
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=5)
    assert_close(beliefs(net, st, ev.n_cases), want, *TOL["fp64"], f"{name} fused first sweep")


def _flush_groups(src):
    return [(int(a), int(b)) for a, b in re.findall(r"BNBP_FLUSH\((\d+),(\d+)\)", src.split("#define BNBP_WALK", 1)[1].split("\n", 1)[0])]


def _expected_groups(net):
    """Consecutive nodes whose marginals fit the 32 columns of the tile, greedily."""
    groups, x = [], 0
    while x < net.n_nodes:
        j0, w = int(net.belief_off[x]), 0
        while x < net.n_nodes and w + int(net.card[x]) <= 32:
            w += int(net.card[x])
            x += 1
        groups.append((j0, w))
    return groups


@pytest.mark.parametrize("name", E.NAMES)
def test_last_sweep_fused_with_the_beliefs(engine, oracle_mod, tmp_path, name):
    """Variants 6 (fp64) and 7 (fp32 kernel, double marginals): the marginal tile groups and the case-major rows they
    write, five guard rows behind a ragged batch."""
    net = NETS[name]
    ev = E.evidence(net, 150, seed=22)

    def last(precision, variant):
        src = _source(engine, net, precision, variant, UNROLLED)
        assert _flush_groups(src) == _expected_groups(net)
        cu, so = str(tmp_path / f"last_{precision}_{variant}.cu"), str(tmp_path / f"last_{precision}_{variant}.so")
        open(cu, "w").write(src)
        cmd = ["g++", "-O0", "-std=c++17", "-ffp-contract=off", "-fvisibility=hidden", "-fno-gnu-unique", "-Wno-unknown-pragmas",
               "-I", os.path.join(HERE, "emul"), f'-DBNBP_GENERATED="{cu}"', "-shared", "-fPIC", "-pthread", "-o", so,
               os.path.join(HERE, "emul", "spec_block_emul.cpp")]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        return C.CDLL(so)

    plan = [("fp64", 6), ("fp32", 7)]
    made = _parallel([lambda p=p, v=v: last(p, v) for p, v in plan] +
                     [lambda p=p, v=v: Emulated(engine, net, p, v, False, str(tmp_path)) for p, _ in plan for v in (3, 0)])
    libs, ks = made[:2], made[2:]
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=6)
    for i, (precision, variant) in enumerate(plan):
        lib, k3, k0 = libs[i], ks[2 * i], ks[2 * i + 1]
        OUT = np.float32 if lib.emul_out_bytes() == 4 else np.float64
        assert OUT == np.float64 and lib.emul_v() == net.belief_values
        cpt = np.ascontiguousarray(net.cpt, dtype=k0.T)
        lib.emul_set_cpt(cpt.ctypes.data_as(C.c_void_p), C.c_longlong(cpt.size))
        st = initial_state(net, ev, k0)
        cur, nxt = st["msg"]
        k3.launch(st, cur, nxt)
        for _ in range(4):
            cur, nxt = nxt, cur
            k0.launch(st, cur, nxt)
        cur, nxt = nxt, cur
        out = np.full((ev.n_cases + 5, net.belief_values), -7.0, OUT)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        lib.emul_launch_last(p(st["pl"]), p(cur), p(nxt), p(st["evbits"]), C.c_int(st["tiles"]), p(out), C.c_longlong(ev.n_cases))
        assert_close(out[:ev.n_cases], want, *TOL[precision], f"{name} fused last sweep {precision} v{variant}")
        assert (out[ev.n_cases:] == -7.0).all()


def test_tile_groups_of_exactly_32_columns(engine):
    net = NETS["tile32"]
    for variant in (6, 7):
        assert _flush_groups(_source(engine, net, "fp32", variant, UNROLLED)) == [(0, 32), (32, 32), (64, 5)]


@pytest.mark.parametrize("name", E.NAMES)
def test_onchip_kernel_matches_the_oracle(engine, oracle_mod, tmp_path, name):
    """Variants 8 / 9 in both precisions, with the default number of roles (warps per case group) and with one.  With
    one role a single warp walks every node, so nothing a role reads can have been overwritten by another role."""
    net = NETS[name]
    ev = E.evidence(net, 77, seed=13)                               # two full groups of 32 and a ragged one
    try:
        _source(engine, net, "fp64", 8, UNROLLED)
    except engine.BnbpError as e:
        assert name in E.ONCHIP_REFUSED and E.ONCHIP_REFUSED[name] in str(e), str(e)
        return
    specs = [(p, v, r) for p in ("fp64", "fp32") for v in (8, 9) for r in (None, 1)]
    made = _parallel([lambda p=p, v=v, r=r: OnchipEmulated(engine, net, p, v, str(tmp_path), env=dict(UNROLLED, BNBP_OC_ROLES=str(r)) if r else UNROLLED)
                      for p, v, r in specs])
    ks = dict(zip(specs, made))
    for roles in (None, 1):
        what = f"{name} on chip, {roles or 'default'} roles"
        for precision in ("fp64", "fp32"):
            for sweeps in (1, 2, 9):
                want, osw, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=sweeps)
                got, sw, conv = ks[(precision, 8, roles)].run(ev, 0.0, sweeps)
                assert np.array_equal(sw, osw) and not conv.any()
                assert_close(got, want, *TOL[precision], f"{what}, {precision}, {sweeps} sweeps")
            # the check flavour at a fixed count (damping needs the time-t messages)
            want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=7, damping=0.25)
            got, _, _ = ks[(precision, 9, roles)].run(ev, 0.0, 7, damping=0.25)
            assert_close(got, want, *TOL[precision], f"{what}, {precision}, damped")
        want, osw, ocv = oracle_mod.run_port(net, ev, eps=1e-7, max_sweeps=300)
        got, sw, conv = ks[("fp64", 9, roles)].run(ev, 1e-7, 300)
        assert np.array_equal(sw, osw), (what, np.nonzero(sw != osw)[0][:8])
        assert np.array_equal(conv, ocv), what
        assert_close(got, want, *TOL["fp64"], f"{what}, eps mode")
    # a query list with the card-1 / card-16 nodes (and the first and last node)
    query = sorted({0, net.n_nodes - 1} | {x for x in range(net.n_nodes) if int(net.card[x]) in (1, 16)})
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=9)
    cols = np.concatenate([np.arange(net.belief_off[x], net.belief_off[x + 1]) for x in query])
    got, _, _ = ks[("fp64", 8, None)].run(ev, 0.0, 9, query=query)
    assert_close(got, want[:, cols], *TOL["fp64"], f"{name} on chip, query {query}")
    assert name not in E.ONCHIP_REFUSED


def test_hub_of_65_children_on_chip(engine, oracle_mod, tmp_path):
    """A hub with more children than the on-chip kernel keeps in registers would read its children's lambda-messages
    after the sweep barrier, when the warps that own the children may already have overwritten them with the next
    sweep's: a Gauss-Seidel step in a Jacobi schedule, wrong beliefs from the second sweep on with the default 6 roles.
    Such a network is refused with a reason; were the kernel changed to accept it, it must match the oracle."""
    net = NETS["hub65"]
    ev = E.evidence(net, 64)
    try:
        k = OnchipEmulated(engine, net, "fp64", 8, str(tmp_path), env=UNROLLED)
    except engine.BnbpError as e:
        assert "a hub with more than 64 children: its inbox cannot be read before the sweep barrier" in str(e)
        return
    for sweeps in (1, 2, 9):
        want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=sweeps)
        got, _, _ = k.run(ev, 0.0, sweeps)
        assert_close(got, want, *TOL["fp64"], f"hub65 on chip, {sweeps} sweeps")


@pytest.mark.parametrize("net,variant,env,reason", E.REFUSED, ids=[f"{r[0].name}_v{r[1]}" for r in E.REFUSED])
def test_refused_shapes_name_their_reason(engine, monkeypatch, net, variant, env, reason):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    with pytest.raises(engine.BnbpError, match=re.escape(reason)):
        engine.spec_source(net, "fp64", variant)


def test_class_looped_walk_takes_a_hub_of_64_children(engine, monkeypatch):
    """The other side of the 64-children limit of the class-looped walk (hub65_wide in edge_networks.REFUSED)."""
    from bayesiannetwork_b200 import synth
    monkeypatch.setenv("BNBP_CLASSLOOP", "2")
    net = synth._assemble([16] + [8] * 64, [[]] + [[0]] * 64, 22, "hub64_wide")
    assert "#define BNBP_CLASSLOOP 1" in engine.spec_source(net, "fp64", 0)


@pytest.mark.parametrize("name", [n for n in E.NAMES if E.is_polytree(NETS[n]) and np.prod(NETS[n].card.astype(float)) <= 4e5])
def test_oracle_is_exact_on_polytree_members(oracle_mod, name):
    """BP is exact on a polytree once the messages have crossed it: the oracle equals brute-force enumeration."""
    from test_lw import exact_posteriors
    net = NETS[name]
    ev = E.evidence(net, 12, seed=5)
    want = exact_posteriors(net, ev)
    got, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=net.n_nodes + 2)
    assert_close(got, want, *TOL["fp64"], f"{name} oracle vs enumeration")
