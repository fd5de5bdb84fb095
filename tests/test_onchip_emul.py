"""The ON-CHIP multi-sweep kernel (bnbp_onchip.cuh: the headline kernel of cfg 2) emulated on the host -- one OS thread
per CUDA thread of one CTA, pthread barriers for `bar.sync` and for the warp collectives (tests/emul/onchip_emul.cpp) --
and run against the oracle WITHOUT a GPU.  One persistent group of 32 lanes takes every case of the batch from the
ticket counter, so the case hand-out, the two-phase sweep over one message buffer, the in-kernel stopping rule, the
retire / refill batches and the belief write are all exercised.  The GPU tests of the same kernel are
tests/test_gpu_onchip.py (-m gpu)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from bayesiannetwork_b200 import synth
from helpers import assert_close
from test_netcompiler_emul import generated_source

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

PTX = [('asm volatile("bar.sync 1, %0;" ::"n"(OC_THREADS) : "memory");', "emul_cta_barrier();"),
       ('asm("mov.u32 %0, %%smid;" : "=r"(smid));', "smid = 0;"),
       ('asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(s));', "x = 1.0 / s;")]


@pytest.fixture(scope="module")
def engine():
    from bayesiannetwork_b200 import _build, engine
    _build.build()
    return engine


class OnchipEmulated:
    def __init__(self, engine, net, precision, variant, workdir, extra=(), env=None):
        """env: generator knobs for this kernel (e.g. BNBP_OC_ROLES), set while its source is generated."""
        env = env or {}
        src = generated_source(engine, net, precision, variant, env)
        for ptx, host in PTX:                       # the three inline-PTX statements of the kernel, see onchip_emul.cpp
            assert src.count(ptx) == 1, ptx
            src = src.replace(ptx, host)
        tag = f"{net.name}_{precision}_v{variant}" + "".join(f"_{k}{v}" for k, v in sorted(env.items()))
        cu, so = os.path.join(workdir, tag + ".cu"), os.path.join(workdir, tag + ".so")
        with open(cu, "w") as f:
            f.write(src)
        cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fvisibility=hidden", "-fno-gnu-unique", "-Wno-unknown-pragmas",
               *extra, "-I", os.path.join(HERE, "emul"), f'-DBNBP_GENERATED="{cu}"', "-shared", "-fPIC", "-pthread", "-o", so,
               os.path.join(HERE, "emul", "onchip_emul.cpp")]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        self.lib = C.CDLL(so)
        self.net = net
        self.T = np.float32 if precision == "fp32" else np.float64
        self.cT = C.c_float if precision == "fp32" else C.c_double
        assert self.lib.emul_value_bytes() == np.dtype(self.T).itemsize
        self.OUT = np.float32 if self.lib.emul_out_bytes() == 4 else np.float64
        cpt = np.ascontiguousarray(net.cpt, dtype=self.T)
        self.lib.emul_set_cpt(cpt.ctypes.data_as(C.c_void_p), C.c_longlong(cpt.size))

    def run(self, ev, eps, max_sweeps, interval=1, damping=0.0, query=None):
        net = self.net
        bel_col = np.full(net.n_nodes, -1, np.int32)
        if query is None:
            bel_col[:] = net.belief_off[:-1]
            stride = net.belief_values
        else:
            col = 0
            for x in query:
                bel_col[x] = col
                col += int(net.card[x])
            stride = col
        out = np.full((ev.n_cases, stride), -7.0, self.OUT)
        sweeps = np.zeros(ev.n_cases, np.int32)
        conv = np.zeros(ev.n_cases, np.uint8)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = self.lib.emul_run(p(ev.ev_off), p(ev.ev_node), p(ev.ev_state), C.c_longlong(ev.n_cases), p(out), p(bel_col),
                               C.c_longlong(stride), p(sweeps), p(conv), self.cT(eps), self.cT(damping), C.c_int(max_sweeps),
                               C.c_int(interval))
        assert rc == 0
        return out, sweeps, conv


def _net(name):
    net = {"alarm37": synth.alarm37, "pearl": synth.pearl_network, "grid5": lambda: synth.grid(5),
           "polytree24": lambda: synth.random_polytree(24, card_hi=4, max_parents=3, seed=6)}[name]()
    net.name = name
    return net


@pytest.mark.parametrize("name", ["alarm37", "grid5", "polytree24"])
def test_fixed_sweep_flavour_matches_the_oracle(engine, oracle_mod, tmp_path, name):
    net = _net(name)
    ev = synth.make_evidence(net, 203, seed=13, **(dict(exact_k=4) if name == "alarm37" else dict(p=0.2)))   # 6 refills + a ragged tail
    k = OnchipEmulated(engine, net, "fp64", 8, str(tmp_path))
    for sweeps in (1, 2, 20):
        want, osw, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=sweeps)
        got, sw, conv = k.run(ev, 0.0, sweeps)
        assert np.array_equal(sw, osw) and not conv.any()
        assert_close(got, want, 1e-9, 1e-12, f"{name} on chip, {sweeps} sweeps")


@pytest.mark.parametrize("name", ["alarm37", "grid5"])
def test_epsilon_flavour_stops_where_the_oracle_stops(engine, oracle_mod, tmp_path, name):
    """Lanes stop at different sweeps, wait frozen for a retire batch of 8, and are refilled while the others carry on."""
    net = _net(name)
    ev = synth.make_evidence(net, 170, seed=14, **(dict(exact_k=4) if name == "alarm37" else dict(p=0.2)))
    k = OnchipEmulated(engine, net, "fp64", 9, str(tmp_path))
    want, osw, ocv = oracle_mod.run_port(net, ev, eps=1e-6, max_sweeps=200)
    got, sw, conv = k.run(ev, 1e-6, 200)
    assert np.array_equal(sw, osw), np.nonzero(sw != osw)[0][:8]
    assert np.array_equal(conv, ocv)
    assert_close(got, want, 1e-9, 1e-12, f"{name} on chip, epsilon mode")
    # a sweep cap below what some cases need, tested every 3rd sweep, with damping (extensions; same definitions as the port)
    want, osw, ocv = oracle_mod.run_port(net, ev, eps=1e-6, max_sweeps=9, damping=0.25, check_interval=3)
    got, sw, conv = k.run(ev, 1e-6, 9, interval=3, damping=0.25)
    assert np.array_equal(sw, osw) and np.array_equal(conv, ocv) and not conv.all()
    assert_close(got, want, 1e-9, 1e-12, f"{name} on chip, capped / damped / interval 3")


def test_query_nodes_and_impossible_evidence(engine, oracle_mod, ref_fixtures, tmp_path):
    """Only the queried columns are written; an all-zero row becomes NaN exactly where the reference's does
    (unnormalised pi / lambda on chip, DESIGN section 4 K1c)."""
    from helpers import load_fixture
    net = _net("alarm37")
    ev = synth.make_evidence(net, 64, seed=15, exact_k=4)
    k = OnchipEmulated(engine, net, "fp64", 8, str(tmp_path))
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=12)
    query = [3, 17, 30]
    got, _, _ = k.run(ev, 0.0, 12, query=query)
    off = net.belief_off
    cols = np.concatenate([np.arange(off[x], off[x + 1]) for x in query])
    assert_close(got, want[:, cols], 1e-9, 1e-12, "query nodes")
    f = load_fixture(ref_fixtures, "pearl_nan_fixed6")
    f["net"].name = "pearl_nan"
    k2 = OnchipEmulated(engine, f["net"], "fp64", 8, str(tmp_path))
    got, sw, _ = k2.run(f["ev"], 0.0, f["max_sweeps"])
    assert np.isnan(f["marginals"]).any()
    assert_close(got, f["marginals"], 1e-9, 1e-12, "pearl_nan_fixed6 on chip")


@pytest.mark.parametrize("variant,eps,damage", [(8, 0.0, False), (9, 1e-6, False), (8, 0.0, True)],
                         ids=["fixed", "epsilon", "control_without_the_phase_barrier"])
def test_barrier_placement_under_thread_sanitizer(engine, oracle_mod, tmp_path, variant, eps, damage):
    """A host-side race check of the kernel's barrier discipline: the same emulation built with -fsanitize=thread (every
    CUDA thread an OS thread, `bar.sync` a pthread barrier).  Two warps touching one shared-memory word without a barrier
    between them -- an inbox overwritten before its owner has read it, a partial delta read before it is written, a
    ticket slot reused too early -- is a data race ThreadSanitizer reports; the results must still equal the oracle's."""
    net = _net("alarm37")
    ev = synth.make_evidence(net, 77, seed=16, exact_k=4)
    src = engine.spec_source(net, "fp64", variant)
    for ptx, host in PTX:
        src = src.replace(ptx, host)
    if damage:
        # negative control: without the barrier between "every warp has read its inboxes" and "the inboxes are overwritten"
        # the checker must speak up -- otherwise its silence on the real kernel would mean nothing
        assert src.count("#define BNBP_SYNC oc_barrier();") == 1
        src = src.replace("#define BNBP_SYNC oc_barrier();", "#define BNBP_SYNC")
    cu, exe = str(tmp_path / "oc.cu"), str(tmp_path / "oc_tsan")
    open(cu, "w").write(src)
    cmd = ["g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-fsanitize=thread", "-Wno-unknown-pragmas", "-DEMUL_MAIN",
           "-I", os.path.join(HERE, "emul"), f'-DBNBP_GENERATED="{cu}"', "-pthread", "-o", exe, os.path.join(HERE, "emul", "onchip_emul.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0 and "tsan" in r.stderr.lower() and "cannot find" in r.stderr:
        pytest.skip("libtsan not installed")
    assert r.returncode == 0, r.stderr[-3000:]
    cap = 20 if eps == 0.0 else 200
    stride = net.belief_values
    with open(tmp_path / "in.bin", "wb") as f:
        f.write(np.array([ev.n_cases, ev.nnz, net.n_nodes, net.cpt.size, stride, cap, 1], np.int64).tobytes())
        f.write(np.array([eps, 0.0], np.float64).tobytes())
        f.write(ev.ev_off.astype(np.int64).tobytes() + ev.ev_node.astype(np.int32).tobytes() + ev.ev_state.astype(np.int32).tobytes())
        f.write(net.belief_off[:-1].astype(np.int32).tobytes() + net.cpt.astype(np.float64).tobytes())
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=0:report_signal_unsafe=0")
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True, env=env, timeout=900)
    if "FATAL: ThreadSanitizer" in r.stderr and "unexpected memory mapping" in r.stderr:
        pytest.skip("ThreadSanitizer cannot map its shadow memory in this container")
    if damage:
        assert r.stderr.count("WARNING: ThreadSanitizer: data race") >= 1
        return
    assert "WARNING: ThreadSanitizer" not in r.stderr, r.stderr[:4000]
    assert r.returncode == 0, r.stderr[-2000:]
    raw = open(tmp_path / "out.bin", "rb").read()
    n = ev.n_cases
    got = np.frombuffer(raw[:n * stride * 8], np.float64).reshape(n, stride)
    sw = np.frombuffer(raw[n * stride * 8:n * stride * 8 + 4 * n], np.int32)
    want, osw, _ = oracle_mod.run_port(net, ev, eps=eps, max_sweeps=cap)
    assert np.array_equal(sw, osw)
    assert_close(got, want, 1e-9, 1e-12, "on chip under ThreadSanitizer")


def test_float_handles_on_chip_hold_the_fp32_bar(engine, oracle_mod, tmp_path):
    net = _net("alarm37")
    ev = synth.make_evidence(net, 130, seed=17, exact_k=4)
    k = OnchipEmulated(engine, net, "fp32", 8, str(tmp_path))
    assert k.OUT == np.float32                                    # marginals in the handle's precision (bnbp_run_params.out_precision)
    want, osw, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=20)
    got, sw, _ = k.run(ev, 0.0, 20)
    assert np.array_equal(sw, osw)
    assert_close(got, want, 1e-5, 1e-7, "alarm37 on chip, fp32")


def test_edge_batches_and_the_reference_fixtures_on_chip(engine, oracle_mod, ref_fixtures, tmp_path):
    """Batches around the group width (1 ... 65 cases: lanes without a case, one refill with a single case), no evidence
    at all, every node observed, a sweep cap below the test interval, an epsilon nothing undercuts -- and the reference's own
    test graphs (Pearl, the resume graph, the impossible-evidence case) from the outputs of the compiled reference."""
    from bayesiannetwork_b200.flat import EvidenceBatch
    from helpers import load_fixture
    net = _net("alarm37")
    k8 = OnchipEmulated(engine, net, "fp64", 8, str(tmp_path))
    k9 = OnchipEmulated(engine, net, "fp64", 9, str(tmp_path))

    def check(k, ev, eps, cap, **kw):
        want, osw, ocv = oracle_mod.run_port(net, ev, eps=eps, max_sweeps=cap, damping=kw.get("damping", 0.0),
                                             check_interval=kw.get("interval", 1))
        got, sw, conv = k.run(ev, eps, cap, **kw)
        assert np.array_equal(sw, osw) and np.array_equal(conv, ocv)
        assert_close(got, want, 1e-9, 1e-12, f"{ev.n_cases} cases, eps {eps}, cap {cap}, {kw}")

    for n in (1, 31, 33, 65):
        ev = synth.make_evidence(net, n, seed=n, exact_k=4)
        check(k8, ev, 0.0, 5)
        check(k9, ev, 1e-6, 200)
    check(k9, EvidenceBatch.empty(40), 1e-6, 100)
    everything = EvidenceBatch.from_cases(net, [{x: int((x + c) % net.card[x]) for x in range(net.n_nodes)} for c in range(5)])
    check(k8, everything, 0.0, 3)
    ev = synth.make_evidence(net, 50, seed=3, exact_k=4)
    check(k9, ev, 0.0, 7, damping=0.3)                  # a fixed count with damping takes the check flavour
    check(k9, ev, 1e-6, 3, interval=5)                  # the cap comes before the first tested sweep
    check(k9, ev, 1e-13, 60)
    check(k9, ev, 10.0, 30)                             # every case stops after its first sweep
    for name in ("pearl_tests", "pearl_nan", "resume_tests", "pearl_one_sweep"):
        f = load_fixture(ref_fixtures, name)
        f["net"].name = name
        kk = OnchipEmulated(engine, f["net"], "fp64", 9 if f["eps"] > 0 else 8, str(tmp_path))
        got, sw, conv = kk.run(f["ev"], f["eps"], f["max_sweeps"] if f["max_sweeps"] > 0 else 1 << 20)
        assert np.array_equal(sw, f["sweeps"]) and np.array_equal(conv, f["converged"]), name
        assert_close(got, f["marginals"], 1e-9, 1e-12, name)
