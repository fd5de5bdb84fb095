"""The source the network compiler generates (bnbp_jit.cu: trait structs / class tables + bnbp_spec.cuh), compiled
as ORDINARY HOST CODE by g++ (tests/emul/cuda_host_shim.h) and run against the oracle -- WITHOUT a GPU.

The streaming sweep kernel gives a case to one thread and no thread reads what another wrote, so one call of the
kernel function per (block, thread) is the kernel.  That checks, on the CPU box, everything but timing: the generated
offsets / class records, the walk order (node by node, or class by class -- BNBP_CLASSLOOP), the one-pass node
arithmetic, first/last-sweep variants and the delta of the check variant.  The GPU parity tests of the same kernels
are tests/test_gpu_spec.py and tests/test_gpu_fullsize.py (-m gpu).
"""
import ctypes as C
import os
import shutil
import subprocess
import threading

import numpy as np
import pytest

from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.flat import EvidenceBatch
from helpers import assert_close

HERE = os.path.dirname(os.path.abspath(__file__))
# the generator reads its knobs from the environment: one source generation at a time, so that kernels can be built
# from several threads (the g++ runs are what takes the time)
SOURCE_LOCK = threading.Lock()
pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")


def generated_source(engine, net, precision, variant, env):
    """engine.spec_source with generator knobs (BNBP_CLASSLOOP, BNBP_OC_ROLES, ...) set in the environment meanwhile."""
    with SOURCE_LOCK:
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            return engine.spec_source(net, precision, variant)
        finally:
            for k, v in saved.items():
                if v is None:
                    del os.environ[k]
                else:
                    os.environ[k] = v


@pytest.fixture(scope="module")
def engine():
    from bayesiannetwork_b200 import _build, engine
    _build.build()
    return engine


class Emulated:
    """One generated kernel (network x precision x variant x walk mode) as a host shared object."""

    def __init__(self, engine, net, precision, variant, classloop, workdir, vec=1):
        src = generated_source(engine, net, precision, variant, {"BNBP_CLASSLOOP": "2" if classloop else "0", "BNBP_SPEC_VEC": str(vec)})
        assert ("#define BNBP_CLASSLOOP 1" in src) == classloop
        tag = f"{net.name}_{precision}_v{variant}_{'cls' if classloop else 'unr'}_x{vec}"
        cu = os.path.join(workdir, tag + ".cu")
        so = os.path.join(workdir, tag + ".so")
        with open(cu, "w") as f:
            f.write(src)
        cmd = ["g++", "-O0", "-std=c++17", "-ffp-contract=off", "-fvisibility=hidden", "-fno-gnu-unique", "-Wno-unknown-pragmas", "-I", os.path.join(HERE, "emul"),
               f'-DBNBP_GENERATED="{cu}"', "-shared", "-fPIC", "-o", so, os.path.join(HERE, "emul", "spec_emul.cpp")]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        self.lib = C.CDLL(so)
        self.src = src
        self.T = np.float32 if precision == "fp32" else np.float64
        self.cT = C.c_float if precision == "fp32" else C.c_double
        assert self.lib.emul_value_bytes() == np.dtype(self.T).itemsize and self.lib.emul_variant() == variant
        self.PL, self.M, self.W, self.TBC = (self.lib.emul_pl(), self.lib.emul_m(), self.lib.emul_w(), self.lib.emul_tbc())
        cpt = np.ascontiguousarray(net.cpt, dtype=self.T)
        self.lib.emul_set_cpt(cpt.ctypes.data_as(C.c_void_p), C.c_longlong(cpt.size))

    def launch(self, st, cur, nxt, n_inner=1, eps=0.0, damping=0.0, sweep_index=0, prev_tested=0, per_case=None, node_slices=1,
               evst=None):
        p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        pc = per_case or {}
        self.lib.emul_launch(p(st["pl"]), p(cur), p(nxt), p(st["evbits"]), C.c_int(st["tiles"]), C.c_int(n_inner),
                             self.cT(eps), self.cT(damping), C.c_int(sweep_index), C.c_int(prev_tested),
                             p(pc.get("delta_prev")), p(pc.get("delta_cur")), p(pc.get("delta_next")),
                             p(pc.get("status")), p(pc.get("sweeps")), p(pc.get("last_active")), C.c_int(node_slices), p(evst))


def initial_state(net, ev, k):
    """Time-0 arena the way K0 (init_kernel, belief_propagation.hpp:33-73) leaves it: batch-minor tiles
    state[tile][slot][TBC]; pi = lambda = 1, a root's pi = its prior row, an observed node's pi = lambda = the one-hot
    row, every message 1; observed-node bits [tile][W][TBC]."""
    tbc, tiles = k.TBC, (ev.n_cases + k.TBC - 1) // k.TBC
    n = net.n_nodes
    pl_off = np.concatenate([[0], np.cumsum(2 * net.card.astype(np.int64))])
    assert pl_off[-1] == k.PL and net.msg_values == k.M and (n + 31) // 32 == k.W
    pl = np.ones((tiles, k.PL, tbc), dtype=k.T)
    for x in range(n):
        if net.parent_off[x + 1] == net.parent_off[x]:
            r = int(net.card[x])
            pl[:, pl_off[x]:pl_off[x] + r, :] = net.cpt[net.cpt_off[x]:net.cpt_off[x] + r].astype(k.T)[None, :, None]
    evbits = np.zeros((tiles, k.W, tbc), dtype=np.uint32)
    for c in range(ev.n_cases):
        t, j = divmod(c, tbc)
        for e in range(int(ev.ev_off[c]), int(ev.ev_off[c + 1])):
            x, s = int(ev.ev_node[e]), int(ev.ev_state[e])
            r = int(net.card[x])
            row = np.zeros(r, dtype=k.T)
            row[s] = 1
            pl[t, pl_off[x]:pl_off[x] + r, j] = row
            pl[t, pl_off[x] + r:pl_off[x] + 2 * r, j] = row
            evbits[t, x >> 5, j] |= np.uint32(1 << (x & 31))
    msg = [np.ones((tiles, k.M, tbc), dtype=k.T), np.full((tiles, k.M, tbc), 7.0, dtype=k.T)]   # 7: never read before written
    return dict(pl=pl, msg=msg, evbits=evbits, tiles=tiles, pl_off=pl_off)


def beliefs(net, st, n_cases):
    """normalize(pi .* lambda) per node (belief_propagation.hpp:151-158) from the arena, case-major rows."""
    tbc = st["pl"].shape[2]
    out = np.empty((n_cases, net.belief_values), dtype=np.float64)
    boff = net.belief_off
    for x in range(net.n_nodes):
        r, o = int(net.card[x]), int(st["pl_off"][x])
        prod = st["pl"][:, o:o + r, :].astype(np.float64) * st["pl"][:, o + r:o + 2 * r, :].astype(np.float64)
        with np.errstate(invalid="ignore", divide="ignore"):
            b = prod / prod.sum(axis=1, keepdims=True)
        out[:, boff[x]:boff[x] + r] = b.transpose(0, 2, 1).reshape(-1, r)[:n_cases]
    return out


def run_fixed(kernels, net, ev, sweeps):
    """The launch sequence of a fixed-count run (bnbp_api.cu): variant 3 (first), 0 ..., 4 (last)."""
    st = initial_state(net, ev, kernels[0])
    cur, nxt = st["msg"]
    for t in range(sweeps):
        v = 0 if sweeps < 2 else (3 if t == 0 else (4 if t == sweeps - 1 else 0))
        kernels[v].launch(st, cur, nxt)
        cur, nxt = nxt, cur
    return st, cur


def _networks():
    yield "pearl", synth.pearl_network(), dict(p=0.3)
    yield "grid6", synth.grid(6), dict(p=0.15)
    yield "polytree40", synth.random_polytree(40, card_hi=4, max_parents=3, seed=11), dict(p=0.15)
    yield "dag30", synth.random_dag(30, max_parents=3, card_lo=2, card_hi=4, seed=5), dict(p=0.2)


@pytest.mark.parametrize("classloop", [False, True], ids=["unrolled", "classloop"])
@pytest.mark.parametrize("name,net,evkw", list(_networks()), ids=[n[0] for n in _networks()])
def test_generated_sweeps_match_the_oracle_on_the_host(engine, oracle_mod, tmp_path, name, net, evkw, classloop):
    net.name = name
    ev = synth.make_evidence(net, 150, seed=3, **evkw)                 # two tiles, the second one ragged
    ks = {v: Emulated(engine, net, "fp64", v, classloop, str(tmp_path)) for v in (0, 3, 4)}
    for sweeps in (1, 2, 7):
        st, _ = run_fixed(ks, net, ev, sweeps)
        want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=sweeps)
        assert_close(beliefs(net, st, ev.n_cases), want, 1e-9, 1e-12, f"{name} {sweeps} sweeps")


def test_classloop_equals_unrolled_bit_for_bit_and_loops_in_kernel(engine, tmp_path):
    """Same arithmetic per node in both code generators: the arenas agree bit for bit; the in-kernel loop over
    sweeps (variant 0, n_inner) equals separate launches; two cases per thread (16-byte accesses) equal one; node slices
    in grid.y (small batches) equal the unsliced walk."""
    net = synth.random_dag(30, max_parents=3, card_lo=2, card_hi=4, seed=5)
    net.name = "dag30"
    ev = synth.make_evidence(net, 300, seed=4, p=0.2)
    res = {}
    for mode, cl, vec, inner, slices in (("unrolled", False, 1, 1, 1), ("classloop", True, 1, 1, 1), ("classloop_inner", True, 1, 6, 1),
                                         ("classloop_vec2", True, 2, 1, 1), ("classloop_slices3", True, 1, 1, 3),
                                         ("classloop_slices16", True, 1, 1, 16)):     # 16 slices: more than most classes have nodes
        k = Emulated(engine, net, "fp64", 0, cl, str(tmp_path), vec=vec)
        st = initial_state(net, ev, k)
        cur, nxt = st["msg"]
        if inner > 1:
            k.launch(st, cur, nxt, n_inner=inner)             # buffers swapped per inner sweep: 6 sweeps end in `cur`
        else:
            for _ in range(6):
                k.launch(st, cur, nxt, node_slices=slices)    # grid.y: block (tile, y) walks the y-th slice of every class
                cur, nxt = nxt, cur
        # case-major copies, so that the tile width (128 x cases per thread) does not matter
        res[mode] = (st["pl"].transpose(0, 2, 1).reshape(-1, k.PL)[:ev.n_cases].copy(),
                     cur.transpose(0, 2, 1).reshape(-1, k.M)[:ev.n_cases].copy())
    for mode in ("classloop", "classloop_inner", "classloop_vec2", "classloop_slices3", "classloop_slices16"):
        assert np.array_equal(res[mode][0], res["unrolled"][0]), mode
        assert np.array_equal(res[mode][1], res["unrolled"][1]), mode


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_classloop_check_variant_delta_freeze_and_evidence_rows(engine, tmp_path, precision):
    """Variant 2 (freeze + check) in a class-looped walk: the per-case delta is max |new - old| over the messages
    (:105-131), frozen cases keep their state, observed nodes keep their rows (:177,:223)."""
    net = synth.grid(5)
    net.name = "grid5"
    ev = synth.make_evidence(net, 128, seed=9, p=0.2)
    k = Emulated(engine, net, precision, 2, True, str(tmp_path))
    st = initial_state(net, ev, k)
    cur, nxt = st["msg"]
    n = st["tiles"] * k.TBC
    floor = np.finfo(k.T).tiny
    pc = dict(delta_prev=np.full(n, floor, k.T), delta_cur=np.full(n, floor, k.T), delta_next=np.zeros(n, k.T),
              status=np.zeros(n, np.uint8), sweeps=np.zeros(n, np.int32), last_active=np.zeros(1, np.int32))
    pc["status"][5] = 1                                              # a case frozen by an earlier sweep
    pl0 = st["pl"].copy()
    k.launch(st, cur, nxt, eps=1e-6, sweep_index=0, prev_tested=0, per_case=pc)
    d = np.abs(nxt - cur)                                            # in the kernel's precision; every time-0 message is 1
    want = np.maximum(np.nanmax(d, axis=1).reshape(-1), floor).astype(np.float64)
    live = np.ones(n, bool)
    live[5] = False
    got = pc["delta_cur"].astype(np.float64)
    assert np.array_equal(got[live], want[live])
    assert np.all(nxt[0, :, 5] == 7.0) and np.array_equal(st["pl"][0, :, 5], pl0[0, :, 5])      # frozen: nothing written
    assert np.all(pc["delta_next"] == floor)
    # observed nodes keep their one-hot rows in both pi and lambda
    for c in range(ev.n_cases):
        for e in range(int(ev.ev_off[c]), int(ev.ev_off[c + 1])):
            x = int(ev.ev_node[e])
            o, r = int(st["pl_off"][x]), int(net.card[x])
            assert np.array_equal(st["pl"][c // k.TBC, o:o + 2 * r, c % k.TBC], pl0[c // k.TBC, o:o + 2 * r, c % k.TBC])


def test_grid100_is_walked_class_by_class(engine):
    """cfg 3: 10 000 nodes, 6 shape classes; the record table names every node once and carries its slots."""
    net = synth.grid(100)
    src = engine.spec_source(net, "fp64", 0)
    assert "#define BNBP_CLASSLOOP 1" in src
    classes = [l for l in src.splitlines() if l.startswith("struct C") and "static constexpr int R=" in l]
    assert 4 <= len(classes) <= 9
    walk = [l for l in src.splitlines() if l.startswith("#define BNBP_WALK")][0]
    assert walk.count("BNBP_CLASS(") == len(classes)
    body = src[src.index("__device__ const int bnbp_rec["):]
    body = body[body.index("{") + 1:body.index("};")]
    vals = np.array([int(t) for t in body.replace("\n", "").split(",") if t.strip()], dtype=np.int64)
    # walk the table with the (first, count) pairs of the walk and the K / M of each class
    import re
    seen = []
    for cl, (first, count) in zip(classes, re.findall(r"BNBP_CLASS\(C\d+,(\d+),(\d+)\)", walk)):
        kk, mm = int(re.search(r"K=(\d+)", cl).group(1)), int(re.search(r",M=(\d+)", cl).group(1))
        rec = vals[int(first):int(first) + int(count) * (5 + kk + mm)].reshape(int(count), 5 + kk + mm)
        for row in rec:
            x = int(row[0])
            seen.append(x)
            assert net.parent_off[x + 1] - net.parent_off[x] == kk
            assert row[4] == net.cpt_off[x] and row[1] == 2 * int(net.card[:x].sum())
    assert sorted(seen) == list(range(net.n_nodes))
    with pytest.raises(engine.BnbpError, match="variants 0-4"):
        engine.spec_source(net, "fp64", 6)


def run_eps(k, net, ev, eps, cap, interval=1, k_unchecked=None):
    """The host loop of an epsilon-mode run (bnbp_api.cu run_chunk): launch t runs the freeze + check variant when its sweep
    is tested (every `interval`-th sweep and the last one) and the freeze variant otherwise; a launch freezes the cases whose
    delta of a TESTED launch t-1 was below epsilon (status / sweeps), three delta buffers rotate; what is still running
    after the last launch is settled from its last delta."""
    st = initial_state(net, ev, k)
    n = st["tiles"] * k.TBC
    floor = np.finfo(k.T).tiny
    delta = [np.full(n, floor, k.T) for _ in range(3)]
    status, sweeps, last_active = np.zeros(n, np.uint8), np.zeros(n, np.int32), np.full(1, -1, np.int32)
    msg = st["msg"]
    t = 0
    prev_tested = False
    while t < cap:
        tested = (t + 1) % interval == 0 or t + 1 >= cap
        pc = dict(delta_prev=delta[(t + 2) % 3], delta_cur=delta[t % 3], delta_next=delta[(t + 1) % 3],
                  status=status, sweeps=sweeps, last_active=last_active)
        (k if tested else k_unchecked).launch(st, msg[t & 1], msg[(t + 1) & 1], eps=eps, sweep_index=t,
                                              prev_tested=1 if prev_tested else 0, per_case=pc)
        t += 1
        if last_active[0] < t - 1:                            # the launch found every case frozen: nothing ran
            t -= 1
            break
        prev_tested = tested
    last = delta[(t - 1) % 3]
    conv = status.astype(bool) | ((last < eps) & prev_tested)
    sw = np.where(status.astype(bool), sweeps, t)
    return st, sw[:ev.n_cases], conv[:ev.n_cases]


@pytest.mark.parametrize("name,classloop", [("alarm37", False), ("alarm37", True), ("grid6", True), ("polytree40", True)])
def test_epsilon_mode_on_the_host_stops_where_the_oracle_stops(engine, oracle_mod, tmp_path, name, classloop):
    net = {"alarm37": synth.alarm37, "grid6": lambda: synth.grid(6), "polytree40": lambda: synth.random_polytree(40, card_hi=4, max_parents=3, seed=11)}[name]()
    net.name = name
    ev = synth.make_evidence(net, 140, seed=5, **(dict(exact_k=4) if name == "alarm37" else dict(p=0.15)))
    eps = 1e-6
    want, osw, ocv = oracle_mod.run_port(net, ev, eps=eps, max_sweeps=300)
    k = Emulated(engine, net, "fp64", 2, classloop, str(tmp_path))
    st, sw, conv = run_eps(k, net, ev, eps, 300)
    assert np.array_equal(sw, osw), np.nonzero(sw != osw)[0][:8]
    assert np.array_equal(conv, ocv.astype(bool))
    assert_close(beliefs(net, st, ev.n_cases), want, 1e-9, 1e-12, f"{name} eps mode")


@pytest.mark.parametrize("classloop", [False, True], ids=["unrolled", "classloop"])
def test_float_kernels_on_the_host_hold_the_fp32_bar(engine, oracle_mod, tmp_path, classloop):
    """fp32 handles: the same generated code with T = float against the double-precision oracle at the fp32 bar of
    BASELINE.json (1e-5 relative + 1e-7 absolute) after 12 sweeps of a loopy network."""
    net = synth.grid(6)
    net.name = "grid6"
    ev = synth.make_evidence(net, 200, seed=8, p=0.15)
    ks = {v: Emulated(engine, net, "fp32", v, classloop, str(tmp_path)) for v in (0, 3, 4)}
    st, _ = run_fixed(ks, net, ev, 12)
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=12)
    assert_close(beliefs(net, st, ev.n_cases), want, 1e-5, 1e-7, "grid6 fp32")


@pytest.mark.parametrize("name", ["alarm37", "grid6"])
def test_first_sweep_fused_with_the_initialisation(engine, oracle_mod, tmp_path, name):
    """Variant 5 (unrolled walks): the time-0 pi / lambda (belief_propagation.hpp:33-73) are formed in registers from one
    evidence-state byte per (node, case) -- nothing of time 0 is read, so the arena may hold garbage when the run starts."""
    net = synth.alarm37() if name == "alarm37" else synth.grid(6)
    net.name = name
    ev = synth.make_evidence(net, 150, seed=21, **(dict(exact_k=4) if name == "alarm37" else dict(p=0.2)))
    ks = {v: Emulated(engine, net, "fp64", v, False, str(tmp_path)) for v in (5, 0)}
    st = initial_state(net, ev, ks[0])
    evst = np.zeros((st["tiles"], net.n_nodes, ks[0].TBC), np.uint8)
    for c in range(ev.n_cases):
        for e in range(int(ev.ev_off[c]), int(ev.ev_off[c + 1])):
            evst[c // ks[0].TBC, int(ev.ev_node[e]), c % ks[0].TBC] = int(ev.ev_state[e]) + 1
    st["pl"][:] = np.nan                                      # what K0 would have written is never read ...
    cur, nxt = st["msg"]
    cur[:] = np.nan                                           # ... nor are the time-0 messages
    ks[5].launch(st, cur, nxt, evst=evst)
    for _ in range(5):
        cur, nxt = nxt, cur
        ks[0].launch(st, cur, nxt)
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=6)
    assert_close(beliefs(net, st, ev.n_cases), want, 1e-9, 1e-12, f"{name} fused first sweep")


def test_epsilon_mode_tested_every_third_sweep(engine, oracle_mod, tmp_path):
    """check_interval = 3 (extension): untested sweeps run the freeze variant (1), tested ones the freeze + check variant (2)."""
    net = synth.alarm37()
    net.name = "alarm37"
    ev = synth.make_evidence(net, 140, seed=6, exact_k=4)
    want, osw, ocv = oracle_mod.run_port(net, ev, eps=1e-6, max_sweeps=300, check_interval=3)
    k1, k2 = (Emulated(engine, net, "fp64", v, False, str(tmp_path)) for v in (1, 2))
    st, sw, conv = run_eps(k2, net, ev, 1e-6, 300, interval=3, k_unchecked=k1)
    assert np.array_equal(sw, osw) and (osw % 3 == 0).all()
    assert np.array_equal(conv, ocv.astype(bool))
    assert_close(beliefs(net, st, ev.n_cases), want, 1e-9, 1e-12, "alarm37 eps mode, interval 3")


@pytest.mark.parametrize("precision,variant", [("fp64", 6), ("fp32", 6), ("fp32", 7)], ids=["fp64", "fp32", "fp32_double_marginals"])
def test_last_sweep_fused_with_the_beliefs(engine, oracle_mod, tmp_path, precision, variant):
    """Variants 6 / 7: the new pi / lambda of the last sweep stay in registers and BEL = normalize(pi .* lambda)
    (belief_propagation.hpp:151-158) leaves through a per-warp shared-memory tile as contiguous row segments of the
    case-major marginals -- a warp-cooperative kernel, emulated with one OS thread per CUDA thread of a block
    (tests/emul/spec_block_emul.cpp).  A ragged last tile: rows beyond the batch are never written."""
    net = synth.alarm37()
    net.name = "alarm37"
    ev = synth.make_evidence(net, 150, seed=22, exact_k=4)
    ks = {v: Emulated(engine, net, precision, v, False, str(tmp_path)) for v in (3, 0)}
    src = engine.spec_source(net, precision, variant)
    cu, so = str(tmp_path / f"last{variant}.cu"), str(tmp_path / f"last{variant}.so")
    open(cu, "w").write(src)
    cmd = ["g++", "-O0", "-std=c++17", "-ffp-contract=off", "-fvisibility=hidden", "-fno-gnu-unique", "-Wno-unknown-pragmas",
           "-I", os.path.join(HERE, "emul"), f'-DBNBP_GENERATED="{cu}"', "-shared", "-fPIC", "-pthread", "-o", so,
           os.path.join(HERE, "emul", "spec_block_emul.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    lib = C.CDLL(so)
    T = ks[0].T
    OUT = np.float32 if lib.emul_out_bytes() == 4 else np.float64
    assert OUT == (np.float64 if variant == 7 or precision == "fp64" else np.float32) and lib.emul_v() == net.belief_values
    cpt = np.ascontiguousarray(net.cpt, dtype=T)
    lib.emul_set_cpt(cpt.ctypes.data_as(C.c_void_p), C.c_longlong(cpt.size))
    st = initial_state(net, ev, ks[0])
    cur, nxt = st["msg"]
    ks[3].launch(st, cur, nxt)
    for _ in range(4):
        cur, nxt = nxt, cur
        ks[0].launch(st, cur, nxt)
    cur, nxt = nxt, cur
    out = np.full((ev.n_cases + 5, net.belief_values), -7.0, OUT)          # five guard rows behind the batch
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    lib.emul_launch_last(p(st["pl"]), p(cur), p(nxt), p(st["evbits"]), C.c_int(st["tiles"]), p(out), C.c_longlong(ev.n_cases))
    want, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=6)
    tol = (1e-9, 1e-12) if precision == "fp64" else (1e-5, 1e-7)
    assert_close(out[:ev.n_cases], want, *tol, f"fused last sweep {precision} v{variant}")
    assert (out[ev.n_cases:] == -7.0).all()
