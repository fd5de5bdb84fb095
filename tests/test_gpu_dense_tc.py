"""Tensor-core variant of the dense contraction path (csrc/bnbp_dense_tc.cuh: tcgen05 MMAs with fp32
accumulators in TMEM, every operand split hi + lo into two tf32 values) -- needs a B200 (-m gpu).

fp32 handles only; the bar is the library's fp32 tolerance against the fp64 oracle (1e-5 / 1e-7) at
fixed sweep counts, the same bar the CUDA-core products meet.  `dense_tensor=1` sends EVERY dense
product through the tensor-core kernel, so small networks cover ragged K and N, one-step products,
odd tile counts, both state-tile widths, frozen tiles (epsilon mode) and CPT refresh."""
import os
import subprocess

import numpy as np
import pytest

from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.flat import FlatNetwork
from helpers import assert_close
from test_gpu_parity import TOL

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def BP():
    from bayesiannetwork_b200.engine import BeliefPropagation
    return BeliefPropagation


def test_kernel_against_host_product():
    """The kernel alone: T = A x B against a double-precision host product (tests/cuda/test_dense_tc.cu)."""
    exe = os.path.join(ROOT, "tests", "cuda", "_build", "test_dense_tc")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "dense_tc ok" in r.stdout, r.stdout[-3000:] + r.stderr[-1000:]


def _cases():
    # (name, network, evidence kwargs, sweeps, dense_min_cpt, n_cases)
    yield "card8_k3", synth.high_card(12, card=8, n_parents=3, seed=31), dict(p=0.15), 6, 0, 300
    yield "card16_k2", synth.high_card(10, card=16, n_parents=2, seed=9), dict(p=0.2), 6, 256, 300
    yield "card32_k2", synth.high_card(6, card=32, n_parents=2, seed=10), dict(p=0.2), 5, 1024, 520
    yield "card12_k3", synth.random_dag(24, 3, 2, 12, seed=8), dict(p=0.1), 8, 64, 300
    yield "dag80_card8_all", synth.random_dag(80, 4, 2, 8, seed=7), dict(p=0.1), 9, 2, 129
    yield "wide_parents_k7", synth.random_dag(40, 7, 2, 3, seed=12), dict(p=0.1), 6, 16, 300
    yield "alarm37_vec2_soft", synth.alarm37(), dict(exact_k=4, soft=True), 15, 8, 700
    yield "grid8", synth.grid(8, seed=4), dict(p=0.1), 30, 2, 1


@pytest.mark.parametrize("name,net,evkw,cap,dmin,n", list(_cases()), ids=[c[0] for c in _cases()])
def test_every_product_on_tensor_cores_vs_oracle(BP, oracle_mod, name, net, evkw, cap, dmin, n):
    ev = synth.make_evidence(net, n, seed=17, **evkw)
    om, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=cap, threads=0)
    bp = BP(net, "fp32", dense_min_cpt=dmin, dense_tensor=1)
    st = bp.stats()
    assert st["dense_nodes"] > 0 and st["dense_tensor_jobs"] == 2 * st["dense_nodes"], (name, st)
    res = bp(ev, 0.0, max_sweeps=cap)
    assert bp.stats()["last_dense_tensor_launches"] >= cap
    assert_close(res.marginals, om, what=name, **TOL["fp32"])


def test_default_thresholds_and_cuda_core_equivalence(BP, oracle_mod):
    """card 16 / 3 parents: 256 x 256 products take the tensor cores by default; the same handle with
    dense_tensor=-1 (FMA products) agrees to fp32 rounding; fp64 handles never use the path."""
    net = synth.high_card(8, card=16, n_parents=3, seed=5)
    ev = synth.make_evidence(net, 256, p=0.15, seed=3)
    a, b = BP(net, "fp32"), BP(net, "fp32", dense_tensor=-1)
    assert a.stats()["dense_tensor_jobs"] == 2 * a.stats()["dense_nodes"] > 0
    assert b.stats()["dense_tensor_jobs"] == 0 and BP(net, "fp64").stats()["dense_tensor_jobs"] == 0
    ra, rb = a(ev, 0.0, max_sweeps=8), b(ev, 0.0, max_sweeps=8)
    assert a.stats()["last_dense_tensor_launches"] == 8 and b.stats()["last_dense_tensor_launches"] == 0
    assert_close(ra.marginals, rb.marginals, rtol=2e-5, atol=2e-7, what="tensor vs FMA products")
    om, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=8, threads=0)
    assert_close(ra.marginals, om, what="card16_k3 default", **TOL["fp32"])


def test_epsilon_mode_frozen_tiles_and_refresh(BP, oracle_mod):
    net = synth.random_dag(60, 4, 2, 6, seed=13)
    ev = synth.make_evidence(net, 600, p=0.1, seed=2)
    bp = BP(net, "fp32", dense_min_cpt=2, dense_tensor=1)
    om, osw, _ = oracle_mod.run_port(net, ev, eps=1e-4, max_sweeps=100, threads=0)
    res = bp(ev, 1e-4, max_sweeps=100)
    # fp32 sweep counts may differ by one where a delta sits on the threshold; beliefs agree to eps scale
    assert np.all(np.abs(res.sweeps.astype(int) - osw.astype(int)) <= 1)
    assert_close(res.marginals, om, rtol=1e-3, atol=1e-4, what="eps mode")
    rng = np.random.default_rng(5)
    cpt = net.cpt.copy()
    for x in range(net.n_nodes):
        rows = cpt[net.cpt_off[x]:net.cpt_off[x + 1]].reshape(-1, int(net.card[x]))
        rows[:] = 0.05 + rng.random(rows.shape)
        rows /= rows.sum(axis=1, keepdims=True)
    net2 = FlatNetwork(net.card, net.parent_off, net.parents, net.cpt_off, cpt, name="refreshed")
    bp.refresh_cpt(net2.cpt)
    om2, _, _ = oracle_mod.run_port(net2, ev, eps=0.0, max_sweeps=10, threads=0)
    assert_close(bp(ev, 0.0, max_sweeps=10).marginals, om2, what="refreshed", **TOL["fp32"])


def test_destroy_returns_the_tensor_core_arena(BP):
    """Creating and destroying handles leaves the free device memory where it was, the pre-tiled tensor-core CPT
    arena included: 13 nodes of 32 states with 3 parents are 26 products of 1024 x 1024, each pre-tiled hi | lo into
    8 MiB, so 12 handles hold 2.4 GiB of arena between them."""
    import torch
    net = synth.high_card(16, card=32, n_parents=3, seed=5)
    bp = BP(net, "fp32", device=0, dense_tensor=1)      # warm-up: context, modules, shared-memory opt-ins
    assert bp.stats()["dense_tensor_jobs"] == 26
    bp.close()
    free0, _ = torch.cuda.mem_get_info(0)
    for _ in range(12):
        BP(net, "fp32", device=0, dense_tensor=1).close()
    free1, _ = torch.cuda.mem_get_info(0)
    assert free0 - free1 < 256 << 20, f"{(free0 - free1) / 2**20:.0f} MiB of device memory not returned by bnbp_destroy"


def test_card32_full_size_sample(BP, oracle_mod):
    """BASELINE config 5 at full size (64 nodes, card 32, 3 parents: 61 CPTs of 32^4 entries, products of
    depth K = 1024): a small sample of cases against the oracle, fp32 on the tensor cores and fp64."""
    net = synth.high_card()
    ev = synth.make_evidence(net, 8, p=0.1, seed=3)
    om, _, _ = oracle_mod.run_port(net, ev, eps=0.0, max_sweeps=3, threads=0)
    bp = BP(net, "fp32")
    st = bp.stats()
    assert st["dense_nodes"] == 61 and st["dense_tensor_jobs"] == 122
    assert_close(bp(ev, 0.0, max_sweeps=3).marginals, om, what="card32 fp32 tensor", **TOL["fp32"])
    del bp
    assert_close(BP(net, "fp64")(ev, 0.0, max_sweeps=3).marginals, om, what="card32 fp64", **TOL["fp64"])
