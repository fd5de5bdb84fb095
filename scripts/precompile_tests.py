"""Fill the in-tree cubin cache with the specialised kernels the GPU tests will ask for, so the
GPU box spends its minutes on running them (NVRTC works without a GPU).  Purely an optimisation:
a missing cache entry is compiled on the box on first use."""
import os
import sys
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def jobs():
    import numpy as np
    import test_gpu_spec as t
    from helpers import load_fixture
    out = []
    for name, net, evkw, eps, cap in t._cases():
        for prec in ("fp64", "fp32"):
            if prec == "fp32" and eps > 0:
                continue
            out.append((net, prec, 0b00100 if eps > 0 else 0b11111001))
    fx = np.load(os.path.join(ROOT, "tests", "golden", "ref_fixtures.npz"), allow_pickle=False)
    for name in ["pearl_tests", "pearl_nan_fixed6", "resume_tests"]:   # (0b...1 also serves the split eps path)
        f = load_fixture(fx, name)
        out.append((f["net"], "fp64", 0b11111101))
    from bayesiannetwork_b200 import synth
    out.append((synth.grid(5, seed=8), "fp64", 0b11111111))
    out.append((synth.alarm37(), "fp64", 0b00000110))           # eps-mode compaction tests
    out.append((synth.alarm37(), "fp32", 0b00000110))
    # the on-chip kernel (tests/test_gpu_onchip.py): bit 8 fixed sweeps, 9 the same with double marginals from a
    # float kernel (host-buffer call), 10 / 11 the epsilon / damping flavours
    import test_gpu_onchip as oc
    for name, net, evkw, eps, cap in oc._cases():
        out.append((net, "fp64", 1 << (10 if eps > 0 else 8)))
        if not eps > 0:
            out.append((net, "fp32", 1 << 9))
    for name in ["pearl_tests", "resume_tests"]:
        f = load_fixture(fx, name)
        out.append((f["net"], "fp64", (1 << 8) | (1 << 10)))
    out.append((synth.random_dag(20, 3, 2, 4, seed=31), "fp64", 1 << 8))
    # class-looped walks (tests/test_gpu_classloop.py): the small networks forced through the class generator, alarm37 for
    # the bit-for-bit comparison with the unrolled walk, and the network the mode exists for (cfg 3, the 100 x 100 grid)
    import test_gpu_classloop as cl
    force = {"BNBP_CLASSLOOP": "2"}
    for name, net, evkw, eps, cap in cl._cases():
        for prec in ("fp64", "fp32"):
            if prec == "fp32" and eps > 0:
                continue
            out.append((net, prec, 0b00100 if eps > 0 else 0b11001, force))
    out.append((synth.alarm37(), "fp64", 0b11101, force))
    out.append((synth.grid(100), "fp64", 0b11101))
    out.append((synth.grid(100), "fp32", 0b11001))
    # the shape-boundary networks (tests/test_gpu_edge_shapes.py): unrolled walks (fused variants included), class-looped
    # walks, the on-chip kernel (fixed / epsilon in fp64, double marginals from a float kernel; refused for hub65: reported
    # as not compiled), and hub65 the way AUTO lays it out
    import edge_networks as en
    unrolled = {"BNBP_CLASSLOOP": "0"}
    for net in en.catalogue().values():
        out.append((net, "fp64", 0b01111111, unrolled))
        out.append((net, "fp32", 0b11111111, unrolled))
        out.append((net, "fp64", 0b11111, force))
        out.append((net, "fp32", 0b11111, force))
        out.append((net, "fp64", (1 << 8) | (1 << 10), unrolled))
        out.append((net, "fp32", 1 << 9, unrolled))
    out.append((en.catalogue()["hub65"], "fp64", 0b01111111))
    # expected counts (tests/test_gpu_em.py): the polytree checked against enumeration, and the 20 x 20 grid class-looped
    for prec in ("fp64", "fp32"):
        out.append((synth.random_polytree(8, card_hi=4, max_parents=3, seed=9), prec, 0b11111))
        out.append((synth.grid(20), prec, 0b11001, force))
    return out


def one(job):
    from bayesiannetwork_b200 import engine
    net, prec, mask = job[:3]
    env = job[3] if len(job) > 3 else {}
    os.environ.update(env)                 # knobs the library reads when it lays the network out (one job per worker call)
    try:
        engine.precompile(net, prec, mask)
    except engine.BnbpError as e:          # e.g. a test network whose state does not fit the on-chip kernel: the test skips it
        return net.name, prec, mask, f"not compiled: {e}"
    finally:
        for k in env:
            os.environ.pop(k, None)
    return net.name, prec, mask


if __name__ == "__main__":
    with ProcessPoolExecutor(8) as ex:
        for r in ex.map(one, jobs()):
            print(r, flush=True)
