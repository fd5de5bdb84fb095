"""ctypes binding of tests/em_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The expected-counts reference: oracle/bp_oracle.c's BP restatement (included unchanged through logev_oracle.c), each
case's Bethe log-evidence, and its family posteriors added serially in case order.  Compiled on first use into a
private temporary directory, so a read-only checkout works and nothing is left in the tree."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "em_oracle.c")
_lib = None


def _load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="bnbp_em_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libem_oracle.so")
        # gcc from PATH, as oracle/Makefile does; the counts loop is serial, OpenMP is not needed
        subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-Wall", "-Wextra", "-Wno-unknown-pragmas", "-o", so,
                        SRC, "-lm"], check=True, capture_output=True)
        _lib = C.CDLL(so)
        _lib.bp_oracle_run_expected_counts.restype = C.c_int
    return _lib


def _ptr(a, ctype):
    return None if a is None else a.ctypes.data_as(C.POINTER(ctype))


def run(net, ev, eps=1e-3, max_sweeps=0, damping=0.0, check_interval=1, weights=None, counts=None):
    """The oracle's sum-product BP on hard evidence, each case's log-evidence, and the expected family counts added
    into ``counts`` (a fresh zero array when None).  Returns (counts [cpt_values], marginals [B, sum r], sweeps [B],
    converged [B], log-evidence [B])."""
    if ev.is_soft:
        raise ValueError("expected counts take hard evidence")
    lib = _load()
    if counts is None:
        counts = np.zeros(int(net.cpt_off[-1]), dtype=np.float64)
    assert counts.dtype == np.float64 and counts.size == int(net.cpt_off[-1]) and counts.flags.c_contiguous
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
    assert w is None or w.shape == (ev.n_cases,)
    out = np.empty((ev.n_cases, net.belief_values), dtype=np.float64)
    sweeps = np.empty(ev.n_cases, dtype=np.int32)
    conv = np.empty(ev.n_cases, dtype=np.uint8)
    logev = np.empty(ev.n_cases, dtype=np.float64)
    cpt = np.ascontiguousarray(net.cpt, dtype=np.float64)
    rc = lib.bp_oracle_run_expected_counts(
        C.c_int32(net.n_nodes), _ptr(net.card, C.c_int32), _ptr(net.parent_off, C.c_int32),
        _ptr(net.parents, C.c_int32), _ptr(net.cpt_off, C.c_int64), _ptr(cpt, C.c_double),
        C.c_int64(ev.n_cases), _ptr(ev.ev_off, C.c_int64), _ptr(ev.ev_node, C.c_int32), _ptr(ev.ev_state, C.c_int32),
        _ptr(w, C.c_double), C.c_double(eps), C.c_int32(max_sweeps), C.c_double(damping), C.c_int32(check_interval),
        _ptr(counts, C.c_double), _ptr(out, C.c_double), _ptr(sweeps, C.c_int32), _ptr(conv, C.c_uint8),
        _ptr(logev, C.c_double))
    if rc != 0:
        raise RuntimeError("bp_oracle_run_expected_counts failed")
    return counts, out, sweeps, conv, logev
