"""ctypes binding of tests/logev_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The log-evidence reference: oracle/bp_oracle.c's BP restatement (included unchanged) plus the Bethe log-evidence of
each case from the state it ends with.  Compiled on first use into a private temporary directory, so a read-only
checkout works and nothing is left in the tree."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "logev_oracle.c")
_lib = None


def _load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="bnbp_logev_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "liblogev_oracle.so")
        # gcc from PATH, as oracle/Makefile does; without OpenMP where the compiler has none
        base = ["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", so, SRC, "-lm"]
        if subprocess.run(base[:6] + ["-fopenmp"] + base[6:], capture_output=True).returncode != 0:
            subprocess.run(base[:6] + ["-Wno-unknown-pragmas"] + base[6:], check=True, capture_output=True)
        _lib = C.CDLL(so)
        _lib.bp_oracle_run_log_evidence.restype = C.c_int
    return _lib


def _ptr(a, ctype):
    return None if a is None else a.ctypes.data_as(C.POINTER(ctype))


def run(net, ev, eps=1e-3, max_sweeps=0, damping=0.0, check_interval=1, threads=0):
    """The oracle's sum-product BP on hard evidence, plus each case's log-evidence.
    Returns (marginals [B, sum r], sweeps [B], converged [B], log-evidence [B])."""
    if ev.is_soft:
        raise ValueError("log-evidence takes hard evidence")
    lib = _load()
    out = np.empty((ev.n_cases, net.belief_values), dtype=np.float64)
    sweeps = np.empty(ev.n_cases, dtype=np.int32)
    conv = np.empty(ev.n_cases, dtype=np.uint8)
    logev = np.empty(ev.n_cases, dtype=np.float64)
    rc = lib.bp_oracle_run_log_evidence(
        C.c_int32(net.n_nodes), _ptr(net.card, C.c_int32), _ptr(net.parent_off, C.c_int32),
        _ptr(net.parents, C.c_int32), _ptr(net.cpt_off, C.c_int64), _ptr(net.cpt, C.c_double),
        C.c_int64(ev.n_cases), _ptr(ev.ev_off, C.c_int64), _ptr(ev.ev_node, C.c_int32), _ptr(ev.ev_state, C.c_int32),
        C.c_double(eps), C.c_int32(max_sweeps), C.c_double(damping), C.c_int32(check_interval), C.c_int32(threads),
        _ptr(out, C.c_double), _ptr(sweeps, C.c_int32), _ptr(conv, C.c_uint8), _ptr(logev, C.c_double))
    if rc != 0:
        raise RuntimeError("bp_oracle_run_log_evidence failed")
    return out, sweeps, conv, logev
