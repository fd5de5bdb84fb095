"""Host-side mirror of ``bn::inference::belief_propagation`` (belief_propagation.hpp:12-34) for
batches of evidence cases.  Construction flattens nothing itself -- it takes a ``FlatNetwork`` --
and uploads the device arena through ``bnbp_create``; calls go through ``bnbp_run_batch`` (host
buffers) or ``bnbp_run_batch_device`` (torch CUDA tensors: device memory and streams are the only
things torch is used for)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _capi
from ._capi import BnbpError  # noqa: F401
from .flat import EvidenceBatch, FlatNetwork

FP64, FP32 = 0, 1
SPECIALIZE = {"auto": 0, "always": 1, "never": 2}
ONCHIP = {"auto": 0, "always": 1, "never": -1}


def _net_c(net: FlatNetwork):
    return _capi.FlatNetworkC(net.n_nodes, _vp(net.card), _vp(net.parent_off), _vp(net.parents),
                              _vp(net.cpt_off), _vp(net.cpt))


def precompile(net: FlatNetwork, precision: str = "fp64", variants: int = 0b11111) -> None:
    """Run the network compiler without a GPU: generate the specialised sweep kernels of ``net``
    and leave their cubins in the cache (``bnbp_precompile``)."""
    lib = _capi.load()
    opt = _capi.OptionsC({"fp64": FP64, "fp32": FP32}[precision], -1, 0, 0)
    _capi.check(lib.bnbp_precompile(C.byref(_net_c(net)), C.byref(opt), variants))


def spec_source(net: FlatNetwork, precision: str = "fp64", variant: int = 0) -> str:
    """CUDA source the network compiler generates for ``net`` (``bnbp_spec_source``)."""
    lib = _capi.load()
    opt = _capi.OptionsC({"fp64": FP64, "fp32": FP32}[precision], -1, 0, 0)
    need = C.c_int64(0)
    _capi.check(lib.bnbp_spec_source(C.byref(_net_c(net)), C.byref(opt), variant, None, 0, C.byref(need)))
    buf = C.create_string_buffer(need.value)
    _capi.check(lib.bnbp_spec_source(C.byref(_net_c(net)), C.byref(opt), variant, buf, need.value, C.byref(need)))
    return buf.value.decode()


def estimate_cpt(net: FlatNetwork, samples: np.ndarray, multiplicity: Optional[np.ndarray] = None,
                 device: int = -1) -> np.ndarray:
    """``sampler::make_cpt`` (sampler.hpp:81-163) on the GPU (``bnbp_estimate_cpt``): the CPT arena of
    ``net``'s topology estimated from ``samples`` [n_rows, N] (state of every node per distinct sample)
    and their multiplicities.  ``net.cpt`` is not read; the result has its layout."""
    lib = _capi.load()
    samples = np.ascontiguousarray(samples, dtype=np.int32)
    if samples.ndim != 2 or samples.shape[1] != net.n_nodes:
        raise ValueError("samples must be [n_rows, n_nodes]")
    mult = None if multiplicity is None else np.ascontiguousarray(multiplicity, dtype=np.int64)
    if mult is not None and mult.shape != (samples.shape[0],):
        raise ValueError("multiplicity must be [n_rows]")
    out = np.empty(int(net.cpt_off[-1]), dtype=np.float64)
    _capi.check(lib.bnbp_estimate_cpt(C.byref(_net_c(net)), _vp(samples), _vp(mult), int(samples.shape[0]),
                                      int(device), _vp(out)))
    return out


@dataclass
class BPResult:
    marginals: np.ndarray      # [n_cases, sum r_X] (float64 on the host path)
    sweeps: np.ndarray         # [n_cases] int32
    converged: np.ndarray      # [n_cases] uint8
    log_evidence: Optional[np.ndarray] = None   # [n_cases] float64, Bethe estimate of ln P(e) (log_evidence=True)
    expected_counts: Optional[np.ndarray] = None   # [cpt_values] float64, expected family counts (expected_counts=True)

    def node(self, net: FlatNetwork, x: int) -> np.ndarray:
        off = net.belief_off
        return self.marginals[:, off[x]:off[x + 1]]


def _vp(a) -> Optional[int]:
    return None if a is None else a.ctypes.data


def m_step(net: FlatNetwork, counts: np.ndarray, pseudo_count: float = 0.0) -> np.ndarray:
    """The M-step of EM: ``sampler::make_cpt``'s normalisation (sampler.hpp:147-163) of expected family counts in the
    CPT-arena layout of ``net`` (``BPResult.expected_counts``).  ``pseudo_count`` is added to every entry first; a row
    whose total is 0 becomes uniform 1/r, as make_cpt does for a parent configuration never seen."""
    counts = np.asarray(counts, dtype=np.float64)
    if counts.shape != (int(net.cpt_off[-1]),):
        raise ValueError("counts must have cpt_off[-1] entries")
    if not (np.isfinite(pseudo_count) and pseudo_count >= 0.0):
        raise ValueError("pseudo_count must be finite and >= 0")
    out = np.empty_like(counts)
    for x in range(net.n_nodes):
        a, b, r = int(net.cpt_off[x]), int(net.cpt_off[x + 1]), int(net.card[x])
        rows = counts[a:b].reshape(-1, r) + pseudo_count
        tot = rows.sum(axis=1, keepdims=True)
        zero = tot[:, 0] == 0.0
        dst = out[a:b].reshape(-1, r)
        dst[~zero] = rows[~zero] / tot[~zero]
        dst[zero] = 1.0 / r
    return out


@dataclass
class EMResult:
    cpt: np.ndarray                # [cpt_values] the CPT after the last M-step (the handle holds it)
    log_likelihood: np.ndarray     # [iterations] sum_c w_c ln Z_B(e_c) over the counted cases, under the CPT going in
    skipped: np.ndarray            # [iterations] cases whose evidence was impossible under that CPT (counted nowhere)
    iterations: int


class BeliefPropagation:
    """``bp = BeliefPropagation(net); bp(evidence, epsilon)`` -- the reference call shape
    (belief_propagation.hpp:24,31) with a batch in place of one evidence map."""

    def __init__(self, net: FlatNetwork, precision: str = "fp64", device: int = -1,
                 max_resident_cases: int = 0, specialize: str = "auto", dense_min_cpt: int = 0,
                 dense_tensor: int = 0, onchip: str = "auto", devices: Optional[Sequence[int]] = None):
        self.net = net
        self.precision = {"fp64": FP64, "fp32": FP32, "f64": FP64, "f32": FP32}[precision]
        lib = _capi.load()
        self._lib = lib
        self._h = C.c_void_p()
        fn = _net_c(net)
        # dense_min_cpt: CPT size from which a node takes the dense contraction path (0 = default
        # 256 entries, < 0 = never); see include/bnbp.h
        # dense_tensor: fp32 handles run large dense products on the tensor cores (tcgen05, 3xTF32);
        # 0 = default, 1 = every dense product, -1 = never
        # onchip: the on-chip multi-sweep kernel ("auto": eligible networks with specialize="auto" and >= 4096
        # hard-evidence cases; "always" / "never")
        opt = _capi.OptionsC(self.precision, device, max_resident_cases, SPECIALIZE[specialize], int(dense_min_cpt),
                             int(dense_tensor), ONCHIP[onchip])
        # devices: several GPUs of this box behind one handle (bnbp_create_multi): a call shards its cases over them
        # ([] = every visible device); host-buffer calls only
        self.devices = None if devices is None else [int(d) for d in devices]
        if self.devices is None:
            _capi.check(lib.bnbp_create(C.byref(fn), C.byref(opt), C.byref(self._h)))
        else:
            arr = np.asarray(self.devices, dtype=np.int32)
            _capi.check(lib.bnbp_create_multi(C.byref(fn), C.byref(opt), _vp(arr) if arr.size else None, int(arr.size),
                                              C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.bnbp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- host buffers ---------------------------------------------------------------------------
    def __call__(self, evidence: Optional[EvidenceBatch] = None, epsilon: float = 0.001, *,
                 max_sweeps: int = 0, damping: float = 0.0, check_interval: int = 1,
                 out: Optional[np.ndarray] = None, out_sweeps: Optional[np.ndarray] = None,
                 out_converged: Optional[np.ndarray] = None, query_nodes: Optional[Sequence[int]] = None,
                 out_dtype=np.float64, semiring: str = "sum", log_evidence: bool = False,
                 marginals: bool = True, expected_counts: bool = False, weights: Optional[np.ndarray] = None,
                 counts_out: Optional[np.ndarray] = None) -> BPResult:
        """``query_nodes``: only these nodes' marginals are returned (columns in the given order);
        ``out_dtype=np.float32`` (fp32 handles): float marginals, half the device-to-host copy;
        ``semiring="max"``: max-product (max-marginals) instead of the reference's sum-product;
        ``log_evidence=True``: also each case's Bethe estimate of ln P(e) (``bnbp_run_batch_log_evidence``; exact on
        polytrees run to convergence; hard evidence only) in ``BPResult.log_evidence``;
        ``marginals=False`` (with ``log_evidence`` or ``expected_counts``): no marginals are computed into or copied to
        the host, the result's marginals are an (n, 0) array;
        ``expected_counts=True``: also the E-step of EM (``bnbp_run_batch_expected_counts``): sum_c w_c P(x, u | e_c)
        per CPT entry from the family beliefs of the final state, in ``BPResult.expected_counts`` (CPT-arena layout;
        ``weights`` [n_cases], default 1; added into ``counts_out`` when given, else into zeros)."""
        if not marginals and not log_evidence and not expected_counts:
            raise ValueError("marginals=False needs log_evidence=True or expected_counts=True (the call would return nothing)")
        if not expected_counts and (weights is not None or counts_out is not None):
            raise ValueError("weights / counts_out belong to expected_counts=True")
        if evidence is None:
            evidence = EvidenceBatch.empty(1)   # operator()(epsilon) by-pass (:24-28)
        ev = evidence
        q = None if query_nodes is None else np.ascontiguousarray(query_nodes, dtype=np.int32)
        n = ev.n_cases
        if q is not None and q.size and (int(q.min()) < 0 or int(q.max()) >= self.net.n_nodes):
            raise BnbpError(1, "query node id out of range")
        V = self.net.belief_values if q is None or q.size == 0 else int(self.net.card[q].sum())
        out_dtype = np.dtype(out_dtype)
        if not marginals:
            out = np.empty((n, 0), dtype=out_dtype)
        elif out is None:
            out = np.empty((n, V), dtype=out_dtype)
        if marginals:
            assert out.dtype == out_dtype and out.size == n * V and out.flags.c_contiguous
        # caller-owned result buffers (all three optional) keep a hot loop free of multi-megabyte
        # allocations: every fresh array is an mmap + page faults + munmap on the calling thread
        sweeps = np.empty(n, dtype=np.int32) if out_sweeps is None else out_sweeps
        conv = np.empty(n, dtype=np.uint8) if out_converged is None else out_converged
        assert sweeps.dtype == np.int32 and sweeps.size == n and sweeps.flags.c_contiguous
        assert conv.dtype == np.uint8 and conv.size == n and conv.flags.c_contiguous
        evc = _capi.EvidenceC(n, _vp(ev.ev_off), _vp(ev.ev_node),
                              None if ev.is_soft else _vp(ev.ev_state),
                              _vp(ev.ev_val_off) if ev.is_soft else None,
                              _vp(ev.ev_values) if ev.is_soft else None)
        prm = _capi.RunParamsC(float(epsilon), int(max_sweeps), float(damping), int(check_interval),
                               2 if out_dtype == np.float32 else 0, 0, 0 if q is None else int(q.size), _vp(q),
                               {"sum": 0, "max": 1}[semiring])
        if expected_counts:
            nv = int(self.net.cpt_off[-1])
            counts = np.zeros(nv, dtype=np.float64) if counts_out is None else counts_out
            assert counts.dtype == np.float64 and counts.size == nv and counts.flags.c_contiguous
            w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
            if w is not None and w.shape != (n,):
                raise ValueError("weights must be [n_cases]")
            logev = np.empty(n, dtype=np.float64) if log_evidence else None
            _capi.check(self._lib.bnbp_run_batch_expected_counts(self._h, C.byref(evc), C.byref(prm), _vp(w), _vp(counts),
                                                                 _vp(out) if marginals else None, _vp(sweeps), _vp(conv),
                                                                 _vp(logev)))
            return BPResult(out.reshape(n, V if marginals else 0), sweeps, conv, logev, counts)
        if log_evidence:
            logev = np.empty(n, dtype=np.float64)
            _capi.check(self._lib.bnbp_run_batch_log_evidence(self._h, C.byref(evc), C.byref(prm),
                                                              _vp(out) if marginals else None, _vp(sweeps), _vp(conv),
                                                              _vp(logev)))
            return BPResult(out.reshape(n, V if marginals else 0), sweeps, conv, logev)
        _capi.check(self._lib.bnbp_run_batch(self._h, C.byref(evc), C.byref(prm), _vp(out), _vp(sweeps), _vp(conv)))
        return BPResult(out.reshape(n, V), sweeps, conv)

    # ---- device-resident buffers (torch tensors on the handle's device) --------------------------
    def run_device(self, n_cases: int, ev_off, ev_node, ev_state, out, *, ev_val_off=None, ev_values=None,
                   epsilon: float = 0.0, max_sweeps: int = 20, damping: float = 0.0, check_interval: int = 1,
                   out_sweeps=None, out_converged=None, stream: int = 0, gather: bool = False,
                   query_nodes: Optional[Sequence[int]] = None, out_log_evidence=None, out_counts=None,
                   case_weights=None) -> None:
        """All tensor arguments are CUDA tensors (int64 / int32 / float64 offsets and values as in
        ``bnbp_evidence``); ``out`` has the handle's precision, shape [n_cases, sum r_X].
        Work is enqueued on ``stream`` (a raw cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream).
        ``out_log_evidence``: a float64 CUDA tensor [n_cases] that receives each case's Bethe log-evidence
        (``bnbp_run_batch_device_log_evidence``); ``out`` may then be None (no marginals).
        ``out_counts``: a float64 CUDA tensor [cpt_values] that the expected family counts are ADDED into, in stream
        order (``bnbp_run_batch_device_expected_counts``), with ``case_weights`` a float64 CUDA tensor [n_cases] (finite
        and >= 0, not checked) or None; ``out`` and ``out_log_evidence`` may then be None."""
        def dp(t):
            return None if t is None else int(t.data_ptr())
        evc = _capi.EvidenceC(int(n_cases), dp(ev_off), dp(ev_node), dp(ev_state), dp(ev_val_off), dp(ev_values))
        q = None if query_nodes is None else np.ascontiguousarray(query_nodes, dtype=np.int32)
        # gather: ``out`` is [world * n_cases, row] on every rank (comm_init first); this rank's rows are written in
        # place and exchanged over NCCL inside the call
        prm = _capi.RunParamsC(float(epsilon), int(max_sweeps), float(damping), int(check_interval), 0,
                               1 if gather else 0, 0 if q is None else int(q.size), _vp(q))
        st = C.c_void_p(stream) if stream else None
        if out_counts is not None or case_weights is not None:
            if out_counts is None:
                raise ValueError("case_weights belong to out_counts")
            for t, m in ((out_counts, int(self.net.cpt_off[-1])), (case_weights, int(n_cases)),
                         (out_log_evidence, int(n_cases))):
                if t is not None:
                    assert t.dtype.itemsize == 8 and t.is_floating_point() and t.is_cuda and t.numel() == m and t.is_contiguous()
            _capi.check(self._lib.bnbp_run_batch_device_expected_counts(self._h, C.byref(evc), C.byref(prm), dp(case_weights),
                                                                        dp(out_counts), dp(out), dp(out_sweeps),
                                                                        dp(out_converged), dp(out_log_evidence), st))
            return
        if out_log_evidence is not None:
            assert out_log_evidence.dtype.itemsize == 8 and out_log_evidence.is_floating_point() and out_log_evidence.is_cuda
            assert out_log_evidence.numel() == int(n_cases) and out_log_evidence.is_contiguous()
            _capi.check(self._lib.bnbp_run_batch_device_log_evidence(self._h, C.byref(evc), C.byref(prm), dp(out), dp(out_sweeps),
                                                                     dp(out_converged), dp(out_log_evidence), st))
            return
        _capi.check(self._lib.bnbp_run_batch_device(self._h, C.byref(evc), C.byref(prm), dp(out), dp(out_sweeps),
                                                    dp(out_converged), st))

    # ---- several processes, one GPU each: the communicator lives in the library (SURVEY 8e) --------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(_capi.COMM_ID_BYTES)
        _capi.check(_capi.load().bnbp_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, world: int, rank: int, unique_id: bytes) -> None:
        """Join the NCCL communicator rank 0 drew with ``comm_unique_id`` (ship the 128 bytes with the
        launcher's own means, e.g. a ``torch.distributed`` broadcast)."""
        assert len(unique_id) == _capi.COMM_ID_BYTES
        buf = C.create_string_buffer(unique_id, _capi.COMM_ID_BYTES)
        _capi.check(self._lib.bnbp_comm_init(self._h, int(world), int(rank), buf))

    def comm_summary(self, d_sweeps, d_converged, n_cases: int, stream: int = 0) -> dict:
        """All-reduce (in the library, NCCL) of the per-case counts the last ``run_device`` left in the two CUDA
        tensors: totals over every rank."""
        sm = _capi.SummaryC()
        _capi.check(self._lib.bnbp_comm_summary(self._h, int(d_sweeps.data_ptr()), int(d_converged.data_ptr()), int(n_cases),
                                                C.byref(sm), C.c_void_p(stream) if stream else None))
        return {k: int(getattr(sm, k)) for k, _ in sm._fields_}

    def summary(self) -> dict:
        """Group handle (``devices=...``): totals of the last call over all devices (``bnbp_get_summary``)."""
        sm = _capi.SummaryC()
        _capi.check(self._lib.bnbp_get_summary(self._h, C.byref(sm)))
        return {k: int(getattr(sm, k)) for k, _ in sm._fields_}

    def check_errors(self, stream: int = 0) -> None:
        """After synchronising with a ``run_device`` call: raise if it skipped malformed evidence
        (``bnbp_check_errors``; the asynchronous call itself cannot report it)."""
        _capi.check(self._lib.bnbp_check_errors(self._h, C.c_void_p(stream) if stream else None))

    # ---- likelihood weighting (SURVEY 8 f2) ------------------------------------------------------
    def likelihood_weighting(self, evidence: EvidenceBatch, n_samples: int = 10000, seed: int = 1,
                             return_weight: bool = False):
        """``likelihood_weighting::operator()(evidence_list, sample_num)`` (likelihood_weighting.hpp:28-59)
        for a batch of hard-evidence cases on the GPU (``bnbp_lw_run_batch``): marginals [n_cases, sum r_X]
        (and the total sample weight per case).  Reproducible: the variates are a function of ``seed``."""
        ev = evidence
        if ev.is_soft:
            raise ValueError("likelihood weighting takes hard evidence (vertex -> state)")
        n, V = ev.n_cases, self.net.belief_values
        out = np.empty((n, V), dtype=np.float64)
        wsum = np.empty(n, dtype=np.float64)
        evc = _capi.EvidenceC(n, _vp(ev.ev_off), _vp(ev.ev_node), _vp(ev.ev_state), None, None)
        _capi.check(self._lib.bnbp_lw_run_batch(self._h, C.byref(evc), int(n_samples), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                                _vp(out), _vp(wsum)))
        return (out, wsum) if return_weight else out

    def stats(self) -> dict:
        st = _capi.StatsC()
        _capi.check(self._lib.bnbp_get_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_ if k != "reserved"}

    def refresh_cpt(self, cpt: np.ndarray) -> None:
        cpt = np.ascontiguousarray(cpt, dtype=np.float64)
        _capi.check(self._lib.bnbp_refresh_cpt(self._h, _vp(cpt), cpt.size))

    # ---- EM parameter learning from incomplete evidence -----------------------------------------------
    def em(self, evidence: EvidenceBatch, *, iterations: int = 50, tol: float = 1e-6, pseudo_count: float = 0.0,
           epsilon: float = 1e-6, max_sweeps: int = 200, damping: float = 0.0,
           weights: Optional[np.ndarray] = None, cpt: Optional[np.ndarray] = None) -> EMResult:
        """Expectation-maximisation of the CPTs from the hard-evidence cases ``evidence`` (``weights`` [n_cases]: each
        case's multiplicity, default 1).  Each iteration: the E-step on the GPU (expected family counts and the Bethe
        log-evidence of every case, one ``expected_counts`` call), ``m_step`` on the host and ``refresh_cpt``.  Starts
        from ``cpt`` (default ``self.net.cpt``; ``self.net`` is never modified) and stops after ``iterations`` or once
        the log-likelihood gains no more than ``tol * |L|``.  ``log_likelihood[i]`` is sum_c w_c ln Z_B(e_c) over the
        cases counted in iteration i, under the CPT going into it (exact on polytrees run to convergence, the Bethe
        approximation on loopy networks).  The handle is left holding the returned CPT."""
        if iterations < 1:
            raise ValueError("iterations must be >= 1")
        n = evidence.n_cases
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        if w is not None and (w.shape != (n,) or not np.isfinite(w).all() or (w < 0).any()):
            raise ValueError("weights must be [n_cases], finite and >= 0")
        cur = np.array(self.net.cpt if cpt is None else cpt, dtype=np.float64)
        self.refresh_cpt(cur)            # the handle may hold another CPT from an earlier refresh_cpt
        counts = np.zeros(int(self.net.cpt_off[-1]), dtype=np.float64)
        lls, skipped = [], []
        for it in range(iterations):
            counts[:] = 0.0
            res = self(evidence, epsilon, max_sweeps=max_sweeps, damping=damping, marginals=False, log_evidence=True,
                       expected_counts=True, weights=w, counts_out=counts)
            ok = np.isfinite(res.log_evidence)
            le = res.log_evidence[ok]
            lls.append(float(le.sum() if w is None else (w[ok] * le).sum()))
            skipped.append(int((~ok).sum()))
            cur = m_step(self.net, counts, pseudo_count)
            self.refresh_cpt(cur)
            if it > 0 and lls[-1] - lls[-2] <= tol * abs(lls[-1]):
                break
        return EMResult(cur, np.array(lls), np.array(skipped, dtype=np.int64), len(lls))


# the name the north star uses (SURVEY.md section 0.1: the reference class is belief_propagation)
loopy_belief_propagation = BeliefPropagation


def device_count() -> int:
    return int(_capi.load().bnbp_device_count())
