"""Trial scoring with the reference's signatures and return objects (sidekit/iv_scoring.py:52-113 cosine,
:159-212 two-covariance, :215-269 PLDA dispatcher, :370-477 fast PLDA).

Host side (numpy, like the reference): id matching -- an O(N) hash join instead of the reference's O(N^2)
``item in ndarray`` scans, with identical ordering semantics (rows follow ``ndx.modelset`` restricted to the
enrolled ids, first occurrence wins, every occurrence in the ndx kept) -- and the D x D PLDA algebra.  Device
side (CUDA, csrc/scoring.cu): centring, the Psi / Phi folds, the quadratic row / column terms and the
Ne x Nt score matrix.  The result stays on the device until ``Scores.scoremat`` is read.
"""
import collections
import copy
import ctypes
import logging

import numpy
import torch

from . import _lib
from .bosaris import Ndx, Scores, TrialScores
from .statserver import StatServer


def _check_missing_model(enroll, test, ndx):
    """iv_scoring.py:52-60."""
    clean_ndx = ndx.filter(enroll.modelset, test.segset, True)
    enroll.align_models(clean_ndx.modelset)
    test.align_segments(clean_ndx.segset)
    return clean_ndx


def _device(device=None):
    if not torch.cuda.is_available():
        raise RuntimeError("sidekit_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


def _dev32(a, device):
    return torch.as_tensor(numpy.ascontiguousarray(a, dtype=numpy.float32)).to(device, non_blocking=True)


def _operands(name, E, T, vectors=()):
    """The checks every score GEMM wrapper makes before a library call, which reads its operands through bare pointers:
    ``E`` (Ne, D) and ``T`` (Nt, D) 2-D float32 tensors on one CUDA device (``T`` may be a ``PackedEmbeddings`` of width
    D there), and every ``(vector, length)`` of ``vectors`` None or float32 of shape (length,) on that device.  Raises
    ``ValueError``; returns ``E``, ``T`` and the vectors made contiguous."""
    packed = isinstance(T, PackedEmbeddings)
    for X in (E,) if packed else (E, T):
        if not torch.is_tensor(X) or X.dim() != 2 or X.dtype != torch.float32 or X.device.type != "cuda":
            raise ValueError("%s: E and T must be 2-D float32 CUDA tensors" % name)
    dev = E.device
    if T.device != dev:
        raise ValueError("%s: E is on %s, T on %s" % (name, dev, T.device))
    D_t = T.D if packed else T.shape[1]
    if E.shape[1] != D_t:
        raise ValueError("%s: E and T must be (Ne, D) and (Nt, D), got D = %d and %d" % (name, E.shape[1], D_t))
    for t, n in vectors:
        if t is not None and (not torch.is_tensor(t) or t.dtype != torch.float32 or t.device != dev or tuple(t.shape) != (n,)):
            raise ValueError("%s: per-row vectors must be float32 on %s, one value per row" % (name, dev))
    return (E.contiguous(), T if packed else T.contiguous()) + tuple(None if t is None else t.contiguous() for t, _ in vectors)


def _rows(T):
    return T.rows if isinstance(T, PackedEmbeddings) else T.shape[0]


def score_matrix(E, T, rowterm=None, colterm=None, cst=0.0, alpha=1.0, passes=0, out_dtype=torch.float32, out=None):
    """S = alpha*(rowterm_i + colterm_j + cst) + alpha * E T^T on the device (all arguments torch CUDA fp32; ``T`` may be a
    ``PackedEmbeddings``).  ``out_dtype`` float32, float64 or float16 (half the HBM-bound write; 11-bit mantissa); ``out``
    an (Ne, Nt) tensor of one of those types with unit column stride (a view into a wider matrix is fine).

    ``passes``: 3 multiplies split fp16 operands (hi*hi + hi*lo + lo*hi) for float32-class accuracy; 1 multiplies fp16
    operands once; 0 picks 1 when an error estimate for operands whose fp16 rounding errors are uncorrelated stays below
    2.5e-4 (on S, alpha included), else 3.  Operands whose rounding errors add coherently (e.g. rows of one repeated value) can exceed
    that with 1 pass; ``passes=3`` is the bound for them."""
    E, T, rowterm, colterm = _operands("score_matrix", E, T, [(rowterm, E.shape[0]), (colterm, _rows(T))])
    Ne, D = E.shape
    Nt = _rows(T)
    if out is None:
        if out_dtype not in _OUT_DTYPE:
            raise ValueError("score_matrix: out_dtype must be float32, float64 or float16")
        out = torch.empty((Ne, Nt), dtype=out_dtype, device=E.device)
    elif (not torch.is_tensor(out) or out.dtype not in _OUT_DTYPE or out.device != E.device or tuple(out.shape) != (Ne, Nt) or
          out.stride(1) != 1):
        raise ValueError("score_matrix: out must be an (Ne, Nt) = (%d, %d) float32 / float64 / float16 tensor on %s with unit "
                         "column stride" % (Ne, Nt, E.device))
    if isinstance(T, PackedEmbeddings):
        with torch.cuda.device(E.device):
            _lib.check(_lib.lib().skb_score_gemm_packed(
                E.data_ptr(), Ne, T._ptr, None if rowterm is None else rowterm.data_ptr(),
                None if colterm is None else colterm.data_ptr(), float(cst), float(alpha), int(passes),
                _OUT_DTYPE[out.dtype], out.data_ptr(), out.stride(0), _lib.stream_ptr()))
        return out
    with torch.cuda.device(E.device):
        _lib.check(_lib.lib().skb_score_gemm(
            E.data_ptr(), T.data_ptr(), Ne, Nt, D, None if rowterm is None else rowterm.data_ptr(),
            None if colterm is None else colterm.data_ptr(), float(cst), float(alpha), int(passes),
            _OUT_DTYPE[out.dtype], out.data_ptr(), out.stride(0), _lib.stream_ptr()))
    return out


class PackedEmbeddings:
    """A test-side operand prepared once for ``score_matrix`` (``skb_packed_create``): scaled, split into fp16 hi / lo
    planes and tiled for the tcgen05 GEMM.  Scoring many enrol panels against it (row-panel sharding over GPUs, repeated
    calls) then pays only for the enrol side."""

    def __init__(self, T):
        T = T.to(torch.float32).contiguous()
        self.rows, self.D, self.device = int(T.shape[0]), int(T.shape[1]), T.device
        self._ptr = ctypes.c_void_p()
        with torch.cuda.device(T.device):
            _lib.check(_lib.lib().skb_packed_create(T.data_ptr(), self.rows, self.D, ctypes.byref(self._ptr), _lib.stream_ptr()))
            torch.cuda.current_stream().synchronize()          # T may be freed by the caller after this returns

    def __del__(self):
        try:
            if self._ptr:
                _lib.lib().skb_packed_destroy(self._ptr)
                self._ptr = None
        except Exception:
            pass


_OUT_DTYPE = {torch.float32: 0, torch.float64: 1, torch.float16: 2}


class TrialIndex:
    """Bit words + prefix counts of an (Ne, Nt) trial mask on the device (``skb_trial_index_create``), for
    ``score_trials``.  ``n_trials`` = number of selected trials; their order is numpy's ``mask.nonzero()`` order."""

    def __init__(self, mask, device=None):
        dev = _device(device)
        m = torch.as_tensor(numpy.ascontiguousarray(mask, dtype=numpy.uint8) if not torch.is_tensor(mask) else mask)
        m = m.to(dev, torch.uint8).contiguous()
        self.Ne, self.Nt, self.device = int(m.shape[0]), int(m.shape[1]), dev
        self._ptr = ctypes.c_void_p()
        n = ctypes.c_int64(0)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().skb_trial_index_create(m.data_ptr(), self.Ne, self.Nt, m.stride(0), ctypes.byref(self._ptr),
                                                         ctypes.byref(n), _lib.stream_ptr()))
        self.n_trials = int(n.value)

    def __del__(self):
        try:
            if self._ptr:
                _lib.lib().skb_trial_index_destroy(self._ptr)
                self._ptr = None
        except Exception:
            pass


def score_trials(E, T, trials, rowterm=None, colterm=None, cst=0.0, alpha=1.0, passes=0):
    """The scores of the trials of a mask only, as a 1-D float32 CUDA tensor in row-major mask order -- what the reference
    selects with ``scoremat[trialmask]`` (xvector.py:243-245) -- without the Ne x Nt matrix ever reaching HBM.
    ``trials``: a ``TrialIndex`` or an (Ne, Nt) bool mask; ``T`` may be a ``PackedEmbeddings``."""
    E, T, rowterm, colterm = _operands("score_trials", E, T, [(rowterm, E.shape[0]), (colterm, _rows(T))])
    if not isinstance(trials, TrialIndex):
        trials = TrialIndex(trials, E.device)
    Ne, D = E.shape
    out = torch.empty((max(trials.n_trials, 1),), dtype=torch.float32, device=E.device)
    if isinstance(T, PackedEmbeddings):
        with torch.cuda.device(E.device):
            _lib.check(_lib.lib().skb_score_gemm_trials_packed(
                E.data_ptr(), Ne, T._ptr, None if rowterm is None else rowterm.data_ptr(),
                None if colterm is None else colterm.data_ptr(), float(cst), float(alpha), int(passes), trials._ptr, out.data_ptr(),
                _lib.stream_ptr()))
        return out[:trials.n_trials]
    with torch.cuda.device(E.device):
        _lib.check(_lib.lib().skb_score_gemm_trials(
            E.data_ptr(), T.data_ptr(), Ne, T.shape[0], D, None if rowterm is None else rowterm.data_ptr(),
            None if colterm is None else colterm.data_ptr(), float(cst), float(alpha), int(passes), trials._ptr, out.data_ptr(),
            _lib.stream_ptr()))
    return out[:trials.n_trials]


def score_pairs(E, T, rows, cols, rowterm=None, colterm=None, cst=0.0, alpha=1.0):
    """The scores of the trials ``(rows[p], cols[p])`` as a 1-D float32 CUDA tensor: entry p is
    ``alpha * (rowterm[i] + colterm[j] + cst) + alpha * E[i] . T[j]`` with ``i = rows[p]``, ``j = cols[p]`` -- the
    ``score_matrix`` entry (i, j) -- at O(trials) cost, for lists too large for an (Ne, Nt) mask (VoxCeleb1-E / -H).
    ``E`` (Ne, D), ``T`` (Nt, D), ``rowterm`` (Ne,), ``colterm`` (Nt,): CUDA float32; ``rows`` / ``cols``: integer arrays
    (numpy or torch).  The dot products are float32 FMAs over the float32 rows in a fixed order, so a trial's score has the
    same bits wherever it sits in whichever list.  An index out of range gives NaN."""
    return _score_pairs(E, T, rows, cols, rowterm, colterm, cst, alpha)


def _score_pairs(E, T, rows, cols, rowterm=None, colterm=None, cst=0.0, alpha=1.0, asnorm_stats=None):
    """``score_pairs``; ``asnorm_stats = (mean_e, std_e, mean_t, std_t)`` (float32 CUDA, indexed like ``E`` / ``T``)
    normalises every score with the symmetric as-norm formula in the same kernel."""
    if not torch.is_tensor(E) or not torch.is_tensor(T) or E.dim() != 2 or T.dim() != 2:
        raise ValueError("score_pairs: E and T must be (Ne, D) and (Nt, D)")
    vectors = [(rowterm, E.shape[0]), (colterm, T.shape[0])]
    if asnorm_stats is not None:
        vectors += [(asnorm_stats[0], E.shape[0]), (asnorm_stats[1], E.shape[0]), (asnorm_stats[2], T.shape[0]), (asnorm_stats[3], T.shape[0])]
    E, T, rowterm, colterm, *stats = _operands("score_pairs", E, T, vectors)
    dev = E.device
    rows = torch.as_tensor(rows).to(dev, torch.int32).contiguous()
    cols = torch.as_tensor(cols).to(dev, torch.int32).contiguous()
    if rows.dim() != 1 or rows.shape != cols.shape:
        raise ValueError("score_pairs: rows and cols must be 1-D arrays of one length")
    ptr = lambda t: None if t is None else t.data_ptr()
    me, se, mt, st = stats if asnorm_stats is not None else (None,) * 4
    out = torch.empty((rows.shape[0],), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().skb_score_pairs(E.data_ptr(), T.data_ptr(), E.shape[0], T.shape[0], E.shape[1], rows.data_ptr(),
                                              cols.data_ptr(), rows.shape[0], ptr(rowterm), ptr(colterm), float(cst), float(alpha),
                                              ptr(me), ptr(se), ptr(mt), ptr(st), out.data_ptr(), _lib.stream_ptr()))
    return out


def _referenced(rows, cols, shared):
    """The rows a trial list references and the trials' positions among them: ``(ref_e, ref_t, r, c)`` with ``ref_e`` /
    ``ref_t`` sorted row numbers and ``r`` / ``c`` int32 indices into them.  ``shared``: enrolment and test rows index one
    matrix, so one set serves both sides (one upload, one preparation)."""
    if shared:
        ref, inv = numpy.unique(numpy.concatenate([rows, cols]), return_inverse=True)
        inv = inv.astype(numpy.int32)
        return ref, ref, inv[:rows.shape[0]], inv[rows.shape[0]:]
    ref_e, r = numpy.unique(rows, return_inverse=True)
    ref_t, c = numpy.unique(cols, return_inverse=True)
    return ref_e, ref_t, r.astype(numpy.int32), c.astype(numpy.int32)


def _trial_rows(server, ref):
    """A StatServer holding rows ``ref`` of ``server.stat1`` only (for the StatServer methods, which rebind ``stat1``)."""
    out = StatServer()
    out.stat1 = server.stat1[ref]
    return out


def cosine_scoring_trials(enroll, test, trials, wccn=None):
    """Cosine similarities of the trials of a ``TrialList`` -- ``cosine_scoring`` at O(trials) cost.  Trials whose ids are
    not in ``enroll.modelset`` / ``test.segset`` are dropped (the first occurrence of an id wins, as in
    ``cosine_scoring``).  Rows are WCCN-rotated and length-normalised like ``cosine_scoring``; when ``enroll`` and
    ``test`` share their embeddings (one StatServer for both, the VoxCeleb1-E / -H case) they are prepared once.
    Returns ``TrialScores`` with float32 scores; the caller's objects are not modified."""
    assert isinstance(enroll, StatServer), 'First parameter should be a StatServer'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    rows, cols, keep = trials.index(enroll.modelset, test.segset)
    shared = enroll.stat1 is test.stat1
    ref_e, ref_t, r, c = _referenced(rows, cols, shared)
    dev = _device()
    sides = []
    for server, ref in ((enroll, ref_e), (test, ref_t))[:1 if shared else 2]:
        part = _trial_rows(server, ref)
        if wccn is not None:
            part.rotate_stat1(wccn)
        part.norm_stat1()
        sides.append(_dev32(part.stat1, dev))
    E, T = sides[0], sides[-1]
    return TrialScores(trials.subset(keep), _score_pairs(E, T, r, c))


def PLDA_scoring_trials(enroll, test, trials, mu, F, Sigma, scaling_factor=1.):
    """Simplified PLDA log-likelihood ratios of the trials of a ``TrialList`` -- ``fast_PLDA_scoring`` at O(trials) cost:
    duplicate enrolment ids are averaged first (``mean_stat_per_model``), trials with unknown ids are dropped, and the
    row / column terms come from the same device preparation (``_quadratic_prepare``).  Returns ``TrialScores`` with
    float64 scores like the PLDA scorers (float32-class precision); the caller's objects are not modified."""
    assert isinstance(enroll, StatServer), 'First parameter should be a StatServer'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    assert enroll.stat1.shape[1] == test.stat1.shape[1], 'I-vectors dimension mismatch'
    enroll_ctr = _unique_models(enroll)
    rows, cols, keep = trials.index(enroll_ctr.modelset, test.segset)
    kept = trials.subset(keep)
    dev = _device()
    if not keep.any():
        return TrialScores(kept, torch.empty((0,), dtype=torch.float32, device=dev), numpy.float64)
    shared = enroll_ctr.stat1 is test.stat1
    ref_e, ref_t, r, c = _referenced(rows, cols, shared)
    Phi, Psi, plda_cst = _simplified_plda_terms(F, Sigma, scaling_factor)
    E = _dev32(enroll_ctr.stat1[ref_e], dev)
    T = E if shared else _dev32(test.stat1[ref_t], dev)
    Ep, model_part = _quadratic_prepare(E, mu, Psi, Phi)
    Tc, seg_part = _quadratic_prepare(T, mu, None, Phi)
    return TrialScores(kept, _score_pairs(Ep, Tc, r, c, model_part, seg_part, cst=plda_cst, alpha=scaling_factor), numpy.float64)


TOPK_MAX = 1024


def score_topk(E, T, k, rowterm=None, colterm=None, cst=0.0, alpha=1.0, passes=0):
    """The ``k`` largest entries of every row of ``score_matrix(E, T, rowterm, colterm, cst, alpha, passes)`` as CUDA tensors
    ``(values (Ne, k) float32, indices (Ne, k) int64)``, ordered by score descending and, among equal scores, by lower column
    -- each value equals its ``score_matrix`` entry bit for bit.  ``T`` may be a ``PackedEmbeddings`` (a gallery packed once
    and searched by many query batches).  For ``k <= 32`` and ``D <= 256`` the selection runs inside the GEMM epilogue and
    the (Ne, Nt) matrix never reaches memory; otherwise row panels of it pass through a bounded scratch.  The order of NaN
    scores is undefined."""
    E, T, rowterm, colterm = _operands("score_topk", E, T, [(rowterm, E.shape[0]), (colterm, _rows(T))])
    Ne, D = E.shape
    Nt = _rows(T)
    k = int(k)
    if not 1 <= k <= min(Nt, TOPK_MAX):
        raise ValueError("score_topk: need 1 <= k <= min(Nt, %d), got k = %d with Nt = %d" % (TOPK_MAX, k, Nt))
    values = torch.empty((Ne, k), dtype=torch.float32, device=E.device)
    indices = torch.empty((Ne, k), dtype=torch.int64, device=E.device)
    r = None if rowterm is None else rowterm.data_ptr()
    q = None if colterm is None else colterm.data_ptr()
    with torch.cuda.device(E.device):
        if isinstance(T, PackedEmbeddings):
            _lib.check(_lib.lib().skb_score_gemm_topk_packed(E.data_ptr(), Ne, T._ptr, r, q, float(cst), float(alpha), int(passes), k,
                                                             values.data_ptr(), indices.data_ptr(), _lib.stream_ptr()))
        else:
            _lib.check(_lib.lib().skb_score_gemm_topk(E.data_ptr(), T.data_ptr(), Ne, Nt, D, r, q, float(cst), float(alpha), int(passes),
                                                      k, values.data_ptr(), indices.data_ptr(), _lib.stream_ptr()))
    return values, indices


def _quadratic_prepare(X, mu, Psi, Phi):
    """xc = X - mu; returns (xc . Psi, 0.5 * diag(xc Phi xc^T)) on the device."""
    N, D = X.shape
    Xout = torch.empty_like(X)
    rowterm = torch.empty((N,), dtype=torch.float32, device=X.device)
    psi_t = None if Psi is None else _dev32(numpy.asarray(Psi).T, X.device)
    phi = _dev32(Phi, X.device)
    mu_d = None if mu is None else _dev32(mu, X.device)
    with torch.cuda.device(X.device):
        _lib.check(_lib.lib().skb_quadratic_prepare(X.data_ptr(), None if mu_d is None else mu_d.data_ptr(),
                                                    None if psi_t is None else psi_t.data_ptr(), phi.data_ptr(), N, D,
                                                    Xout.data_ptr(), rowterm.data_ptr(), _lib.stream_ptr()))
    return Xout, rowterm


def _finish(clean_ndx, mat_dev, np_dtype=None):
    """``Scores`` whose matrix stays on the device until ``scoremat`` is read.  ``np_dtype=float64``: the reference's PLDA /
    two-covariance / Mahalanobis scorers return float64; the GEMM writes float32 (its accuracy class: fp32 accumulation
    of split fp16 products, <= 1e-3 absolute against the reference as north_star asks, typically 4e-5) and the widening
    happens on the way to the host, so the HBM-bound kernel does not write 8 bytes per trial."""
    score = Scores()
    score.modelset = clean_ndx.modelset
    score.segset = clean_ndx.segset
    score.scoremask = clean_ndx.trialmask
    score.scoremat_device = mat_dev
    score.scoremat_dtype = np_dtype
    score.scoremat = None           # materialised lazily from the device tensor
    return score


def cosine_scoring(enroll, test, ndx, wccn=None, check_missing=True, device=None):
    """Cosine similarities for the trials of ``ndx`` (iv_scoring.py:63-113); ``scoremat`` is float32."""
    assert isinstance(enroll, StatServer), 'First parameter should be a StatServer'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    assert isinstance(ndx, Ndx), 'Third parameter should be an Ndx'
    enroll_copy = copy.copy(enroll)            # shallow: every StatServer method used below REBINDS its arrays, none writes in place,
    test_copy = copy.copy(test)                # so the caller's objects are untouched without two (N, D) float64 copies
    clean_ndx = _check_missing_model(enroll_copy, test_copy, ndx) if check_missing else ndx
    if wccn is not None:
        enroll_copy.rotate_stat1(wccn)
        test_copy.rotate_stat1(wccn)
    enroll_copy.norm_stat1()
    test_copy.norm_stat1()
    dev = _device(device)
    E, T = _dev32(enroll_copy.stat1, dev), _dev32(test_copy.stat1, dev)
    # the reference multiplies fp32 operands (torch.einsum on FloatTensors): split mode keeps fp32-class accuracy
    return _finish(clean_ndx, score_matrix(E, T, passes=3))


def fast_PLDA_scoring(enroll, test, ndx, mu, F, Sigma, test_uncertainty=None, Vtrans=None, p_known=0.0,
                      scaling_factor=1., check_missing=True):
    """Simplified PLDA log-likelihood ratios (iv_scoring.py:370-477); ``scoremat`` is float64 like the reference
    (fp32-class precision, see ``_finish``)."""
    enroll_ctr = copy.copy(enroll)             # shallow: every StatServer method used below REBINDS its arrays, none writes in place,
    test_ctr = copy.copy(test)                 # so the caller's objects are untouched without two (N, D) float64 copies
    if not numpy.unique(enroll_ctr.modelset).shape == enroll_ctr.modelset.shape:
        logging.warning("Enrollment models are not unique, average i-vectors")
        enroll_ctr = enroll_ctr.mean_stat_per_model()
    clean_ndx = _check_missing_model(enroll_ctr, test_ctr, ndx) if check_missing else ndx
    if not numpy.unique(enroll_ctr.modelset).shape == enroll_ctr.modelset.shape:
        # the reference averages a second time after alignment (:422-425); see oracle/scoring_ref.py
        logging.warning("Enrollment models are not unique, average i-vectors")
        enroll_ctr = enroll_ctr.mean_stat_per_model()

    Phi, Psi, plda_cst = _simplified_plda_terms(F, Sigma, scaling_factor)

    dev = _device()
    E, T = _dev32(enroll_ctr.stat1, dev), _dev32(test_ctr.stat1, dev)
    Ep, model_part = _quadratic_prepare(E, mu, Psi, Phi)           # (E - mu) Psi ; 0.5 diag((E-mu) Phi (E-mu)^T)
    Tc, seg_part = _quadratic_prepare(T, mu, None, Phi)
    S = score_matrix(Ep, Tc, model_part, seg_part, cst=plda_cst, alpha=scaling_factor, passes=0)
    if p_known != 0:
        S = _open_set(S.double(), p_known)
    return _finish(clean_ndx, S, numpy.float64)


def _simplified_plda_terms(F, Sigma, scaling_factor):
    """The three model-dependent quantities of the two-covariance log-likelihood ratio (what the reference derives at
    iv_scoring.py:429-448), D x D float64 algebra on the host.  With the between-class covariance ``B = F F'``, the total
    covariance ``T = B + Sigma`` and the Schur complement ``M = T - B T^-1 B`` of the stacked (enrol, test) covariance:

        llr(e, t) = e' Psi t + (e' Phi e + t' Phi t) / 2 + cst,   Psi = T^-1 B M^-1,   Phi = T^-1 - M^-1,
        cst = log det(I + K) - log det(I + 2 K) / 2,              K = s F' Sigma^-1 F.

    ``numpy.linalg`` throughout: the matrix products run on numpy's BLAS threads, and alternating between numpy's and
    scipy's thread pools inside one function cost 0.25-0.4 s per call on a many-core host (tools/api_probe.py)."""
    F = numpy.asarray(F, dtype=numpy.float64)
    Sigma = numpy.asarray(Sigma, dtype=numpy.float64)
    rank = F.shape[1]
    cst = 0.0
    if rank:
        K = scaling_factor * (F.T @ numpy.linalg.solve(Sigma, F))
        eye = numpy.eye(rank)
        cst = numpy.linalg.slogdet(eye + K)[1] - 0.5 * numpy.linalg.slogdet(eye + 2.0 * K)[1]
    between = F @ F.T
    total = between + Sigma
    total_inv = numpy.linalg.inv(total)
    ti_b = total_inv @ between
    schur_inv = numpy.linalg.inv(total - between @ ti_b)
    return total_inv - schur_inv, ti_b @ schur_inv, cst


def _open_set(S, p_known):
    """Open-set correction (iv_scoring.py:356-366, :467-475), vectorised: sum_{k != i} exp(S_kj) = colsum_j - exp(S_ij)."""
    N = S.shape[0]
    tmp = torch.exp(S)
    return S - torch.log(p_known * (tmp.sum(dim=0, keepdim=True) - tmp) / (N - 1) + (1 - p_known))


def _full_plda_terms(F, G, Sigma, scaling_factor):
    """``(Psi, Phi, cst)`` of the PLDA model with a channel subspace (the quantities of iv_scoring.py:296-313), D x D float64
    algebra on the host.  ``P = s Sigma^-1`` is the residual precision; marginalising the channel factor turns it into
    ``Pc = P - P G (I + G' P G)^-1 G' P`` (Woodbury), the speaker factor then sees ``B = F' Pc`` and ``K = B F``, and

        llr(e, t) = e' Psi t + (e' Phi e + t' Phi t) / 2 + cst,   Psi = B' (I + 2K)^-1 B,   Phi = Psi - B' (I + K)^-1 B,
        cst = log det(I + K) - log det(I + 2 K) / 2."""
    F = numpy.asarray(F, dtype=numpy.float64)
    G = numpy.asarray(G, dtype=numpy.float64)
    P = scaling_factor * numpy.linalg.inv(numpy.asarray(Sigma, dtype=numpy.float64))
    PG = P @ G
    Pc = P - PG @ numpy.linalg.solve(numpy.eye(G.shape[1]) + G.T @ PG, PG.T) if G.shape[1] else P
    B = F.T @ Pc
    K = B @ F
    eye = numpy.eye(F.shape[1])
    inv1, inv2 = numpy.linalg.inv(eye + K), numpy.linalg.inv(eye + 2.0 * K)
    cst = numpy.linalg.slogdet(eye + K)[1] - 0.5 * numpy.linalg.slogdet(eye + 2.0 * K)[1]
    Psi = B.T @ inv2 @ B
    return Psi, Psi - B.T @ inv1 @ B, cst


def full_PLDA_scoring(enroll, test, ndx, mu, F, G, Sigma, p_known=0.0, scaling_factor=1., check_missing=True):
    """PLDA with a channel subspace ``G`` (iv_scoring.py:272-368); ``scoremat`` is float64 like the reference.

    The reference projects the i-vectors with ``B`` (speaker space after channel compensation) and loops over the
    models; expanding ``(e+t)' K2 (e+t)/2 - t' K1 t/2 - e' K1 e/2`` gives ``e' K2 t + e'(K2-K1)e/2 + t'(K2-K1)t/2``,
    i.e. the same row-term / column-term / GEMM form as the simplified scorer with ``Psi = B' K2 B`` and
    ``Phi = B' (K2 - K1) B`` (D x D algebra on the host in float64, the trial matrix on the device).  Note that --
    unlike ``fast_PLDA_scoring`` -- duplicate enrolment models are NOT averaged (the reference has that block
    commented out, :290-294)."""
    enroll_copy = copy.copy(enroll)            # shallow: every StatServer method used below REBINDS its arrays, none writes in place,
    test_copy = copy.copy(test)                # so the caller's objects are untouched without two (N, D) float64 copies
    clean_ndx = _check_missing_model(enroll_copy, test_copy, ndx) if check_missing else ndx
    Psi, Phi, constant = _full_plda_terms(F, G, Sigma, scaling_factor)
    Phi = 0.5 * (Phi + Phi.T)                      # symmetric up to rounding; the device routine assumes it
    dev = _device()
    E, T = _dev32(enroll_copy.stat1, dev), _dev32(test_copy.stat1, dev)
    Ep, model_part = _quadratic_prepare(E, mu, Psi, Phi)
    Tc, seg_part = _quadratic_prepare(T, mu, None, Phi)
    S = score_matrix(Ep, Tc, model_part, seg_part, cst=constant, alpha=scaling_factor, passes=0)
    if p_known != 0:
        S = _open_set(S.double(), p_known)
    return _finish(clean_ndx, S, numpy.float64)


def PLDA_scoring(enroll, test, ndx, mu, F, G, Sigma, test_uncertainty=None, Vtrans=None, p_known=0.0,
                 scaling_factor=1., full_model=False):
    """PLDA dispatcher (iv_scoring.py:215-269)."""
    assert isinstance(enroll, StatServer), 'First parameter should be a StatServer'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    assert isinstance(ndx, Ndx), 'Third parameter should be an Ndx'
    assert enroll.stat1.shape[1] == test.stat1.shape[1], 'I-vectors dimension mismatch'
    assert enroll.stat1.shape[1] == F.shape[0], 'I-vectors and co-variance matrix dimension mismatch'
    assert enroll.stat1.shape[1] == G.shape[0], 'I-vectors and co-variance matrix dimension mismatch'
    if not full_model:
        return fast_PLDA_scoring(enroll, test, ndx, mu, F, Sigma, test_uncertainty, Vtrans, p_known=p_known,
                                 scaling_factor=scaling_factor, check_missing=True)
    return full_PLDA_scoring(enroll, test, ndx, mu, F, G, Sigma, p_known=p_known, scaling_factor=scaling_factor)


def mahalanobis_scoring(enroll, test, ndx, m, check_missing=True):
    """``-0.5 (e_i - t_j)' m (e_i - t_j)`` (iv_scoring.py:116-156), float64 like the reference.

    Like the reference it aligns (reorders / shrinks) the caller's ``enroll`` / ``test`` in place.  Expanded for the score GEMM: ``0.5 e'(m + m')t - 0.5 e'me - 0.5 t'mt``."""
    assert isinstance(enroll, StatServer), 'First parameter should be a StatServer'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    assert isinstance(ndx, Ndx), 'Third parameter should be an Ndx'
    assert enroll.stat1.shape[1] == test.stat1.shape[1], 'I-vectors dimension mismatch'
    assert enroll.stat1.shape[1] == m.shape[0], 'I-vectors and Mahalanobis matrix dimension mismatch'
    if not numpy.unique(enroll.modelset).shape == enroll.modelset.shape:
        logging.warning("Enrollment models are not unique, average i-vectors")
        enroll = enroll.mean_stat_per_model()
    clean_ndx = _check_missing_model(enroll, test, ndx) if check_missing else ndx
    m = numpy.asarray(m, dtype=numpy.float64)
    dev = _device()
    E, T = _dev32(enroll.stat1, dev), _dev32(test.stat1, dev)
    Ep, model_part = _quadratic_prepare(E, None, 0.5 * (m + m.T), -m)          # rowterm = 0.5 * e'(-m)e
    Tc, seg_part = _quadratic_prepare(T, None, None, -m)
    # split mode always: e'me + t'mt - 2 e'mt cancels when e is close to t, so the cross term needs fp32-class products
    S = score_matrix(Ep, Tc, model_part, seg_part, passes=3)
    return _finish(clean_ndx, S, numpy.float64)


def two_covariance_scoring(enroll, test, ndx, W, B, check_missing=True):
    """Two-covariance scores (iv_scoring.py:159-212).  Like the reference it works on the caller's objects:
    ``enroll`` / ``test`` are aligned (reordered / shrunk) in place."""
    assert isinstance(enroll, StatServer), 'First parameter should be a directory'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    assert isinstance(ndx, Ndx), 'Third parameter should be an Ndx'
    assert enroll.stat1.shape[1] == test.stat1.shape[1], 'I-vectors dimension mismatch'
    assert enroll.stat1.shape[1] == W.shape[0], 'I-vectors and co-variance matrix dimension mismatch'
    assert enroll.stat1.shape[1] == B.shape[0], 'I-vectors and co-variance matrix dimension mismatch'
    if not numpy.unique(enroll.modelset).shape == enroll.modelset.shape:
        logging.warning("Enrollment models are not unique, average i-vectors")
        enroll = enroll.mean_stat_per_model()
    clean_ndx = _check_missing_model(enroll, test, ndx) if check_missing else ndx
    # W^-1 (B^-1 + c W^-1)^-1 W^-1 = (W B^-1 W + c W)^-1: one solve and two inverses (numpy.linalg, see _simplified_plda_terms)
    W = numpy.asarray(W, dtype=numpy.float64)
    WBW = W @ numpy.linalg.solve(numpy.asarray(B, dtype=numpy.float64), W)
    G = numpy.linalg.inv(WBW + 2.0 * W)
    H = numpy.linalg.inv(WBW + W)
    # (e+t)' G (e+t) - t' H t - e' H e  =  e'(G-H)e + t'(G-H)t + 2 e' G t
    dev = _device()
    E, T = _dev32(enroll.stat1, dev), _dev32(test.stat1, dev)
    Ep, model_part = _quadratic_prepare(E, None, 2.0 * G, 2.0 * (G - H))
    Tc, seg_part = _quadratic_prepare(T, None, None, 2.0 * (G - H))
    S = score_matrix(Ep, Tc, model_part, seg_part, passes=0)
    return _finish(clean_ndx, S, numpy.float64)


TopK = collections.namedtuple("TopK", ["segset", "models", "scores"])
TopK.__doc__ = """Best enrolled models per test segment: ``models[i]`` / ``scores[i]`` (both (Nt, k)) are the k best model ids of
``segset[i]`` and their scores, best first (equal scores: the model listed first in the enrolment wins)."""


def _unique_models(enroll):
    """One row per model id: duplicate ids averaged with ``mean_stat_per_model``, as ``fast_PLDA_scoring`` does (a model
    must appear once in a ranking).  The caller's object is not modified."""
    if numpy.unique(enroll.modelset).shape == enroll.modelset.shape:
        return copy.copy(enroll)
    logging.warning("Enrollment models are not unique, average i-vectors")
    return enroll.mean_stat_per_model()


def _check_k(k, n_models):
    k = int(k)
    if not 1 <= k <= min(n_models, TOPK_MAX):
        raise ValueError("need 1 <= k <= min(number of models, %d), got k = %d with %d models" % (TOPK_MAX, k, n_models))
    return k


def cosine_topk(enroll, test, k, wccn=None, device=None):
    """For every test segment (in ``test.segset`` order) the ``k`` enrolled models of highest cosine score -- speaker
    identification / embedding search over the scores ``cosine_scoring`` computes, without the (models x segments) matrix.
    The reference has no such function.  Duplicate model ids are averaged first (``mean_stat_per_model``, before the WCCN
    rotation and length normalisation), so each model appears once.  Returns ``TopK(segset, models, scores)`` with float32
    scores; the caller's objects are not modified."""
    assert isinstance(enroll, StatServer), 'First parameter should be a StatServer'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    enroll_copy = _unique_models(enroll)
    test_copy = copy.copy(test)                # shallow: the StatServer methods below rebind their arrays
    k = _check_k(k, enroll_copy.modelset.shape[0])
    if wccn is not None:
        enroll_copy.rotate_stat1(wccn)
        test_copy.rotate_stat1(wccn)
    enroll_copy.norm_stat1()
    test_copy.norm_stat1()
    dev = _device(device)
    Q, M = _dev32(test_copy.stat1, dev), _dev32(enroll_copy.stat1, dev)
    # queries are the GEMM rows, models the columns; split mode like cosine_scoring
    values, indices = score_topk(Q, M, k, passes=3)
    return TopK(numpy.asarray(test.segset).copy(), enroll_copy.modelset[indices.cpu().numpy()], values.cpu().numpy())


def PLDA_topk(enroll, test, k, mu, F, Sigma, scaling_factor=1.):
    """For every test segment (in ``test.segset`` order) the ``k`` enrolled models of highest simplified-PLDA log-likelihood
    ratio (the scores of ``fast_PLDA_scoring``), without the (models x segments) matrix.  The reference has no such function.
    Duplicate model ids are averaged first (``mean_stat_per_model``, as ``fast_PLDA_scoring`` does).  The LLR is symmetric in
    (enrol, test), so Psi is folded into the query side.  Returns ``TopK(segset, models, scores)`` with float64 scores like
    the PLDA scorers (fp32-class precision); the caller's objects are not modified."""
    assert isinstance(enroll, StatServer), 'First parameter should be a StatServer'
    assert isinstance(test, StatServer), 'Second parameter should be a StatServer'
    assert enroll.stat1.shape[1] == test.stat1.shape[1], 'I-vectors dimension mismatch'
    enroll_ctr = _unique_models(enroll)
    k = _check_k(k, enroll_ctr.modelset.shape[0])
    Phi, Psi, plda_cst = _simplified_plda_terms(F, Sigma, scaling_factor)
    dev = _device()
    Q, M = _dev32(test.stat1, dev), _dev32(enroll_ctr.stat1, dev)
    Qp, seg_part = _quadratic_prepare(Q, mu, Psi.T, Phi)         # (t - mu) Psi' ; e' Psi t = t' Psi' e
    Mc, model_part = _quadratic_prepare(M, mu, None, Phi)
    values, indices = score_topk(Qp, Mc, k, seg_part, model_part, cst=plda_cst, alpha=scaling_factor, passes=0)
    return TopK(numpy.asarray(test.segset).copy(), enroll_ctr.modelset[indices.cpu().numpy()], values.double().cpu().numpy())
