"""Score normalisation: z-norm, t-norm, zt-norm (sidekit/score_normalization.py:44-117) and the adaptive symmetric
as-norm (:120-140).  Statistics and normalisation run on the device (csrc/evaltail.cu, csrc/scoring.cu)."""
import copy

import numpy
import torch

from . import _lib


def _dev_matrix(a):
    if not torch.cuda.is_available():
        raise RuntimeError("sidekit_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    a = numpy.ascontiguousarray(a)
    if a.dtype not in (numpy.float32, numpy.float64):
        a = a.astype(numpy.float64)
    return torch.from_numpy(a).cuda()


def _stats(mat, axis, sym=False):
    """(mean, std) device doubles along ``axis`` of a device matrix."""
    M, N = mat.shape
    n = M if axis == 1 else N
    mean = torch.empty((n,), dtype=torch.float64, device=mat.device)
    std = torch.empty((n,), dtype=torch.float64, device=mat.device)
    _lib.check(_lib.lib().skb_scoremat_stats(mat.data_ptr(), M, N, mat.stride(0), int(mat.dtype == torch.float64), axis, int(sym),
                                             mean.data_ptr(), std.data_ptr(), _lib.stream_ptr()))
    return mean, std


def _normalise(mat, sub, div):
    """(mat - sub) / div with the (N,) vectors broadcast against the last axis, like numpy."""
    M, N = mat.shape
    if sub.shape[0] != N:
        raise ValueError("operands could not be broadcast together with shapes (%d,%d) (%d,)" % (M, N, sub.shape[0]))
    out = torch.empty_like(mat)
    _lib.check(_lib.lib().skb_scoremat_normalise(mat.data_ptr(), M, N, mat.stride(0), int(mat.dtype == torch.float64), sub.data_ptr(),
                                                 div.data_ptr(), out.data_ptr(), out.stride(0), _lib.stream_ptr()))
    return out


def znorm(enrol_test_scores, enrol_imp_scores, sym=False):
    """score_normalization.py:44-74.  Like the reference: sorts ``enrol_imp_scores`` in place, returns a sorted deep copy
    of ``enrol_test_scores``, divides by the VARIANCE when ``sym`` (:66), and subtracts the per-model statistics with
    numpy's last-axis broadcasting (:70), i.e. it needs as many test segments as models."""
    scores_znorm = copy.deepcopy(enrol_test_scores)
    scores_znorm.sort()
    enrol_imp_scores.sort()
    mean, std = _stats(_dev_matrix(enrol_imp_scores.scoremat), 1, sym)
    scores_znorm.scoremat = _normalise(_dev_matrix(scores_znorm.scoremat), mean, std).cpu().numpy()
    return scores_znorm


def tnorm(enrol_test_scores, imp_test_scores):
    """score_normalization.py:77-95."""
    scores_tnorm = copy.deepcopy(enrol_test_scores)
    scores_tnorm.sort()
    imp_test_scores.sort()
    mean, std = _stats(_dev_matrix(imp_test_scores.scoremat), 0)
    scores_tnorm.scoremat = _normalise(_dev_matrix(scores_tnorm.scoremat), mean, std).cpu().numpy()
    return scores_tnorm


def ztnorm(enrol_test_scores, enrol_imp_scores, imp_test_scores, imp_imp_scores):
    """score_normalization.py:98-117: z-norm of both score sets, then t-norm."""
    z_enrol_test_scores = znorm(enrol_test_scores, enrol_imp_scores)
    z_imp_test_scores = znorm(imp_test_scores, imp_imp_scores, sym=True)
    return tnorm(z_enrol_test_scores, z_imp_test_scores)


def asnorm(enrol_xv, cohort_xv, ndx=None, topk=200, return_device=False):
    """Same contract as the reference: ``enrol_xv`` (N, D) unit-norm embeddings, ``cohort_xv`` (C, D) raw cohort
    vectors (normalised here, :124), ``ndx`` unused; returns the (N, N) float32 normalised score matrix as numpy."""
    if not torch.cuda.is_available():
        raise RuntimeError("sidekit_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = enrol_xv.device if enrol_xv.is_cuda else torch.device("cuda", torch.cuda.current_device())
    X = enrol_xv.to(dev, torch.float32).contiguous()
    coh = torch.nn.functional.normalize(cohort_xv.to(dev, torch.float32), dim=1).contiguous()
    N, D = X.shape
    C = coh.shape[0]
    mean = torch.empty((N,), dtype=torch.float32, device=dev)
    std = torch.empty((N,), dtype=torch.float32, device=dev)
    out = torch.empty((N, N), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        l = _lib.lib()
        _lib.check(l.skb_asnorm_stats(X.data_ptr(), coh.data_ptr(), N, C, D, int(topk), mean.data_ptr(), std.data_ptr(),
                                      _lib.stream_ptr()))
        _lib.check(l.skb_asnorm_apply(X.data_ptr(), N, D, mean.data_ptr(), std.data_ptr(), out.data_ptr(), _lib.stream_ptr()))
    if return_device:
        return out
    from .bosaris import _device_to_numpy
    return _device_to_numpy(out)                     # pinned, PCIe-speed path for large matrices


def _ids_and_rows(side, ids_attr):
    """``(ids, embeddings)`` of an ``asnorm_trials`` operand: a StatServer (``ids_attr``, ``stat1``) or an ``(ids, X)`` pair."""
    from .statserver import StatServer
    if isinstance(side, StatServer):
        return getattr(side, ids_attr), side.stat1
    ids, X = side
    return ids, X


def _rows_on_device(X, ref, dev):
    """Rows ``ref`` (sorted) of ``X`` (numpy or torch, any device) as a contiguous float32 tensor on ``dev``; the whole
    matrix as it is when every row is referenced."""
    if ref.shape[0] != X.shape[0]:
        X = X[ref] if not torch.is_tensor(X) else X[torch.from_numpy(ref).to(X.device)]
    return torch.as_tensor(X).to(dev, torch.float32).contiguous()


def asnorm_trials(enroll, test, trials, cohort_xv, topk=200):
    """Symmetric adaptive s-norm of the cosine scores of the trials of a ``TrialList``: per trial (e, t),
    ``0.5 (s - mu_e) / sigma_e + 0.5 (s - mu_t) / sigma_t`` with ``s = e . t``, the entry of ``asnorm``'s N x N matrix
    without the matrix (VoxCeleb1-E / -H: 145 000 utterances, 84 GB as a float32 matrix).  ``asnorm``'s conventions: rows
    are taken as given (unit-norm embeddings expected, no normalisation here), the cohort is L2-normalised, mu / sigma are
    the mean and unbiased std of a row's ``topk`` best cohort scores, which needs ``topk <= C <= 51 200`` cohort rows.

    ``enroll`` / ``test``: StatServers (ids ``enroll.modelset`` / ``test.segset``, rows ``stat1``) or ``(ids, X)`` pairs
    with X an (N, D) numpy array or torch tensor.  The statistics are computed for the rows the kept trials reference, once
    when both sides are the same object or share their embeddings.  Trials with unknown ids are dropped.  Returns
    ``TrialScores`` with float32 scores."""
    from . import bulk
    from .bosaris import TrialScores
    from .iv_scoring import _device, _referenced, _score_pairs
    ids_e, Xe = _ids_and_rows(enroll, "modelset")
    ids_t, Xt = _ids_and_rows(test, "segset")
    rows, cols, keep = trials.index(ids_e, ids_t)
    shared = enroll is test or Xe is Xt
    dev = Xe.device if torch.is_tensor(Xe) and Xe.is_cuda else _device()
    ref_e, ref_t, r, c = _referenced(rows, cols, shared)
    E = _rows_on_device(Xe, ref_e, dev)
    T = E if shared else _rows_on_device(Xt, ref_t, dev)
    coh = torch.nn.functional.normalize(torch.as_tensor(cohort_xv).to(dev, torch.float32), dim=1).contiguous()
    mean_e, std_e = bulk._asnorm_stats_cuda(E, coh, topk)
    mean_t, std_t = (mean_e, std_e) if shared else bulk._asnorm_stats_cuda(T, coh, topk)
    return TrialScores(trials.subset(keep), _score_pairs(E, T, r, c, asnorm_stats=(mean_e, std_e, mean_t, std_t)))
