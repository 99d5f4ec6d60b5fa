"""Embedding conditioning for embeddings held in GPU memory: the scatter matrices, LDA / WCCN / Mahalanobis, whitening
and EFR / SphNorm spectral normalisation that a SIDEKIT recipe applies before PLDA training and scoring
(statserver.py:789-1054, :1279-1333), without a round trip through numpy.

The statistics and the row transforms run in float64 on the device (``csrc/conditioning.cu``): ``skb_class_stats`` (column
mean, per-class sums and counts), ``skb_gram_f64`` (every scatter matrix as one weighted, shifted Gram matrix, centred
while it is loaded) and ``skb_affine_rows`` (centre, scale, rotate and optionally length-normalise every row in one pass).
The D x D algebra (eigendecompositions, inverses, Cholesky factors) stays on the host in float64 and is the same code the
``StatServer`` methods use.  Inputs are CUDA tensors (float32 or float64, rows may have a stride), typically what
``Xtractor.extract_*`` / ``bulk.extract_embeddings`` return; there is no CPU fallback.
"""
from dataclasses import dataclass
from typing import Optional

import numpy
import scipy.linalg
import torch

from . import _lib
from .statserver import _cholesky_whitener, _inverse_sqrt_factor, _lda_from_scatter, _wccn_from_scatter

MAX_DIM = 1024


@dataclass
class ScatterStats:
    """What ``scatter`` returns.  ``models`` (numpy, C) are the sorted unique model ids (or ``arange(C)`` for integer
    labels); ``counts`` (C), ``class_means`` (C, D), ``mean`` (D) and the (D, D) matrices are float64 CUDA tensors:
    ``total`` / ``within`` / ``between`` covariances (statserver.py:920-980), ``class_normalised`` = sum_c (1 / n_c)
    sum_{x in c} (x - m_c)(x - m_c)' (the Sw of the LDA and the WCCN accumulator) and ``Sb`` = sum_c (m_c - mu)(m_c - mu)'
    (the LDA's unweighted between-class scatter).  Without labels only ``mean`` and ``total`` are set."""
    n: int
    mean: torch.Tensor
    total: torch.Tensor
    models: Optional[numpy.ndarray] = None
    counts: Optional[torch.Tensor] = None
    class_means: Optional[torch.Tensor] = None
    within: Optional[torch.Tensor] = None
    between: Optional[torch.Tensor] = None
    class_normalised: Optional[torch.Tensor] = None
    Sb: Optional[torch.Tensor] = None


class _Classes:
    """Class index of every row plus the CSR lists (rows of each class in input order) the class kernels take."""

    def __init__(self, labels, n, device):
        if isinstance(labels, torch.Tensor):
            if labels.dtype.is_floating_point or labels.dtype == torch.bool or labels.dim() != 1:
                raise ValueError("integer class indices must be a 1-D integer tensor")
            if labels.shape[0] != n:
                raise ValueError("%d labels for %d rows" % (labels.shape[0], n))
            idx = labels.to(device=device, dtype=torch.int64)
            lo, hi = (int(v) for v in torch.stack([idx.min(), idx.max()]).tolist())
            if lo < 0:
                raise ValueError("class index %d out of range (class indices are 0 .. C-1)" % lo)
            self.models = numpy.arange(hi + 1)
        else:
            labels = numpy.asarray(labels)
            if labels.ndim != 1 or labels.shape[0] != n:
                raise ValueError("%s labels for %d rows" % (labels.shape, n))
            self.models, inv = numpy.unique(labels, return_inverse=True)      # the class order of the host path
            idx = torch.from_numpy(inv.reshape(-1).astype(numpy.int64)).to(device)
        n_cls = self.models.shape[0]
        sessions = torch.bincount(idx, minlength=n_cls)
        if not bool((sessions > 0).all()):
            raise ValueError("class indices out of range: every class 0 .. C-1 needs at least one row")
        self.n_cls = n_cls
        self.idx = idx.to(torch.int32)
        self.rows = torch.sort(idx, stable=True).indices.to(torch.int32)
        self.ptr = torch.zeros(n_cls + 1, dtype=torch.int32, device=device)
        self.ptr[1:] = torch.cumsum(sessions, 0)


def _check(X):
    if not isinstance(X, torch.Tensor):
        raise TypeError("expected a torch.Tensor, got %s" % type(X).__name__)
    if not X.is_cuda:
        raise RuntimeError("sidekit_b200.conditioning needs CUDA tensors (B200, sm_100a); there is no CPU fallback")
    if X.dim() != 2:
        raise ValueError("expected a 2-D (N, D) tensor, got %d dimensions" % X.dim())
    if X.dtype not in (torch.float32, torch.float64):
        raise ValueError("expected float32 or float64 rows, got %s" % X.dtype)
    if X.shape[0] < 1 or X.shape[1] < 1 or X.shape[1] > MAX_DIM:
        raise ValueError("shape %s: need N >= 1 and 1 <= D <= %d" % (tuple(X.shape), MAX_DIM))
    if X.stride(1) != 1 or X.stride(0) < X.shape[1]:
        X = X.contiguous()
    return X


def _f64(a, device):
    """A host array / tensor as a contiguous float64 tensor on ``device`` (None stays None)."""
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=torch.float64).contiguous()
    return torch.from_numpy(numpy.ascontiguousarray(a, dtype=numpy.float64)).to(device)


def _ptr(t):
    return None if t is None else t.data_ptr()


def gram(X, shift=None, shift_idx=None, w=None, scale=1.0):
    """``scale * sum_i w_i (x_i - shift[shift_idx[i]]) (x_i - shift[shift_idx[i]])'`` (D, D) float64 (``skb_gram_f64``)."""
    X = _check(X)
    D = X.shape[1]
    G = torch.empty((D, D), dtype=torch.float64, device=X.device)
    _lib.check(_lib.lib().skb_gram_f64(X.data_ptr(), int(X.dtype == torch.float64), X.shape[0], D, X.stride(0), _ptr(shift),
                                       _ptr(shift_idx), _ptr(w), float(scale), G.data_ptr(), _lib.stream_ptr()))
    return G


def _class_stats(X, classes=None):
    """(mean, class sums, class counts) in one launch sequence: two passes over X."""
    lib = _lib.lib()
    N, D = X.shape
    mean = torch.empty((D,), dtype=torch.float64, device=X.device)
    sums = counts = None
    if classes is not None:
        sums = torch.empty((classes.n_cls, D), dtype=torch.float64, device=X.device)
        counts = torch.empty((classes.n_cls,), dtype=torch.float64, device=X.device)
    _lib.check(lib.skb_class_stats(X.data_ptr(), int(X.dtype == torch.float64), N, D, X.stride(0),
                                   _ptr(classes.ptr if classes else None), _ptr(classes.rows if classes else None),
                                   classes.n_cls if classes else 0, mean.data_ptr(), _ptr(sums), _ptr(counts), _lib.stream_ptr()))
    return mean, sums, counts


def scatter(X, labels=None):
    """Mean and scatter matrices of the rows of ``X`` (N, D), a float32 / float64 CUDA tensor.  ``labels``: an array of
    model ids (as ``StatServer.modelset``; classes in ``numpy.unique`` order) or an integer CUDA tensor of class indices
    0 .. C-1.  Two passes over X for the mean and the class statistics, then one Gram launch per scatter matrix."""
    X = _check(X)
    N = X.shape[0]
    if labels is None:
        mean, _, _ = _class_stats(X)
        return ScatterStats(n=N, mean=mean, total=gram(X, mean, scale=1.0 / N))
    classes = _Classes(labels, N, X.device)
    mean, sums, counts = _class_stats(X, classes)
    class_means = sums / counts[:, None]
    row_w = (1.0 / counts)[classes.idx.long()]
    return ScatterStats(n=N, mean=mean, models=classes.models, counts=counts, class_means=class_means,
                        total=gram(X, mean, scale=1.0 / N),
                        within=gram(X, class_means, classes.idx, scale=1.0 / N),
                        class_normalised=gram(X, class_means, classes.idx, row_w),
                        between=gram(class_means, mean, w=counts, scale=1.0 / N),
                        Sb=gram(class_means, mean))


def _host(t):
    return t.cpu().numpy()


def lda_matrix(stats, rank):
    """``StatServer.get_lda_matrix_stat1(rank)`` from ``scatter(X, labels)``: (D, rank) numpy float64."""
    return _lda_from_scatter(_host(stats.Sb), _host(stats.class_normalised), rank)


def wccn_cholesky(stats):
    """``StatServer.get_wccn_choleski_stat1()`` from ``scatter(X, labels)``: (D, D) numpy float64."""
    return _wccn_from_scatter(_host(stats.class_normalised), stats.models.shape[0])


def mahalanobis_matrix(stats):
    """``StatServer.get_mahalanobis_matrix_stat1()`` from ``scatter(X, labels)``: (D, D) numpy float64."""
    return scipy.linalg.inv(_host(stats.within))


def _affine(X, mu=None, d=None, W=None, unit_norm=False, out_dtype=None):
    X = _check(X)
    N, D = X.shape
    dev = X.device
    mu, d, W = _f64(mu, dev), _f64(d, dev), _f64(W, dev)
    for name, v in (("mean", mu), ("scaling", d)):
        if v is not None and v.shape != (D,):
            raise ValueError("%s of shape %s for %d-dimensional rows" % (name, tuple(v.shape), D))
    if W is not None and (W.dim() != 2 or W.shape[0] != D):
        raise ValueError("matrix of shape %s for %d-dimensional rows" % (tuple(W.shape), D))
    D_out = D if W is None else W.shape[1]
    Y = torch.empty((N, D_out), dtype=out_dtype or X.dtype, device=dev)
    _lib.check(_lib.lib().skb_affine_rows(X.data_ptr(), int(X.dtype == torch.float64), N, D, X.stride(0), _ptr(mu), _ptr(d),
                                          _ptr(W), D_out, int(unit_norm), Y.data_ptr(), int(Y.dtype == torch.float64),
                                          Y.stride(0), _lib.stream_ptr()))
    return Y


def _out_dtype(X, out_dtype):
    if out_dtype not in (None, torch.float32, torch.float64):
        raise ValueError("out_dtype must be torch.float32 or torch.float64")
    return out_dtype or X.dtype


def _whitening(sigma, is_sqr_inv_sigma, factor):
    """(diagonal scaling, matrix) of statserver.py:852-918 for a 1-D or 2-D ``sigma``."""
    sigma = _host(sigma) if isinstance(sigma, torch.Tensor) else numpy.asarray(sigma, dtype=numpy.float64)
    if sigma.ndim == 1:
        return 1.0 / numpy.sqrt(sigma.astype(numpy.float64)), None
    if sigma.ndim == 2:
        return None, sigma if is_sqr_inv_sigma else factor(sigma)
    raise ValueError("Wrong dimension of Sigma, must be 1 or 2")


def whiten(X, mu, sigma, is_sqr_inv_sigma=False, out_dtype=None):
    """``StatServer.whiten_stat1`` on device rows: ``(X - mu) / sqrt(sigma)`` for a 1-D ``sigma``, ``(X - mu) V
    diag(lambda^-1/2)`` for a 2-D one (``sigma`` itself with ``is_sqr_inv_sigma``).  Returns a new tensor, dtype of X
    unless ``out_dtype`` is given."""
    X = _check(X)
    d, W = _whitening(sigma, is_sqr_inv_sigma, _inverse_sqrt_factor)
    return _affine(X, mu, d, W, out_dtype=_out_dtype(X, out_dtype))


def whiten_cholesky(X, mu, sigma, out_dtype=None):
    """``StatServer.whiten_cholesky_stat1`` on device rows (lower Cholesky factor of the precision)."""
    X = _check(X)
    d, W = _whitening(sigma, False, _cholesky_whitener)
    return _affine(X, mu, d, W, out_dtype=_out_dtype(X, out_dtype))


def estimate_spectral_norm(X, labels=None, it=1, mode="efr"):
    """``StatServer.estimate_spectral_norm_stat1(it, mode)`` on device rows: the (mean, covariance) of ``it`` rounds of
    "whiten, then length-normalise", each estimated on the output of the round before ('efr': total covariance,
    'sphNorm': within-class, needs ``labels``).  Returns ``(means, covs)``, lists of numpy float64 arrays, the types the
    host method returns.  The working copy stays on the device (float64) between rounds."""
    X = _check(X)
    if mode not in ("efr", "sphNorm"):
        raise ValueError("mode must be 'efr' or 'sphNorm'")
    classes = None
    if mode == "sphNorm":
        if labels is None:
            raise ValueError("mode 'sphNorm' needs the labels")
        classes = _Classes(labels, X.shape[0], X.device)
    N = X.shape[0]
    work, means, covs = X, [], []
    for _ in range(it):
        mean, sums, counts = _class_stats(work, classes)
        if mode == "efr":
            cov = gram(work, mean, scale=1.0 / N)
        else:
            cov = gram(work, sums / counts[:, None], classes.idx, scale=1.0 / N)
        means.append(_host(mean))
        covs.append(_host(cov))
        work = _affine(work, means[-1], None, _inverse_sqrt_factor(covs[-1]), unit_norm=True, out_dtype=torch.float64)
    return means, covs


def spectral_norm(X, means, covs, is_sqr_inv_sigma=False, out_dtype=None):
    """``StatServer.spectral_norm_stat1(means, covs)`` on device rows: per round, whiten then length-normalise (one pass
    over the rows each).  Intermediate rounds are float64; the result has the dtype of X unless ``out_dtype`` is given."""
    X = _check(X)
    if len(means) != len(covs):
        raise ValueError("Number of mean vectors and covariance matrices is different")
    out = _out_dtype(X, out_dtype)
    work = X
    for k, (mean, cov) in enumerate(zip(means, covs)):
        d, W = _whitening(cov, is_sqr_inv_sigma, _inverse_sqrt_factor)
        work = _affine(work, mean, d, W, unit_norm=True, out_dtype=out if k == len(means) - 1 else torch.float64)
    return work if len(means) else X.to(out, copy=True)
