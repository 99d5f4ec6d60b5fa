"""``skb_kernel_launches()`` counts every kernel the library launches: over each call below, its delta equals the number of
the library's kernels (namespace ``skb::``) that ``torch.profiler`` records on the device.  Copies and memsets are not
kernels; torch kernels run by the Python wrappers around a call are not the library's and are left out."""
import json
import os

import numpy
import pytest
import torch

import sidekit_b200 as sk
from sidekit_b200 import _lib, conditioning, synth
from sidekit_b200.iv_scoring import TrialIndex, score_trials
from sidekit_b200.nnet import functional as Fn
from sidekit_b200.nnet.preprocessor import Resample
from tests.models import make_xtractor

pytestmark = pytest.mark.gpu


def _counts(tmp_path, fn):
    """(skb_kernel_launches delta, names of the skb:: kernels the profiler saw) over fn()."""
    lib = _lib.lib()
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        n0 = lib.skb_kernel_launches()
        fn()
        torch.cuda.synchronize()
        n1 = lib.skb_kernel_launches()
    path = os.path.join(str(tmp_path), "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    kernels = [e["name"] for e in events if e.get("cat") == "kernel" and "skb::" in e.get("name", "")]
    return n1 - n0, kernels


def _check(tmp_path, fn):
    counted, kernels = _counts(tmp_path, fn)
    assert kernels, "no library kernel recorded"
    assert counted == len(kernels), (counted, len(kernels), sorted(set(kernels)))


def _rows(n, D, seed, unit=True):
    return torch.from_numpy(synth.synth_embeddings(n, D, seed=seed, unit_norm=unit)).float().cuda()


@pytest.mark.parametrize("archi", ["halfresnet34", "xvector", "fastresnet34"])
def test_extraction_on_a_new_geometry(tmp_path, archi):
    with torch.no_grad():
        m = make_xtractor(archi, 32, 256).cuda()
        m.extract_varlen([synth.synth_wave(1, L, seed=s)[0].cuda() for L, s in ((16000, 1), (9000, 2))])
        ws = [synth.synth_wave(1, L, seed=s)[0].cuda() for L, s in ((21000, 3), (12345, 4), (30001, 5))]     # a batch never seen
        _check(tmp_path, lambda: m.extract_varlen(ws))


@pytest.mark.parametrize("D", [256, 512])
def test_score_matrix(tmp_path, D):
    E, T = _rows(700, D, 1, False), _rows(900, D, 2, False)
    _check(tmp_path, lambda: sk.score_matrix(E, T))


def test_score_trials_and_top_k(tmp_path):
    E, T = _rows(600, 256, 3), _rows(800, 256, 4)
    mask = numpy.random.default_rng(0).random((600, 800)) < 0.05
    _check(tmp_path, lambda: score_trials(E, T, TrialIndex(mask)))
    _check(tmp_path, lambda: sk.score_topk(E, T, 10))                  # selected in the GEMM epilogue
    _check(tmp_path, lambda: sk.score_topk(E, T, 100))                 # row panels through the scratch


def test_pairs_asnorm_stats_and_quadratic_prepare(tmp_path):
    l, st = _lib.lib(), _lib.stream_ptr()
    N, C, D = 500, 300, 128
    E, T, X, coh = _rows(N, D, 5), _rows(400, D, 6), _rows(N, D, 7, False), _rows(C, D, 8)
    rng = numpy.random.default_rng(1)
    rows, cols = rng.integers(0, N, 3000), rng.integers(0, 400, 3000)
    _check(tmp_path, lambda: sk.score_pairs(E, T, rows, cols))
    mean, std = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
    _check(tmp_path, lambda: _lib.check(l.skb_asnorm_stats(X.data_ptr(), coh.data_ptr(), N, C, D, 50, mean.data_ptr(), std.data_ptr(), st)))
    mu = torch.randn(D, device="cuda")
    A = torch.randn(D, D, device="cuda")
    Phi, PsiT = (A + A.T) / D, torch.randn(D, D, device="cuda") / D
    Xout, rowterm = torch.empty(N, D, device="cuda"), torch.empty(N, device="cuda")
    _check(tmp_path, lambda: _lib.check(l.skb_quadratic_prepare(X.data_ptr(), mu.data_ptr(), PsiT.data_ptr(), Phi.data_ptr(), N, D,
                                                                Xout.data_ptr(), rowterm.data_ptr(), st)))


def test_plda_em_two_iterations(tmp_path):
    l, st = _lib.lib(), _lib.stream_ptr()
    rng = numpy.random.default_rng(2)
    D, R, n_cls = 40, 10, 30
    sessions = rng.integers(2, 6, n_cls)
    cls = numpy.repeat(numpy.arange(n_cls), sessions)
    X = torch.from_numpy(rng.standard_normal((cls.size, D)) + 3 * rng.standard_normal((n_cls, D))[cls]).cuda()
    ptr = torch.from_numpy(numpy.concatenate([[0], numpy.cumsum(sessions)]).astype(numpy.int32)).cuda()
    order = torch.arange(cls.size, dtype=torch.int32, device="cuda")
    mean, sigma_obs = torch.empty(D, dtype=torch.float64, device="cuda"), torch.empty(D, D, dtype=torch.float64, device="cuda")
    S1 = torch.empty(n_cls, D, dtype=torch.float64, device="cuda")
    _lib.check(l.skb_plda_stats(X.data_ptr(), cls.size, D, ptr.data_ptr(), order.data_ptr(), n_cls, 1.0, mean.data_ptr(),
                                sigma_obs.data_ptr(), S1.data_ptr(), st))
    F = torch.linalg.eigh(sigma_obs)[1][:, -R:].flip(1).contiguous()
    stat0 = sessions.astype(numpy.float64)
    uniq_n, n_index = numpy.unique(stat0, return_inverse=True)
    counts = numpy.bincount(n_index).astype(numpy.float64)
    n_d, u_d = torch.from_numpy(stat0).cuda(), torch.from_numpy(n_index.astype(numpy.int32)).cuda()
    uq_d, cnt_d = torch.from_numpy(uniq_n).cuda(), torch.from_numpy(counts).cuda()
    Sigma = sigma_obs.clone()
    torch.cuda.synchronize()
    _check(tmp_path, lambda: _lib.check(l.skb_plda_em(S1.data_ptr(), n_d.data_ptr(), u_d.data_ptr(), n_cls, uq_d.data_ptr(),
                                                      cnt_d.data_ptr(), int(uniq_n.size), mean.data_ptr(), sigma_obs.data_ptr(), D, R, 2,
                                                      float(stat0.sum()), F.data_ptr(), Sigma.data_ptr(), st)))


def test_gram_scoremat_stats_and_resample(tmp_path):
    l, st = _lib.lib(), _lib.stream_ptr()
    X = _rows(3000, 96, 9, False)
    _check(tmp_path, lambda: conditioning.gram(X))
    S = torch.randn(300, 300, device="cuda")
    mean, std = torch.empty(300, dtype=torch.float64, device="cuda"), torch.empty(300, dtype=torch.float64, device="cuda")
    for axis, sym in ((1, 1), (0, 0)):
        _check(tmp_path, lambda: _lib.check(l.skb_scoremat_stats(S.data_ptr(), 300, 300, 300, 0, axis, sym, mean.data_ptr(),
                                                                 std.data_ptr(), st)))
    lengths = [44100, 1000, 30000]
    waves = torch.cat([synth.synth_wave(1, L, seed=k)[0] for k, L in enumerate(lengths)]).cuda()
    r = Resample(44100, 16000)
    _check(tmp_path, lambda: r.resample_packed(waves, lengths))


def test_conv2d_bn_act(tmp_path):
    g = torch.Generator().manual_seed(0)
    x = torch.randn(3, 32, 13, 80, generator=g).cuda()
    w = (torch.randn(64, 32, 3, 3, generator=g) / 17).numpy()
    b = (torch.randn(64, generator=g) * 0.1).numpy()
    res, sc = torch.randn(3, 64, 7, 40, generator=g).cuda(), torch.rand(3, 64, generator=g).cuda()
    _check(tmp_path, lambda: Fn.conv2d_bn_act(x, w, b, 2, 0.01, se_scale=sc, residual=res))
