"""Device embedding conditioning (sidekit_b200.conditioning, csrc/conditioning.cu) against the real reference's outputs
(tests/golden/conditioning.npz), against the host StatServer methods at scale, against float64 numpy over odd shapes,
plus determinism, interoperability with the host path and argument errors."""
import numpy
import pytest
import torch

import sidekit_b200 as sk
from sidekit_b200 import _lib, conditioning as cd
from tests.helpers import golden

gpu = pytest.mark.gpu


def _close(a, b, tol=1e-10):
    a, b = (x.cpu().numpy() if isinstance(x, torch.Tensor) else numpy.asarray(x) for x in (a, b))
    return numpy.abs(a - b).max() < tol * max(1.0, numpy.abs(b).max())


def _ss(X, ids):
    return sk.StatServer.from_embeddings(ids, numpy.asarray(X, dtype=numpy.float64))


@pytest.fixture(scope="module")
def ref():
    g = golden("plda_training.npz")
    return g["ids"], g["X"], golden("conditioning.npz")


@pytest.fixture(scope="module")
def big():
    """200 000 x 256 rows in ~2 000 classes of uneven size, singletons included."""
    rng = numpy.random.default_rng(11)
    n, D = 200000, 256
    sizes = numpy.concatenate([numpy.ones(300, int), rng.integers(2, 180, 1700)])
    sizes[-1] += n - sizes.sum()
    assert sizes[-1] > 0
    lab = rng.permutation(numpy.repeat(numpy.arange(sizes.shape[0]), sizes))
    centres = rng.standard_normal((sizes.shape[0], D)) * 0.7
    X = centres[lab] + rng.standard_normal((n, D)) @ (rng.standard_normal((D, D)) * 0.1) + 3.0
    ids = numpy.array(["spk%05d" % v for v in lab])
    return ids, X


# ---------------------------------------------------------------------------------------------------- 1. real reference
@gpu
def test_statistics_match_reference(ref):
    ids, X, g = ref
    st = cd.scatter(torch.from_numpy(X).cuda(), ids)
    assert _close(st.mean, g["mean"]) and _close(st.total, g["total_cov"])
    assert _close(st.within, g["within_cov"]) and _close(st.between, g["between_cov"])
    assert _close(cd.mahalanobis_matrix(st), g["mahalanobis"], 1e-8) and _close(cd.wccn_cholesky(st), g["wccn"], 1e-8)
    lda = cd.lda_matrix(st, 5)
    sign = numpy.sign((lda * g["lda"]).sum(axis=0))
    assert lda.shape == g["lda"].shape and _close(lda * sign, g["lda"], 1e-6)
    assert numpy.array_equal(st.models, g["sum_modelset"])
    assert _close(st.class_means * st.counts[:, None], g["sum_stat1"])
    assert numpy.array_equal(st.counts.cpu().numpy(), g["sum_sessions"])


@gpu
def test_whitening_and_spectral_norm_match_reference(ref):
    ids, X, g = ref
    Xd = torch.from_numpy(X).cuda()
    assert _close(cd.whiten(Xd, g["mean"], g["total_cov"]), g["whiten_full"], 1e-9)
    assert _close(cd.whiten(Xd, g["mean"], numpy.diag(g["total_cov"]).copy()), g["whiten_diag"])
    assert _close(cd.whiten_cholesky(Xd, g["mean"], g["total_cov"]), g["whiten_chol"], 1e-9)
    for mode in ("efr", "sphNorm"):
        means, covs = cd.estimate_spectral_norm(Xd, ids, 2, mode)
        assert _close(means[0], g["sn_%s_mean" % mode][0], 1e-9) and _close(covs[0], g["sn_%s_cov" % mode][0], 1e-9)
        assert _close(numpy.abs(means[1]), numpy.abs(g["sn_%s_mean" % mode][1]), 1e-8)
        assert _close(numpy.abs(covs[1]), numpy.abs(g["sn_%s_cov" % mode][1]), 1e-8)
        out = cd.spectral_norm(Xd, means, covs).cpu().numpy()
        r = g["sn_%s_out" % mode]
        sign = numpy.sign((out * r).sum(axis=0))
        assert _close(out * sign, r, 1e-8) and _close(out @ out.T, r @ r.T, 1e-8)
        assert numpy.allclose(numpy.linalg.norm(out, axis=1), 1.0)


# ---------------------------------------------------------------------------------------------------- 2. host path at scale
def _host_scatters(ss):
    models, means, Sw = ss._class_normalised_scatter()
    cm = means - ss.get_mean_stat1()
    return dict(mean=ss.get_mean_stat1(), total=ss.get_total_covariance_stat1(), within=ss.get_within_covariance_stat1(),
                between=ss.get_between_covariance_stat1(), class_normalised=Sw, Sb=cm.T @ cm, class_means=means)


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_scatter_and_whitening_match_host_at_scale(big, dtype):
    ids, X = big
    Xd = torch.from_numpy(X).to("cuda", dtype)
    ss = _ss(Xd.cpu().double().numpy(), ids)
    st = cd.scatter(Xd, ids)
    for k, v in _host_scatters(ss).items():
        assert _close(getattr(st, k), v), k
    mu, cov = ss.get_mean_stat1(), ss.get_total_covariance_stat1()
    w = _ss(ss.stat1, ids); w.whiten_stat1(mu, cov)
    assert _close(cd.whiten(Xd, mu, cov, out_dtype=torch.float64), w.stat1, 1e-9)
    w = _ss(ss.stat1, ids); w.whiten_stat1(mu, numpy.diag(cov).copy())
    assert _close(cd.whiten(Xd, mu, numpy.diag(cov).copy(), out_dtype=torch.float64), w.stat1, 1e-9)
    w = _ss(ss.stat1, ids); w.whiten_cholesky_stat1(mu, cov)
    assert _close(cd.whiten_cholesky(Xd, mu, cov, out_dtype=torch.float64), w.stat1, 1e-9)


@gpu
def test_centring_on_load_survives_a_large_mean():
    """Mean 1e4 x the spread: the raw-moment shortcut sum xx' - N mu mu' loses every digit here."""
    rng = numpy.random.default_rng(5)
    X = 1e4 + rng.standard_normal((100007, 24))
    ids = numpy.array(["c%d" % v for v in rng.integers(0, 300, X.shape[0])])
    st = cd.scatter(torch.from_numpy(X).cuda(), ids)
    ss = _ss(X, ids)
    for k, v in _host_scatters(ss).items():
        assert _close(getattr(st, k), v), k
    raw = (X.T @ X) / X.shape[0] - numpy.outer(X.mean(0), X.mean(0))
    assert not _close(raw, ss.get_total_covariance_stat1())


# ---------------------------------------------------------------------------------------------------- 3. shapes
SHAPES = [(n, d) for d in (1, 24, 200, 256, 600) for n in (1, 2, 63, 64, 65, 100007)]


@gpu
@pytest.mark.parametrize("n,d", SHAPES)
def test_gram_through_the_abi(n, d):
    rng = numpy.random.default_rng(n * 1000 + d)
    wide = torch.from_numpy(rng.standard_normal((n, d + 5)) + 2.0).cuda()
    X = wide[:, 3:3 + d]                                          # strided rows: a column slice of a wider tensor
    K = 7
    shift = rng.standard_normal((K, d))
    idx = rng.integers(0, K, n).astype(numpy.int32)
    w = rng.random(n) + 0.5
    s_d, i_d, w_d = (torch.from_numpy(a).cuda() for a in (shift, idx, w))
    G = torch.empty((d, d), dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().skb_gram_f64(X.data_ptr(), 1, n, d, X.stride(0), s_d.data_ptr(), i_d.data_ptr(), w_d.data_ptr(),
                                       0.5, G.data_ptr(), _lib.stream_ptr()))
    Xh = X.cpu().numpy() - shift[idx]
    assert _close(G, 0.5 * (Xh * w[:, None]).T @ Xh, 1e-12)
    X32 = X.float()
    G32 = cd.gram(X32, s_d[:1].contiguous())
    Xh = X32.cpu().double().numpy() - shift[0]
    assert _close(G32, Xh.T @ Xh, 1e-12)
    assert torch.equal(G32, G32.T)


@gpu
@pytest.mark.parametrize("n,d", SHAPES)
@pytest.mark.parametrize("d_out", [None, 1, 130, 300])
def test_affine_rows(n, d, d_out):
    rng = numpy.random.default_rng(n + d)
    X = torch.from_numpy(rng.standard_normal((n, d + 3)) + 1.0).cuda()[:, 1:1 + d]
    mu, dsc = rng.standard_normal(d), rng.random(d) + 0.5
    W = None if d_out is None else rng.standard_normal((d, d_out))
    Xh = X.cpu().numpy()
    for m, s in ((None, None), (mu, None), (mu, dsc), (None, dsc)):
        ref = Xh - (0.0 if m is None else m)
        ref = ref * (1.0 if s is None else s)
        ref = ref if W is None else ref @ W
        for norm in (False, True):
            want = ref / numpy.maximum(numpy.linalg.norm(ref, axis=1, keepdims=True), 1e-8) if norm else ref
            got = cd._affine(X, m, s, W, unit_norm=norm, out_dtype=torch.float64)
            assert _close(got, want, 1e-12), (m is None, s is None, norm)
    got32 = cd._affine(X, mu, dsc, W, unit_norm=True, out_dtype=torch.float32)
    assert got32.dtype == torch.float32 and _close(got32, cd._affine(X, mu, dsc, W, unit_norm=True, out_dtype=torch.float64), 1e-6)


# ---------------------------------------------------------------------------------------------------- 4. determinism
@gpu
def test_gram_is_bitwise_reproducible_and_symmetric(big):
    ids, X = big
    Xd = torch.from_numpy(X[:, :200]).float().cuda()
    a, b = cd.scatter(Xd, ids), cd.scatter(Xd, ids)
    for k in ("mean", "total", "within", "between", "class_normalised", "Sb"):
        G1, G2 = getattr(a, k), getattr(b, k)
        assert torch.equal(G1, G2), k
        if G1.dim() == 2:
            assert torch.equal(G1, G1.T), k


# ---------------------------------------------------------------------------------------------------- 5. interop
@gpu
@pytest.mark.parametrize("mode", ["efr", "sphNorm"])
def test_spectral_norm_interoperates_with_host(big, mode):
    ids, X = big
    X = X[:20000, :64]
    ids = ids[:20000]
    Xd = torch.from_numpy(X).cuda()
    means, covs = cd.estimate_spectral_norm(Xd, ids, 2, mode)
    assert all(isinstance(v, numpy.ndarray) for v in means + covs)
    dev = cd.spectral_norm(Xd, means, covs)
    host = _ss(X, ids); host.spectral_norm_stat1(means, covs)
    assert _close(dev, host.stat1, 1e-9)
    hm, hc = _ss(X, ids).estimate_spectral_norm_stat1(2, mode)
    host = _ss(X, ids); host.spectral_norm_stat1(hm, hc)
    assert _close(cd.spectral_norm(Xd, hm, hc), host.stat1, 1e-9)


# ---------------------------------------------------------------------------------------------------- 6. errors
def test_scatter_without_cuda_raises():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="CUDA"):
        cd.scatter(torch.zeros(8, 4))


@gpu
def test_errors():
    X = torch.randn(10, 4, device="cuda")
    with pytest.raises(RuntimeError, match="CUDA"):
        cd.scatter(X.cpu())
    with pytest.raises(ValueError):
        cd.scatter(X[0])
    with pytest.raises(ValueError):
        cd.scatter(torch.randn(3, 1025, device="cuda"))
    with pytest.raises(ValueError):
        cd.scatter(X, numpy.array(["a"] * 9))
    with pytest.raises(ValueError):
        cd.scatter(X, torch.tensor([0, 1, 2, 0, 1, 2, 0, 1, 2, -1], device="cuda"))
    with pytest.raises(ValueError):
        cd.scatter(X, torch.tensor([0, 1, 3, 0, 1, 3, 0, 1, 3, 0], device="cuda"))      # class 2 has no row
    lib, st = _lib.lib(), _lib.stream_ptr()
    G = torch.empty((4, 4), dtype=torch.float64, device="cuda")
    for rc in (lib.skb_gram_f64(None, 0, 10, 4, 4, None, None, None, 1.0, G.data_ptr(), st),
               lib.skb_gram_f64(X.data_ptr(), 0, 10, 4, 3, None, None, None, 1.0, G.data_ptr(), st),
               lib.skb_gram_f64(X.data_ptr(), 0, 10, 1025, 1025, None, None, None, 1.0, G.data_ptr(), st),
               lib.skb_gram_f64(X.data_ptr(), 0, 10, 4, 4, None, X.data_ptr(), None, 1.0, G.data_ptr(), st),
               lib.skb_class_stats(X.data_ptr(), 0, 10, 4, 4, None, None, 3, None, G.data_ptr(), None, st),
               lib.skb_class_stats(X.data_ptr(), 0, 0, 4, 4, None, None, 0, G.data_ptr(), None, None, st),
               lib.skb_affine_rows(X.data_ptr(), 0, 10, 4, 4, None, None, None, 5, 0, G.data_ptr(), 1, 5, st),
               lib.skb_affine_rows(X.data_ptr(), 0, 10, 4, 4, None, None, G.data_ptr(), 4, 0, None, 1, 4, st)):
        assert rc != 0 and lib.skb_last_error()
