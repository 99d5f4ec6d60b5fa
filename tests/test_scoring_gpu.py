"""GPU parity of the scoring path (through the C ABI) against the oracle, the KAT and the golden fixtures.
Scores within 1e-3 absolute; modelset / segset / scoremask bit-exact (BASELINE.json north_star)."""
import copy

import numpy
import pytest
import torch

import sidekit_b200 as sk
from oracle import scoring_ref as S
from sidekit_b200 import synth
from tests import kat
from tests.helpers import golden

pytestmark = pytest.mark.gpu


def _ss(ids, X):
    return sk.StatServer.from_embeddings(numpy.asarray(ids), X)


def _ndx(models, segs, mask):
    n = sk.Ndx()
    n.modelset, n.segset, n.trialmask = numpy.asarray(models), numpy.asarray(segs), numpy.asarray(mask)
    return n


def _check(score, ref, tol, dtype):
    assert numpy.array_equal(score.modelset, ref[0]) and numpy.array_equal(score.segset, ref[1])
    assert numpy.array_equal(score.scoremask, ref[2])
    assert score.scoremat.dtype == dtype
    assert score.scoremat.shape == ref[3].shape
    assert numpy.abs(score.scoremat - ref[3]).max() < tol


def test_kat_vectors():
    k = kat.kat_inputs()
    mk = lambda: (_ss(k["en_ids"], k["en"]), _ss(k["te_ids"], k["te"]), _ndx(k["ndx_models"], k["ndx_segs"], k["trialmask"]))
    B = k["F"] @ k["F"].T + 0.1 * numpy.eye(8)
    res = {
        "plda": sk.PLDA_scoring(*mk(), k["mu"], k["F"], numpy.zeros((8, 0)), k["Sigma"]),
        "plda_sf05": sk.PLDA_scoring(*mk(), k["mu"], k["F"], numpy.zeros((8, 0)), k["Sigma"], scaling_factor=0.5),
        "twocov": sk.two_covariance_scoring(*mk(), k["Sigma"], B),
        "cosine": sk.cosine_scoring(*mk()),
    }
    for name, sc in res.items():
        exp = kat.KAT[name]
        assert sc.modelset.tolist() == kat.KAT_MODELSET and sc.segset.tolist() == kat.KAT_SEGSET
        assert sc.scoremask.sum() == kat.KAT_MASK_SUM and sc.scoremask[0].tolist() == kat.KAT_MASK_ROW0
        assert str(sc.scoremat.dtype) == exp["dtype"] and sc.validate()
        assert numpy.abs(sc.scoremat[0] - numpy.array(exp["row0"])).max() < 1e-4, name
        assert abs(float(sc.scoremat.sum()) - exp["total"]) < 1e-3, name


def test_mahalanobis_scoring_kat_and_random():
    # iv_scoring.py:116-156, float64
    k = kat.kat_inputs()
    M = numpy.linalg.inv(k["Sigma"]) + 0.05 * numpy.triu(k["F"] @ k["F"].T)
    a = (k["en_ids"], k["en"], k["te_ids"], k["te"], k["ndx_models"], k["ndx_segs"], k["trialmask"])
    sc = sk.mahalanobis_scoring(_ss(k["en_ids"], k["en"]), _ss(k["te_ids"], k["te"]), _ndx(k["ndx_models"], k["ndx_segs"], k["trialmask"]), M)
    ref = S.mahalanobis_scoring(*a, M)
    assert sc.modelset.tolist() == kat.KAT_MODELSET and sc.segset.tolist() == kat.KAT_SEGSET
    assert numpy.array_equal(sc.scoremask, ref[2]) and sc.scoremat.dtype == numpy.float64 and sc.scoremat.shape == (4, 3)
    assert numpy.abs(sc.scoremat - ref[3]).max() < 1e-3
    assert numpy.abs(sc.scoremat[0] - numpy.array(kat.KAT_MAHALANOBIS_ROW0)).max() < 1e-3
    rng = numpy.random.default_rng(31)
    D, Ne, Nt = 256, 333, 517
    E, T = synth.synth_embeddings(Ne, D, seed=41), synth.synth_embeddings(Nt, D, seed=42)
    A = rng.standard_normal((D, D)) * 0.05
    M = A @ A.T + numpy.eye(D) + 0.01 * rng.standard_normal((D, D))
    ids_e = numpy.array(["m%04d" % i for i in range(Ne)])
    ids_t = numpy.array(["s%04d" % i for i in range(Nt)])
    mask = rng.random((Ne, Nt)) < 0.5
    sc = sk.mahalanobis_scoring(_ss(ids_e, E), _ss(ids_t, T), _ndx(ids_e, ids_t, mask), M)
    _check(sc, S.mahalanobis_scoring(ids_e, E, ids_t, T, ids_e, ids_t, mask, M), 1e-3, numpy.float64)


def test_mahalanobis_near_identical_vectors_do_not_cancel():
    """The expanded form -0.5 e'me - 0.5 t'mt + e'mt cancels when e is close to t (ADVICE r1): with the split-precision
    cross term and fp32 row / column terms the scores of near-identical pairs (true value ~ -1e-4) stay inside the 1e-3 gate."""
    rng = numpy.random.default_rng(77)
    D, N = 256, 300
    E = synth.synth_embeddings(N, D, seed=43, unit_norm=False)
    T = E + 1e-3 * rng.standard_normal((N, D))
    A = rng.standard_normal((D, D)) * 0.05
    M = A @ A.T + numpy.eye(D)
    ids_e = numpy.array(["m%04d" % i for i in range(N)])
    ids_t = numpy.array(["s%04d" % i for i in range(N)])
    mask = numpy.ones((N, N), dtype=bool)
    sc = sk.mahalanobis_scoring(_ss(ids_e, E), _ss(ids_t, T), _ndx(ids_e, ids_t, mask), M)
    ref = S.mahalanobis_scoring(ids_e, E, ids_t, T, ids_e, ids_t, mask, M)[3]
    assert numpy.abs(numpy.diag(ref)).max() < 1e-3                   # the near-identical pairs: tiny true scores
    assert numpy.abs(numpy.diag(sc.scoremat) - numpy.diag(ref)).max() < 1e-3
    assert numpy.abs(sc.scoremat - ref).max() < 1e-3 * max(1.0, numpy.abs(ref).max() / 100.0)


def test_two_covariance_mutates_callers_objects_like_the_reference():
    k = kat.kat_inputs()
    en, te = _ss(k["en_ids"], k["en"]), _ss(k["te_ids"], k["te"])
    sk.two_covariance_scoring(en, te, _ndx(k["ndx_models"], k["ndx_segs"], k["trialmask"]), k["Sigma"],
                              k["F"] @ k["F"].T + 0.1 * numpy.eye(8))
    assert en.modelset.tolist() == kat.KAT_MODELSET
    en2 = _ss(k["en_ids"], k["en"])
    sk.cosine_scoring(en2, te, _ndx(k["ndx_models"], k["ndx_segs"], k["trialmask"]))
    assert en2.modelset.tolist() == k["en_ids"].tolist()          # cosine / PLDA deep-copy


@pytest.mark.parametrize("name", ["cosine", "plda", "plda_sf", "plda_open", "twocov", "plda_dup"])
def test_golden_scoring(name):
    g = golden("scoring.npz")
    en = _ss(g["en_ids_dup"] if name == "plda_dup" else g["en_ids"], g["E"])
    te = _ss(g["te_ids"], g["T"])
    ndx = _ndx(g["ndx_models"], g["ndx_segs"], g["trialmask"])
    D = g["E"].shape[1]
    if name == "cosine":
        sc = sk.cosine_scoring(en, te, ndx)
    elif name in ("plda", "plda_dup"):
        sc = sk.PLDA_scoring(en, te, ndx, g["mu"], g["F"], numpy.zeros((D, 0)), g["Sigma"])
    elif name == "plda_sf":
        sc = sk.PLDA_scoring(en, te, ndx, g["mu"], g["F"], numpy.zeros((D, 0)), g["Sigma"], scaling_factor=0.7)
    elif name == "plda_open":
        sc = sk.fast_PLDA_scoring(en, te, ndx, g["mu"], g["F"], g["Sigma"], p_known=0.3)
    else:
        sc = sk.two_covariance_scoring(en, te, ndx, g["Sigma"], g["B"])
    ref = (g[name + "_modelset"], g[name + "_segset"], g[name + "_mask"], g[name + "_mat"])
    _check(sc, ref, 1e-3, ref[3].dtype)


@pytest.mark.parametrize("name", ["full", "full_sf", "full_open"])
def test_golden_full_plda(name):
    """full_PLDA_scoring (channel subspace G) against the fixture recorded from the real reference."""
    g = golden("scoring_full.npz")
    en, te = _ss(g["en_ids"], g["E"]), _ss(g["te_ids"], g["T"])
    ndx = _ndx(g["ndx_models"], g["ndx_segs"], g["trialmask"])
    if name == "full":
        sc = sk.PLDA_scoring(en, te, ndx, g["mu"], g["F"], g["G"], g["Sigma"], full_model=True)
    elif name == "full_sf":
        sc = sk.full_PLDA_scoring(en, te, ndx, g["mu"], g["F"], g["G"], g["Sigma"], scaling_factor=0.6)
    else:
        sc = sk.full_PLDA_scoring(en, te, ndx, g["mu"], g["F"], g["G"], g["Sigma"], p_known=0.25)
    ref = (g[name + "_modelset"], g[name + "_segset"], g[name + "_mask"], g[name + "_mat"])
    _check(sc, ref, 1e-3, ref[3].dtype)
    assert en.modelset.tolist() == g["en_ids"].tolist()           # deep copies: the caller's objects are untouched


@pytest.mark.parametrize("unit_norm", [True, False])
@pytest.mark.parametrize("Ne,Nt,D", [(1000, 777, 256), (130, 3000, 256), (257, 129, 200)])
def test_plda_and_cosine_random(Ne, Nt, D, unit_norm):
    """Ragged sizes (tile edges), permuted / missing ids, unit-norm and N(0,1)-scale embeddings (split-precision path)."""
    rng = numpy.random.default_rng(Ne + Nt)
    E = synth.synth_embeddings(Ne, D, seed=1, unit_norm=unit_norm)
    T = synth.synth_embeddings(Nt, D, seed=2, unit_norm=unit_norm)
    mu, F, Sigma = synth.synth_plda(D, D, seed=3)
    en_ids = numpy.array(["m%05d" % i for i in range(Ne)])
    te_ids = numpy.array(["s%05d" % i for i in range(Nt)])
    nm = numpy.concatenate([en_ids[rng.permutation(Ne)[: Ne - 3]], ["nope"]])
    ns = numpy.concatenate([["nope2"], te_ids[rng.permutation(Nt)[: Nt - 5]]])
    mask = rng.random((nm.shape[0], ns.shape[0])) < 0.5
    a = (en_ids, E, te_ids, T, nm, ns, mask)
    sc = sk.PLDA_scoring(_ss(en_ids, E), _ss(te_ids, T), _ndx(nm, ns, mask), mu, F, numpy.zeros((D, 0)), Sigma)
    _check(sc, S.fast_plda_scoring(*a, mu, F, Sigma), 1e-3, numpy.float64)
    sc = sk.cosine_scoring(_ss(en_ids, E), _ss(te_ids, T), _ndx(nm, ns, mask))
    _check(sc, S.cosine_scoring(*a), 2e-5, numpy.float32)
    sc = sk.two_covariance_scoring(_ss(en_ids, E), _ss(te_ids, T), _ndx(nm, ns, mask), Sigma, F @ F.T + 0.1 * numpy.eye(D))
    _check(sc, S.two_covariance_scoring(*a, Sigma, F @ F.T + 0.1 * numpy.eye(D)), 1e-3, numpy.float64)


def test_score_matrix_linearity_and_symmetry_at_scale():
    """Size-independent properties at a size the numpy oracle would take long on: S(E,T) = S(T,E)^T bit-exactly
    is not required (different tilings), but cosine self-scores have a unit diagonal and S is linear in alpha."""
    X = torch.from_numpy(synth.synth_embeddings(6000, 256, seed=9)).float().cuda()
    S1 = sk.score_matrix(X, X, passes=3)
    assert (torch.diagonal(S1) - 1).abs().max().item() < 1e-5
    assert (S1 - S1.t()).abs().max().item() < 1e-5
    S2 = sk.score_matrix(X, X, alpha=2.0, cst=0.25, passes=3)
    assert (S2 - (2 * S1 + 0.5)).abs().max().item() < 1e-5
    S3 = sk.score_matrix(X, X, passes=1)
    assert (S3 - S1).abs().max().item() < 2.5e-4                  # single-pass fp16 on unit-norm rows
    ref = (X[:512].double() @ X[:700].double().t()).float()
    assert (S1[:512, :700] - ref).abs().max().item() < 1e-5


def test_baseline_config3_full_size_plda():
    """BASELINE.json configs[2]: PLDA scoring of the full 20k x 20k x 256 trial matrix through ``PLDA_scoring``.  The numpy
    oracle scores a random 300 x 300 sub-block (every score depends on its own pair only); the whole matrix is checked
    through a checksum of checksums: sum_ij S_ij = Nt sum_i a_i + Ne sum_j b_j + Ne Nt c + (sum_i e_i)' Psi (sum_j t_j),
    evaluated in float64 on the host from the oracle's matrices."""
    Ne = Nt = 20000
    D = 256
    E = synth.synth_embeddings(Ne, D, seed=6)
    T = synth.synth_embeddings(Nt, D, seed=7)
    mu, F, Sigma = synth.synth_plda(D, D, seed=8)
    en_ids = numpy.array(["m%06d" % i for i in range(Ne)])
    te_ids = numpy.array(["s%06d" % i for i in range(Nt)])
    ndx = _ndx(en_ids, te_ids, numpy.ones((Ne, Nt), dtype=bool))
    sc = sk.PLDA_scoring(_ss(en_ids, E), _ss(te_ids, T), ndx, mu, F, numpy.zeros((D, 0)), Sigma)
    dev = sc.scoremat_device
    assert dev.shape == (Ne, Nt) and dev.dtype == torch.float32 and sc.scoremat_dtype == numpy.float64      # widened on the way to the host
    assert sc.modelset.tolist() == en_ids.tolist() and sc.segset.tolist() == te_ids.tolist()
    rng = numpy.random.default_rng(3)
    ri, ci = numpy.sort(rng.choice(Ne, 300, replace=False)), numpy.sort(rng.choice(Nt, 300, replace=False))
    ref = S.fast_plda_scoring(en_ids[ri], E[ri], te_ids[ci], T[ci], en_ids[ri], te_ids[ci], numpy.ones((300, 300), dtype=bool),
                              mu, F, Sigma)[3]
    got = dev[torch.from_numpy(ri).cuda()][:, torch.from_numpy(ci).cuda()].cpu().numpy()
    assert numpy.abs(got - ref).max() < 1e-3
    Phi, Psi, cst = S.plda_matrices(F, Sigma)
    Ec, Tc = E.astype(numpy.float64) - mu, T.astype(numpy.float64) - mu
    a = 0.5 * numpy.einsum("ij,ij->i", Ec @ Phi, Ec)
    b = 0.5 * numpy.einsum("ij,ij->i", Tc @ Phi, Tc)
    total = Nt * a.sum() + Ne * b.sum() + float(Ne) * Nt * cst + Ec.sum(0) @ Psi @ Tc.sum(0)
    got_total = dev.sum(dtype=torch.float64).item()
    assert abs(got_total - total) < 1e-4 * float(Ne) * Nt             # mean absolute deviation per score below 1e-4
    row_ref = Nt * a + b.sum() + Nt * cst + (Ec @ Psi) @ Tc.sum(0)    # row checksums locate a bad row panel
    assert numpy.abs(dev.sum(dim=1, dtype=torch.float64).cpu().numpy() - row_ref).max() < 1e-4 * Nt


def test_asnorm_golden_and_oracle():
    g = golden("scoring.npz")
    out = sk.asnorm(torch.from_numpy(g["asnorm_X"]), torch.from_numpy(g["asnorm_cohort"]), None)
    assert out.dtype == numpy.float32 and out.shape == g["asnorm_out"].shape
    assert numpy.abs(out - g["asnorm_out"]).max() < 1e-3
    rng = numpy.random.default_rng(5)
    X = synth.synth_embeddings(700, 256, seed=21).astype(numpy.float32)
    coh = rng.standard_normal((1500, 256)).astype(numpy.float32)
    out = sk.asnorm(torch.from_numpy(X), torch.from_numpy(coh), None)
    assert numpy.abs(out - S.asnorm(X, coh)).max() < 1e-3


def test_asnorm_row_panels_equal_full_matrix():
    """bulk.asnorm_sharded through the CUDA routines (one process = whole matrix) and two hand-cut row panels."""
    from sidekit_b200 import bulk
    g = torch.Generator().manual_seed(12)
    X = torch.nn.functional.normalize(torch.randn(300, 64, generator=g), dim=1).cuda()
    coh = torch.randn(500, 64, generator=g).cuda()
    full = torch.from_numpy(sk.asnorm(X, coh, None)).cuda()
    lo, hi, panel = bulk.asnorm_sharded(X, coh, topk=200)
    assert (lo, hi) == (0, 300) and torch.equal(panel, full)
    mean, std = bulk._asnorm_stats_cuda(X, torch.nn.functional.normalize(coh, dim=1).contiguous(), 200)
    top = bulk._asnorm_panel_cuda(X, 0, 130, mean, std)
    bot = bulk._asnorm_panel_cuda(X, 130, 300, mean, std)
    assert torch.equal(torch.cat([top, bot]), full)               # panels are bit-identical to the one-shot matrix


def test_scores_device_gather_and_pipelined_copy_equal_the_plain_paths():
    from sidekit_b200.bosaris import _device_to_numpy
    g = torch.Generator().manual_seed(5)
    t = torch.randn(777, 333, generator=g, dtype=torch.float64).cuda()
    assert numpy.array_equal(_device_to_numpy(t, chunk_bytes=1 << 16), t.cpu().numpy())       # many chunks, ragged last one
    assert numpy.array_equal(_device_to_numpy(t.float()), t.float().cpu().numpy())             # small: direct copy
    rng = numpy.random.default_rng(8)
    ids_m = numpy.array(["m%03d" % i for i in range(120)])
    ids_s = numpy.array(["s%03d" % i for i in range(90)])
    en, te = _ss(ids_m, rng.standard_normal((120, 64))), _ss(ids_s, rng.standard_normal((90, 64)))
    ndx = _ndx(ids_m, ids_s, rng.random((120, 90)) < 0.7)
    key = sk.Key.create(ids_m, ids_s, rng.random((120, 90)) < 0.2, rng.random((120, 90)) < 0.5)
    a = sk.cosine_scoring(en, te, ndx)
    tar_d, non_d = a.get_tar_non(key)                 # matrix still on the device: gathered there
    assert a._scoremat is None
    b = sk.cosine_scoring(en, te, ndx)
    _ = b.scoremat                                    # materialise on the host first
    tar_h, non_h = b.get_tar_non(key)
    assert numpy.array_equal(tar_d, tar_h) and numpy.array_equal(non_d, non_h) and tar_d.dtype == tar_h.dtype


def test_cosine_scoring_with_wccn():
    """iv_scoring.py:99-101: both sides rotated by the WCCN matrix before the length normalisation."""
    rng = numpy.random.default_rng(8)
    D, Ne, Nt = 64, 150, 170
    E, T = synth.synth_embeddings(Ne, D, seed=51, unit_norm=False), synth.synth_embeddings(Nt, D, seed=52, unit_norm=False)
    Wc = numpy.linalg.cholesky(numpy.cov(rng.standard_normal((D, 4 * D))) + numpy.eye(D))
    ids_e = numpy.array(["m%04d" % i for i in range(Ne)])
    ids_t = numpy.array(["s%04d" % i for i in range(Nt)])
    mask = rng.random((Ne, Nt)) < 0.5
    sc = sk.cosine_scoring(_ss(ids_e, E), _ss(ids_t, T), _ndx(ids_e[::-1], ids_t, mask), wccn=Wc)
    _check(sc, S.cosine_scoring(ids_e, E, ids_t, T, ids_e[::-1], ids_t, mask, wccn=Wc), 1e-3, numpy.float32)


def test_packed_test_operand_equals_the_plain_call():
    from sidekit_b200.iv_scoring import PackedEmbeddings, score_matrix
    for unit in (True, False):
        E = torch.from_numpy(synth.synth_embeddings(700, 256, seed=61, unit_norm=unit)).float().cuda()
        T = torch.from_numpy(synth.synth_embeddings(900, 256, seed=62, unit_norm=unit)).float().cuda()
        r, q = torch.randn(700, device="cuda"), torch.randn(900, device="cuda")
        plain = score_matrix(E, T, r, q, cst=0.25, alpha=1.5, passes=0)
        Tp = PackedEmbeddings(T)
        for lo, hi in ((0, 700), (128, 391)):                        # the whole matrix and a row panel
            got = score_matrix(E[lo:hi].contiguous(), Tp, r[lo:hi].contiguous(), q, cst=0.25, alpha=1.5, passes=3 if not unit else 1)
            assert (got - plain[lo:hi]).abs().max().item() < 2e-4
        assert torch.equal(score_matrix(E, Tp, r, q, cst=0.25, alpha=1.5, passes=0), plain)      # same arithmetic, same bits


def test_pass_count_decided_on_the_device_is_one_launch_equal_to_the_forced_count():
    """passes=0 equals the call forced to the pass count the operand statistics pick (one pass on unit-norm rows, three on
    N(0,1) rows) bit for bit, and costs the same launches whether the E panel is resident (D = 256) or streamed (D = 512)."""
    from sidekit_b200 import _lib
    lib = _lib.lib()
    launches = {}
    for D in (256, 512):
        for unit, forced in ((True, 1), (False, 3)):
            E = torch.from_numpy(synth.synth_embeddings(300, D, seed=91, unit_norm=unit)).float().cuda()
            T = torch.from_numpy(synth.synth_embeddings(200, D, seed=92, unit_norm=unit)).float().cuda()
            n0 = lib.skb_kernel_launches()
            want = sk.score_matrix(E, T, passes=forced)
            n1 = lib.skb_kernel_launches()
            got = sk.score_matrix(E, T, passes=0)
            launches[D, unit] = lib.skb_kernel_launches() - n1
            assert torch.equal(got, want), (D, unit)
            assert launches[D, unit] == n1 - n0, (D, unit)
    for unit in (True, False):
        assert launches[512, unit] == launches[256, unit]


def test_large_matrix_reaches_the_host_through_the_pinned_path_widened():
    """Scores.scoremat of the PLDA family: float32 on the device, float64 on the host (widened on the way out)."""
    from sidekit_b200.bosaris import _device_to_numpy
    g = torch.Generator(device="cuda").manual_seed(3)
    t = torch.randn((5000, 2048), device="cuda", generator=g)           # 80 MB as float64: pinned, chunked path
    out64 = _device_to_numpy(t, numpy.float64, chunk_bytes=16 << 20)
    assert out64.dtype == numpy.float64 and numpy.array_equal(out64, t.cpu().numpy().astype(numpy.float64))
    out32 = _device_to_numpy(t)
    assert out32.dtype == numpy.float32 and numpy.array_equal(out32, t.cpu().numpy())
    small = _device_to_numpy(t[:7].contiguous(), numpy.float64)
    assert small.dtype == numpy.float64 and numpy.array_equal(small, t[:7].cpu().numpy().astype(numpy.float64))


def test_trial_list_mode_and_fp16_output():
    """VERDICT r1 item 4: the epilogue writes only the masked trials (row-major, the order of scoremat[trialmask]) or a
    16-bit matrix."""
    from sidekit_b200.iv_scoring import TrialIndex, score_matrix, score_trials
    rng = numpy.random.default_rng(12)
    for Ne, Nt, dens, unit in ((700, 900, 0.5, True), (333, 517, 0.01, False), (128, 128, 1.0, True), (1, 33, 0.3, True), (257, 31, 0.0, True)):
        E = torch.from_numpy(synth.synth_embeddings(Ne, 256, seed=71, unit_norm=unit)).float().cuda()
        T = torch.from_numpy(synth.synth_embeddings(Nt, 256, seed=72, unit_norm=unit)).float().cuda()
        r, q = torch.randn(Ne, device="cuda"), torch.randn(Nt, device="cuda")
        mask = rng.random((Ne, Nt)) < dens
        full = score_matrix(E, T, r, q, cst=0.25, alpha=1.5, passes=0)
        idx = TrialIndex(mask)
        assert idx.n_trials == int(mask.sum())
        got = score_trials(E, T, idx, r, q, cst=0.25, alpha=1.5, passes=0)
        assert got.shape == (int(mask.sum()),)
        assert torch.equal(got, full[torch.from_numpy(mask).cuda()])            # same arithmetic, same order
        from sidekit_b200.iv_scoring import PackedEmbeddings
        assert torch.equal(score_trials(E, PackedEmbeddings(T), idx, r, q, cst=0.25, alpha=1.5, passes=0), got)   # test side packed once
        assert torch.equal(score_trials(E, T, idx, r, None, cst=0.25, alpha=1.5, passes=0),
                           score_matrix(E, T, r, None, cst=0.25, alpha=1.5, passes=0)[torch.from_numpy(mask).cuda()])   # no column term
        qu = torch.randn(Nt + 1, device="cuda")[1:]                                 # a column term that is not 16-byte aligned
        assert torch.equal(score_trials(E, T, idx, r, qu, cst=0.25, alpha=1.5, passes=0),
                           score_matrix(E, T, r, qu, cst=0.25, alpha=1.5, passes=0)[torch.from_numpy(mask).cuda()])
        half = score_matrix(E, T, r, q, cst=0.25, alpha=1.5, passes=0, out_dtype=torch.float16)
        assert half.dtype == torch.float16 and torch.equal(half, full.half())


def test_asnorm_statistics_over_more_rows_than_one_scratch_panel():
    """The cohort score matrix is produced in panels of at most 16384 rows: 20000 rows cross a panel boundary."""
    from sidekit_b200.bulk import _asnorm_stats_cuda
    X = torch.nn.functional.normalize(torch.from_numpy(synth.synth_embeddings(20000, 32, seed=81, unit_norm=False)).float(), dim=1).cuda()
    coh = torch.nn.functional.normalize(torch.from_numpy(synth.synth_embeddings(333, 32, seed=82, unit_norm=False)).float(), dim=1).cuda()
    mean, std = _asnorm_stats_cuda(X, coh, 200)
    top = torch.topk(X.double() @ coh.double().T, 200, dim=1)[0]
    assert (mean.double() - top.mean(dim=1)).abs().max().item() < 1e-5
    assert (std.double() - top.std(dim=1)).abs().max().item() < 1e-5
