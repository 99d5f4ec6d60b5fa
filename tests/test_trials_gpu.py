"""GPU checks of pair-list scoring: ``skb_score_pairs`` against float64 numpy, its bit-level determinism, and
``cosine_scoring_trials`` / ``PLDA_scoring_trials`` / ``asnorm_trials`` against the dense scorers and the oracle at
VoxCeleb1-O shape (4 708 utterances, 37 720 trials)."""
import ctypes

import numpy
import pytest
import torch

import sidekit_b200 as sk
from oracle import scoring_ref as S
from sidekit_b200 import _lib, bulk, synth

pytestmark = pytest.mark.gpu

N_UTT, N_TRIALS = 4708, 37720


def _rows(n, D, seed, unit):
    return torch.from_numpy(synth.synth_embeddings(n, D, seed=seed, unit_norm=unit)).float().cuda()


def _ref(E, T, rows, cols, r=None, q=None, cst=0.0, alpha=1.0):
    """float64 numpy scores of the pairs and the scale a float32 dot product's rounding error is relative to."""
    e, t = E.double().cpu().numpy()[rows], T.double().cpu().numpy()[cols]
    terms = cst + (0.0 if r is None else r.double().cpu().numpy()[rows]) + (0.0 if q is None else q.double().cpu().numpy()[cols])
    return alpha * (terms + (e * t).sum(1)), abs(alpha) * (numpy.abs(e * t).sum(1) + numpy.abs(terms))


@pytest.mark.parametrize("D", [64, 200, 256, 512, 203])
@pytest.mark.parametrize("unit", [True, False])
def test_score_pairs_against_float64(D, unit):
    Ne, Nt, n = 1001, 777, 5000
    E, T = _rows(Ne, D, 11, unit), _rows(Nt, D, 12, unit)
    rng = numpy.random.default_rng(D)
    rows, cols = rng.integers(0, Ne, n), rng.integers(0, Nt, n)
    r, q = torch.randn(Ne, device="cuda"), torch.randn(Nt, device="cuda")
    for args in [dict(), dict(rowterm=r, colterm=q, cst=0.25, alpha=1.5), dict(rowterm=r, alpha=-0.5)]:
        out = sk.score_pairs(E, T, rows, cols, **args)
        assert out.dtype == torch.float32 and out.shape == (n,)
        ref, scale = _ref(E, T, rows, cols, args.get("rowterm"), args.get("colterm"), args.get("cst", 0.0), args.get("alpha", 1.0))
        err = numpy.abs(out.double().cpu().numpy() - ref)
        if unit:
            assert err.max() <= 1e-6, err.max()
        else:
            assert (err / scale).max() <= 1e-5, (err / scale).max()
    one = sk.score_pairs(E, T, rows[:1], cols[:1])
    assert one.shape == (1,) and abs(one.item() - _ref(E, T, rows[:1], cols[:1])[0][0]) <= 1e-5 * _ref(E, T, rows[:1], cols[:1])[1][0]
    assert sk.score_pairs(E, T, rows[:0], cols[:0]).shape == (0,)


def test_score_pairs_scalar_path_on_unaligned_rows():
    """A 16-byte-misaligned base takes the scalar loads; the scores are those of the aligned copy (same order of sums)."""
    Ne, Nt, D, n = 300, 200, 256, 4000
    buf = torch.empty(Ne * D + 1, device="cuda")
    E = buf[1:].view(Ne, D)
    E.copy_(_rows(Ne, D, 13, True))
    T = _rows(Nt, D, 14, True)
    rng = numpy.random.default_rng(1)
    rows, cols = rng.integers(0, Ne, n), rng.integers(0, Nt, n)
    out = sk.score_pairs(E, T, rows, cols)
    assert numpy.abs(out.double().cpu().numpy() - _ref(E, T, rows, cols)[0]).max() <= 1e-6


def test_score_pairs_bits_do_not_depend_on_position_or_list_length():
    Ne, Nt, D, n = 2000, 1500, 256, 30001
    E, T = _rows(Ne, D, 15, False), _rows(Nt, D, 16, False)
    rng = numpy.random.default_rng(2)
    rows, cols = rng.integers(0, Ne, n), rng.integers(0, Nt, n)
    r, q = torch.randn(Ne, device="cuda"), torch.randn(Nt, device="cuda")
    base = sk.score_pairs(E, T, rows, cols, r, q, cst=0.5, alpha=2.0)
    perm = rng.permutation(n)
    assert torch.equal(sk.score_pairs(E, T, rows[perm], cols[perm], r, q, cst=0.5, alpha=2.0), base[torch.from_numpy(perm).cuda()])
    longer_r = numpy.concatenate([rows, rng.integers(0, Ne, 77777)])
    longer_c = numpy.concatenate([cols, rng.integers(0, Nt, 77777)])
    assert torch.equal(sk.score_pairs(E, T, longer_r, longer_c, r, q, cst=0.5, alpha=2.0)[:n], base)
    assert torch.equal(sk.score_pairs(E, T, rows[:1], cols[:1], r, q, cst=0.5, alpha=2.0), base[:1])


def test_c_abi_out_of_range_index_gives_nan_and_bad_arguments_are_refused():
    Ne, Nt, D = 50, 40, 64
    E, T = _rows(Ne, D, 17, True), _rows(Nt, D, 18, True)
    rows = torch.tensor([0, 5, Ne, 7, -1, 3], dtype=torch.int32, device="cuda")
    cols = torch.tensor([1, Nt, 2, 39, 4, 0], dtype=torch.int32, device="cuda")
    out = torch.zeros(6, device="cuda")
    l = _lib.lib()
    before = l.skb_kernel_launches()
    _lib.check(l.skb_score_pairs(E.data_ptr(), T.data_ptr(), Ne, Nt, D, rows.data_ptr(), cols.data_ptr(), 6, None, None, 0.0, 1.0,
                                 None, None, None, None, out.data_ptr(), _lib.stream_ptr()))
    assert l.skb_kernel_launches() - before == 1
    got = out.cpu().numpy()
    assert numpy.isnan(got[[1, 2, 4]]).all()
    good = numpy.array([0, 3, 5])
    ref = _ref(E, T, rows.cpu().numpy()[good], cols.cpu().numpy()[good])[0]
    assert numpy.abs(got[good] - ref).max() <= 1e-6

    def call(n=6, Ne_=Ne, E_=E.data_ptr(), stats=(None, None, None, None)):
        return l.skb_score_pairs(E_, T.data_ptr(), Ne_, Nt, D, rows.data_ptr(), cols.data_ptr(), n, None, None, 0.0, 1.0,
                                 *stats, out.data_ptr(), _lib.stream_ptr())
    m = torch.zeros(Ne, device="cuda")
    assert call(Ne_=-1) == -1 and "bad arguments" in l.skb_last_error().decode()
    assert call(n=-1) == -1
    assert call(stats=(m.data_ptr(), m.data_ptr(), None, None)) == -1
    assert call(E_=None) == -1
    assert call(n=0, E_=None) == 0


# ---------------------------------------------------------------------------------------------- VoxCeleb1-O-shaped lists
def _vox_list(seed=0):
    """Ids, a Key and a TrialList of N_TRIALS distinct pairs over N_UTT utterances; every utterance is in some trial."""
    rng = numpy.random.default_rng(seed)
    ids = numpy.array(["id%05d/utt.wav" % i for i in range(N_UTT)])
    first = numpy.stack([numpy.arange(N_UTT), (numpy.arange(N_UTT) + 1) % N_UTT], 1)
    more = rng.integers(0, N_UTT, (3 * N_TRIALS, 2))
    pairs = numpy.concatenate([first, more])
    pairs = pairs[pairs[:, 0] != pairs[:, 1]]
    _, at = numpy.unique(pairs[:, 0] * N_UTT + pairs[:, 1], return_index=True)
    pairs = pairs[numpy.sort(at)][:N_TRIALS]
    tar = numpy.zeros((N_UTT, N_UTT), bool)
    non = numpy.zeros((N_UTT, N_UTT), bool)
    lab = rng.random(N_TRIALS) < 0.5
    tar[pairs[lab, 0], pairs[lab, 1]] = True
    non[pairs[~lab, 0], pairs[~lab, 1]] = True
    key = sk.Key.create(ids, ids, tar, non)
    return ids, key, sk.TrialList.from_key(key)


def _at(models, segs, mat, trials):
    """The entries of a (models x segs) matrix at the trials' ids."""
    mi = {v: i for i, v in enumerate(numpy.asarray(models).tolist())}
    si = {v: i for i, v in enumerate(numpy.asarray(segs).tolist())}
    return mat[[mi[v] for v in trials.enrolset.tolist()], [si[v] for v in trials.testset.tolist()]]


def test_cosine_scoring_trials_against_dense_and_oracle():
    ids, key, trials = _vox_list()
    X = synth.synth_embeddings(N_UTT, 256, seed=21, unit_norm=False)
    ss = sk.StatServer.from_embeddings(ids, X)
    before = ss.stat1.copy()
    res = sk.cosine_scoring_trials(ss, ss, trials)
    assert numpy.array_equal(ss.stat1, before)
    assert res.scores.dtype == numpy.float32 and res.scores.shape == (N_TRIALS,)
    tar, non = res.get_tar_non()
    dtar, dnon = sk.cosine_scoring(ss, ss, key.to_ndx()).get_tar_non(key)
    assert tar.shape == dtar.shape and non.shape == dnon.shape
    assert max(numpy.abs(tar - dtar).max(), numpy.abs(non - dnon).max()) <= 1e-5
    m, s, _, ref = S.cosine_scoring(ids, X, ids, X, key.modelset, key.segset, key.tar | key.non)
    assert numpy.abs(res.scores - _at(m, s, ref, trials)).max() <= 1e-6

    # separate enrolment / test servers: permuted rows, a duplicated enrolment id (first occurrence wins), unknown ids, WCCN
    rng = numpy.random.default_rng(5)
    pe = rng.permutation(N_UTT)
    en_ids = numpy.concatenate([ids[pe][:-10], ids[pe][:3]])
    E = numpy.concatenate([X[pe][:-10], X[pe][:3] + 1.0])
    pt = rng.permutation(N_UTT)[:-20]
    wccn = numpy.linalg.qr(rng.standard_normal((256, 256)))[0] + 0.1 * numpy.eye(256)
    res = sk.cosine_scoring_trials(sk.StatServer.from_embeddings(en_ids, E), sk.StatServer.from_embeddings(ids[pt], X[pt]), trials,
                                   wccn=wccn)
    keep = numpy.isin(trials.enrolset, en_ids) & numpy.isin(trials.testset, ids[pt])
    assert len(res.trials) == keep.sum() < N_TRIALS
    assert numpy.array_equal(res.trials.enrolset, trials.enrolset[keep])
    m, s, _, ref = S.cosine_scoring(en_ids, E, ids[pt], X[pt], key.modelset, key.segset, key.tar | key.non, wccn)
    assert numpy.abs(res.scores - _at(m, s, ref, res.trials)).max() <= 1e-6


def test_plda_scoring_trials_against_dense_and_oracle():
    ids, key, trials = _vox_list(1)
    D = 256
    X = synth.synth_embeddings(N_UTT, D, seed=22)
    mu, F, Sigma = synth.synth_plda(D, D, seed=23)
    ss = sk.StatServer.from_embeddings(ids, X)
    res = sk.PLDA_scoring_trials(ss, ss, trials, mu, F, Sigma)
    assert res.scores.dtype == numpy.float64 and res.scores.shape == (N_TRIALS,)
    dense = sk.PLDA_scoring(ss, ss, key.to_ndx(), mu, F, numpy.zeros((D, 0)), Sigma)
    assert numpy.abs(res.scores - _at(dense.modelset, dense.segset, dense.scoremat, trials)).max() <= 2e-4
    m, s, _, ref = S.fast_plda_scoring(ids, X, ids, X, key.modelset, key.segset, key.tar | key.non, mu, F, Sigma)
    assert numpy.abs(res.scores - _at(m, s, ref, trials)).max() <= 1e-3

    # duplicate enrolment ids are averaged, as fast_PLDA_scoring does; scaling factor
    en_ids = numpy.concatenate([ids, ids[:500]])
    E = numpy.concatenate([X, synth.synth_embeddings(500, D, seed=24)])
    en = sk.StatServer.from_embeddings(en_ids, E)
    res = sk.PLDA_scoring_trials(en, ss, trials, mu, F, Sigma, scaling_factor=0.7)
    dense = sk.PLDA_scoring(en, ss, key.to_ndx(), mu, F, numpy.zeros((D, 0)), Sigma, scaling_factor=0.7)
    assert numpy.abs(res.scores - _at(dense.modelset, dense.segset, dense.scoremat, trials)).max() <= 2e-4
    m, s, _, ref = S.fast_plda_scoring(en_ids, E, ids, X, key.modelset, key.segset, key.tar | key.non, mu, F, Sigma, scaling_factor=0.7)
    assert numpy.abs(res.scores - _at(m, s, ref, trials)).max() <= 1e-3


def test_asnorm_trials_against_dense_and_oracle(monkeypatch):
    ids, key, trials = _vox_list(2)
    X = synth.synth_embeddings(N_UTT, 256, seed=25).astype(numpy.float32)
    coh = synth.synth_embeddings(2000, 256, seed=26, unit_norm=False).astype(numpy.float32)
    calls = []
    stats_fn = bulk._asnorm_stats_cuda

    def recording(Xd, c, k):
        out = stats_fn(Xd, c, k)
        calls.append(out)
        return out
    monkeypatch.setattr(bulk, "_asnorm_stats_cuda", recording)
    ss = sk.StatServer.from_embeddings(ids, X)
    res = sk.asnorm_trials(ss, ss, trials, torch.from_numpy(coh), topk=200)
    assert len(calls) == 1                                  # one StatServer for both sides: the statistics once
    Xd = torch.from_numpy(X).cuda()
    mean, std = stats_fn(Xd, torch.nn.functional.normalize(torch.from_numpy(coh).cuda(), dim=1).contiguous(), 200)
    assert torch.equal(calls[0][0], mean) and torch.equal(calls[0][1], std)
    assert res.scores.dtype == numpy.float32 and res.scores.shape == (N_TRIALS,)
    dense = sk.asnorm(torch.from_numpy(X), torch.from_numpy(coh), None)
    ref_dense = _at(ids, ids, dense, trials)
    assert numpy.abs(res.scores - ref_dense).max() <= 5e-4
    assert numpy.abs(res.scores - _at(ids, ids, S.asnorm(X, coh), trials)).max() <= 1e-3
    tar, non = res.get_tar_non()
    assert tar.shape[0] == trials.labels.sum() and non.shape[0] == (~trials.labels).sum()

    # device tensors given as (ids, X) pairs: the same object is still detected
    calls.clear()
    pair = (ids, Xd)
    res2 = sk.asnorm_trials(pair, pair, trials, coh, topk=200)
    assert len(calls) == 1 and numpy.array_equal(res2.scores, res.scores)

    # separate enrolment / test sets, a subset of rows referenced: two statistics calls over the referenced rows
    calls.clear()
    half = trials.subset(numpy.arange(len(trials)) < 5000)
    res3 = sk.asnorm_trials((ids, X), (ids, X.copy()), half, coh, topk=200)
    assert len(calls) == 2
    assert numpy.abs(res3.scores - ref_dense[:5000]).max() <= 5e-4


def test_score_pairs_at_voxceleb1_e_shape():
    """145 160 x 256 embeddings, 579 818 random pairs; a random subset of 10 000 checked in float64."""
    N, D, n = 145160, 256, 579818
    g = torch.Generator(device="cuda").manual_seed(7)
    X = torch.nn.functional.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
    rows = torch.randint(0, N, (n,), device="cuda", generator=g, dtype=torch.int32)
    cols = torch.randint(0, N, (n,), device="cuda", generator=g, dtype=torch.int32)
    out = sk.score_pairs(X, X, rows, cols)
    pick = torch.from_numpy(numpy.random.default_rng(8).choice(n, 10000, replace=False)).cuda()
    r, c = rows[pick].long(), cols[pick].long()
    ref = (X[r].double() * X[c].double()).sum(1)
    assert (out[pick].double() - ref).abs().max().item() <= 1e-6
