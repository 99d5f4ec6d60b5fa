"""Top-k scoring on the B200: ``score_topk`` equals the first k columns of a stable descending sort of ``score_matrix``
with the same arguments (values bit for bit, indices exactly) on the fused epilogue path (k <= 32, D <= 256) and the
panel path (larger k, D = 512); ties, errors, the StatServer-level functions against the oracle, and the row-panel
sharding (one GPU: hand-cut panels; two GPUs: NCCL)."""
import os
import socket

import numpy
import pytest
import torch

import sidekit_b200 as sk
from sidekit_b200 import bulk, synth
from sidekit_b200.iv_scoring import PackedEmbeddings, score_topk
from oracle import scoring_ref as S

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
SHAPES = [(700, 900), (333, 517), (1, 33), (128, 128), (257, 4097), (5, 200000)]


def _operands(Ne, Nt, D, kind, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    E = torch.randn((Ne, D), generator=g, device=DEV)
    T = torch.randn((Nt, D), generator=g, device=DEV)
    if kind == "unit":
        E, T = torch.nn.functional.normalize(E, dim=1), torch.nn.functional.normalize(T, dim=1)
    r = torch.randn((Ne,), generator=g, device=DEV)
    q = torch.randn((Nt,), generator=g, device=DEV)
    return E.contiguous(), T.contiguous(), r, q


def _ref(E, T, k, r, q, cst, alpha, passes):
    M = sk.score_matrix(E, T, r, q, cst, alpha, passes=passes)
    v, i = torch.sort(M, dim=1, descending=True, stable=True)
    return v[:, :k], i[:, :k]


def _check(got, ref, what):
    v, i = got
    rv, ri = ref
    assert v.dtype == torch.float32 and i.dtype == torch.int64, what
    assert torch.equal(v, rv), (what, (v - rv).abs().max().item())
    assert torch.equal(i, ri), (what, (i != ri).sum().item())


def _ks(Nt):
    return sorted({k for k in (1, 7, 32, 33, 200, min(Nt, 1024)) if k <= Nt})


@pytest.mark.parametrize("D", [64, 200, 256, 512])
@pytest.mark.parametrize("shape", SHAPES, ids=["%dx%d" % s for s in SHAPES])
def test_topk_equals_sorted_score_matrix(D, shape):
    Ne, Nt = shape
    for kind in ("unit", "normal"):
        E, T, r, q = _operands(Ne, Nt, D, kind, seed=D + Ne + Nt)
        for passes in (0, 1, 3):
            refs = {}
            M = sk.score_matrix(E, T, r, q, 0.25, 1.5, passes=passes)
            sv, si = torch.sort(M, dim=1, descending=True, stable=True)
            for k in _ks(Nt):
                refs[k] = (sv[:, :k], si[:, :k])
                _check(score_topk(E, T, k, r, q, 0.25, 1.5, passes), refs[k], (kind, passes, k))
            del M, sv, si
        # the same with the gallery packed once, without a column term, with a column term that is not 16-byte aligned,
        # and with a negative scale
        Tp = PackedEmbeddings(T)
        qbuf = torch.randn((Nt + 1,), device=DEV)
        q_odd = qbuf[1:]
        assert q_odd.data_ptr() % 16 != 0
        for k in sorted({min(7, Nt), min(33, Nt)}):
            _check(score_topk(E, Tp, k, r, q, 0.25, 1.5, 0), _ref(E, T, k, r, q, 0.25, 1.5, 0), ("packed", k))
            _check(score_topk(E, T, k, r, None, 0.0, 1.0, 0), _ref(E, T, k, r, None, 0.0, 1.0, 0), ("no colterm", k))
            _check(score_topk(E, Tp, k, None, q_odd, 0.0, 1.0, 3), _ref(E, T, k, None, q_odd, 0.0, 1.0, 3), ("unaligned colterm", k))
            _check(score_topk(E, T, k, r, q, 1.0, -2.0, 0), _ref(E, T, k, r, q, 1.0, -2.0, 0), ("negative alpha", k))


def _tie_operands():
    g = torch.Generator(device=DEV).manual_seed(3)
    # every row has the same largest |x| (column 0), so a subset of rows is packed with the same scale exponent as all of them
    E = torch.randn((300, 256), generator=g, device=DEV).clamp(-3, 3)
    E[:, 0] = 4.0
    base = torch.randn((400, 256), generator=g, device=DEV).clamp(-3, 3)
    base[:, 0] = 4.0
    dup = torch.randint(0, 400, (2000,), generator=g, device=DEV)
    return E, base[dup].contiguous()                  # a gallery with many duplicated rows: identical scores


@pytest.mark.parametrize("k", [1, 32, 200])
def test_ties_lower_column_first_and_partition_independent(k):
    E, T = _tie_operands()
    v, i = score_topk(E, T, k, passes=3)
    _check((v, i), _ref(E, T, k, None, None, 0.0, 1.0, 3), "ties")
    # equal scores come out lowest column first
    if k > 1:
        same = v[:, 1:] == v[:, :-1]
        assert bool(same.any())
        assert bool((i[:, 1:][same] > i[:, :-1][same]).all())
    else:
        M = sk.score_matrix(E, T, passes=3)
        first = (M == M.max(dim=1, keepdim=True).values).int().argmax(dim=1)
        assert torch.equal(i[:, 0], first)
    v2, i2 = score_topk(E, T, k, passes=3)
    assert torch.equal(v, v2) and torch.equal(i, i2)
    for row in (0, 131, 299):
        v1, i1 = score_topk(E[row:row + 1].contiguous(), T, k, passes=3)
        assert torch.equal(v1[0], v[row]) and torch.equal(i1[0], i[row]), row


def test_bad_k_raises():
    E, T, r, q = _operands(10, 50, 64, "unit", 1)
    for k in (0, 51):
        with pytest.raises(ValueError):
            score_topk(E, T, k)
    E, T, r, q = _operands(10, 2000, 64, "unit", 1)
    with pytest.raises(ValueError):
        score_topk(E, T, 1025)
    with pytest.raises(ValueError):
        score_topk(E, PackedEmbeddings(T), 1025)


def _statservers(n_models=300, n_segs=200, D=256, dup=False):
    E, T = synth.synth_embeddings(n_models, D, seed=1), synth.synth_embeddings(n_segs, D, seed=2)
    ids_e = numpy.array(["m%03d" % i for i in range(n_models)])
    if dup:
        ids_e[7] = ids_e[3]
    ids_t = numpy.array(["s%03d" % i for i in range(n_segs)])
    return ids_e, E, ids_t, T


def _compare_to_reference(res, ids_t, ref_models, ref_S, k):
    St = ref_S.T                                        # (segments, models)
    order = numpy.argsort(-St, axis=1, kind="stable")[:, :k]
    ref_v = numpy.take_along_axis(St, order, axis=1)
    assert numpy.array_equal(res.segset, ids_t)
    assert res.models.shape == res.scores.shape == (len(ids_t), k)
    assert numpy.abs(res.scores - ref_v).max() < 1e-3
    full = -numpy.sort(-St, axis=1)
    gap_prev = numpy.full(ref_v.shape, numpy.inf)
    gap_prev[:, 1:] = full[:, :k - 1] - full[:, 1:k]
    gap_next = full[:, :k] - full[:, 1:k + 1]
    clear = (gap_prev > 2e-3) & (gap_next > 2e-3)
    assert clear.any()
    assert numpy.array_equal(res.models[clear], ref_models[order][clear])


def test_cosine_topk_matches_oracle():
    ids_e, E, ids_t, T = _statservers()
    en, te = sk.StatServer.from_embeddings(ids_e, E), sk.StatServer.from_embeddings(ids_t, T)
    en_before, te_before = en.stat1.copy(), te.stat1.copy()
    wccn = numpy.linalg.qr(numpy.random.default_rng(4).standard_normal((256, 256)))[0]
    for w in (None, wccn):
        res = sk.cosine_topk(en, te, 10, wccn=w)
        assert res.scores.dtype == numpy.float32
        models, segs, mask, ref = S.cosine_scoring(ids_e, E, ids_t, T, ids_e, ids_t, numpy.ones((300, 200), bool), wccn=w)
        _compare_to_reference(res, ids_t, models, ref, 10)
    assert numpy.array_equal(en.stat1, en_before) and numpy.array_equal(te.stat1, te_before)
    assert numpy.array_equal(en.modelset, ids_e)


def test_plda_topk_matches_oracle():
    ids_e, E, ids_t, T = _statservers()
    mu, F, Sigma = synth.synth_plda(256, 256, seed=3)
    en, te = sk.StatServer.from_embeddings(ids_e, E), sk.StatServer.from_embeddings(ids_t, T)
    en_before, te_before = en.stat1.copy(), te.stat1.copy()
    for k in (5, 40):
        res = sk.PLDA_topk(en, te, k, mu, F, Sigma)
        assert res.scores.dtype == numpy.float64
        models, segs, mask, ref = S.fast_plda_scoring(ids_e, E, ids_t, T, ids_e, ids_t, numpy.ones((300, 200), bool), mu, F, Sigma)
        _compare_to_reference(res, ids_t, models, ref, k)
    assert numpy.array_equal(en.stat1, en_before) and numpy.array_equal(te.stat1, te_before)


def test_duplicate_model_ids_appear_once():
    ids_e, E, ids_t, T = _statservers(dup=True)
    en, te = sk.StatServer.from_embeddings(ids_e, E), sk.StatServer.from_embeddings(ids_t, T)
    mu, F, Sigma = synth.synth_plda(256, 256, seed=3)
    for res in (sk.cosine_topk(en, te, 299), sk.PLDA_topk(en, te, 299, mu, F, Sigma)):
        assert res.models.shape == (200, 299)
        for row in res.models:
            assert len(set(row.tolist())) == 299
        assert (res.models == ids_e[3]).sum(axis=1).tolist() == [1] * 200
    with pytest.raises(ValueError):
        sk.cosine_topk(en, te, 300)                   # 299 distinct models


def _panel_operands():
    E, T = _tie_operands()
    return E, T[:1500].contiguous()


def _per_panel(Q, G, k, world):
    parts = [bulk._topk_cuda(Q[lo:hi].contiguous(), G, k, 3) for lo, hi in (bulk.row_panel(Q.shape[0], r, world) for r in range(world))]
    return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])


def test_hand_cut_panels_equal_the_sharded_result():
    Q, G = _panel_operands()
    for k in (10, 100):
        v, i = bulk.topk_sharded(Q, G, k, passes=3)
        pv, pi = _per_panel(Q, G, k, 2)
        assert torch.equal(v, pv) and torch.equal(i, pi)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    Q, G = _panel_operands()
    dev = torch.device("cuda", rank)
    out = {}
    for k in (10, 100):
        v, i = bulk.topk_sharded(Q.to(dev), G.to(dev), k, passes=3)
        out[k] = (v.cpu(), i.cpu())
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_world2_equals_per_panel_calls():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    Q, G = _panel_operands()
    for k in (10, 100):
        pv, pi = _per_panel(Q, G, k, 2)
        for r in range(2):
            assert torch.equal(res[r][k][0], pv.cpu()) and torch.equal(res[r][k][1], pi.cpu())
