"""Bulk extraction / scoring across GPUs (SURVEY.md 8e): one process per GPU, utterances sharded by length
bucket with greedy FLOP balancing, embeddings all-gathered with NCCL ONCE per shard (the path's only collective);
score matrices are sharded by row panel against a test operand that is packed once.  Host logic only -- the
per-rank work goes through ``Xtractor.extract_packed`` / ``extract_stream`` / ``score_matrix`` (CUDA).  Mirrors what
the reference does one utterance at a time in ``extract_embeddings`` (sidekit/nnet/xvector.py:1796-1916) and returns
the same ``StatServer`` layout.

Nothing here needs the whole corpus in memory: a rank only ever touches the waveforms of the batch it is working on
(``waves`` may be a callable ``i -> 1-D tensor`` or a ``load_batch`` function that returns a packed batch), so one
million utterances (704 GB of fp32 audio, BASELINE config 4) are streamed.
"""
import heapq

import numpy
import torch

from .statserver import StatServer


def halfresnet34_macs(n_samples):
    """Algorithmic MACs of one HalfResNet34 embedding (SURVEY.md 8d closed form); used as the balancing weight.
    Accepts a scalar or an integer array."""
    t1 = 1 + n_samples // 160
    t2 = (t1 - 1) // 2 + 1
    t3 = (t2 - 1) // 2 + 1
    t4 = (t3 - 1) // 2 + 1
    return 80 * t1 * 56608 + 40 * t2 * 278528 + 20 * t3 * 1703936 + 10 * t4 * 3276800 + 1310720 * t4 + 1350016


def _costs(lengths, cost):
    lengths = numpy.asarray(lengths, dtype=numpy.int64)
    try:
        c = numpy.asarray(cost(lengths), dtype=numpy.float64)
        if c.shape == lengths.shape:
            return c
    except Exception:
        pass
    return numpy.array([float(cost(int(v))) for v in lengths], dtype=numpy.float64)


def plan_shards(lengths, world_size, cost=halfresnet34_macs):
    """Deterministic assignment of utterances to ranks: longest-first greedy on the MAC count (ties -> lowest rank).
    Returns ``world_size`` index arrays, each sorted by length (so consecutive batches are length buckets).  A pure
    function of ``(lengths, world_size)``: every rank computes the same plan, so no index exchange is ever needed."""
    lengths = numpy.asarray(lengths, dtype=numpy.int64)
    c = _costs(lengths, cost)
    order = numpy.argsort(-lengths, kind="stable")
    heap = [(0.0, r) for r in range(world_size)]
    owner = numpy.empty(lengths.shape[0], dtype=numpy.int64)
    for i in order.tolist():
        load, r = heap[0]
        owner[i] = r
        heapq.heapreplace(heap, (load + c[i], r))
    shards = []
    idx = numpy.arange(lengths.shape[0], dtype=numpy.int64)
    for r in range(world_size):
        s = idx[owner == r]
        shards.append(s[numpy.lexsort((s, lengths[s]))])
    return shards


def make_batches(indices, lengths, max_audio_seconds=1200.0, max_utts=256, sample_rate=16000):
    """Split a length-sorted index list into packed batches bounded by total audio (activation memory) and count."""
    batches, cur, cur_s = [], [], 0.0
    for i in indices:
        s = float(lengths[i]) / sample_rate
        if cur and (cur_s + s > max_audio_seconds or len(cur) >= max_utts):
            batches.append(cur)
            cur, cur_s = [], 0.0
        cur.append(int(i))
        cur_s += s
    if cur:
        batches.append(cur)
    return batches


def make_batches_equal_cost(indices, lengths, n_batches, cost=halfresnet34_macs):
    """Split a length-sorted index list into exactly ``n_batches`` contiguous batches of (nearly) equal MAC count:
    every batch is a length bucket and takes the same time on the GPU.  Empty batches only when there are fewer
    utterances than batches."""
    indices = numpy.asarray(indices, dtype=numpy.int64)
    if indices.shape[0] == 0:
        return [[] for _ in range(n_batches)]
    c = numpy.cumsum(_costs(numpy.asarray(lengths, dtype=numpy.int64)[indices], cost))
    cuts = numpy.searchsorted(c, c[-1] * numpy.arange(1, n_batches) / n_batches, side="left") + 1
    cuts = numpy.minimum(numpy.maximum.accumulate(cuts), indices.shape[0])
    return [[int(v) for v in part] for part in numpy.split(indices, cuts)]


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


def _collective_device(device=None):
    """Device the collectives of this process run on: the given one, else the current CUDA device under NCCL, else CPU."""
    if device is not None:
        return torch.device(device)
    dist, _, _ = _dist()
    if dist is not None and dist.get_backend() == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return None


def gather_embeddings(local, shards, embedding_size, device=None):
    """The one collective of the extraction path: every rank contributes the (n_r, E) embeddings of ITS shard (rows in
    shard order) and receives all N embeddings in input order.  One ``all_gather_into_tensor`` of the padded blocks; the
    shard plan is a pure function of the lengths, so the index vectors are known everywhere.  Single process: a scatter."""
    dist, rank, world = _dist()
    dev = _collective_device(device) or (local.device if local is not None and local.numel() else torch.device("cpu"))
    n = int(sum(len(s) for s in shards))
    if local is None:
        local = torch.zeros((0, embedding_size), dtype=torch.float32, device=dev)
    local = local.to(dev, torch.float32)
    result = torch.empty((n, embedding_size), dtype=torch.float32, device=dev)
    if world == 1:
        result[torch.as_tensor(shards[0], device=dev)] = local
        return result
    n_max = max(len(s) for s in shards)
    block = torch.zeros((n_max, embedding_size), dtype=torch.float32, device=dev)
    block[: local.shape[0]] = local
    gathered = torch.empty((world * n_max, embedding_size), dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(gathered, block)
    for r, s in enumerate(shards):
        if len(s):
            result[torch.as_tensor(s, device=dev)] = gathered[r * n_max: r * n_max + len(s)]
    return result


def extract_embeddings_sharded(extract_fn, waves, embedding_size, max_audio_seconds=1200.0, device=None, lengths=None,
                               max_utts=256, n_batches=None):
    """Embeddings of all utterances on every rank, in input order.

    ``waves`` is a list of 1-D tensors, or a callable ``i -> 1-D tensor`` together with ``lengths`` (so that a rank only
    ever materialises the utterances of the batch it is working on).  ``extract_fn(list_of_waves) -> (n, E) tensor`` is
    ``model.extract_varlen`` in production.  Each rank extracts its shard in length-bucketed packed batches, largest
    first (the engine sizes its work buffers once); ONE ``all_gather`` at the end restores the global order.  With a
    single process this is just the batched local extraction."""
    dist, rank, world = _dist()
    get = waves if callable(waves) else (lambda i: waves[i])
    if lengths is None:
        if callable(waves):
            raise ValueError("a callable wave source needs `lengths`")
        lengths = [int(w.shape[-1]) for w in waves]
    lengths = numpy.asarray(lengths, dtype=numpy.int64)
    shards = plan_shards(lengths, world)
    mine = shards[rank]
    if n_batches is not None:
        batches = [b for b in make_batches_equal_cost(mine, lengths, n_batches) if b]
    else:
        batches = make_batches(mine, lengths, max_audio_seconds, max_utts)
    parts = [None] * len(batches)
    for k in reversed(range(len(batches))):
        parts[k] = extract_fn([get(i) for i in batches[k]]).to(torch.float32)
    dev = _collective_device(device) or (parts[0].device if parts else torch.device("cpu"))
    local = torch.cat([p.to(dev) for p in parts]) if parts else None
    return gather_embeddings(local, shards, embedding_size, dev)


def extract_embeddings(ids, waves, model, max_audio_seconds=1200.0, lengths=None):
    """In-memory counterpart of the reference's ``extract_embeddings``: returns a ``StatServer`` whose ``stat1`` holds
    the embeddings and ``stat0`` ones (xvector.py:1905-1914)."""
    dev = next(model.parameters()).device
    if dev.type == "cuda":
        model.reserve(256, max_audio_seconds, dev)      # the batch budget of make_batches below: no allocation inside the run
    emb = extract_embeddings_sharded(lambda ws: model.extract_varlen([w.to(dev) for w in ws]), waves, model.embedding_size,
                                     max_audio_seconds, lengths=lengths)
    return StatServer.from_embeddings(numpy.asarray(ids), emb.cpu().numpy())


def row_panel(n_rows, rank=None, world=None):
    """Contiguous block of enrol rows scored by this rank (score-matrix sharding; no collective)."""
    dist, r, w = _dist()
    rank = r if rank is None else rank
    world = w if world is None else world
    per = (n_rows + world - 1) // world
    return min(rank * per, n_rows), min((rank + 1) * per, n_rows)


def gather_rows(local_rows, n_rows, device=None):
    """All-gather of a row-sharded (``row_panel`` split) matrix: every rank passes ITS rows and gets all ``n_rows``.
    Used to replicate the test embeddings before tile-sharded scoring (SURVEY.md 8e)."""
    dist, rank, world = _dist()
    if world == 1:
        return local_rows
    per = (n_rows + world - 1) // world
    dev = _collective_device(device) or local_rows.device
    block = torch.zeros((per,) + tuple(local_rows.shape[1:]), dtype=local_rows.dtype, device=dev)
    block[: local_rows.shape[0]] = local_rows.to(dev)
    out = torch.empty((world * per,) + tuple(local_rows.shape[1:]), dtype=local_rows.dtype, device=dev)
    dist.all_gather_into_tensor(out, block)
    return out[:n_rows]


def _asnorm_stats_cuda(X, cohort_normalised, topk):
    from . import _lib
    N, D = X.shape
    mean = torch.empty((N,), dtype=torch.float32, device=X.device)
    std = torch.empty((N,), dtype=torch.float32, device=X.device)
    with torch.cuda.device(X.device):
        _lib.check(_lib.lib().skb_asnorm_stats(X.data_ptr(), cohort_normalised.data_ptr(), N, cohort_normalised.shape[0], D, int(topk),
                                               mean.data_ptr(), std.data_ptr(), _lib.stream_ptr()))
    return mean, std


def _asnorm_panel_cuda(X, lo, hi, mean, std):
    from . import _lib
    N, D = X.shape
    out = torch.empty((hi - lo, N), dtype=torch.float32, device=X.device)
    with torch.cuda.device(X.device):
        _lib.check(_lib.lib().skb_asnorm_apply_panel(X.data_ptr(), N, D, lo, hi - lo, mean.data_ptr(), std.data_ptr(), out.data_ptr(),
                                                     out.stride(0), _lib.stream_ptr()))
    return out


def asnorm_sharded(enrol_xv, cohort_xv, topk=200, stats_fn=_asnorm_stats_cuda, panel_fn=_asnorm_panel_cuda):
    """Adaptive s-norm across ranks (SURVEY.md 8e): every rank computes the top-k cohort statistics of ITS row panel,
    one ``all_gather`` shares the (N,) mean / std vectors (the symmetric formula needs mu_j, sigma_j of every column),
    then every rank normalises its rows.  Returns ``(row_begin, row_end, panel)`` with ``panel`` the (rows, N) block of
    the matrix ``asnorm`` returns; the result stays row-sharded.  ``stats_fn`` / ``panel_fn`` are the CUDA routines in
    production and injectable so the exchange can be tested on CPU."""
    dist, rank, world = _dist()
    X = enrol_xv.to(torch.float32).contiguous()
    coh = torch.nn.functional.normalize(cohort_xv.to(X.device, torch.float32), dim=1).contiguous()
    N = X.shape[0]
    lo, hi = row_panel(N, rank, world)
    per = (N + world - 1) // world
    mean = torch.zeros((world * per,), dtype=torch.float32, device=X.device)
    std = torch.ones((world * per,), dtype=torch.float32, device=X.device)
    if hi > lo:
        m, s = stats_fn(X[lo:hi].contiguous(), coh, topk)
        mean[lo:hi], std[lo:hi] = m, s
    if world > 1:
        both = torch.stack([mean[rank * per:(rank + 1) * per], std[rank * per:(rank + 1) * per]]).contiguous()
        gathered = torch.empty((world * 2, per), dtype=torch.float32, device=X.device)
        dist.all_gather_into_tensor(gathered, both)
        gathered = gathered.view(world, 2, per)
        mean, std = gathered[:, 0, :].reshape(-1).contiguous(), gathered[:, 1, :].reshape(-1).contiguous()
    mean, std = mean[:N].contiguous(), std[:N].contiguous()
    panel = panel_fn(X, lo, hi, mean, std) if hi > lo else torch.zeros((0, N), dtype=torch.float32, device=X.device)
    return lo, hi, panel


def _topk_cuda(queries, gallery, k, passes):
    from .iv_scoring import PackedEmbeddings, score_topk
    G = gallery if isinstance(gallery, PackedEmbeddings) else PackedEmbeddings(gallery.to(queries.device, torch.float32))
    return score_topk(queries, G, k, passes=passes)


def topk_sharded(queries, gallery, k, passes=3, topk_fn=_topk_cuda):
    """The ``k`` best gallery rows of every query across ranks: each rank scores ITS query rows (``row_panel``) against the
    gallery (packed once per call, or passed as a ``PackedEmbeddings``), and ONE ``all_gather_into_tensor`` of values +
    indices gives every rank the full ``(values (N, k) float32, indices (N, k) int64)``.

    ``passes`` is fixed (1 or 3), not decided from the operands: with ``passes=0`` a rank's pass count and operand scale
    would follow its own panel's statistics, so the result would depend on the number of ranks.  With a fixed count the
    rows of rank r equal ``topk_fn`` on that rank's panel.  ``topk_fn(queries, gallery, k, passes) -> (values, indices)`` is
    ``score_topk`` in production and injectable so the exchange can be tested on CPU."""
    if passes not in (1, 3):
        raise ValueError("topk_sharded needs a fixed pass count (1 or 3), got %r" % (passes,))
    dist, rank, world = _dist()
    Q = queries.to(torch.float32).contiguous()
    N = Q.shape[0]
    lo, hi = row_panel(N, rank, world)
    if hi > lo:
        values, indices = topk_fn(Q[lo:hi].contiguous(), gallery, k, passes)
    else:
        values = torch.zeros((0, k), dtype=torch.float32, device=Q.device)
        indices = torch.zeros((0, k), dtype=torch.int64, device=Q.device)
    if world == 1:
        return values, indices
    # one collective: the float32 value bits ride in int64 next to the indices, padded to the panel size
    per = (N + world - 1) // world
    dev = _collective_device() or Q.device
    block = torch.zeros((per, 2 * k), dtype=torch.int64, device=dev)
    block[: hi - lo, :k] = values.to(dev).contiguous().view(torch.int32).to(torch.int64)
    block[: hi - lo, k:] = indices.to(dev)
    gathered = torch.empty((world * per, 2 * k), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(gathered, block)
    gathered = gathered[:N]
    return gathered[:, :k].to(torch.int32).view(torch.float32).contiguous(), gathered[:, k:].contiguous()
