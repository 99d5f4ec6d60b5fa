"""Host logic of corpus extraction from files (sidekit_b200.corpus) on CPU: the block plan, the window pipeline under a
world-2 gloo group with a stub decoder / extractor, the error exchange, and extract_embeddings' row-count exchange."""
import os
import socket
import wave

import numpy
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from sidekit_b200 import bulk, corpus, synth
from sidekit_b200.nnet import xsets


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _spawn(target, args, world=2):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=target, args=(r, world, port, q) + args) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)


def test_plan_blocks_contiguous_balanced_and_pure():
    rng = numpy.random.default_rng(3)
    w = rng.uniform(1e4, 5e5, size=503)
    for world in (1, 2, 3, 8):
        blocks = corpus.plan_blocks(w, world)
        assert blocks == corpus.plan_blocks(w, world)
        assert blocks[0][0] == 0 and blocks[-1][1] == len(w) and all(a[1] == b[0] for a, b in zip(blocks, blocks[1:]))
        loads = numpy.array([w[a:b].sum() for a, b in blocks])
        assert numpy.abs(loads - w.sum() / world).max() <= w.max()
    blocks = corpus.plan_blocks(numpy.ones(3), 8)                   # fewer entries than ranks: empty blocks
    assert sum(b - a for a, b in blocks) == 3 and all(b - a in (0, 1) for a, b in blocks)
    assert corpus.plan_blocks(numpy.zeros(0), 4) == [(0, 0)] * 4


def test_entry_weights_pipes_weigh_the_median(tmp_path):
    paths = []
    for i, n in enumerate((100, 300, 1000)):
        p = os.path.join(str(tmp_path), "f%d" % i)
        open(p, "wb").write(b"x" * n)
        paths.append(p)
    assert corpus.entry_weights(paths + [None]).tolist() == [100, 300, 1000, 300]
    assert corpus.entry_weights([None, None]).tolist() == [1, 1]


def _corpus(d, n=23, bad=None):
    """n short 16-bit WAV files of different lengths and rates; entry ``bad`` is not audio."""
    paths = []
    for i in range(n):
        p = os.path.join(d, "u%02d.wav" % i)
        if i == bad:
            open(p, "wb").write(b"this is not audio" * 40)
        else:
            rate = 8000 if i % 5 == 0 else 16000
            x = (synth.synth_wave(1, 800 + 97 * i, seed=i)[0].numpy() * 32768).astype(numpy.int16)
            with wave.open(p, "wb") as f:
                f.setnchannels(1); f.setsampwidth(2); f.setframerate(rate)
                f.writeframes(x.tobytes())
        paths.append(p)
    return paths


def _stub_embed(win):
    # "decode + extract": a row per entry from its parsed header and bytes, so order and ownership mistakes show
    rows = torch.tensor([[float(f), float(r), float(sum(d[-64:])), float(len(d))] for f, r, d in zip(win.frames, win.rates, win.datas)])
    return lambda: rows


def _pipeline(paths, touched, emitted):
    def read(p):
        touched.append(p)
        return corpus.read_file(p)
    return corpus.extract_sharded(paths, corpus.entry_weights(paths), read, _stub_embed, 4, 0.2, emit_fn=lambda idx, rows: emitted.extend(idx))


def _sharded_worker(rank, world, port, q, paths):
    _init(rank, world, port)
    touched, emitted = [], []
    try:
        out, blocks = _pipeline(paths, touched, emitted)
        q.put((rank, ("ok", out.numpy(), touched, emitted, blocks)))
    except Exception as e:
        q.put((rank, ("error", type(e).__name__, str(e), touched)))
    dist.destroy_process_group()


def test_world2_rows_in_input_order_equal_world1(tmp_path):
    d = str(tmp_path)
    paths = _corpus(d)
    touched, emitted = [], []
    ref, blocks = _pipeline(paths, touched, emitted)
    assert blocks == [(0, len(paths))] and touched == paths and emitted == list(range(len(paths)))
    assert ref.shape == (len(paths), 4) and len({tuple(r) for r in ref.tolist()}) == len(paths)
    res = _spawn(_sharded_worker, (paths,))
    for rank in (0, 1):
        assert res[rank][0] == "ok", res[rank][:3]
        status, out, touched, emitted, blocks = res[rank]
        assert status == "ok" and numpy.array_equal(out, ref.numpy())            # every rank: all rows, input order
        a, b = blocks[rank]
        assert 0 < b - a < len(paths) and touched == paths[a:b]                  # only its own block, in order
        assert emitted == list(range(a, b))


def test_bad_entry_on_rank1_raises_on_both_ranks(tmp_path):
    d = str(tmp_path)
    bad = 20                                           # in rank 1's block (the last ~half of the entries)
    res = _spawn(_sharded_worker, (_corpus(d, bad=bad),))
    name = os.path.join(d, "u%02d.wav" % bad)
    for rank in (0, 1):
        assert res[rank][0] == "error", rank
        assert res[rank][1] == "ValueError" and name in res[rank][2] and "not a FLAC, WAV or NIST SPHERE" in res[rank][2]
    assert name not in res[0][3]                       # rank 0 never opened it


def test_missing_entry_single_process_raises_after_earlier_windows(tmp_path):
    d = str(tmp_path)
    paths = _corpus(d, n=12)
    os.remove(paths[9])
    emitted = []
    with pytest.raises(OSError):
        _pipeline(paths, [], emitted)
    assert emitted and emitted == list(range(len(emitted))) and len(emitted) <= 9


# ----------------------------------------------------------------------------- extract_embeddings' row-count exchange
def _scattered_idmap():
    """Sliding-window segments of four files, one file's segments scattered through the map."""
    import sidekit_b200 as sk
    rows = [("a", "f0", None, None), ("b", "f1", 10, 190), ("a", "f2", None, None), ("c", "f0", 20, 160),
            ("b", "f3", 0, 300), ("c", "f0", 5, 125), ("a", "f1", None, None), ("d", "f0", 0, 100)]
    im = sk.IdMap()
    im.leftids = numpy.array([r[0] for r in rows], dtype="|O")
    im.rightids = numpy.array([r[1] for r in rows], dtype="|O")
    im.start = numpy.array([r[2] for r in rows], dtype="|O")
    im.stop = numpy.array([r[3] for r in rows], dtype="|O")
    return im


FILE_LEN = {"f0": 61000, "f1": 45000, "f2": 52000, "f3": 70000}


def _assemble(owner):
    """What extract_embeddings does after its windows, with a stub row per sliding window (segment index, window)."""
    ds = xsets.IdMapSet(_scattered_idmap(), "/data", "wav", sliding_window=True, window_len=1.0, window_shift=0.5, min_duration=1.0)
    _, rank, _ = bulk._dist()
    mine = [i for i in range(len(ds)) if owner[i] == rank]
    seg_len, parts = {}, []
    for i in mine[::-1]:                               # windows in another order than the map
        n = xsets._segment(ds, i, FILE_LEN[ds.idmap.rightids[i]])[1]
        m = xsets._windows_of(ds, n)[0]
        seg_len[i] = n
        parts.append(([(i, n, m)], torch.tensor([[float(i), float(j)] for j in range(m)])))
    return xsets._assemble(ds, parts, seg_len, None, owner, 2, 0.5)


def _assemble_worker(rank, world, port, q, owner):
    _init(rank, world, port)
    ss = _assemble(owner)
    q.put((rank, (ss.stat1, ss.modelset, ss.segset, ss.start, ss.stop)))
    dist.destroy_process_group()


def test_extract_embeddings_row_exchange_matches_world1():
    owner = numpy.array([1, 0, 0, 1, 0, 1, 0, 1])         # the segments of f0 (rank 1) are scattered through the map
    ref = _assemble(numpy.zeros(8, numpy.int64))
    assert ref.stat1.shape[0] == ref.modelset.shape[0] == ref.start.shape[0]
    assert ref.stat1[:, 0].tolist() == sorted(ref.stat1[:, 0].tolist())          # rows in id-map order
    res = _spawn(_assemble_worker, (owner,))
    for rank in (0, 1):
        stat1, modelset, segset, start, stop = res[rank]
        assert numpy.array_equal(stat1, ref.stat1) and numpy.array_equal(modelset, ref.modelset)
        assert numpy.array_equal(segset, ref.segset) and numpy.array_equal(start, ref.start) and numpy.array_equal(stop, ref.stop)


def test_launch_error_keeps_earlier_windows(tmp_path):
    """A window whose device work fails to launch: the windows before it are still emitted, then the error raises."""
    paths = _corpus(str(tmp_path), n=12)
    emitted, calls = [], []

    def embed(win):
        calls.append(len(win))
        if len(calls) == 3:
            raise RuntimeError("launch failed")
        return _stub_embed(win)

    with pytest.raises(RuntimeError, match="launch failed"):
        corpus.run_windows(paths, corpus.read_file, 0.2, embed, lambda win, rows: emitted.extend(win.index))
    assert emitted == list(range(calls[0] + calls[1]))


def test_pipe_flac_without_frames_is_a_value_error():
    from oracle import flac_ref
    from sidekit_b200 import audio, extract_xvectors as X
    data = flac_ref.encode(numpy.zeros((4096, 1), numpy.int64), 16000, 16)
    head = data[:audio.parse(data)[1].frames_begin]                       # the metadata only
    for name in ("cat x.flac |", "x.flac"):
        with pytest.raises(ValueError, match="no frames"):
            X._parse_source(name, head)
    with pytest.raises(IOError, match="Error processing wav file"):
        X._parse_source("cat x.wav |", b"not audio")
