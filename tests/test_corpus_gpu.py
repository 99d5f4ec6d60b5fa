"""Corpus extraction from files on the device (sidekit_b200.corpus): ``extract_xvectors.main`` over a mixed corpus in
many windows against one window and against direct decoding, the per-window call counts, ``extract_embeddings``
streamed in windows (results and bounded device memory), and the NCCL world-2 runs (skipped with fewer GPUs)."""
import os
import socket

import numpy
import pytest
import torch

import sidekit_b200 as sk
from oracle import flac_ref as F
from oracle import pcm_ref as R
from sidekit_b200 import audio, flac, kaldi_io, pcm, synth
from sidekit_b200.nnet import xsets
from sidekit_b200.nnet.preprocessor import Resample
from tests.models import make_xtractor

pytestmark = pytest.mark.gpu


def _pcm16(L, seed):
    return (synth.synth_wave(1, L, seed=seed)[0].numpy() * 32768.0).clip(-32768, 32767).astype(numpy.int64)[:, None]


def _ulaw(x16):
    table = R.ulaw2lin(numpy.arange(256)).astype(numpy.int64)
    order = numpy.argsort(table)
    return order[numpy.clip(numpy.searchsorted(table[order], x16), 0, 255)].astype(numpy.uint8)


def _mixed_corpus(d, bad=None, corrupt=None):
    """wav.scp over 16- and 24-bit WAV, FLAC, mu-law SPHERE, 8 kHz files and `cat x |` pipes (``bad``: a non-audio entry;
    ``corrupt``: a FLAC entry with a flipped byte in its frames, found by the decoder on the device)."""
    files = []
    for i in range(14):
        L = 9000 + 2311 * i
        x = _pcm16(L, 900 + i)
        kind = i % 6
        if kind == 0:
            data, ext = R.wav_bytes(x, 16000, "pcm", 2), "wav"
        elif kind == 1:
            data, ext = R.wav_bytes(x * 256, 16000, "pcm", 3), "wav"
        elif kind == 2:
            data, ext = F.encode(x, 16000, 16, blocksize=1024), "flac"
        elif kind == 3:
            data, ext = R.sph_bytes(_ulaw(x[:, 0])[:, None], 8000, "ulaw", 1), "sph"
        elif kind == 4:
            data, ext = R.wav_bytes(x, 8000, "pcm", 2), "wav"
        else:
            data, ext = F.encode(x, 8000, 16, blocksize=512), "flac"
        if i == bad:
            data = b"not audio at all " * 100
        if i == corrupt:
            assert ext == "flac"
            data = bytearray(data)
            data[len(data) // 2] ^= 0xFF
            data = bytes(data)
        p = os.path.join(d, "u%02d.%s" % (i, ext))
        with open(p, "wb") as f:
            f.write(data)
        files.append(("utt%02d" % i, "cat %s |" % p if i % 4 == 3 else p))
    with open(os.path.join(d, "wav.scp"), "w") as f:
        f.writelines("%s %s\n" % kv for kv in files)
    with open(os.path.join(d, "spk2utt"), "w") as f:
        f.write("spkA %s\nspkB %s\n" % (" ".join(k for k, _ in files[::2]), " ".join(k for k, _ in files[1::2])))
    return files


def _run_main(model, d, out_dir, window_s, stats=None):
    from sidekit_b200 import extract_xvectors as X
    os.makedirs(out_dir, exist_ok=True)
    emb = X.main(model, os.path.join(d, "wav.scp"), os.path.join(out_dir, "xv.scp"), "cuda", False, 2000, 1500, 16000,
                 os.path.join(out_dir, "spk.scp"), os.path.join(d, "spk2utt"), window_audio_seconds=window_s, stats=stats)
    return emb, _tables(out_dir)


def _tables(out_dir):
    out = {}
    for name in ("xv.ark", "xv.scp", "spk.ark", "spk.scp"):
        p = os.path.join(out_dir, name)
        out[name] = open(p, "rb").read().replace(os.path.realpath(out_dir).encode(), b"<out>") if os.path.exists(p) else None
    return out


class _Counts:
    def __init__(self, monkeypatch):
        self.n = {"h2d": 0, "flac": 0, "pcm": 0, "resample": 0}
        for owner, name, key in ((audio.Staging, "launch", "h2d"), (flac, "launch", "flac"), (pcm, "launch", "pcm"),
                                 (Resample, "launch", "resample")):
            monkeypatch.setattr(owner, name, self._wrap(getattr(owner, name), key))

    def _wrap(self, fn, key):
        def wrapped(*a, **k):
            self.n[key] += 1
            return fn(*a, **k)
        return wrapped


def test_main_windows_pipes_and_formats_bit_exact(tmp_path, monkeypatch):
    d = str(tmp_path)
    files = _mixed_corpus(d)
    model = make_xtractor("halfresnet34", 32, 256).cuda()
    one, t_one = _run_main(model, d, os.path.join(d, "one"), 1e9)
    counts = _Counts(monkeypatch)
    stats = []
    many, t_many = _run_main(model, d, os.path.join(d, "many"), 1.5, stats)
    assert len(stats) >= 6                                          # many windows, read ahead
    assert t_many == t_one and all(v for v in t_one.values())      # ark / scp / speaker means: the same bytes
    assert torch.equal(many, one) and many.shape == (len(files), 256)
    # per window: one host-to-device copy, at most one FLAC and one PCM call, one resampling call (one other rate)
    assert counts.n["h2d"] == len(stats)
    assert counts.n["flac"] <= len(stats) and counts.n["pcm"] <= len(stats) and counts.n["resample"] <= len(stats)
    assert counts.n["resample"] >= 1 and counts.n["flac"] >= 1 and counts.n["pcm"] >= 1
    monkeypatch.undo()
    # the vectors of the decoded and resampled signals, extracted directly
    waves = []
    for _, src in files:
        data = open(src.split()[1] if src.endswith("|") else src, "rb").read()
        x, _, rates = audio.decode([data])
        waves.append(Resample(int(rates[0]), 16000)(x) if rates[0] != 16000 else x)
    assert numpy.array_equal(one.numpy(), model.extract_varlen(waves).cpu().numpy())


def test_main_error_keeps_earlier_windows(tmp_path):
    d = str(tmp_path)
    _mixed_corpus(d, bad=10)
    model = make_xtractor("halfresnet34", 32, 256).cuda()
    with pytest.raises(ValueError, match="u10"):
        _run_main(model, d, os.path.join(d, "out"), 1.5)
    keys = [k for k, _ in kaldi_io.read_scp(os.path.join(d, "out", "xv.scp"))]
    assert keys and keys == ["utt%02d" % i for i in range(len(keys))] and len(keys) <= 10


def test_main_corrupt_flac_is_named_after_earlier_windows(tmp_path):
    """A FLAC entry whose frames fail their CRC on the device: the error names it (not the fp16 guard tripped by the
    unwritten samples), and the windows before it are in the ark."""
    d = str(tmp_path)
    _mixed_corpus(d, corrupt=8)
    model = make_xtractor("halfresnet34", 32, 256).cuda()
    with pytest.raises(ValueError, match="corrupt FLAC: .*u08.flac"):
        _run_main(model, d, os.path.join(d, "out"), 1.5)
    keys = [k for k, _ in kaldi_io.read_scp(os.path.join(d, "out", "xv.scp"))]
    assert keys and keys == ["utt%02d" % i for i in range(len(keys))] and len(keys) <= 8
    # extract_embeddings on the same file
    rows = [("a", "u02", None, None), ("b", "u08", None, None)]
    with pytest.raises(ValueError, match="corrupt FLAC: .*u08.flac"):
        sk.nnet.extract_embeddings(_idmap(rows), model, d, torch.device("cuda"), win_duration=1.0, file_extension="flac")
    # the engine is usable afterwards: no stale overflow count is left to trip the next call
    x = torch.from_numpy(_pcm16(20000, 5)[:, 0].astype(numpy.float32) / 32768).cuda()
    assert model.extract_varlen([x]).shape == (1, 256)


def _idmap(rows):
    im = sk.IdMap()
    im.leftids = numpy.array([r[0] for r in rows], dtype="|O")
    im.rightids = numpy.array([r[1] for r in rows], dtype="|O")
    im.start = numpy.array([r[2] for r in rows], dtype="|O")
    im.stop = numpy.array([r[3] for r in rows], dtype="|O")
    return im


def _wav_files(d, n, L, seed=0):
    for i in range(n):
        with open(os.path.join(d, "f%d.wav" % i), "wb") as f:
            f.write(R.wav_bytes(_pcm16(L + 313 * i, seed + i), 16000, "pcm", 2))


def _seg_rows(n):
    rows = []
    for i in range(n):
        rows += [("m%d" % i, "f%d" % i, None, None), ("m%d" % (i + 1), "f%d" % i, 30 * (i % 3), 30 * (i % 3) + 150)]
    return rows[::-1]                                          # a file's segments are not next to each other


def test_extract_embeddings_windows_equal_one_call(tmp_path):
    d = str(tmp_path)
    _wav_files(d, 6, 40000)
    model = make_xtractor("halfresnet34", 32, 256).cuda()
    for sliding in (False, True):
        kw = dict(win_duration=1.0, win_shift=0.5, sliding_window=sliding)
        one = sk.nnet.extract_embeddings(_idmap(_seg_rows(6)), model, d, torch.device("cuda"), **kw)
        many = sk.nnet.extract_embeddings(_idmap(_seg_rows(6)), model, d, torch.device("cuda"), window_audio_seconds=2.0, **kw)
        for f in ("stat1", "modelset", "segset", "start", "stop", "stat0"):
            assert numpy.array_equal(getattr(one, f), getattr(many, f)), (sliding, f)
        # the items of IdMapSet, embedded one by one
        ds = xsets.IdMapSet(_idmap(_seg_rows(6)), d, "wav", sliding_window=sliding, window_len=1.0, window_shift=0.5, min_duration=1.0)
        waves = []
        for i in range(len(ds)):
            speech = ds[i][0]
            waves.extend(speech if sliding else [speech])
        assert numpy.array_equal(many.stat1, model.extract_varlen([w.contiguous().cuda() for w in waves]).cpu().numpy())


def test_extract_embeddings_device_memory_follows_the_window(tmp_path):
    model = make_xtractor("halfresnet34", 32, 256).cuda()
    peaks = []
    for n in (4, 40):
        d = os.path.join(str(tmp_path), "c%d" % n)
        os.makedirs(d)
        _wav_files(d, n, 128000)
        rows = [("m%d" % i, "f%d" % i, None, None) for i in range(n)]
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        sk.nnet.extract_embeddings(_idmap(rows), model, d, torch.device("cuda"), window_audio_seconds=32.0, win_duration=1.0)
        peaks.append(torch.cuda.max_memory_allocated() - base)
    assert peaks[1] < 2 * peaks[0], peaks


# ----------------------------------------------------------------------------- two GPUs, NCCL
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, q, d, bad_d):
    import torch.distributed as dist
    from sidekit_b200 import extract_xvectors as X
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    model = make_xtractor("halfresnet34", 32, 256).to(dev)
    out = os.path.join(d, "world2")
    os.makedirs(out, exist_ok=True)
    emb = X.main(model, os.path.join(d, "wav.scp"), os.path.join(out, "xv.scp"), dev, False, 2000, 1500, 16000,
                 os.path.join(out, "spk.scp"), os.path.join(d, "spk2utt"), window_audio_seconds=1.5)
    ss = sk.nnet.extract_embeddings(_idmap(_seg_rows(6)), model, d, dev, win_duration=1.0, win_shift=0.5, sliding_window=True,
                                    window_audio_seconds=2.0)
    try:
        X.main(model, os.path.join(bad_d, "wav.scp"), os.path.join(bad_d, "xv.scp"), dev, window_audio_seconds=1.5)
        err = None
    except Exception as e:
        err = (type(e).__name__, str(e))
    q.put((rank, emb.numpy(), (ss.stat1, ss.modelset, ss.segset, ss.start, ss.stop), err))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_world2_main_and_extract_embeddings(tmp_path):
    import torch.multiprocessing as mp
    d, bad_d = os.path.join(str(tmp_path), "good"), os.path.join(str(tmp_path), "bad")
    os.makedirs(d)
    os.makedirs(bad_d)
    _mixed_corpus(d)
    _wav_files(d, 6, 40000)
    _mixed_corpus(bad_d, bad=12)                      # in rank 1's block
    model = make_xtractor("halfresnet34", 32, 256).cuda()
    one, t_one = _run_main(model, d, os.path.join(d, "world1"), 1.5)
    ref = sk.nnet.extract_embeddings(_idmap(_seg_rows(6)), model, d, torch.device("cuda"), win_duration=1.0, win_shift=0.5,
                                     sliding_window=True)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q, d, bad_d)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=900) for _ in range(2)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert _tables(os.path.join(d, "world2")) == t_one            # rank 0 wrote the world-1 bytes
    for rank, emb, ss, err in res:
        assert numpy.array_equal(emb, one.numpy()), rank
        for got, want in zip(ss, (ref.stat1, ref.modelset, ref.segset, ref.start, ref.stop)):
            assert numpy.array_equal(got, want), rank
        assert err is not None and err[0] == "ValueError" and "u12" in err[1], (rank, err)
