"""WAV / NIST SPHERE decoding on the device (csrc/pcm.cu through sidekit_b200.audio) against the numpy decoder of
oracle/pcm_ref.py, bit for bit; mixed FLAC / WAV / SPHERE batches; bad files named; and the feed path (IdMapSet,
extract_embeddings, extract_xvectors.main) on every encoding against extraction from the oracle's waveforms."""
import os

import numpy
import pytest
import torch

import sidekit_b200 as sk
from oracle import flac_ref as F, pcm_ref as R
from sidekit_b200 import _lib, audio, flac, synth
from sidekit_b200.nnet import xsets
from tests.models import make_xtractor

pytestmark = pytest.mark.gpu

FORMATS = [("wav", "u8", 1), ("wav", "pcm", 2), ("wav", "pcm", 3), ("wav", "pcm", 4), ("wav", "float", 4), ("wav", "float", 8),
           ("wav", "ulaw", 1), ("wav", "alaw", 1), ("wavex", "pcm", 3), ("wavex", "float", 4), ("sph", "pcm", 2),
           ("sph_be", "pcm", 2), ("sph", "pcm", 1), ("sph_be", "pcm", 3), ("sph", "ulaw", 1), ("sph", "alaw", 1)]
LENGTHS = (0, 1, 1001, 100003)


def _file(kind, enc, nb, values, rate=16000):
    if kind.startswith("sph"):
        return R.sph_bytes(values, rate, enc, nb, big_endian=kind == "sph_be")
    return R.wav_bytes(values, rate, enc, nb, extensible=kind == "wavex")


@pytest.fixture(scope="module")
def matrix():
    rng = numpy.random.default_rng(5)
    return [_file(kind, enc, nb, R.synth(rng, L, ch, enc, nb)) for kind, enc, nb in FORMATS for ch in (1, 2, 6) for L in LENGTHS]


def test_exact_decode_batch_and_alone(matrix):
    out, n, rates = audio.decode(matrix)
    parts = torch.split(out, n.tolist())
    for data, x, r in zip(matrix, parts, rates.tolist()):
        rate, ref = R.decode(data)
        assert r == rate and x.shape[0] == ref.shape[0] and numpy.array_equal(x.cpu().numpy().view(numpy.uint32), ref.view(numpy.uint32))
    for data, x in zip(matrix, parts):
        alone, _, _ = audio.decode([data])
        assert torch.equal(alone, x)                                  # bit-identical whatever the batch


def test_16_and_32_bit_wav_equal_read_wav(tmp_path):
    rng = numpy.random.default_rng(6)
    paths = []
    for i, (nb, ch, L) in enumerate([(2, 1, 100003), (2, 2, 777), (4, 1, 5000), (4, 3, 4097), (2, 1, 256), (2, 1, 255)]):
        paths.append(os.path.join(str(tmp_path), "w%d.wav" % i))
        with open(paths[-1], "wb") as f:
            f.write(R.wav_bytes(R.synth(rng, L, ch, "pcm", nb), 16000, "pcm", nb))
    out, n, _ = audio.decode(paths)
    for p, x in zip(paths, torch.split(out, n.tolist())):
        assert torch.equal(x.cpu(), xsets.read_wav(p)[0])


def _launches(files):
    lib = _lib.lib()
    torch.cuda.synchronize()
    n0 = lib.skb_kernel_launches()
    audio.decode(files)
    torch.cuda.synchronize()
    return lib.skb_kernel_launches() - n0


def test_one_launch_per_call(matrix):
    assert _launches(matrix[2:3]) == 1
    assert _launches((matrix * 2)[:200]) == 1


def _flac(pcm16, rate=16000):
    return F.encode(pcm16, rate, 16, blocksize=1024)


def test_mixed_batch_in_input_order(matrix):
    rng = numpy.random.default_rng(7)
    flacs = [_flac(F.synth_pcm(rng, 3000 + 700 * i, 1 + i % 2, 16)) for i in range(4)]
    pcms = matrix[2::5]
    files = []
    for i in range(max(len(flacs), len(pcms))):
        files += ([flacs[i]] if i < len(flacs) else []) + ([pcms[i]] if i < len(pcms) else [])
    out, n, rates = audio.decode(files)
    parts = torch.split(out, n.tolist())
    fo, fn, fr = flac.decode(flacs)
    fparts = torch.split(fo, fn.tolist())
    k = 0
    for data, x, r in zip(files, parts, rates.tolist()):
        if flac.is_flac(data):
            assert torch.equal(x, fparts[k]) and r == fr[k]
            k += 1
        else:
            assert torch.equal(x, audio.decode([data])[0]) and r == R.decode(data)[0]
    assert k == len(flacs)
    assert _launches(files) == 4                                       # three FLAC launches and one PCM launch


def test_bad_files_are_named_exactly(tmp_path):
    rng = numpy.random.default_rng(8)
    v = R.synth(rng, 500, 1, "pcm", 2)
    good = {"a.wav": R.wav_bytes(v, 16000, "pcm", 2), "b.sph": R.sph_bytes(R.synth(rng, 500, 1, "ulaw", 1), 8000, "ulaw", 1),
            "c.flac": _flac(F.synth_pcm(rng, 4000, 1, 16))}
    offs = F.decode(good["c.flac"])[0]["frame_offsets"]
    corrupt_flac = bytearray(good["c.flac"])
    corrupt_flac[(offs[1] + offs[2]) // 2] ^= 0x10
    bad = {"rf64.wav": b"RF64" + good["a.wav"][4:], "adpcm.wav": good["a.wav"].replace(b"fmt \x10\x00\x00\x00\x01\x00", b"fmt \x10\x00\x00\x00\x02\x00"),
           "short.sph": R.sph_bytes(v, 8000, "pcm", 2)[:300], "junk.wav": b"not audio at all",
           "frame.flac": bytes(corrupt_flac), "shorten.sph": R.sph_bytes(v, 8000, "pcm,embedded-shorten-v2.00", 2)}
    paths = {}
    for name, data in list(good.items()) + list(bad.items()):
        paths[name] = os.path.join(str(tmp_path), name)
        with open(paths[name], "wb") as f:
            f.write(data)
    order = ["a.wav", "rf64.wav", "b.sph", "frame.flac", "adpcm.wav", "short.sph", "c.flac", "junk.wav", "shorten.sph"]
    with pytest.raises(ValueError) as e:
        audio.decode([paths[k] for k in order])
    named = {k for k in order if paths[k] in str(e.value)}
    assert named == set(bad), str(e.value)
    with pytest.raises(NotImplementedError) as e:                     # only unsupported formats: NotImplementedError
        audio.decode([paths["a.wav"], paths["rf64.wav"], paths["shorten.sph"]])
    assert paths["rf64.wav"] in str(e.value) and paths["shorten.sph"] in str(e.value) and paths["a.wav"] not in str(e.value)
    out, n, _ = audio.decode([paths[k] for k in good])                # the good files alone decode
    assert n.tolist() == [500, 500, 4000]
    with pytest.raises(FileNotFoundError, match="missing.wav"):       # a file that cannot be read keeps its OSError
        audio.decode([paths["a.wav"], os.path.join(str(tmp_path), "missing.wav")])
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------- the feed path, end to end
def _idmap(rows):
    im = sk.IdMap()
    im.leftids = numpy.array([r[0] for r in rows], dtype="|O")
    im.rightids = numpy.array([r[1] for r in rows], dtype="|O")
    im.start = numpy.array([r[2] for r in rows], dtype="|O")
    im.stop = numpy.array([r[3] for r in rows], dtype="|O")
    return im


def _pcm16(L, seed):
    return (synth.synth_wave(1, L, seed=seed)[0].numpy() * 32768.0).clip(-32768, 32767).astype(numpy.int64)[:, None]


def _lin2ulaw_codes(x16):
    """Nearest mu-law code of each int16 value (by search over the 256 expansions): realistic telephone-band codes."""
    table = R.ulaw2lin(numpy.arange(256)).astype(numpy.int64)
    order = numpy.argsort(table)
    k = numpy.clip(numpy.searchsorted(table[order], x16), 0, 255)
    return order[k].astype(numpy.uint8)


def test_sphere_ulaw_8k_idmapset_and_extract_embeddings(tmp_path):
    d = str(tmp_path)
    waves = {}
    for i, L in enumerate((32000, 40000, 25000)):
        codes = _lin2ulaw_codes(_pcm16(L, 700 + i)[:, 0])[:, None]
        data = R.sph_bytes(codes, 8000, "ulaw", 1)
        with open(os.path.join(d, "t%d.sph" % i), "wb") as f:
            f.write(data)
        waves["t%d" % i] = torch.from_numpy(R.decode(data)[1])
    m = make_xtractor("halfresnet34", 32, 256).cuda()
    whole = [("s%d" % i, "t%d" % i, None, None) for i in range(3)]
    ss = sk.nnet.extract_embeddings(_idmap(whole), m, d, torch.device("cuda"), win_duration=1.0, file_extension="sph")
    rs = sk.nnet.Resample(8000, 16000)
    ref = m.extract_varlen([rs(waves["t%d" % i].cuda()) for i in range(3)]).cpu().numpy()
    assert numpy.array_equal(ss.stat1, ref)
    # segments, at the files' own rate: IdMapSet items are the oracle's samples, and the embeddings those of the segments
    segs = [("s0", "t0", 100, 300), ("s1", "t1", 0, 50), ("s2", "t2", 200, 210), ("s1", "t1", 50, None)]
    ds = xsets.IdMapSet(_idmap(segs), d, "sph", sample_rate=8000, min_duration=1.0)
    cut = []
    for i, (_, f, a, b) in enumerate(segs):
        speech, _, _, s0, s1 = ds[i]
        if b is None:
            assert torch.equal(speech, waves[f])
            cut.append(waves[f])
        else:
            assert torch.equal(speech, waves[f][s0:s1])
            cut.append(waves[f][s0:s1])
    sg = sk.nnet.extract_embeddings(_idmap(segs), m, d, torch.device("cuda"), win_duration=1.0, file_extension="sph", sample_rate=8000)
    assert numpy.array_equal(sg.stat1, m.extract_varlen([c.cuda() for c in cut]).cpu().numpy())


@pytest.mark.parametrize("enc,nb,kind", [("float", 4, "wav"), ("pcm", 3, "wav"), ("alaw", 1, "wav"), ("float", 8, "wavex")])
def test_wav_encodings_extract_embeddings(tmp_path, enc, nb, kind):
    d = str(tmp_path)
    rng = numpy.random.default_rng(9)
    waves = []
    for i, L in enumerate((24000, 37000)):
        v = R.synth(rng, L, 2, enc, nb)
        if enc == "float":
            v = (synth.synth_wave(2, L, seed=40 + i).numpy().T * 0.5).astype(numpy.float32 if nb == 4 else numpy.float64)
        data = _file(kind, enc, nb, v)
        with open(os.path.join(d, "u%d.wav" % i), "wb") as f:
            f.write(data)
        waves.append(torch.from_numpy(R.decode(data)[1]).cuda())
    m = make_xtractor("halfresnet34", 32, 256).cuda()
    ss = sk.nnet.extract_embeddings(_idmap([("a", "u0", None, None), ("b", "u1", None, None)]), m, d, torch.device("cuda"),
                                    win_duration=1.0)
    assert numpy.array_equal(ss.stat1, m.extract_varlen(waves).cpu().numpy())


def _wav16(x16, rate):
    return R.wav_bytes(x16, rate, "pcm", 2)


def test_extract_xvectors_main_paths_and_pipes(tmp_path):
    """ark / scp from .sph / .wav of every encoding, as paths and as pipes declaring 0xFFFFFFFF data sizes, are byte-identical
    to the tables written from the same samples stored as 16-bit WAV."""
    from sidekit_b200 import extract_xvectors as X
    d = str(tmp_path)
    entries = []                                                       # (key, coded file, rate, int16 values, pipe?)
    x = _pcm16(30000, 801)
    entries.append(("a", R.sph_bytes(_lin2ulaw_codes(x[:, 0])[:, None], 8000, "ulaw", 1), 8000, True))
    entries.append(("b", R.sph_bytes(x, 16000, "pcm", 2, big_endian=True), 16000, False))
    entries.append(("c", R.wav_bytes(_pcm16(20000, 802), 16000, "pcm", 2, declared=0xFFFFFFFF), 16000, True))
    entries.append(("d", R.wav_bytes(R.synth(numpy.random.default_rng(3), 18000, 1, "alaw", 1), 16000, "alaw", 1), 16000, True))
    entries.append(("e", R.wav_bytes((_pcm16(22000, 803) * 256), 16000, "pcm", 3), 16000, False))
    entries.append(("f", R.wav_bytes(_pcm16(26000, 804).astype(numpy.float32) / 32768, 16000, "float", 4, declared=0xFFFFFFFF), 16000, True))
    coded, ref = [], []
    for key, data, rate, pipe in entries:
        ext = ".sph" if data[:4] == b"NIST" else ".wav"
        p = os.path.join(d, key + ext)
        with open(p, "wb") as f:
            f.write(data)
        x16 = numpy.round(R.decode(data)[1].astype(numpy.float64) * 32768).astype(numpy.int64)[:, None]
        assert numpy.array_equal(x16.astype(numpy.float32)[:, 0] / numpy.float32(32768), R.decode(data)[1])   # representable
        q = os.path.join(d, key + "_16.wav")
        with open(q, "wb") as f:
            f.write(_wav16(x16, rate))
        coded.append("%s cat %s |" % (key, p) if pipe else "%s %s" % (key, p))
        ref.append("%s %s" % (key, q))
        sig, sr = X.prepare(["cat", p, "|"] if pipe else p)
        assert sr == rate and numpy.array_equal(sig.numpy(), R.decode(data)[1])
    for name, lines in (("coded.scp", coded), ("ref.scp", ref)):
        with open(os.path.join(d, name), "w") as f:
            f.write("\n".join(lines) + "\n")
    m = make_xtractor("halfresnet34", 32, 256).cuda()
    out = os.path.join(d, "out", "xv.scp")
    os.makedirs(os.path.dirname(out))
    tables = []
    for scp in ("ref.scp", "coded.scp"):
        X.main(m, os.path.join(d, scp), out, "cuda")
        tables.append((open(out, "rb").read(), open(out[:-4] + ".ark", "rb").read()))
    assert tables[0] == tables[1]
    X.main(m, os.path.join(d, "coded.scp"), out, "cuda", window_audio_seconds=1.0)   # one decode call per small window
    assert (open(out, "rb").read(), open(out[:-4] + ".ark", "rb").read()) == tables[0]
