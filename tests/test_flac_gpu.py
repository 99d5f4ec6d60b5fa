"""FLAC decoding on the device (csrc/flac.cu through sidekit_b200.flac) against the reference decoder of
oracle/flac_ref.py, bit for bit; corrupt streams; and the feed path (IdMapSet, extract_embeddings, extract_xvectors.main)
on .flac files against the same audio as 16-bit .wav."""
import os
import wave

import numpy
import pytest
import torch

import sidekit_b200 as sk
from oracle import flac_ref as R
from sidekit_b200 import _lib, flac, synth
from sidekit_b200.nnet import xsets
from tests.models import make_xtractor
from tests.test_flac import HAND_LEFT, hand_stream

pytestmark = pytest.mark.gpu

N_BATCH = 210


def _expected(pcm, bps):
    return (pcm[:, 0].astype(numpy.float32) / numpy.float32(2 ** (bps - 1))).astype(numpy.float32)


@pytest.fixture(scope="module")
def matrix():
    return [R.matrix_case(i, seed=1) for i in range(N_BATCH)]


def test_hand_assembled_stream_on_device():
    out, n, rates = flac.decode([hand_stream()])
    assert n.tolist() == [20] and rates.tolist() == [16000]
    assert numpy.array_equal(out.cpu().numpy(), numpy.array(HAND_LEFT, numpy.float32) / 8)


def test_exact_decode_batch_and_alone(matrix):
    datas = [m[0] for m in matrix]
    out, n, rates = flac.decode(datas)
    parts = torch.split(out, n.tolist())
    for (data, pcm, rate, bps), x, r in zip(matrix, parts, rates.tolist()):
        ref = _expected(R.decode(data)[1], bps)
        assert numpy.array_equal(ref, _expected(pcm, bps))
        assert r == rate and numpy.array_equal(x.cpu().numpy(), ref)
    for (data, pcm, rate, bps), x in zip(matrix, parts):
        alone, _, _ = flac.decode([data])
        assert torch.equal(alone, x)                                  # bit-identical whatever the batch


def test_launch_count_independent_of_file_count(matrix):
    lib = _lib.lib()
    counts = []
    for k in (1, 200):
        torch.cuda.synchronize()
        n0 = lib.skb_kernel_launches()
        flac.decode([m[0] for m in matrix[:k]])
        counts.append(lib.skb_kernel_launches() - n0)
    assert counts[0] == counts[1] == 3


def _corrupt_set(tmp_path):
    rng = numpy.random.default_rng(11)
    good = []
    for i in range(4):
        pcm = R.synth_pcm(rng, 6000 + 500 * i, 1 + i % 2, 16)
        good.append((R.encode(pcm, 16000, 16, blocksize=1024), pcm))
    data = good[0][0]
    offs = R.decode(data)[0]["frame_offsets"]
    b = bytearray(data)
    b[(offs[2] + offs[3]) // 2] ^= 0x10                               # a bit in the residual of frame 2
    residual = bytes(b)
    b = bytearray(data)
    b[offs[1] + 4] ^= 0x01                                            # the coded frame number of frame 1
    header = bytes(b)
    truncated = data[:len(data) - 300]
    garbage = data[:offs[2]] + bytes(rng.integers(0, 256, 77, dtype=numpy.uint8)) + data[offs[2]:]
    # a VERBATIM subframe whose samples spell a frame header with a valid CRC-8 (8-bit mono: one byte per sample)
    pcm8 = R.synth_pcm(rng, 1024, 1, 8)
    fake = bytearray([0xFF, 0xF8, 0x80, 0x02, 0x02])
    fake.append(R.crc8(fake))
    pcm8[40:46, 0] = numpy.frombuffer(bytes(fake), dtype=numpy.int8)
    trap = R.encode(pcm8, 16000, 8, blocksize=256, plan=lambda k: R.FramePlan(size_code="explicit", subs=[R.SubPlan(kind="verbatim")]))
    assert bytes(fake) in trap[trap.index(b"\xff\xf8") + 6:]
    files = {"good0.flac": good[1][0], "residual.flac": residual, "good1.flac": good[2][0], "header.flac": header,
             "truncated.flac": truncated, "garbage.flac": garbage, "trap.flac": trap, "good2.flac": good[3][0]}
    paths = {}
    for name, d in files.items():
        paths[name] = os.path.join(str(tmp_path), name)
        with open(paths[name], "wb") as f:
            f.write(d)
    return paths, pcm8


def test_corrupt_streams_are_named(tmp_path):
    paths, pcm8 = _corrupt_set(tmp_path)
    bad = {"residual.flac", "header.flac", "truncated.flac", "garbage.flac"}
    with pytest.raises(ValueError) as e:
        flac.decode(list(paths.values()))
    named = {os.path.basename(p) for p in paths.values() if p in str(e.value)}
    assert named == bad, str(e.value)
    for name in bad:
        with pytest.raises(ValueError, match=name):
            flac.decode([paths[name]])
    out, _, _ = flac.decode([paths["trap.flac"]])                    # the fake header inside the data is not a frame
    assert numpy.array_equal(out.cpu().numpy(), _expected(pcm8, 8))
    torch.cuda.synchronize()


def _write_pair(d, name, pcm16, rate=16000):
    with wave.open(os.path.join(d, name + ".wav"), "wb") as f:
        f.setnchannels(1); f.setsampwidth(2); f.setframerate(rate)
        f.writeframes(pcm16.astype("<i2").tobytes())
    with open(os.path.join(d, name + ".flac"), "wb") as f:
        f.write(R.encode(pcm16, rate, 16, blocksize=4096, plan=lambda k: R.FramePlan(subs=[R.SubPlan(order=8, porder=4)])))


def _pcm(L, seed):
    return (synth.synth_wave(1, L, seed=seed)[0].numpy() * 32768.0).clip(-32768, 32767).astype(numpy.int16)


def _idmap(rows):
    im = sk.IdMap()
    im.leftids = numpy.array([r[0] for r in rows], dtype="|O")
    im.rightids = numpy.array([r[1] for r in rows], dtype="|O")
    im.start = numpy.array([r[2] for r in rows], dtype="|O")
    im.stop = numpy.array([r[3] for r in rows], dtype="|O")
    return im


def test_idmapset_and_extract_embeddings_flac_equal_wav(tmp_path):
    d = str(tmp_path)
    for i, L in enumerate((64000, 80000, 50000)):
        _write_pair(d, "f%d" % i, _pcm(L, 900 + i))
    rows = [("spk0", "f0", None, None), ("spk1", "f1", 100, 450), ("spk1", "f1", 200, 260), ("spk2", "f2", 0, 20),
            ("spk0", "f0", 50, None)]
    dw = xsets.IdMapSet(_idmap(rows), d, "wav", min_duration=1.0)
    df = xsets.IdMapSet(_idmap(rows), d, "flac", min_duration=1.0)
    for i in range(len(rows)):
        a, b = dw[i], df[i]
        assert a[1:] == b[1:] and torch.equal(a[0], b[0].cpu())
    m = make_xtractor("halfresnet34", 32, 256).cuda()
    sw = sk.nnet.extract_embeddings(_idmap(rows), m, d, torch.device("cuda"), win_duration=1.0)
    sf = sk.nnet.extract_embeddings(_idmap(rows), m, d, torch.device("cuda"), win_duration=1.0, file_extension="flac")
    assert numpy.array_equal(sw.stat1, sf.stat1) and numpy.array_equal(sw.start, sf.start) and numpy.array_equal(sw.stop, sf.stop)
    assert list(sw.segset) == list(sf.segset)


def test_48k_24bit_stereo_flac(tmp_path):
    rng = numpy.random.default_rng(21)
    pcm = R.synth_pcm(rng, 96000, 2, 24)
    with open(os.path.join(str(tmp_path), "hi.flac"), "wb") as f:
        f.write(R.encode(pcm, 48000, 24, blocksize=4608, plan=lambda k: R.FramePlan(assign="mid_side", subs=[R.SubPlan(order=12, precision=15)] * 2)))
    m = make_xtractor("halfresnet34", 32, 256).cuda()
    ss = sk.nnet.extract_embeddings(_idmap([("s", "hi", None, None)]), m, str(tmp_path), torch.device("cuda"), win_duration=1.0,
                                    file_extension="flac")
    x = torch.from_numpy(pcm[:, 0].astype(numpy.float32) / numpy.float32(2 ** 23)).cuda()
    ref = m.extract_varlen([sk.nnet.Resample(48000, 16000)(x)]).cpu().numpy()
    assert numpy.array_equal(ss.stat1, ref)


def test_extract_xvectors_main_flac_equals_wav(tmp_path):
    from sidekit_b200 import extract_xvectors as X
    d = str(tmp_path)
    for i, L in enumerate((40000, 56000, 30000)):
        _write_pair(d, "u%d" % i, _pcm(L, 950 + i))
    with open(os.path.join(d, "wav.scp"), "w") as f:
        f.write("a %s/u0.wav\nb %s/u1.wav\nc cat %s/u2.wav |\n" % (d, d, d))
    with open(os.path.join(d, "flac.scp"), "w") as f:
        f.write("a %s/u0.flac\nb cat %s/u1.flac |\nc cat %s/u2.flac |\n" % (d, d, d))
    sig, sr = X.prepare(["cat", os.path.join(d, "u1.flac"), "|"])
    assert sr == 16000 and numpy.array_equal(sig.numpy(), X.prepare(os.path.join(d, "u1.wav"))[0].numpy())
    m = make_xtractor("halfresnet34", 32, 256).cuda()
    out = os.path.join(d, "out", "xv.scp")
    os.makedirs(os.path.dirname(out))
    tables = []
    for scp in ("wav.scp", "flac.scp"):
        X.main(m, os.path.join(d, scp), out, "cuda")
        tables.append((open(out, "rb").read(), open(out[:-4] + ".ark", "rb").read()))
    assert tables[0] == tables[1]
