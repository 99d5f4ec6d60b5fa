"""WAV / NIST SPHERE input of the feed path on the host: the container parser of sidekit_b200/pcm.py over every supported
container and encoding, its rejections, the numpy oracle of oracle/pcm_ref.py against scipy and audioop, and the
single-file reader's host path."""
import os
import struct
import warnings

import numpy
import pytest
import scipy.io.wavfile

from oracle import pcm_ref as R
from sidekit_b200 import audio, pcm
from sidekit_b200.nnet.xsets import read_wav

WAV_FORMATS = [("u8", 1), ("pcm", 2), ("pcm", 3), ("pcm", 4), ("float", 4), ("float", 8), ("ulaw", 1), ("alaw", 1)]


def _values(seed, frames, channels, enc, nb):
    return R.synth(numpy.random.default_rng(seed), frames, channels, enc, nb)


def test_g711_oracle_matches_audioop_on_every_code():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)
        import audioop
    codes = numpy.arange(256, dtype=numpy.uint8)
    for ref, mine in ((audioop.ulaw2lin, R.ulaw2lin), (audioop.alaw2lin, R.alaw2lin)):
        expected = numpy.frombuffer(ref(codes.tobytes(), 2), dtype="<i2")
        assert numpy.array_equal(mine(codes), expected)


SCIPY_FORMATS = [(enc, nb, ext) for enc, nb in WAV_FORMATS if enc in ("u8", "float") or nb in (2, 4) for ext in (False, True)
                 if not (ext and enc == "u8")]


@pytest.mark.parametrize("enc,nb,extensible", SCIPY_FORMATS)
@pytest.mark.parametrize("channels", [1, 2, 6])
def test_oracle_matches_scipy(tmp_path, enc, nb, extensible, channels):
    v = _values(7, 1001, channels, enc, nb)
    path = os.path.join(str(tmp_path), "x.wav")
    with open(path, "wb") as f:
        f.write(R.wav_bytes(v, 22050, enc, nb, extensible=extensible))
    rate, s = scipy.io.wavfile.read(path)
    s = s.reshape(len(s), -1)
    assert rate == 22050 and s.shape == v.shape and numpy.array_equal(s, v)
    with open(path, "rb") as f:
        r, x = R.decode(f.read())
    assert r == 22050 and numpy.array_equal(x, R.to_float(s[:, 0], enc, nb))


def _check(info, rate, channels, enc, nb, big, begin, frames, container, truncated=False):
    assert (info.sample_rate, info.channels, info.encoding, info.bytes_per_sample, info.big_endian, info.data_begin,
            info.frames, info.container, info.truncated) == (rate, channels, enc, nb, big, begin, frames, container, truncated)


@pytest.mark.parametrize("enc,nb", WAV_FORMATS)
@pytest.mark.parametrize("channels", [1, 2, 6])
@pytest.mark.parametrize("extensible", [False, True])
def test_parse_wav_matrix(enc, nb, channels, extensible):
    if extensible and enc in ("ulaw", "alaw"):
        return
    v = _values(3, 37, channels, enc, nb)
    data = R.wav_bytes(v, 44100, enc, nb, extensible=extensible)
    fmt_size = 40 if extensible else (16 if enc in ("pcm", "u8") else 18)
    info = pcm.parse(data, "x.wav")
    _check(info, 44100, channels, enc, nb, False, 12 + 8 + fmt_size + 8, 37, "wavex" if extensible else "wav")
    _, vals, e, b = R.decode_all(data)
    assert numpy.array_equal(vals, v) and (e, b) == (enc, nb)


def test_parse_skips_chunks_and_pad_bytes():
    v = _values(4, 11, 1, "pcm", 2)
    data = R.wav_bytes(v, 16000, "pcm", 2, before_data=[(b"LIST", b"INFOISFT\x05\x00\x00\x00abcd\x00"), (b"fact", b"\x0b\x00\x00\x00"),
                                                       (b"cue ", b"odd"), (b"junk", b"")])
    assert data.count(b"odd\x00junk") == 1                       # the odd-sized chunk is followed by its pad byte
    info = pcm.parse(data, "x.wav")
    assert info.data_begin == data.index(b"data") + 8 and info.frames == 11 and not info.truncated
    # fmt after an unknown chunk, and a chunk after data
    body = b"WAVE" + struct.pack("<4sI", b"bext", 3) + b"abc\x00" + data[12:] + b"LIST\x02\x00\x00\x00zz"
    info2 = pcm.parse(b"RIFF" + struct.pack("<I", len(body)) + body, "y.wav")
    assert info2.frames == 11 and info2.data_begin == info.data_begin + 12


def test_parse_data_size_past_the_end_is_cut_to_whole_frames():
    v = _values(5, 100, 2, "pcm", 3)
    data = R.wav_bytes(v, 8000, "pcm", 3, declared=0xFFFFFFFF)
    info = pcm.parse(data, "pipe")
    assert info.frames == 100 and info.truncated
    info = pcm.parse(data[:-4], "pipe")                            # a partial last frame is dropped
    assert info.frames == 99 and info.truncated
    assert pcm.parse(R.wav_bytes(v, 8000, "pcm", 3, declared=6 * 50), "p").frames == 50


@pytest.mark.parametrize("coding,enc,nb", [("pcm", "pcm", 2), ("pcm", "pcm", 1), ("pcm", "pcm", 3), ("pcm", "pcm", 4),
                                           ("ulaw", "ulaw", 1), ("mu-law", "ulaw", 1), ("alaw", "alaw", 1)])
@pytest.mark.parametrize("big", [False, True])
@pytest.mark.parametrize("channels", [1, 2])
def test_parse_sphere(coding, enc, nb, big, channels):
    v = _values(6, 53, channels, enc, nb)
    data = R.sph_bytes(v, 8000, coding, nb, big_endian=big)
    info = pcm.parse(data, "x.sph")
    _check(info, 8000, channels, enc, nb, big and nb > 1, 1024, 53, "sph")
    _, vals, e, b = R.decode_all(data)
    assert numpy.array_equal(vals, v) and (e, b) == (enc, nb)


def test_parse_sphere_defaults_and_short_data():
    v = _values(8, 20, 1, "pcm", 2)
    data = R.sph_bytes(v, 16000, "pcm", 2, fields={"sample_coding": ("-s%d", None), "channel_count": ("-i", None)})
    _check(pcm.parse(data, "x.sph"), 16000, 1, "pcm", 2, False, 1024, 20, "sph")
    data = R.sph_bytes(v, 16000, "pcm", 2, sample_count=1000)
    info = pcm.parse(data, "x.sph")
    assert info.frames == 20 and info.truncated


def _wav_with_fmt(fmt, data=b"\x00\x00"):
    body = b"WAVE" + R._chunk(b"fmt ", fmt) + R._chunk(b"data", data)
    return b"RIFF" + struct.pack("<I", len(body)) + body


def _rejections():
    v = _values(9, 8, 1, "pcm", 2)
    good = R.wav_bytes(v, 16000, "pcm", 2)
    ext = bytearray(R.wav_bytes(v, 16000, "pcm", 2, extensible=True))
    g = ext.index(R.EXT_GUID_TAIL)
    ext[g + 3] ^= 0xFF
    sph = R.sph_bytes(v, 8000, "pcm", 2)
    return {
        "rf64.wav": (b"RF64" + good[4:], NotImplementedError, "RF64"),
        "rifx.wav": (b"RIFX" + good[4:], NotImplementedError, "RIFX"),
        "adpcm.wav": (_wav_with_fmt(struct.pack("<HHIIHHH", 2, 1, 8000, 4000, 256, 4, 0)), NotImplementedError, "0x0002"),
        "gsm.wav": (_wav_with_fmt(struct.pack("<HHIIHHH", 0x31, 1, 8000, 1625, 65, 0, 0)), NotImplementedError, "0x0031"),
        "guid.wav": (bytes(ext), NotImplementedError, "subformat"),
        "shorten.sph": (R.sph_bytes(v, 8000, "pcm,embedded-shorten-v2.00", 2), NotImplementedError, "sph2pipe -f wav"),
        "noorder.sph": (R.sph_bytes(v, 8000, "pcm", 2, fields={"sample_byte_format": ("-s%d", None)}), ValueError, "byte order"),
        "truncated.wav": (good[:30], ValueError, "truncated fmt"),
        "tiny.wav": (good[:10], ValueError, "WAVE"),
        "truncated.sph": (sph[:500], ValueError, "truncated SPHERE header"),
        "nofmt.wav": (b"RIFF" + struct.pack("<I", 12) + b"WAVE" + R._chunk(b"data", b"\x00" * 4), ValueError, "before the fmt"),
        "nodata.wav": (good[:good.index(b"data")], ValueError, "no data chunk"),
        "rate0.wav": (_wav_with_fmt(struct.pack("<HHIIHH", 1, 1, 0, 0, 2, 16)), ValueError, "sample rate is 0"),
        "chan0.wav": (_wav_with_fmt(struct.pack("<HHIIHH", 1, 0, 8000, 0, 2, 16)), ValueError, "channel count is 0"),
        "align.wav": (_wav_with_fmt(struct.pack("<HHIIHH", 1, 2, 8000, 32000, 2, 16)), ValueError, "block align"),
        "float16.wav": (_wav_with_fmt(struct.pack("<HHIIHH", 3, 1, 8000, 16000, 2, 16)), ValueError, "IEEE float"),
        "rate0.sph": (R.sph_bytes(v, 0, "pcm", 2), ValueError, "sample_rate"),
        "garbage.wav": (b"hello world" * 4, ValueError, "not a WAV or NIST SPHERE"),
    }


@pytest.mark.parametrize("name", sorted(_rejections()))
def test_rejections_name_the_file(name):
    data, exc, what = _rejections()[name]
    with pytest.raises(exc) as e:
        pcm.parse(data, name)
    assert type(e.value) is exc and str(e.value).startswith(name + ":") and what in str(e.value), str(e.value)


def test_sniffing_by_content():
    v = _values(10, 5, 1, "pcm", 2)
    assert audio.parse(R.wav_bytes(v, 16000, "pcm", 2), "a")[0] == "pcm"
    assert audio.parse(R.sph_bytes(v, 16000, "pcm", 2), "a")[0] == "pcm"
    from oracle import flac_ref as F
    assert audio.parse(F.encode(numpy.zeros((16, 1), numpy.int64), 16000, 16), "a")[0] == "flac"
    with pytest.raises(ValueError, match="^junk.wav: not a FLAC, WAV or NIST SPHERE file"):
        audio.parse(b"\x00" * 64, "junk.wav")


@pytest.mark.parametrize("nb", [2, 4])
@pytest.mark.parametrize("channels", [1, 3])
def test_read_host_path_is_read_wav(tmp_path, nb, channels):
    """16- and 32-bit PCM WAV is read on the host by read_wav itself (no device needed); other encodings are not."""
    v = _values(11, 999, channels, "pcm", nb)
    path = os.path.join(str(tmp_path), "x.wav")
    with open(path, "wb") as f:
        f.write(R.wav_bytes(v, 16000, "pcm", nb))
    for off, n in ((0, -1), (100, 50), (990, 100), (2000, 5)):
        a, ra = audio.read(path, off, n)
        b, rb = read_wav(path, off, n)
        assert ra == rb == 16000 and a.dtype == b.dtype and numpy.array_equal(a.numpy(), b.numpy())
    assert numpy.array_equal(audio.read(path)[0].numpy(), R.decode(open(path, "rb").read())[1])
    assert pcm.host_readable(pcm.parse(R.wav_bytes(v, 16000, "pcm", nb), "x"))
    for other in (R.wav_bytes(v, 16000, "pcm", nb, extensible=True), R.wav_bytes(v, 16000, "pcm", nb, declared=0xFFFFFFFF),
                  R.sph_bytes(v, 16000, "pcm", nb), R.wav_bytes(_values(1, 9, 1, "pcm", 3), 16000, "pcm", 3)):
        assert not pcm.host_readable(pcm.parse(other, "x"))


def test_read_sniffs_a_wav_path_from_its_header(tmp_path):
    """A host-readable WAV path is recognised from its first bytes and read by read_wav from the segment on; a header
    that lies past those bytes is recognised from the whole file, with the same result."""
    v = _values(12, 70000, 2, "pcm", 2)
    near = os.path.join(str(tmp_path), "near.wav")
    far = os.path.join(str(tmp_path), "far.wav")
    with open(near, "wb") as f:
        f.write(R.wav_bytes(v, 16000, "pcm", 2))
    with open(far, "wb") as f:
        f.write(R.wav_bytes(v, 16000, "pcm", 2, before_data=[(b"LIST", b"x" * (audio._HEAD + 10))]))
    assert audio._host_wav(near, "near.wav") and not audio._host_wav(far, "far.wav")
    for path in (near, far):
        a, ra = audio.read(path, 60000, 500)
        b, rb = read_wav(near, 60000, 500)
        assert ra == rb and numpy.array_equal(a.numpy(), b.numpy())
