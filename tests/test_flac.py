"""FLAC input, CPU side: the CRCs against their published check values, a stream assembled bit by bit from RFC 9639,
the test encoder against the reference decoder over the tool matrix (oracle/flac_ref.py), the STREAMINFO MD5, and the
container parser of sidekit_b200.flac."""
import hashlib

import numpy
import pytest

from oracle import flac_ref as R
from sidekit_b200 import flac


def test_crc_check_values():
    assert R.crc8(b"123456789") == 0xF4            # CRC-8/SMBUS: poly 0x07, init 0, not reflected
    assert R.crc16(b"123456789") == 0xFEE8         # CRC-16/UMTS (BUYPASS): poly 0x8005, init 0, not reflected


def _bits(*fields):
    s = "".join(f.replace(" ", "") for f in fields)
    assert len(s) % 8 == 0 and set(s) <= {"0", "1"}
    return int(s, 2).to_bytes(len(s) // 8, "big")


def _frame(header_bits, body_bits):
    hdr = _bits(*header_bits)
    hdr += bytes([R.crc8(hdr)])                                  # section 9.1.8
    body = hdr + _bits(*body_bits)
    return body + R.crc16(body).to_bytes(2, "big")               # section 9.3


def hand_stream():
    """Two frames, 4 bits per sample (from STREAMINFO), 2 channels, 20 samples."""
    streaminfo = _bits(
        "0000000000010000",            # minimum block size 16 (section 8.2)
        "0000000000010000",            # maximum block size 16
        "000000000000000000000000",    # minimum frame size unknown
        "000000000000000000000000",    # maximum frame size unknown
        "00000011111010000000",        # sample rate 16000
        "001",                         # channels - 1
        "00011",                       # bits per sample - 1 = 3
        "000000000000000000000000000000010100")   # total samples 20
    md5 = bytes(16)                                              # unknown (section 8.2: all zeros allowed)
    meta = b"fLaC" + _bits("1", "0000000", "000000000000000000100010") + streaminfo + md5   # last block, STREAMINFO, 34 bytes
    frame0 = _frame(
        ["11111111111110", "0", "0",   # sync code, reserved, fixed blocking (section 9.1)
         "0110", "0000",               # block size: 8-bit (size - 1) follows; sample rate from STREAMINFO
         "1010", "000", "0",           # mid/side stereo; sample size from STREAMINFO; reserved
         "00000000",                   # coded frame number 0
         "00001111"],                  # block size - 1 = 15
        ["0", "000000", "0", "0011",   # subframe 0 (mid, 4 bits): CONSTANT 3, no wasted bits (section 9.2.3)
         "0", "000001", "0",           # subframe 1 (side, 4 + 1 bits): VERBATIM (section 9.2.4)
         "00000 00001 11111 00010 11110 00011 11101 00100 11100 00101 11011 00110 11010 00111 11001 00001",
         "0000"])                      # zero padding to the byte boundary
    frame1 = _frame(
        ["11111111111110", "0", "0",
         "0110", "0000",
         "0001", "000", "0",           # two independent channels
         "00000001",                   # coded frame number 1
         "00000011"],                  # block size - 1 = 3
        ["0", "001010", "1", "1",      # subframe 0: FIXED order 2, wasted bits flag, unary 0 -> 1 wasted bit (section 9.2.2)
         "001", "010",                 # warm-up 1, 2 (3 bits: 4 - 1 wasted)
         "00", "0000", "1111", "00011",  # residual: 4-bit parameters, partition order 0, escape code, 3-bit raw (9.2.7)
         "101", "000",                 # residuals -3, 0
         "0", "001001", "0",           # subframe 1: FIXED order 1, no wasted bits
         "0101",                       # warm-up 5
         "01", "0000", "00001",        # residual: 5-bit parameters, partition order 0, Rice parameter 1
         "010", "011", "00010",        # zigzag 2, 3, 6 = residuals 1, -2, 3
         "00"])
    return meta + frame0 + frame1


# mid = 3, side = the verbatim values: left = (((mid << 1) | (side & 1)) + side) >> 1, right = that - side ... >> 1
HAND_LEFT = [3, 4, 3, 4, 2, 5, 2, 5, 1, 6, 1, 6, 0, 7, 0, 4] + [2, 4, 0, -4]
HAND_RIGHT = [3, 3, 4, 2, 4, 2, 5, 1, 5, 1, 6, 0, 6, 0, 7, 3] + [5, 6, 4, 7]


def test_hand_assembled_stream():
    info, x = R.decode(hand_stream())
    assert (info["rate"], info["channels"], info["bps"], info["total"]) == (16000, 2, 4, 20)
    assert x[:, 0].tolist() == HAND_LEFT and x[:, 1].tolist() == HAND_RIGHT
    fi = flac.parse(hand_stream())
    assert (fi.sample_rate, fi.channels, fi.bits_per_sample, fi.total_samples) == (16000, 2, 4, 20)
    assert fi.frames_begin == 42


N_MATRIX = 48


@pytest.mark.parametrize("i", range(N_MATRIX))
def test_encoder_reference_decoder_round_trip(i):
    data, pcm, rate, bps = R.matrix_case(i)
    info, x = R.decode(data)
    assert numpy.array_equal(x, pcm)
    assert info["md5"] == R.pcm_md5(x, bps)                      # STREAMINFO MD5 = MD5 of the decoded PCM
    assert (info["rate"], info["bps"], info["channels"], info["total"]) == (rate, bps, pcm.shape[1], pcm.shape[0])
    fi = flac.parse(data)
    assert (fi.sample_rate, fi.channels, fi.bits_per_sample, fi.total_samples) == (rate, pcm.shape[1], bps, pcm.shape[0])
    assert (fi.min_blocksize, fi.max_blocksize) == (info["min_bs"], info["max_bs"])
    assert fi.frames_begin == info["frame_offsets"][0] and fi.frames_end == len(data)


def test_matrix_covers_every_tool():
    """the matrix above exercises every bit depth, channel count, blocking strategy, channel assignment, subframe type,
    residual method, escaped partition and wasted-bit case the decoder has to handle"""
    seen = set()
    for i in range(N_MATRIX):
        data, pcm, rate, bps = R.matrix_case(i)
        info, _ = R.decode(data)
        seen.add(("bps", bps))
        seen.add(("ch", pcm.shape[1]))
        for p in info["frame_offsets"]:
            seen.add(("variable", data[p + 1] & 1))
            seen.add(("assign", data[p + 3] >> 4))
            seen.add(("bs_code", data[p + 2] >> 4 in (6, 7)))
            seen.add(("rate_code", data[p + 2] & 15))
        seen.add(("short", pcm.shape[0] < 16))
    for bps in (8, 12, 16, 20, 24):
        assert ("bps", bps) in seen
    for ch in range(1, 9):
        assert ("ch", ch) in seen
    assert {("variable", 0), ("variable", 1), ("short", True), ("bs_code", True), ("bs_code", False)} <= seen
    assert {("assign", a) for a in (8, 9, 10)} <= seen
    assert {("rate_code", c) for c in (0, 5, 12, 13, 14)} <= seen


def test_md5_matches_hashlib_layout():
    pcm = numpy.array([[1, -1], [-32768, 32767]])
    raw = b"\x01\x00\xff\xff\x00\x80\xff\x7f"                     # interleaved little-endian 16-bit
    assert R.pcm_md5(pcm, 16) == hashlib.md5(raw).digest()


def _with_streaminfo(data, **fields):
    """data with STREAMINFO fields replaced (a stream without ID3 whose first block is STREAMINFO)"""
    b = bytearray(data)
    v = int.from_bytes(b[8:26], "big")
    if "total" in fields:
        v = (v & ~((1 << 36) - 1)) | fields["total"]
    if "bps" in fields:
        v = (v & ~(31 << 36)) | ((fields["bps"] - 1) << 36)
    b[8:26] = v.to_bytes(18, "big")
    return bytes(b)


def test_parser_skips_id3_and_unknown_blocks():
    rng = numpy.random.default_rng(3)
    pcm = R.synth_pcm(rng, 5000, 2, 16)
    plain = R.encode(pcm, 16000, 16, blocksize=1024)
    tagged = R.encode(pcm, 16000, 16, blocksize=1024, id3=b"\x00" * 37,
                      extra_blocks=[(1, bytes(100)), (4, b"\x05\x00\x00\x00hello\x00\x00\x00\x00"), (9, b"unknown"), (2, b"APPLdata")])
    a, b = flac.parse(plain), flac.parse(tagged)
    assert (a.sample_rate, a.channels, a.bits_per_sample, a.total_samples) == (b.sample_rate, b.channels, b.bits_per_sample, b.total_samples)
    assert plain[a.frames_begin:] == tagged[b.frames_begin:]
    assert numpy.array_equal(R.decode(tagged)[1], pcm)


def test_parser_rejects_bad_inputs():
    rng = numpy.random.default_rng(4)
    good = R.encode(R.synth_pcm(rng, 3000, 1, 16), 16000, 16, blocksize=1024)
    with pytest.raises(ValueError, match="bad.flac.*fLaC"):
        flac.parse(b"RIFF" + good[4:], "bad.flac")
    with pytest.raises(ValueError, match="x.flac.*STREAMINFO missing"):
        flac.parse(b"fLaC" + bytes([0x81, 0, 0, 4]) + bytes(4), "x.flac")                  # a lone PADDING block
    with pytest.raises(ValueError, match="STREAMINFO too short"):
        flac.parse(b"fLaC" + bytes([0x80, 0, 0, 20]) + bytes(20), "s.flac")
    with pytest.raises(ValueError, match="past the end"):
        flac.parse(good[:30], "cut.flac")
    with pytest.raises(NotImplementedError, match="z.flac.*unknown length"):
        flac.parse(_with_streaminfo(good, total=0), "z.flac")
    with pytest.raises(NotImplementedError, match="w.flac.*32 bits"):
        flac.parse(_with_streaminfo(good, bps=32), "w.flac")
    assert flac.parse(_with_streaminfo(good, bps=24)).bits_per_sample == 24


def test_slice_samples_clamps_like_read_wav():
    x = numpy.arange(10)
    assert flac.slice_samples(x, 3, 4).tolist() == [3, 4, 5, 6]
    assert flac.slice_samples(x, 8, 5).tolist() == [8, 9]
    assert flac.slice_samples(x, 12).tolist() == [] and flac.slice_samples(x, -2, 2).tolist() == [0, 1]
