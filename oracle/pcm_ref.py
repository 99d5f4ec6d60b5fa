"""Test infrastructure for the WAV / NIST SPHERE input of the feed path (sidekit_b200/pcm.py, csrc/pcm.cu): writers for
every supported container and encoding, and a separately written numpy decoder of the files they produce.

``decode(data) -> (sample_rate, float32 channel 0)`` gives what ``soundfile.read`` / ``torchaudio.load`` give: signed
integers ``x / 2^(8 bytes - 1)`` (int32 rounded to float32 first), unsigned 8-bit ``(x - 128) / 128``, float32 as is,
float64 rounded to float32, G.711 expanded with the Sun g711.c arithmetic (``ulaw2lin`` / ``alaw2lin``) then ``/ 2^15``.
"""
import struct

import numpy

EXT_GUID_TAIL = b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"
WAV_TAGS = {"pcm": 1, "u8": 1, "float": 3, "alaw": 6, "ulaw": 7}


def ulaw2lin(codes):
    """G.711 mu-law codes (uint8) -> int16, Sun g711.c ``ulaw2linear``."""
    u = ~numpy.asarray(codes, numpy.int64) & 0xFF
    t = (((u & 0x0F) << 3) + 0x84) << ((u & 0x70) >> 4)
    return numpy.where(u & 0x80, 0x84 - t, t - 0x84).astype(numpy.int16)


def alaw2lin(codes):
    """G.711 A-law codes (uint8) -> int16, Sun g711.c ``alaw2linear``."""
    a = numpy.asarray(codes, numpy.int64) ^ 0x55
    t = (a & 0x0F) << 4
    seg = (a & 0x70) >> 4
    t = numpy.where(seg == 0, t + 8, (t + 0x108) << numpy.maximum(seg - 1, 0))
    return numpy.where(a & 0x80, t, -t).astype(numpy.int16)


def to_float(values, encoding, nbytes):
    """Sample values (any shape) -> float32 with the readers' scaling."""
    if encoding == "pcm":
        return values.astype(numpy.float32) / numpy.float32(2.0 ** (8 * nbytes - 1))
    if encoding == "u8":
        return (values.astype(numpy.float32) - numpy.float32(128)) / numpy.float32(128)
    if encoding == "float":
        return values.astype(numpy.float32)
    lin = ulaw2lin(values) if encoding == "ulaw" else alaw2lin(values)
    return lin.astype(numpy.float32) / numpy.float32(32768)


# ----------------------------------------------------------------------------- sample values and their bytes
def synth(rng, frames, channels, encoding, nbytes):
    """Random sample values (frames, channels) covering the full range of the encoding."""
    shape = (frames, channels)
    if encoding == "pcm":
        lo = -(1 << (8 * nbytes - 1))
        v = rng.integers(lo, -lo, size=shape, dtype=numpy.int64)
        if frames >= 2:
            v[0, 0], v[1, 0] = lo, -lo - 1                       # the extremes
        return v
    if encoding in ("u8", "ulaw", "alaw"):
        return rng.integers(0, 256, size=shape, dtype=numpy.int64).astype(numpy.uint8)
    dt = numpy.float32 if nbytes == 4 else numpy.float64
    return (rng.standard_normal(shape) * 0.3).astype(dt)


def sample_bytes(values, encoding, nbytes, big_endian=False):
    """Interleaved frame bytes of ``values`` (frames, channels)."""
    if encoding == "float":
        return values.astype((">" if big_endian else "<") + ("f4" if nbytes == 4 else "f8")).tobytes()
    v = values.astype(numpy.int64).reshape(-1)
    b = ((v[:, None] >> (8 * numpy.arange(nbytes))) & 0xFF).astype(numpy.uint8)
    return (b[:, ::-1] if big_endian else b).tobytes()


def _chunk(cid, body):
    return cid + struct.pack("<I", len(body)) + body + (b"\x00" if len(body) & 1 else b"")


def wav_bytes(values, rate, encoding, nbytes, extensible=False, before_data=(), declared=None):
    """A RIFF/WAVE file: ``fmt `` (EXTENSIBLE with ``extensible``), the ``(id, body)`` chunks of ``before_data``, then
    ``data``.  ``declared`` overrides the data chunk's size field (and sets the RIFF size to 0xFFFFFFFF, as a streaming
    writer does)."""
    channels = values.shape[1]
    tag = WAV_TAGS[encoding]
    bits = 8 * nbytes
    common = struct.pack("<HIIHH", channels, rate, rate * channels * nbytes, channels * nbytes, bits)
    if extensible:
        fmt = struct.pack("<H", 0xFFFE) + common + struct.pack("<HHI", 22, bits, 0) + struct.pack("<H", tag) + EXT_GUID_TAIL
    else:
        fmt = struct.pack("<H", tag) + common + (struct.pack("<H", 0) if tag != 1 else b"")
    body = b"WAVE" + _chunk(b"fmt ", fmt) + b"".join(_chunk(c, b) for c, b in before_data)
    data = sample_bytes(values, encoding, nbytes)
    if declared is None:
        body += _chunk(b"data", data)
        return b"RIFF" + struct.pack("<I", len(body)) + body
    return b"RIFF" + struct.pack("<I", 0xFFFFFFFF) + body + b"data" + struct.pack("<I", declared) + data


def sph_bytes(values, rate, coding, nbytes, big_endian=False, fields=None, sample_count=None):
    """A NIST SPHERE file (1024-byte header).  ``coding``: ``pcm``, ``ulaw``, ``mu-law`` or ``alaw``; ``fields`` adds or
    replaces header fields ({key: (type, value)}, value None drops the field)."""
    channels = values.shape[1]
    f = {"sample_count": ("-i", values.shape[0] if sample_count is None else sample_count), "sample_rate": ("-i", rate),
         "channel_count": ("-i", channels), "sample_n_bytes": ("-i", nbytes),
         "sample_byte_format": ("-s%d", "1" if nbytes == 1 else ("10" if big_endian else "01")), "sample_coding": ("-s%d", coding)}
    f.update(fields or {})
    lines = [b"NIST_1A", b"   1024"]
    for k, (t, v) in f.items():
        if v is None:
            continue
        if "%d" in t:
            t = t % len(str(v))
        lines.append(("%s %s %s" % (k, t, v)).encode())
    lines.append(b"end_head")
    head = b"\n".join(lines) + b"\n"
    head += b" " * (1024 - len(head))
    enc = "pcm" if coding == "pcm" else coding.replace("mu-law", "ulaw")
    return head + sample_bytes(values, enc, nbytes, big_endian)


# ----------------------------------------------------------------------------- decoder
def _decode_wav(data):
    p, fmt = 12, None
    while p + 8 <= len(data):
        cid, size = data[p:p + 4], struct.unpack("<I", data[p + 4:p + 8])[0]
        if cid == b"fmt ":
            tag, ch, rate, _, align, bits = struct.unpack("<HHIIHH", data[p + 8:p + 24])
            if tag == 0xFFFE:
                tag = struct.unpack("<H", data[p + 32:p + 34])[0]
            nb = bits // 8
            enc = {1: "u8" if nb == 1 else "pcm", 3: "float", 6: "alaw", 7: "ulaw"}[tag]
            fmt = (rate, ch, enc, nb)
        elif cid == b"data":
            rate, ch, enc, nb = fmt
            raw = data[p + 8:p + 8 + size]
            frames = len(raw) // (ch * nb)
            return rate, _values(raw[:frames * ch * nb], enc, nb, False, ch), enc, nb
        p += 8 + size + (size & 1)
    raise ValueError("no data chunk")


def _values(raw, enc, nb, big, ch):
    if enc == "float":
        v = numpy.frombuffer(raw, (">" if big else "<") + ("f4" if nb == 4 else "f8"))
    elif enc in ("u8", "ulaw", "alaw") or nb == 1:
        v = numpy.frombuffer(raw, numpy.uint8)
        if enc == "pcm":
            v = v.astype(numpy.int8)
    else:
        b = numpy.frombuffer(raw, numpy.uint8).reshape(-1, nb).astype(numpy.int64)
        if big:
            b = b[:, ::-1]
        v = (b << (8 * numpy.arange(nb))).sum(axis=1)
        v = numpy.where(v >= 1 << (8 * nb - 1), v - (1 << (8 * nb)), v)
    return v.reshape(-1, ch)


def _decode_sph(data):
    head = int(data[8:16].split(b"\n")[0])
    f = {}
    for line in data[:head].split(b"\n")[2:]:
        parts = line.split(None, 2)
        if parts == [b"end_head"]:
            break
        if len(parts) == 3:
            f[parts[0].decode()] = parts[2].decode()
    coding = f.get("sample_coding", "pcm").lower()
    enc = "ulaw" if coding in ("ulaw", "mu-law") else ("alaw" if coding == "alaw" else "pcm")
    nb, ch = int(f.get("sample_n_bytes", 2 if enc == "pcm" else 1)), int(f.get("channel_count", 1))
    frames = min(int(f["sample_count"]), (len(data) - head) // (nb * ch))
    raw = data[head:head + frames * nb * ch]
    return int(f["sample_rate"]), _values(raw, enc, nb, f.get("sample_byte_format") == "10", ch), enc, nb


def decode_all(data):
    """``(sample_rate, values (frames, channels), encoding, bytes per sample)`` of a WAV or SPHERE file."""
    return _decode_wav(data) if data[:4] == b"RIFF" else _decode_sph(data)


def decode(data):
    """``(sample_rate, float32 channel 0)`` of a WAV or SPHERE file."""
    rate, v, enc, nb = decode_all(data)
    return rate, to_float(v[:, 0], enc, nb)
