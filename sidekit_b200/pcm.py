"""Uncompressed audio of the feed path: what ``torchaudio.load`` (sidekit/nnet/xsets.py:419-464) and ``soundfile.read``
(sidekit/bin/extract_xvectors.py:37-72) give for a WAV or NIST SPHERE file, decoded on the device (csrc/pcm.cu).

The host parses the container only (``parse``); no sample is touched here.  Supported:

- RIFF/WAVE with format tag 1 (8-bit unsigned, 16/24/32-bit signed PCM), 3 (32/64-bit IEEE float), 6 (A-law), 7 (mu-law)
  and 0xFFFE (EXTENSIBLE with a PCM or IEEE-float subformat), any channel count.  Chunks other than ``fmt `` and ``data``
  are skipped (odd-sized ones with their pad byte).  A ``data`` chunk whose declared size runs past the end of the stream
  (``0xFFFFFFFF``, as streaming writers declare on a pipe) is cut to the whole frames present.
- NIST SPHERE (``NIST_1A``): PCM (signed, 1-4 bytes), mu-law or A-law, either byte order.

RF64, RIFX, compressed WAV tags (ADPCM, GSM, ...) and shorten-compressed SPHERE raise ``NotImplementedError``; any other
malformed header raises ``ValueError``.  Both name the file.  Channel 0 comes out as float32 with the scaling of
``soundfile.read``: signed ``x / 2^(8 bytes - 1)``, unsigned 8-bit ``(x - 128) / 128``, float copied (float64 rounded),
G.711 expanded to 16 bits then ``/ 2^15``.
"""
import struct
from dataclasses import dataclass

import numpy

from . import _lib

# encodings, as the kernel's SKB_PCM_* codes
ENCODINGS = {"pcm": 0, "u8": 1, "float": 2, "ulaw": 3, "alaw": 4}
TILE = 256                          # frames per tile of skb_pcm_decode

# WAVE_FORMAT_EXTENSIBLE subformat GUIDs: the format tag followed by this fixed tail
_GUID_TAIL = b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"


@dataclass
class PcmInfo:
    sample_rate: int
    channels: int
    encoding: str            # "pcm" (signed), "u8", "float", "ulaw" or "alaw"
    bytes_per_sample: int
    big_endian: bool
    data_begin: int          # first byte of the first frame
    frames: int              # whole frames present
    container: str           # "wav" (format tag 1, 3, 6 or 7), "wavex" (EXTENSIBLE) or "sph"
    truncated: bool          # the declared data size runs past the end of the stream (the frames present are kept)


def _fmt_encoding(tag, bits, name):
    nbytes = (bits + 7) // 8
    if tag == 1:
        if not 1 <= nbytes <= 4:
            raise ValueError("%s: %d-bit PCM is invalid" % (name, bits))
        return ("u8" if nbytes == 1 else "pcm"), nbytes
    if tag == 3:
        if bits not in (32, 64):
            raise ValueError("%s: %d-bit IEEE float is invalid (32 or 64)" % (name, bits))
        return "float", nbytes
    if tag in (6, 7):
        if bits != 8:
            raise ValueError("%s: %d-bit G.711 is invalid (8)" % (name, bits))
        return ("alaw" if tag == 6 else "ulaw"), 1
    raise NotImplementedError("%s: compressed WAV format tag 0x%04x (ADPCM, GSM, MP3, ...) is not supported" % (name, tag))


def _parse_wav(data, name, n):
    fmt = None
    p = 12
    while True:
        if p + 8 > n:
            raise ValueError("%s: no data chunk" % name if fmt else "%s: no fmt chunk" % name)
        cid, size = data[p:p + 4], struct.unpack_from("<I", data, p + 4)[0]
        body = p + 8
        if cid == b"fmt ":
            if size < 16 or body + size > n:
                raise ValueError("%s: truncated fmt chunk" % name)
            tag, channels, rate, _, align, bits = struct.unpack_from("<HHIIHH", data, body)
            container = "wav"
            if tag == 0xFFFE:
                if size < 40:
                    raise ValueError("%s: EXTENSIBLE fmt chunk of %d bytes (40 needed)" % (name, size))
                guid = data[body + 24:body + 40]
                sub = struct.unpack_from("<H", guid)[0]
                if guid[2:] != _GUID_TAIL or sub not in (1, 3):
                    raise NotImplementedError("%s: EXTENSIBLE subformat %s is not supported (PCM or IEEE float)" % (name, guid.hex()))
                tag, container = sub, "wavex"
            encoding, nbytes = _fmt_encoding(tag, bits, name)
            if channels == 0:
                raise ValueError("%s: channel count is 0" % name)
            if rate == 0:
                raise ValueError("%s: sample rate is 0" % name)
            if align != channels * nbytes:
                raise ValueError("%s: block align %d does not match %d channels of %d bytes" % (name, align, channels, nbytes))
            fmt = (rate, channels, encoding, nbytes, container)
        elif cid == b"data":
            if fmt is None:
                raise ValueError("%s: data chunk before the fmt chunk" % name)
            rate, channels, encoding, nbytes, container = fmt
            avail = min(size, n - body)
            return PcmInfo(rate, channels, encoding, nbytes, False, body, avail // (channels * nbytes), container, size > n - body)
        p = body + size + (size & 1)


def _parse_sphere(data, name, n):
    end = data.find(b"\n", 8)
    try:
        head_size = int(data[8:end]) if end > 8 else -1
    except ValueError:
        raise ValueError("%s: bad SPHERE header size line" % name) from None
    if head_size < 16 or head_size > n:
        raise ValueError("%s: truncated SPHERE header (%d bytes declared, %d present)" % (name, head_size, n))
    fields = {}
    for line in data[end + 1:head_size].split(b"\n"):
        line = line.strip()
        if line == b"end_head":
            break
        parts = line.split(None, 2)
        if len(parts) < 3 or not parts[1].startswith(b"-"):
            continue
        key, typ, value = parts[0].decode("latin-1"), parts[1], parts[2]
        if typ.startswith(b"-s"):
            try:
                value = value[:int(typ[2:])]
            except ValueError:
                raise ValueError("%s: bad SPHERE field %r" % (name, line)) from None
            fields[key] = value.decode("latin-1")
        else:
            try:
                fields[key] = int(value) if typ == b"-i" else float(value)
            except ValueError:
                raise ValueError("%s: bad SPHERE field %r" % (name, line)) from None
    else:
        raise ValueError("%s: SPHERE header has no end_head" % name)
    coding = str(fields.get("sample_coding", "pcm")).lower()
    if "shorten" in coding:
        raise NotImplementedError("%s: shorten-compressed SPHERE is not supported; decompress it in the wav.scp entry, as "
                                  "Kaldi recipes do: 'sph2pipe -f wav %s |'" % (name, name))
    if coding.startswith("pcm"):
        encoding = "pcm"
    elif coding in ("ulaw", "mu-law"):
        encoding = "ulaw"
    elif coding == "alaw":
        encoding = "alaw"
    else:
        raise NotImplementedError("%s: SPHERE sample_coding %r is not supported" % (name, coding))
    rate = int(fields.get("sample_rate", 0))
    channels = int(fields.get("channel_count", 1))
    nbytes = int(fields.get("sample_n_bytes", 2 if encoding == "pcm" else 1))
    if rate <= 0:
        raise ValueError("%s: SPHERE sample_rate missing or 0" % name)
    if channels <= 0:
        raise ValueError("%s: SPHERE channel_count is %d" % (name, channels))
    if not 1 <= nbytes <= 4 or (encoding != "pcm" and nbytes != 1):
        raise ValueError("%s: SPHERE sample_n_bytes %d is invalid for %s" % (name, nbytes, encoding))
    order = str(fields.get("sample_byte_format", "")).strip()
    if nbytes > 1 and order not in ("01", "10"):
        raise ValueError("%s: SPHERE sample_byte_format %r does not give the byte order of %d-byte samples" % (name, order, nbytes))
    avail = (n - head_size) // (channels * nbytes)
    declared = int(fields.get("sample_count", avail))
    if declared < 0:
        raise ValueError("%s: SPHERE sample_count is negative" % name)
    return PcmInfo(rate, channels, encoding, nbytes, order == "10", head_size, min(declared, avail), "sph", declared > avail)


def parse(data, name="<bytes>", size=None):
    """Container parse of a WAV or NIST SPHERE file held in ``data`` (bytes) -> ``PcmInfo``; no sample is touched.
    ``size``: the length of the whole stream when ``data`` holds only its first bytes (then a header that runs past
    ``data`` raises ``struct.error``)."""
    if data[:4] in (b"RF64", b"RIFX"):
        raise NotImplementedError("%s: %s files are not supported" % (name, data[:4].decode()))
    if data[:4] == b"RIFF":
        if len(data) < 12 or data[8:12] != b"WAVE":
            raise ValueError("%s: RIFF file without a WAVE header" % name)
        return _parse_wav(data, name, len(data) if size is None else size)
    if data[:8] == b"NIST_1A\n":
        return _parse_sphere(data, name, len(data) if size is None else size)
    raise ValueError("%s: not a WAV or NIST SPHERE file" % name)


def is_pcm(data):
    """True when ``data`` (bytes) starts a RIFF/RF64/RIFX or NIST SPHERE header."""
    return data[:4] in (b"RIFF", b"RF64", b"RIFX") or data[:8] == b"NIST_1A\n"


def host_readable(info):
    """True for the files ``read_wav`` decodes on the host: complete 16- or 32-bit PCM WAV of format tag 1."""
    return info.container == "wav" and info.encoding == "pcm" and info.bytes_per_sample in (2, 4) and not info.truncated


def data_bytes(info):
    return info.frames * info.channels * info.bytes_per_sample


def table(infos, byte_offsets, out_offsets):
    """Rows of ``skb_pcm_decode``'s file table (int64, (n, 8)) and the tile total."""
    frames = numpy.array([i.frames for i in infos], dtype=numpy.int64)
    tiles = -(-frames // TILE)
    t = numpy.zeros((len(infos), 8), dtype=numpy.int64)
    t[:, 0], t[:, 1] = byte_offsets, frames
    t[:, 2] = [i.channels for i in infos]
    t[:, 3] = [ENCODINGS[i.encoding] for i in infos]
    t[:, 4] = [i.bytes_per_sample for i in infos]
    t[:, 5] = [int(i.big_endian) for i in infos]
    t[:, 6] = out_offsets
    t[:, 7] = numpy.cumsum(tiles) - tiles
    return t, int(tiles.sum())


def launch(bytes_ptr, table_ptr, n_files, n_tiles, out_ptr):
    """One ``skb_pcm_decode`` call on the current stream (no synchronisation)."""
    lib = _lib.lib()
    _lib.check(lib.skb_pcm_decode(bytes_ptr, table_ptr, n_files, n_tiles, out_ptr, _lib.stream_ptr()))
