"""FLAC input of the feed path: what ``torchaudio.load`` (sidekit/nnet/xsets.py:419-464) and ``soundfile.read``
(sidekit/bin/extract_xvectors.py:37-72) give for a ``.flac`` file, decoded on the device (csrc/flac.cu).

The host parses the container only (the ``fLaC`` marker, an optional leading ID3v2 tag and the metadata blocks, of which
STREAMINFO is required); frames are found, checked (CRC-8 and CRC-16, frame numbers, block sizes summing to STREAMINFO's
total) and decoded on the device, a whole batch of files in one call of three launches.  Channel 0 comes out as float32
``int / 2^(bps - 1)``, the scaling of ``torchaudio.load`` / ``soundfile.read``.  Up to 24 bits per sample; streams of
unknown length (total samples = 0) are not supported.
"""
from dataclasses import dataclass

import numpy
import torch

from . import _lib

_STATUS = {1: "no valid frame where the stream continues (bad header CRC-8, subframe or frame CRC-16, or truncated)",
           2: "frame or sample number out of sequence",
           3: "block sizes do not add up to STREAMINFO's total samples"}


@dataclass
class FlacInfo:
    sample_rate: int
    channels: int
    bits_per_sample: int
    min_blocksize: int
    max_blocksize: int
    total_samples: int
    frames_begin: int        # first byte after the metadata
    frames_end: int          # end of the file


def _name(src, i):
    return src if isinstance(src, str) else "<bytes #%d>" % i


def parse(data, name="<bytes>"):
    """Container parse of a FLAC stream held in ``data`` (bytes) -> ``FlacInfo``; no frame is touched."""
    n = len(data)
    p = 0
    if data[:3] == b"ID3":
        if n < 10:
            raise ValueError("%s: truncated ID3v2 tag" % name)
        p = 10 + ((data[6] & 0x7F) << 21 | (data[7] & 0x7F) << 14 | (data[8] & 0x7F) << 7 | (data[9] & 0x7F))
        p += 10 if data[5] & 0x10 else 0                         # footer
    if data[p:p + 4] != b"fLaC":
        raise ValueError("%s: not a FLAC stream (no fLaC marker)" % name)
    p += 4
    info, first, last = None, True, False
    while not last:
        if p + 4 > n:
            raise ValueError("%s: metadata runs past the end of the file" % name)
        last, btype, length = data[p] >> 7, data[p] & 0x7F, int.from_bytes(data[p + 1:p + 4], "big")
        if btype == 127:
            raise ValueError("%s: invalid metadata block type 127" % name)
        if p + 4 + length > n:
            raise ValueError("%s: metadata block runs past the end of the file" % name)
        if first:
            if btype != 0:
                raise ValueError("%s: STREAMINFO missing (first metadata block has type %d)" % (name, btype))
            if length < 34:
                raise ValueError("%s: STREAMINFO too short (%d bytes)" % (name, length))
            v = int.from_bytes(data[p + 4:p + 4 + 18], "big")       # 144 bits: everything before the MD5
            info = dict(min_bs=v >> 128, max_bs=(v >> 112) & 0xFFFF, rate=(v >> 44) & 0xFFFFF,
                        channels=((v >> 41) & 7) + 1, bps=((v >> 36) & 31) + 1, total=v & ((1 << 36) - 1))
        p += 4 + length
        first = False
    if info["rate"] == 0:
        raise ValueError("%s: STREAMINFO sample rate is 0" % name)
    if info["bps"] > 24:
        raise NotImplementedError("%s: %d bits per sample (up to 24 are supported)" % (name, info["bps"]))
    if info["bps"] < 4:
        raise ValueError("%s: STREAMINFO bits per sample %d is invalid" % (name, info["bps"]))
    if info["total"] == 0:
        raise NotImplementedError("%s: STREAMINFO total samples is 0 (streams of unknown length are not supported)" % name)
    return FlacInfo(info["rate"], info["channels"], info["bps"], info["min_bs"], info["max_bs"], info["total"], p, n)


def _read(src):
    if isinstance(src, (bytes, bytearray, memoryview)):
        return bytes(src)
    with open(src, "rb") as f:
        return f.read()


_work = {}          # device -> workspace tensor, grown when a call needs more


def _workspace(device, nbytes):
    w = _work.get(device)
    if w is None or w.numel() < nbytes:
        w = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _work[device] = w
    return w


def device_of(device):
    """``device`` (None: the current CUDA device) as a ``torch.device`` with an index; raises without CUDA."""
    if not torch.cuda.is_available():
        raise RuntimeError("sidekit_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def table(infos, byte_begin, out_begin):
    """Rows of ``skb_flac_decode``'s file table (int64, (n, 9)) for files whose frame bytes start at ``byte_begin`` of the
    byte buffer and whose samples go to ``out_begin`` of the output, and the frame-slot total."""
    nbytes = numpy.array([i.frames_end - i.frames_begin for i in infos], dtype=numpy.int64)
    totals = numpy.array([i.total_samples for i in infos], dtype=numpy.int64)
    # frame slots per file: an upper bound on its frame count (every frame but the last holds at least STREAMINFO's minimum
    # block size, and no frame is shorter than 10 bytes); a stream that needs more is corrupt
    min_bs = numpy.array([max(i.min_blocksize, 1) for i in infos], dtype=numpy.int64)
    caps = numpy.minimum(-(-totals // min_bs) + 1, nbytes // 10 + 1)
    t = numpy.zeros((len(infos), 9), dtype=numpy.int64)
    t[:, 0], t[:, 1] = byte_begin, numpy.asarray(byte_begin) + nbytes
    t[:, 2], t[:, 3] = out_begin, totals
    t[:, 4], t[:, 5] = numpy.cumsum(caps) - caps, caps
    t[:, 6] = [i.sample_rate for i in infos]
    t[:, 7] = [i.channels for i in infos]
    t[:, 8] = [i.bits_per_sample for i in infos]
    return t, int(caps.sum())


def launch(device, bytes_ptr, n_bytes, table_ptr, n_files, n_slots, out_ptr):
    """One ``skb_flac_decode`` call on the current stream of ``device``; returns the per-file status (device int32)."""
    lib = _lib.lib()
    status = torch.empty(n_files, dtype=torch.int32, device=device)
    work = _workspace(device, int(lib.skb_flac_workspace_bytes(n_bytes, n_files, n_slots)))
    _lib.check(lib.skb_flac_decode(bytes_ptr, n_bytes, table_ptr, n_files, n_slots, work.data_ptr(), work.numel(), out_ptr,
                                   status.data_ptr(), _lib.stream_ptr()))
    return status


def status_errors(names, status):
    """``["name: reason", ...]`` for the files whose status (host int array) is not OK."""
    return ["%s: %s" % (names[i], _STATUS.get(int(status[i]), "status %d" % status[i])) for i in numpy.nonzero(status)[0]]


def decode(files, device=None):
    """Decode a batch of FLAC files (paths or bytes) on ``device`` (default: the current CUDA device) in one native call.

    Returns ``(packed, lengths, sample_rates)``: ``packed`` a float32 CUDA tensor holding channel 0 of every file back to
    back, ``lengths`` (int64 numpy) the files' sample counts and ``sample_rates`` (int64 numpy) their rates.  The
    compressed bytes go to the device in one copy; a corrupt or truncated file raises ``ValueError`` naming every bad
    file of the call."""
    device = device_of(device)
    files = list(files)
    if not files:
        return torch.empty(0, dtype=torch.float32, device=device), numpy.zeros(0, numpy.int64), numpy.zeros(0, numpy.int64)
    names = [_name(f, i) for i, f in enumerate(files)]
    datas = [_read(f) for f in files]
    infos = [parse(d, nm) for d, nm in zip(datas, names)]
    nf = len(files)
    nbytes = numpy.array([i.frames_end - i.frames_begin for i in infos], dtype=numpy.int64)
    totals = numpy.array([i.total_samples for i in infos], dtype=numpy.int64)
    table_, n_slots = table(infos, numpy.cumsum(nbytes) - nbytes, numpy.cumsum(totals) - totals)
    n_bytes = int(nbytes.sum())
    if n_bytes == 0:
        raise ValueError("corrupt FLAC: " + "; ".join("%s: no frames" % nm for nm in names))
    # one pinned staging buffer, one host-to-device copy: the file table, then the frame bytes
    head = table_.nbytes
    host = torch.empty(head + n_bytes, dtype=torch.uint8, pin_memory=True)
    hv = host.numpy()
    hv[:head] = table_.view(numpy.uint8).reshape(-1)
    o = head
    for d, info in zip(datas, infos):
        hv[o:o + info.frames_end - info.frames_begin] = numpy.frombuffer(d, dtype=numpy.uint8, offset=info.frames_begin)
        o += info.frames_end - info.frames_begin
    with torch.cuda.device(device):
        staged = host.to(device, non_blocking=True)
        out = torch.empty(int(totals.sum()), dtype=torch.float32, device=device)
        st = launch(device, staged.data_ptr() + head, n_bytes, staged.data_ptr(), nf, n_slots, out.data_ptr()).cpu().numpy()
    bad = status_errors(names, st)
    if bad:
        raise ValueError("corrupt FLAC: " + "; ".join(bad))
    return out, totals, table_[:, 6].copy()


def read_flac(path, frame_offset=0, num_frames=-1):
    """``read_wav``'s contract for a FLAC file: ``(float32 CPU tensor (n,), sample_rate)``, channel 0, scaled
    ``int / 2^(bps - 1)``, samples ``[frame_offset, frame_offset + num_frames)`` (clamped to the file; ``num_frames < 0``:
    to the end).  Decoded on the current CUDA device."""
    out, lengths, rates = decode([path])
    return slice_samples(out, frame_offset, num_frames).cpu(), int(rates[0])


def slice_samples(x, frame_offset=0, num_frames=-1):
    """``x[frame_offset : frame_offset + num_frames]`` with ``read_wav``'s clamping."""
    total = int(x.shape[0])
    frame_offset = min(max(0, int(frame_offset)), total)
    n = total - frame_offset if num_frames is None or num_frames < 0 else min(int(num_frames), total - frame_offset)
    return x[frame_offset:frame_offset + n]


def is_flac(data):
    """True when ``data`` (bytes) starts a FLAC stream (``fLaC``, possibly behind an ID3v2 tag)."""
    return data[:4] == b"fLaC" or (data[:3] == b"ID3" and b"fLaC" in data[:1 << 16])
