"""Audio input of the feed path, whatever the container: FLAC (``sidekit_b200.flac``), WAV and NIST SPHERE in every PCM
encoding (``sidekit_b200.pcm``).  Files are recognised by their first bytes, not by their names.

``decode`` is the batch entry point: a batch of mixed files goes to the device in one copy and is decoded by at most one
FLAC call and one PCM call, both writing into one packed output in input order.  ``read`` is the single-file reader with
``read_wav``'s contract: 16- and 32-bit PCM WAV is decoded on the host by ``read_wav`` itself, everything else on the
device.
"""
import io
import os
import struct

import numpy
import torch

from . import flac, pcm


def _name(src, i, names):
    if names is not None:
        return names[i]
    return src if isinstance(src, str) else "<bytes #%d>" % i


def _read(src):
    if isinstance(src, (bytes, bytearray, memoryview)):
        return bytes(src)
    with open(src, "rb") as f:
        return f.read()


def parse(data, name="<bytes>"):
    """``("flac", FlacInfo)`` or ``("pcm", PcmInfo)`` for the file held in ``data``; raises ``ValueError`` naming it when it
    is neither FLAC nor WAV nor NIST SPHERE, and whatever the container's parser raises."""
    if flac.is_flac(data):
        return "flac", flac.parse(data, name)
    if pcm.is_pcm(data):
        return "pcm", pcm.parse(data, name)
    raise ValueError("%s: not a FLAC, WAV or NIST SPHERE file" % name)


def length(kind, info):
    """(frames, sample rate) of a parsed file."""
    return (info.total_samples, info.sample_rate) if kind == "flac" else (info.frames, info.sample_rate)


def _align16(x):
    return (x + 15) & ~15


def no_frames(kind, info):
    """True for a FLAC stream whose metadata ends the file: ``decode`` names it ``"<name>: no frames"``."""
    return kind == "flac" and info.frames_end <= info.frames_begin


class Staging:
    """Host side of one decode call: the native calls' file tables and the files' frame / sample bytes in one pinned
    buffer, laid out as ``head`` (int64 rows of the caller's own device tables), FLAC table, PCM table, FLAC frame bytes,
    then each PCM file's sample bytes at a 16-byte boundary.  Files whose ``kind`` is None are left out."""

    def __init__(self, datas, kinds, infos, out_offsets, head=None):
        head = numpy.zeros((0,), numpy.int64) if head is None else numpy.ascontiguousarray(head, dtype=numpy.int64)
        self.fl = [i for i, k in enumerate(kinds) if k == "flac"]
        self.pc = [i for i, k in enumerate(kinds) if k == "pcm"]
        out_offsets = numpy.asarray(out_offsets, dtype=numpy.int64)
        fl_bytes = numpy.array([infos[i].frames_end - infos[i].frames_begin for i in self.fl], numpy.int64)
        pc_bytes = numpy.array([pcm.data_bytes(infos[i]) for i in self.pc], numpy.int64)
        self.fl_bytes = int(fl_bytes.sum())
        pc_begin = numpy.zeros(len(self.pc), numpy.int64)
        o = 0
        for k, nb in enumerate(pc_bytes.tolist()):
            pc_begin[k] = o
            o = _align16(o + nb)
        fl_table, self.n_slots = flac.table([infos[i] for i in self.fl], numpy.cumsum(fl_bytes) - fl_bytes, out_offsets[self.fl])
        pc_table, self.n_tiles = pcm.table([infos[i] for i in self.pc], pc_begin, out_offsets[self.pc])
        self.fl_table_at = head.nbytes
        self.pc_table_at = self.fl_table_at + fl_table.nbytes
        self.fl_at = self.pc_table_at + pc_table.nbytes
        self.pc_at = _align16(self.fl_at + self.fl_bytes)
        self.host = torch.empty(max(self.pc_at + o, 1), dtype=torch.uint8, pin_memory=True)
        hv = self.host.numpy()
        hv[:self.fl_table_at] = head.view(numpy.uint8)
        hv[self.fl_table_at:self.pc_table_at] = fl_table.view(numpy.uint8).reshape(-1)
        hv[self.pc_table_at:self.fl_at] = pc_table.view(numpy.uint8).reshape(-1)
        p = self.fl_at
        for i, nb in zip(self.fl, fl_bytes.tolist()):
            hv[p:p + nb] = numpy.frombuffer(datas[i], dtype=numpy.uint8, count=nb, offset=infos[i].frames_begin)
            p += nb
        for i, b0, nb in zip(self.pc, pc_begin.tolist(), pc_bytes.tolist()):
            hv[self.pc_at + b0:self.pc_at + b0 + nb] = numpy.frombuffer(datas[i], dtype=numpy.uint8, count=nb, offset=infos[i].data_begin)

    def launch(self, out, device):
        """The device side, on the current stream of ``device``: ONE host-to-device copy of the buffer, at most one FLAC and
        one PCM native call writing ``out`` (float32 CUDA tensor) at the offsets given to the constructor.  Returns
        ``(staged, status)``: the device copy (its first bytes are ``head``) and the FLAC calls' per-file status (device
        int32, None without FLAC files), to be read with ``flac_errors`` once the stream has run."""
        with torch.cuda.device(device):
            staged = self.host.to(device, non_blocking=True)
            base = staged.data_ptr()
            status = None
            if self.fl:
                status = flac.launch(device, base + self.fl_at, self.fl_bytes, base + self.fl_table_at, len(self.fl), self.n_slots,
                                     out.data_ptr())
            if self.pc:
                pcm.launch(base + self.pc_at, base + self.pc_table_at, len(self.pc), self.n_tiles, out.data_ptr())
        return staged, status

    def flac_errors(self, status, names):
        """``{file index: ValueError}`` for the FLAC files whose status (host int array) is not OK."""
        return {self.fl[k]: ValueError("corrupt FLAC: " + flac.status_errors([names[self.fl[k]]], status[k:k + 1])[0])
                for k in numpy.nonzero(status)[0]}


def decode(files, device=None, names=None):
    """Decode a batch of audio files (paths or bytes; FLAC, WAV or NIST SPHERE, mixed freely) on ``device`` (default: the
    current CUDA device).  ``names`` (optional) name the files in error messages instead of their paths.

    Returns ``(packed, lengths, sample_rates)`` as ``flac.decode`` does: ``packed`` a float32 CUDA tensor holding channel 0
    of every file back to back in input order, ``lengths`` and ``sample_rates`` int64 numpy arrays.  The files' sample or
    frame bytes go to the device in one copy from one pinned buffer, and at most one FLAC and one PCM native call are made.
    A file that cannot be decoded -- unknown, malformed, unsupported or corrupt -- does not stop the others: after the
    call, one exception names every such file (``NotImplementedError`` when all of them are unsupported formats,
    ``ValueError`` otherwise).  A file that cannot be opened or read raises its ``OSError`` before any decoding."""
    device = flac.device_of(device)
    files = list(files)
    if not files:
        return torch.empty(0, dtype=torch.float32, device=device), numpy.zeros(0, numpy.int64), numpy.zeros(0, numpy.int64)
    names = [_name(f, i, names) for i, f in enumerate(files)]
    datas = [_read(f) for f in files]
    kinds, infos, errors = [], [], {}
    for i, data in enumerate(datas):
        try:
            kind, info = parse(data, names[i])
        except (ValueError, NotImplementedError) as e:
            kind, info, errors[i] = None, None, e
        kinds.append(kind)
        infos.append(info)
    lengths = numpy.zeros(len(files), numpy.int64)
    rates = numpy.zeros(len(files), numpy.int64)
    for i, (kind, info) in enumerate(zip(kinds, infos)):
        if kind is not None:
            lengths[i], rates[i] = length(kind, info)
        if no_frames(kind, info):
            errors[i] = ValueError("%s: no frames" % names[i])
            kinds[i] = None
    staging = Staging(datas, kinds, infos, numpy.cumsum(lengths) - lengths)
    with torch.cuda.device(device):
        out = torch.empty(int(lengths.sum()), dtype=torch.float32, device=device)
    _, status = staging.launch(out, device)
    if status is not None:
        errors.update(staging.flac_errors(status.cpu().numpy(), names))
    if errors:
        kinds_of = {type(e) for e in errors.values()}
        raise (NotImplementedError if kinds_of == {NotImplementedError} else ValueError)(
            "; ".join(str(errors[i]) for i in sorted(errors)))
    return out, lengths, rates


_HEAD = 1 << 16          # bytes read to recognise a file before deciding how to read the rest


def _host_wav(path, name):
    """True when the file at ``path`` is complete 16- or 32-bit PCM WAV, judged from its first ``_HEAD`` bytes and its
    size (a header the first bytes do not hold is judged from the whole file, by the caller)."""
    with open(path, "rb") as f:
        head = f.read(_HEAD)
    if head[:4] != b"RIFF":
        return False
    try:
        return pcm.host_readable(pcm.parse(head, name, size=os.path.getsize(path)))
    except (ValueError, NotImplementedError, struct.error):
        return False


def read(src, frame_offset=0, num_frames=-1, name=None):
    """``read_wav``'s contract for any supported file (a path or bytes): ``(float32 CPU tensor (n,), sample_rate)``,
    channel 0, samples ``[frame_offset, frame_offset + num_frames)`` clamped to the file (``num_frames < 0``: to the end).
    Complete 16- and 32-bit PCM WAV goes through ``read_wav`` on the host (a path is read from the segment's first frame,
    not in full); every other format is decoded on the current CUDA device."""
    from .nnet.xsets import read_wav
    name = name or _name(src, 0, None)
    if isinstance(src, str) and _host_wav(src, name):
        return read_wav(src, frame_offset, num_frames)
    data = _read(src)
    kind, info = parse(data, name)
    if kind == "pcm" and pcm.host_readable(info):
        return read_wav(io.BytesIO(data), frame_offset, num_frames)
    out, _, rates = decode([data], names=[name])
    return flac.slice_samples(out, frame_offset, num_frames).cpu(), int(rates[0])
