"""Corpus extraction from files on every rank of a process group: the window pipeline that ``extract_xvectors.main`` and
``nnet.extract_embeddings`` share.

* **Sharding** (``plan_blocks``): the entry list is cut into one contiguous block per rank, balanced by file size
  (``entry_weights``).  Like ``bulk.plan_shards`` the plan is a pure function of the inputs and the world size, so no
  index is exchanged; rank 0's block comes first, so it can write its rows in input order as they are produced, and a
  rank opens (or runs, for a pipe) only the entries of its own block.
* **Windows** (``run_windows``): a rank's entries are processed in windows of ``window_audio_seconds`` of audio.  One
  background thread reads and parses window k+1 (pipe commands run there, in input order) and stages it in pinned memory
  while window k is on the device; at most one window is read ahead, so host memory holds two windows.  The device side
  of a window is enqueued without a synchronisation, and the host writes window k's rows while window k+1 runs.
* **Exchange** (``exchange``): after its windows, every rank shares its error (or None) and a small payload in ONE
  ``all_gather_object``, so that a bad entry on any rank makes every rank raise, naming it, instead of leaving the others
  waiting in the embedding gather.

The device work of a window is passed in (``prepare_fn`` / ``embed_fn``), the way ``bulk`` takes ``extract_fn``, so the
host logic runs on the CPU with a stub.
"""
import os
import queue
import threading
import time

import numpy
import torch

from . import audio


def entry_weights(paths):
    """Balancing weight of every entry: its file size (``os.stat``).  ``None`` stands for an entry without a file (a pipe
    command); it weighs the median known size, or one unit when no size is known.  A file that cannot be stat'ed weighs
    the same (its rank reports the error when it reads it)."""
    sizes = []
    for p in paths:
        try:
            sizes.append(None if p is None else float(os.stat(p).st_size))
        except OSError:
            sizes.append(None)
    known = [s for s in sizes if s is not None]
    fill = float(numpy.median(known)) if known else 1.0
    return numpy.maximum(numpy.array([fill if s is None else s for s in sizes], dtype=numpy.float64), 1.0)


def plan_blocks(weights, world_size):
    """``world_size`` contiguous ``(begin, end)`` blocks covering the entries in order, rank r's block r.  Every boundary is
    the entry boundary nearest to ``r / world_size`` of the total weight, so a block's weight is within the largest
    entry's weight of the mean.  Ranks past the last entry get empty blocks."""
    w = numpy.asarray(weights, dtype=numpy.float64)
    c = numpy.concatenate([[0.0], numpy.cumsum(w)])
    bounds = [0]
    for r in range(1, world_size):
        t = c[-1] * r / world_size
        i = int(numpy.searchsorted(c, t, side="left"))
        if i > 0 and t - c[i - 1] <= c[i] - t:
            i -= 1
        bounds.append(max(i, bounds[-1]))
    bounds.append(w.shape[0])
    return [(bounds[r], bounds[r + 1]) for r in range(world_size)]


def read_file(path):
    """``(path, bytes)`` of a file."""
    with open(path, "rb") as f:
        return path, f.read()


def parse_entry(name, data):
    """``(kind, info)`` of one file's bytes, as ``audio.decode`` judges them (``ValueError`` / ``NotImplementedError``
    naming the file)."""
    kind, info = audio.parse(data, name)
    if audio.no_frames(kind, info):
        raise ValueError("%s: no frames" % name)
    return kind, info


class Window:
    """Entries of one window: their positions in the rank's list, names, bytes and parsed headers; ``error`` is the
    exception that ended the rank's stream at the entry after the last one here (then the window is not processed);
    ``prepared`` is what ``prepare_fn`` made of it; ``stats`` the host seconds spent on it."""

    def __init__(self):
        self.index, self.names, self.datas, self.kinds, self.infos = [], [], [], [], []
        self.frames, self.rates = [], []
        self.error = None
        self.prepared = None
        self.stats = {"read_s": 0.0, "parse_s": 0.0, "stage_s": 0.0}

    def __len__(self):
        return len(self.index)


def read_windows(items, read_fn, window_audio_seconds, prepare_fn=None, parse_fn=parse_entry):
    """Generator of the ``Window`` s of ``items``, read on a background thread one window ahead.

    ``read_fn(item) -> (name, bytes)`` reads an entry, ``parse_fn(name, bytes) -> (kind, info)`` parses it, and
    ``prepare_fn(window)`` (optional) sets ``window.prepared`` on the same thread.  A window closes once its entries hold
    ``window_audio_seconds`` of audio.  The first entry that fails to read or parse ends the stream: the window in
    progress is yielded with that ``error`` and without the failing entry."""
    q = queue.Queue(maxsize=1)
    stop = threading.Event()

    def put(x):
        q.put(x)
        q.join()                 # the consumer has taken it: only then read the next window

    def close(win):
        if prepare_fn is not None and win.error is None and len(win):
            t0 = time.perf_counter()
            try:
                prepare_fn(win)
            except Exception as e:           # surfaces on the consumer's side like a read error
                win.error = e
            win.stats["stage_s"] += time.perf_counter() - t0
        put(win)

    def work():
        try:
            win, seconds = Window(), 0.0
            for i, item in enumerate(items):
                if stop.is_set():
                    return
                t0 = time.perf_counter()
                try:
                    name, data = read_fn(item)
                    t1 = time.perf_counter()
                    kind, info = parse_fn(name, data)
                except Exception as e:
                    win.error = e
                    break
                t2 = time.perf_counter()
                win.stats["read_s"] += t1 - t0
                win.stats["parse_s"] += t2 - t1
                frames, sr = audio.length(kind, info)
                for field, v in zip(("index", "names", "datas", "kinds", "infos", "frames", "rates"), (i, name, data, kind, info, frames, sr)):
                    getattr(win, field).append(v)
                seconds += float(frames) / sr
                if seconds >= window_audio_seconds:
                    close(win)
                    win, seconds = Window(), 0.0
            if len(win) or win.error is not None:
                close(win)
        except Exception as e:                   # never end the stream silently
            win = Window()
            win.error = e
            put(win)
        finally:
            if not stop.is_set():
                put(None)

    thread = threading.Thread(target=work, daemon=True)
    thread.start()
    try:
        while True:
            win = q.get()
            q.task_done()
            if win is None:
                return
            yield win
    finally:
        stop.set()
        while thread.is_alive():
            try:
                q.get(timeout=0.05)
                q.task_done()
            except queue.Empty:
                pass
        thread.join()


def run_windows(items, read_fn, window_audio_seconds, embed_fn, emit_fn, prepare_fn=None, parse_fn=parse_entry, stats=None):
    """The window pipeline of one rank.  ``embed_fn(window)`` enqueues the window's device work and returns a function
    that waits for it and returns its rows (host tensor); ``emit_fn(window, rows)`` takes them in window order.  Window
    k's rows are emitted while window k+1 runs on the device.  The first error raises after the windows before the
    failing entry's window have been emitted.

    ``stats`` (a list, optional) receives one dict per window: the host seconds of reading, parsing and staging (on the
    reading thread), ``wait_s`` (the main thread waiting for the reading thread), and with CUDA ``device_s`` (device
    time from the window's first launch to its last kernel, CUDA events) and ``files`` / ``audio_s``."""
    timing = stats is not None and torch.cuda.is_available()
    done = None                          # (window, rows) emitted once the next window is on the device
    windows = read_windows(items, read_fn, window_audio_seconds, prepare_fn, parse_fn)
    try:
        while True:
            t0 = time.perf_counter()
            win = next(windows, None)
            wait = time.perf_counter() - t0
            if win is None or win.error is not None:
                if done is not None:
                    emit_fn(*done)
                if win is None:
                    return
                raise win.error
            if timing:
                ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev[0].record()
            try:
                finish = embed_fn(win)
            except Exception:
                if done is not None:                      # the windows before the failing one are emitted
                    emit_fn(*done)
                raise
            if timing:
                ev[1].record()
            if done is not None:
                emit_fn(*done)
            done = (win, finish())
            if stats is not None:
                s = dict(win.stats, wait_s=wait, files=len(win), audio_s=float(sum(f / r for f, r in zip(win.frames, win.rates))))
                if timing:
                    s["device_s"] = ev[0].elapsed_time(ev[1]) / 1e3
                stats.append(s)
            win.datas = win.prepared = None       # the window's bytes are on the device or done with
    finally:
        windows.close()


def extract_sharded(items, weights, read_fn, embed_fn, embedding_size, window_audio_seconds, prepare_fn=None, emit_fn=None,
                    parse_fn=parse_entry, device=None, stats=None):
    """One row per item on every rank, in input order: ``(rows (n, E) float32 host tensor, blocks)``.

    This rank embeds its block of ``plan_blocks(weights, world)`` through ``run_windows`` (``emit_fn(indices, rows)``, if
    given, sees its rows window by window, with their positions in ``items``), then ONE ``exchange`` of errors and ONE
    ``bulk.gather_embeddings`` of the blocks (on ``device``; None: the collective's default).  Without a process group
    this is ``run_windows`` over all items."""
    from . import bulk
    dist, rank, world = bulk._dist()
    blocks = plan_blocks(weights, world)
    lo, hi = blocks[rank]
    parts = []

    def emit(win, rows):
        parts.append(rows)
        if emit_fn is not None:
            emit_fn([lo + i for i in win.index], rows)
    error = None
    try:
        run_windows(items[lo:hi], read_fn, window_audio_seconds, embed_fn, emit, prepare_fn, parse_fn, stats)
    except Exception as e:
        if dist is None:
            raise
        error = e
    local = torch.cat(parts) if parts else torch.zeros((0, embedding_size), dtype=torch.float32)
    if dist is None:
        return local, blocks
    exchange(error, None)
    return bulk.gather_embeddings(local, [numpy.arange(a, b) for a, b in blocks], embedding_size, device).cpu(), blocks


_RAISE_AS = {"OSError": OSError, "FileNotFoundError": OSError, "PermissionError": OSError, "IsADirectoryError": OSError,
             "ValueError": ValueError, "NotImplementedError": NotImplementedError}


def exchange(error, payload):
    """ONE ``all_gather_object`` of ``(error, payload)`` over the ranks of the current process group; returns every rank's
    payload.  When any rank passes an error, every rank raises one exception naming each rank's error: ``IOError`` if
    one of them is an ``OSError``, ``NotImplementedError`` if all of them are, else ``ValueError`` (or ``RuntimeError``
    for errors of other kinds).  Without a process group: re-raises ``error`` or returns ``[payload]``."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        if error is not None:
            raise error
        return [payload]
    mine = (None if error is None else (type(error).__name__, isinstance(error, OSError), str(error)), payload)
    everyone = [None] * dist.get_world_size()
    dist.all_gather_object(everyone, mine)
    bad = [(r, e) for r, (e, _) in enumerate(everyone) if e is not None]
    if bad:
        kinds = {_RAISE_AS.get(name, OSError if is_os else RuntimeError) for _, (name, is_os, _) in bad}
        kind = OSError if OSError in kinds else kinds.pop() if len(kinds) == 1 else ValueError
        raise kind("; ".join("rank %d: %s" % (r, msg) for r, (_, _, msg) in bad))
    return [p for _, p in everyone]


# ----------------------------------------------------------------------------- device side of a window (CUDA)
def model_lengths(frames, rates, model_rate):
    """Sample counts at ``model_rate`` (what ``preprocessor.Resample`` returns for files at another rate)."""
    frames, rates = numpy.asarray(frames, numpy.int64), numpy.asarray(rates, numpy.int64)
    return -(-frames * model_rate // rates)


_resamplers = {}


def _resampler(rate, model_rate):
    from .nnet.preprocessor import Resample
    if (rate, model_rate) not in _resamplers:
        _resamplers[rate, model_rate] = Resample(int(rate), int(model_rate))
    return _resamplers[rate, model_rate]


class WindowDecode:
    """Decode of a window's files into one float32 device buffer, every file at the model rate at ``slots[i]`` of its
    first ``n_out`` samples.  Files at the model rate are decoded there directly; the others are decoded into a side
    region after ``n_out`` and resampled into their slots, one ``skb_resample`` call per distinct rate.  The resampler's
    rows and ``extra`` (int64, the caller's own device table) travel in the head of the decode's staging buffer: one
    host-to-device copy, at most one FLAC and one PCM call per window.  Built on the reading thread; ``launch`` runs on
    the main one."""

    def __init__(self, win, model_rate, slots, n_out, extra=None):
        frames, rates = numpy.asarray(win.frames, numpy.int64), numpy.asarray(win.rates, numpy.int64)
        slots = numpy.asarray(slots, numpy.int64)
        other = numpy.nonzero(rates != model_rate)[0]
        side = numpy.cumsum(frames[other]) - frames[other] + n_out
        out_off = slots.copy()
        out_off[other] = side
        self.n_total = int(n_out + frames[other].sum())
        rows, self.groups = [], []
        for r in sorted(set(rates[other].tolist())):
            k = numpy.nonzero(rates[other] == r)[0]
            sel = other[k]
            m = model_lengths(frames[sel], rates[sel], model_rate)
            self.groups.append((r, len(rows), m))
            rows.extend(numpy.stack([side[k], frames[sel], slots[sel], m], axis=1).tolist())
        head = numpy.array(rows, dtype=numpy.int64).reshape(-1)
        self.extra_at = head.shape[0]
        extra = numpy.zeros(0, numpy.int64) if extra is None else numpy.asarray(extra, numpy.int64).reshape(-1)
        self.extra_n = extra.shape[0]
        self.model_rate = model_rate
        self.staging = audio.Staging(win.datas, win.kinds, win.infos, out_off, numpy.concatenate([head, extra]))

    def launch(self, device):
        """``(buffer, extra table on the device, FLAC status)``, enqueued on the current stream of ``device``."""
        with torch.cuda.device(device):
            buf = torch.empty(self.n_total, dtype=torch.float32, device=device)
            staged, status = self.staging.launch(buf, device)
            table = staged[:8 * (self.extra_at + self.extra_n)].view(torch.int64)
            meta = table[:self.extra_at].view(-1, 4)
            for rate, r0, m in self.groups:
                for c in range(0, len(m), 65535):           # the kernel's grid takes up to 65535 waveforms
                    n = min(65535, len(m) - c)
                    _resampler(rate, self.model_rate).launch(buf, meta[r0 + c:r0 + c + n], buf, int(m[c:c + n].max()))
        return buf, table[self.extra_at:], status

    def errors(self, status, names):
        """The exception of a window whose FLAC status (device tensor, or None) reports corrupt files, else None."""
        if status is None:
            return None
        bad = self.staging.flac_errors(status.cpu().numpy(), names)
        return ValueError("; ".join(str(bad[i]) for i in sorted(bad))) if bad else None


def check_window(xtractor, dec, status, names):
    """Waits for a window's device work and raises its errors: first a ``ValueError`` naming every corrupt FLAC file (the
    decoder leaves such a file's output range unwritten, so what the model made of the window means nothing, an fp16
    overflow included: that overflow is consumed here, not reported), then the extractor's fp16 range guard."""
    err = dec.errors(status, names)
    if err is not None:
        try:
            xtractor.check_overflow()
        except OverflowError:
            pass
        raise err
    xtractor.check_overflow()


def extract_batches(xtractor, wave, lengths, batches, emb, norm_embedding=True):
    """Enqueue ``Xtractor.extract_packed`` on consecutive slices of ``wave`` (the utterances of ``batches`` back to back,
    in that order) into consecutive rows of ``emb``; no synchronisation."""
    off = row = 0
    for b in batches:
        n = int(lengths[b].sum())
        xtractor.extract_packed(wave[off:off + n], lengths[b], norm_embedding=norm_embedding, out=emb[row:row + len(b)])
        off, row = off + n, row + len(b)
