"""Feed path of the extractor (SURVEY.md 8f rank 1): ``IdMap``, ``IdMapSet`` and ``extract_embeddings`` with the
reference's signatures (sidekit/bosaris/idmap.py:43-73, sidekit/nnet/xsets.py:368-480,
sidekit/nnet/xvector.py:1796-1916).

What changes against the reference: a single 16- or 32-bit PCM wav file is read with the standard library
(``torchaudio.load`` needs torchcodec), other audio is decoded on the device; and instead of one ``forward`` per file --
a few hundred small launches and a device-to-host sync each -- the segments / sliding windows are cut on the device, length-bucketed and pushed through
``Xtractor.extract_packed`` as packed batches (``bulk.make_batches``): the engine's packed layout makes a batch of
different lengths exact, so the embeddings are the same as the one-by-one loop, bit for bit.  Augmentation
(``transform_pipeline``) and HDF5 IO are out of scope and raise; files at another sample rate are resampled on the
device (``preprocessor.Resample``); ``IdMap`` reads / writes the reference's text format.  Files are recognised by their
content, whatever ``file_extension`` says: FLAC, WAV and NIST SPHERE in every PCM encoding (``sidekit_b200.audio``);
``extract_embeddings`` streams the dataset's files through the window pipeline of ``sidekit_b200.corpus``.
"""
import os
import wave as _wave

import numpy
import torch

from ..statserver import StatServer


class IdMap:
    """idmap.py:43-73: ``leftids`` (model ids), ``rightids`` (file ids), ``start`` / ``stop`` in centiseconds or None."""

    def __init__(self, idmap_filename=''):
        if idmap_filename != '':
            raise NotImplementedError("HDF5 IdMap files need h5py (not in this image); use IdMap.read_txt or set the fields directly")
        self.leftids = numpy.empty(0, dtype="|O")
        self.rightids = numpy.empty(0, dtype="|O")
        self.start = numpy.empty(0, dtype="|O")
        self.stop = numpy.empty(0, dtype="|O")

    def validate(self, warn=False):
        ok = self.leftids.shape == self.rightids.shape == self.start.shape == self.stop.shape
        return bool(ok and self.leftids.ndim == 1)

    def set(self, left, right, start=None, stop=None):
        """idmap.py:261-280: fill the map from arrays (deep copies); absent boundaries become None."""
        import copy
        self.leftids, self.rightids = copy.deepcopy(left), copy.deepcopy(right)
        self.start = copy.deepcopy(start) if start is not None else numpy.empty(self.rightids.shape, "|O")
        self.stop = copy.deepcopy(stop) if stop is not None else numpy.empty(self.rightids.shape, "|O")

    def _map(self, keys, values, wanted):
        # idmap.py:128-188: ids of `wanted` found in `keys`, in the order of `wanted`, mapped through the LAST pair of a key
        table = dict(zip(keys, values))
        inter = set(numpy.intersect1d(keys, wanted).tolist())
        out = [table[w] for w in numpy.asarray(wanted).tolist() if w in inter]
        if len(out) > len(inter):
            raise IndexError("index %d is out of bounds for axis 0 with size %d" % (len(inter), len(inter)))   # duplicates in the query
        res = numpy.empty(len(inter), "|O")
        res[:len(out)] = out
        return res

    def map_left_to_right(self, leftidlist):
        return self._map(self.leftids, self.rightids, leftidlist)

    def map_right_to_left(self, rightidlist):
        return self._map(self.rightids, self.leftids, rightidlist)

    def _filter(self, ids, idlist, keep):
        keepids = numpy.unique(idlist) if keep else numpy.setdiff1d(ids, idlist)
        keep_idx = numpy.isin(ids, keepids)
        out = IdMap()
        out.leftids, out.rightids = self.leftids[keep_idx], self.rightids[keep_idx]
        out.start, out.stop = self.start[keep_idx], self.stop[keep_idx]
        return out

    def filter_on_left(self, idlist, keep):
        """idmap.py:190-215: the sessions whose left id is (keep=True) / is not (keep=False) in ``idlist``, in map order."""
        return self._filter(self.leftids, idlist, keep)

    def filter_on_right(self, idlist, keep):
        """idmap.py:217-241."""
        return self._filter(self.rightids, idlist, keep)

    @staticmethod
    def merge(self, idmap2):
        """idmap.py:341-373 (a static method taking both maps, as in the reference): ``self`` followed by the sessions of
        ``idmap2`` whose (left, right) pair is not in ``self``."""
        idmap = IdMap()
        if not (self.validate() and idmap2.validate()):
            raise Exception("Cannot merge IdMaps, wrong type")
        have = set(zip(self.leftids.tolist(), self.rightids.tolist()))
        new = numpy.array([p not in have for p in zip(idmap2.leftids.tolist(), idmap2.rightids.tolist())], dtype=bool)
        idmap.leftids = numpy.concatenate((self.leftids, idmap2.leftids[new]), axis=0)
        idmap.rightids = numpy.concatenate((self.rightids, idmap2.rightids[new]), axis=0)
        idmap.start = numpy.concatenate((self.start, idmap2.start[new]), axis=0)
        idmap.stop = numpy.concatenate((self.stop, idmap2.stop[new]), axis=0)
        if not idmap.validate():
            raise Exception("Wrong format of IdMap")
        return idmap

    def split(self, N):
        """idmap.py:375-392: N maps of (nearly) equal size, ``numpy.array_split`` order."""
        out = []
        for idx in numpy.array_split(numpy.arange(self.leftids.shape[0]), N):
            im = IdMap()
            im.leftids, im.rightids, im.start, im.stop = self.leftids[idx], self.rightids[idx], self.start[idx], self.stop[idx]
            assert im.validate(), "Error: wrong IdMap format"
            out.append(im)
        return out

    def write_txt(self, output_file_name):
        """idmap.py:118-126: ``left right start stop`` per line; absent boundaries are written as the string ``None``
        (which ``read_txt`` cannot parse back -- a reference quirk kept as is)."""
        with open(output_file_name, "w") as f:
            for left, right, start, stop in zip(self.leftids, self.rightids, self.start, self.stop):
                f.write(" ".join(filter(None, (left, right, str(start), str(stop)))) + "\n")

    @classmethod
    def read_txt(cls, input_file_name):
        """idmap.py:312-340: two columns (ids only, ``start`` / ``stop`` = None) or four (integer boundaries); the column
        count is taken from the first line split on single spaces, like the reference.  Returns the object (the
        reference's ``check_path_existance`` decorator swallows the return value)."""
        idmap = cls()
        with open(input_file_name, "r") as f:
            columns = len(f.readline().split(" "))
        with open(input_file_name, "r") as f:
            rows = [l.split() for l in f if l.strip()]
        if columns == 2:
            idmap.leftids = numpy.array([r[0] for r in rows], dtype="|O")
            idmap.rightids = numpy.array([r[1] for r in rows], dtype="|O")
            idmap.start = numpy.empty(idmap.rightids.shape, "|O")
            idmap.stop = numpy.empty(idmap.rightids.shape, "|O")
        elif columns == 4:
            idmap.leftids = numpy.array([r[0] for r in rows], dtype="|O")
            idmap.rightids = numpy.array([r[1] for r in rows], dtype="|O")
            try:
                idmap.start = numpy.array([int(r[2]) for r in rows], dtype="int")
                idmap.stop = numpy.array([int(r[3]) for r in rows], dtype="int")
            except ValueError as e:
                raise ValueError("could not convert string to int64: %s" % e)
        if not idmap.validate():
            raise Exception("Wrong format of IdMap")
        return idmap


def read_wav(path, frame_offset=0, num_frames=-1):
    """PCM wav -> (float32 tensor (n,), sample_rate), scaled like ``torchaudio.load`` (int16 / 32768); first channel."""
    with _wave.open(path, "rb") as f:
        rate, width, chans, total = f.getframerate(), f.getsampwidth(), f.getnchannels(), f.getnframes()
        if width not in (2, 4):
            raise NotImplementedError("read_wav: only 16- and 32-bit PCM is supported (%s)" % path)
        frame_offset = min(max(0, int(frame_offset)), total)
        f.setpos(frame_offset)
        n = total - frame_offset if num_frames is None or num_frames < 0 else min(int(num_frames), total - frame_offset)
        raw = f.readframes(n)
    a = numpy.frombuffer(raw, dtype=numpy.int16 if width == 2 else numpy.int32).reshape(-1, chans)[:, 0]
    scale = 32768.0 if width == 2 else 2147483648.0
    return torch.from_numpy(a.astype(numpy.float32) / numpy.float32(scale)), rate


class IdMapSet:
    """xsets.py:368-480 without the augmentation branch: item ``index`` -> (speech, leftid, rightid, start, stop),
    ``speech`` a (n,) tensor or, with ``sliding_window``, the (n_windows, window_len) unfolded view."""

    def __init__(self, idmap_name, data_path, file_extension, transform_pipeline={}, transform_number=1,
                 sliding_window=False, window_len=3., window_shift=1.5, sample_rate=16000, min_duration=0.165):
        if not isinstance(idmap_name, IdMap):
            raise NotImplementedError("HDF5 IdMap files need h5py (not in this image); pass an IdMap object (IdMap.read_txt)")
        if len(transform_pipeline):
            raise NotImplementedError("data augmentation is out of scope of the inference path")
        self.idmap = idmap_name
        self.data_path = data_path
        self.file_extension = file_extension
        self.len = self.idmap.leftids.shape[0]
        self.min_duration = min_duration
        self.sample_rate = sample_rate
        self.sliding_window = sliding_window
        self.window_len = int(window_len * self.sample_rate)
        self.window_shift = int(window_shift * self.sample_rate)
        self._resamplers = {}
        from ..audio import read
        self._read = read

    def __len__(self):
        return self.len

    def _resampler(self, fs):
        if fs not in self._resamplers:
            from .preprocessor import Resample
            self._resamplers[fs] = Resample(fs, self.sample_rate)
        return self._resamplers[fs]

    def _path(self, index):
        return f"{self.data_path}/{self.idmap.rightids[index]}.{self.file_extension}"

    def __getitem__(self, index):
        start = 0 if self.idmap.start[index] is None else int(self.idmap.start[index] * 0.01 * self.sample_rate)
        if self.idmap.stop[index] is None:
            # whole file (xsets.py:430-435; note: the file is NOT cut at `start` in this branch, only `duration` is)
            speech, fs = self._read(self._path(index))
            if fs != self.sample_rate:
                # torchaudio.transforms.Resample(nfo.sample_rate, self.sample_rate) of :434-435, on the device
                speech = self._resampler(fs)(speech.cuda(non_blocking=True))
            duration = int(speech.shape[0] - start)
        else:
            duration = int(self.idmap.stop[index] * 0.01 * self.sample_rate) - start
            if duration <= self.min_duration * self.sample_rate:     # too short: recentre a min_duration window (:443-446)
                middle = start + duration // 2
                start = int(max(0, int(middle - (self.min_duration * self.sample_rate / 2))))
                duration = int(self.min_duration * self.sample_rate)
            speech, fs = self._read(self._path(index), frame_offset=start, num_frames=duration)
            assert fs == self.sample_rate
        stop = start + duration
        if self.sliding_window:
            speech = speech.unfold(0, self.window_len, self.window_shift)
        return speech, self.idmap.leftids[index], self.idmap.rightids[index], start, stop


def load_checkpoint(model_path, device, embedding_size=None):
    """Checkpoint file -> ``Xtractor`` in eval mode on ``device``, as ``extract_embeddings`` (xvector.py:1834-1843) and
    ``extract_xvectors.py:load_model`` (:74-91) do it: ``torch.load`` of a dict holding ``speaker_number``,
    ``model_archi`` (``model_type``, ``loss.type``, optional ``embedding_size``) and ``model_state_dict``, loaded with
    ``strict=True``.  ``embedding_size=None`` takes the checkpoint's value (256 when absent, like ``load_model``)."""
    from .xvector import Xtractor
    checkpoint = torch.load(model_path, map_location="cpu", weights_only=False)
    model_opts = checkpoint["model_archi"]
    if embedding_size is None:
        embedding_size = model_opts.get("embedding_size", 256)
    model = Xtractor(checkpoint["speaker_number"], model_archi=model_opts["model_type"], loss=model_opts["loss"]["type"],
                     embedding_size=embedding_size)
    model.load_state_dict(checkpoint["model_state_dict"], strict=True)
    model.eval()
    return model.to(device)


def _segment(dataset, index, file_len):
    """``IdMapSet.__getitem__``'s cut of item ``index`` from its file (``file_len`` samples at the model rate):
    ``(offset, length, start, stop)`` of the segment within the file, ``start`` / ``stop`` as the item returns them."""
    sr = dataset.sample_rate
    start = 0 if dataset.idmap.start[index] is None else int(dataset.idmap.start[index] * 0.01 * sr)
    if dataset.idmap.stop[index] is None:
        return 0, file_len, start, file_len                       # whole file: NOT cut at `start` (xsets.py:430-435)
    duration = int(dataset.idmap.stop[index] * 0.01 * sr) - start
    if duration <= dataset.min_duration * sr:
        middle = start + duration // 2
        start = int(max(0, int(middle - (dataset.min_duration * sr / 2))))
        duration = int(dataset.min_duration * sr)
    off = min(max(0, start), file_len)                            # read_wav's clamping
    return off, min(duration, file_len - off), start, start + duration


def _windows_of(dataset, seg_len):
    """(number of sliding windows, window length, shift) of a segment of ``seg_len`` samples (``Tensor.unfold``)."""
    wl, ws = dataset.window_len, dataset.window_shift
    if seg_len < wl:
        raise RuntimeError("maximum size for tensor at dimension 0 is %d but size is %d" % (seg_len, wl))
    return (seg_len - wl) // ws + 1, wl, ws


def extract_embeddings(idmap_name, model_filename, data_root_name, device, batch_size=1, file_extension="wav",
                       transform_pipeline={}, sliding_window=False, win_duration=3., win_shift=1.5, num_thread=1,
                       sample_rate=16000, mixed_precision=False, norm_embeddings=True, max_audio_seconds=1200.0,
                       window_audio_seconds=4800.0):
    """xvector.py:1796-1916: a ``StatServer`` with one embedding per segment (or per sliding window).

    ``model_filename`` is an ``Xtractor`` or the path of a checkpoint written by the reference's training loop
    (``speaker_number`` / ``model_archi`` / ``model_state_dict``, xvector.py:1834-1843); ``batch_size``, ``num_thread`` and
    ``mixed_precision`` are accepted and ignored: batches are formed by total audio (``max_audio_seconds``) and the
    kernels pick their own precision.  ``start`` / ``stop`` follow the reference, including its sliding-window
    ``stop = start + <number of 100-window chunks of the last segment>`` (xvector.py:1897, :1911).

    The id map's files are streamed through the window pipeline of ``sidekit_b200.corpus`` in windows of
    ``window_audio_seconds`` of audio: only one window's waveforms are on the device at a time (plus the next window in
    host memory), so an id map of any size is extracted in one call.  A window's files are decoded on the device in one
    batched call, resampled to ``sample_rate`` where needed, and its segments / sliding windows are cut from them by one
    device gather per length-bucketed packed batch.  Under an initialised ``torch.distributed`` process group the
    files are sharded over the ranks in contiguous blocks balanced by size, each segment goes with its file, and every
    rank returns the same ``StatServer`` as one process.
    """
    from .. import bulk, corpus, flac
    model = model_filename
    if isinstance(model, str):
        model = load_checkpoint(model, device, embedding_size=256)          # xvector.py:1838: the size is forced to 256
    dataset = IdMapSet(idmap_name, data_root_name, file_extension, transform_pipeline, 0, sliding_window, win_duration, win_shift,
                       sample_rate, min_duration=win_duration)
    model.eval()
    device = flac.device_of(device)
    model.to(device)
    E = model.embedding_size
    n_seg = len(dataset)
    paths = [dataset._path(i) for i in range(n_seg)]
    files = list(dict.fromkeys(paths))
    file_of = {p: k for k, p in enumerate(files)}
    segs_of = [[] for _ in files]
    for i, p in enumerate(paths):
        segs_of[file_of[p]].append(i)
    dist, rank, world = bulk._dist()
    blocks = corpus.plan_blocks(corpus.entry_weights(files), world)
    lo, hi = blocks[rank]
    seg_len = {}                                   # this rank's segments -> length at the model rate

    def prepare(win):
        """Reading thread: files at the model rate back to back in window order, then the segments / sliding windows
        (in id-map order) cut from them into length-sorted packed batches."""
        flen = corpus.model_lengths(win.frames, win.rates, sample_rate)
        foff = numpy.cumsum(flen) - flen
        segs, src, lens = [], [], []
        for i, k in sorted((i, k) for k, f in enumerate(win.index) for i in segs_of[lo + f]):
            off, n, _, _ = _segment(dataset, i, int(flen[k]))
            if dataset.idmap.stop[i] is not None:
                assert win.rates[k] == sample_rate
            rows = [(off, n)]
            if sliding_window:
                m, wl, ws = _windows_of(dataset, n)
                rows = [(off + j * ws, wl) for j in range(m)]
            segs.append((i, n, len(rows)))
            src.extend(int(foff[k]) + o for o, _ in rows)
            lens.extend(l for _, l in rows)
        lens = numpy.array(lens, dtype=numpy.int64)
        order = numpy.argsort(lens, kind="stable")
        batches = list(reversed(bulk.make_batches(order.tolist(), lens, max_audio_seconds, sample_rate=sample_rate)))
        packed = numpy.array([i for b in batches for i in b], dtype=numpy.int64)
        table = numpy.stack([numpy.array(src, dtype=numpy.int64)[packed], lens[packed]]) if len(packed) else numpy.zeros((2, 0), numpy.int64)
        with torch.cuda.device(device):
            dec = corpus.WindowDecode(win, sample_rate, foff, int(flen.sum()), extra=table)
        win.prepared, win.segs = (dec, lens, batches, packed), segs

    def embed(win):
        dec, lens, batches, packed = win.prepared
        buf, table, status = dec.launch(device)
        emb = torch.empty((len(lens), E), dtype=torch.float32, device=device)
        if len(lens):
            with torch.cuda.device(device):
                src, n = table.view(2, -1)                 # per wave, in packed order: offset in buf, length
                row = 0
                for b in batches:
                    # the batch's waves cut from buf by one gather: its sample t is buf[src of its wave + (t - first sample
                    # of its wave)]; built batch by batch, the index never outgrows one batch (max_audio_seconds)
                    k, total = len(b), int(lens[b].sum())
                    s, m = src[row:row + k], n[row:row + k]
                    idx = torch.repeat_interleave(s - (torch.cumsum(m, 0) - m), m, output_size=total)
                    idx += torch.arange(total, device=device)
                    model.extract_packed(buf[idx], lens[b], norm_embedding=norm_embeddings, out=emb[row:row + k])
                    row += k

        def finish():
            corpus.check_window(model, dec, status, win.names)
            rows = torch.empty((len(lens), E), dtype=torch.float32)
            rows[torch.from_numpy(packed)] = emb.cpu()
            return rows
        return finish

    parts = []

    def emit(win, rows):
        parts.append((win.segs, rows))
        for i, n, _ in win.segs:
            seg_len[i] = n

    error = None
    with torch.no_grad(), torch.cuda.device(device):
        try:
            corpus.run_windows(files[lo:hi], corpus.read_file, window_audio_seconds, embed, emit, prepare)
        except Exception as e:
            if dist is None:
                raise
            error = e
        owner = numpy.searchsorted(numpy.array([b for _, b in blocks]), [file_of[p] for p in paths], side="right")
        return _assemble(dataset, parts, seg_len, error, owner, E, win_shift, device)


def _assemble(dataset, parts, seg_len, error, owner, embedding_size, win_shift, device=None):
    """The ``StatServer`` of ``extract_embeddings`` on every rank from this rank's ``parts`` (``(segments, rows)`` per
    window: ``(index, length, rows)`` of its segments in id-map order and their rows), ``seg_len`` (its segments' lengths
    at the model rate) and ``error`` (None, or what stopped its windows); ``owner``: the rank of every segment.

    One small exchange shares the errors and every segment's length, from which every rank knows every segment's row
    count (sliding windows depend on it) and so where each rank's rows go; then one gather of the rows."""
    from .. import bulk, corpus
    dist, rank, world = bulk._dist()
    n_seg, sliding = len(dataset), dataset.sliding_window
    lengths = {}
    for part in corpus.exchange(error, seg_len):
        lengths.update(part)
    n_rows = numpy.array([_windows_of(dataset, lengths[i])[0] if sliding else 1 for i in range(n_seg)], dtype=numpy.int64)
    row0 = numpy.cumsum(n_rows) - n_rows
    # local rows come window by window; the gather takes this rank's segments in id-map order
    pieces = {}
    for segs, rows in parts:
        r = 0
        for i, _, m in segs:
            pieces[i] = rows[r:r + m]
            r += m
    local = torch.cat([pieces[i] for i in sorted(pieces)]) if pieces else None
    if dist is None:
        emb = local if local is not None else torch.zeros((0, embedding_size), dtype=torch.float32)
    else:
        shards = [numpy.concatenate([numpy.arange(row0[i], row0[i] + n_rows[i]) for i in range(n_seg) if owner[i] == r] or
                                    [numpy.zeros(0, numpy.int64)]).astype(numpy.int64) for r in range(world)]
        emb = bulk.gather_embeddings(local, shards, embedding_size, device).cpu()
    sample_rate = dataset.sample_rate
    modelset, segset, starts, stops = [], [], [], []
    last_chunks = 1
    for i in range(n_seg):
        _, _, start, _ = _segment(dataset, i, lengths[i])
        n = int(n_rows[i])
        modelset.extend([dataset.idmap.leftids[i]] * n)
        segset.extend([dataset.idmap.rightids[i]] * n)
        if sliding:
            starts.extend((numpy.arange(0, n * win_shift, win_shift) * sample_rate + start).tolist())
            last_chunks = len(range(0, n, max(1, n // max(1, n // 100))))          # len(torch.split(...)) of :1885
        else:
            starts.append(start)
            stops.append(lengths[i])
    embeddings = StatServer()
    embeddings.stat1 = emb.numpy().astype(numpy.float32)
    embeddings.modelset = numpy.array(modelset).astype('>U')
    embeddings.segset = numpy.array(segset).astype('>U')
    embeddings.start = numpy.array(starts).squeeze()
    embeddings.stop = embeddings.start + (last_chunks if sliding else numpy.array(stops).squeeze())
    embeddings.stat0 = numpy.ones((embeddings.modelset.shape[0], 1))
    return embeddings
