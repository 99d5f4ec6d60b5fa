"""Light BOSARIS containers used as argument / return types of the scoring functions
(sidekit/bosaris/ndx.py:48-182, sidekit/bosaris/key.py:49-110, sidekit/bosaris/scores.py:52-81, :157-240, :304-313,
:469-478): same attribute names, same ``validate()`` rules, no HDF5 / plotting (out of scope of the hot path).
Id matching is an O(N) hash join with the reference's ordering semantics (first occurrence wins).
"""
import logging

import os

import numpy

try:
    import torch as _torch
    _NP_DTYPE = {_torch.float32: numpy.float32, _torch.float64: numpy.float64, _torch.float16: numpy.float16}
except ImportError:          # the containers themselves do not need torch
    _NP_DTYPE = {}


def _first_index(ids):
    """id -> index of its first occurrence."""
    table = {}
    for i, v in enumerate(numpy.asarray(ids).tolist()):
        table.setdefault(v, i)
    return table


def _device_to_numpy(t, np_dtype=None, chunk_bytes=256 << 20):
    """Device tensor -> numpy array.  Large matrices land in a PINNED host block taken from torch's caching host allocator
    (the numpy array is a view of it and gives the block back to the cache when it is garbage collected, so a scoring loop
    re-uses one block): the copy runs at PCIe speed straight into the result, with no pageable bounce (a plain ``.cpu()`` of a
    20k x 20k float64 matrix takes 1.5 s).  ``np_dtype=float64`` on a float32 tensor widens on the DEVICE, chunk by chunk
    (``skb_widen_f32_f64``), on the way out: the reference's PLDA scorers return float64, the score GEMM keeps float32."""
    import torch
    from . import _lib
    t = t.contiguous()
    np_dtype = numpy.dtype(np_dtype or _NP_DTYPE[t.dtype])
    widen = t.dtype == torch.float32 and np_dtype == numpy.float64
    if not widen and np_dtype != numpy.dtype(_NP_DTYPE[t.dtype]):
        raise TypeError("unsupported conversion %s -> %s" % (t.dtype, np_dtype))
    nbytes = t.numel() * np_dtype.itemsize
    if nbytes < (32 << 20) or t.dim() != 2:
        out = t.cpu().numpy()
        return out.astype(np_dtype) if widen else out
    host = torch.empty(tuple(t.shape), dtype=torch.float64 if widen else t.dtype, pin_memory=True)
    if not widen:
        host.copy_(t, non_blocking=True)
    else:
        rows_per = max(1, chunk_bytes // (t.shape[1] * 8))
        stage = [torch.empty((min(rows_per, t.shape[0]), t.shape[1]), dtype=torch.float64, device=t.device) for _ in range(2)]
        lib = _lib.lib()
        with torch.cuda.device(t.device):
            for k, lo in enumerate(range(0, t.shape[0], rows_per)):
                hi = min(t.shape[0], lo + rows_per)
                st = stage[k % 2][:hi - lo]
                _lib.check(lib.skb_widen_f32_f64(t[lo:hi].data_ptr(), st.data_ptr(), (hi - lo) * t.shape[1], _lib.stream_ptr()))
                host[lo:hi].copy_(st, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return host.numpy()


def _read_columns(path, n_min):
    """Whitespace-separated columns of a text file (lines are ``rstrip().split()`` like ndx.py:216 / scores.py:379)."""
    with open(path, "r") as f:
        rows = [l.rstrip().split() for l in f]
    rows = [r for r in rows if len(r)]
    for r in rows:
        if len(r) < n_min:
            raise IndexError("list index out of range")            # what the reference's lines[ii][k] raises
    return rows


def _expand(mat, own_models, own_segs, new_models, new_segs, dtype):
    """Place ``mat`` (own_models x own_segs) into the (new_models x new_segs) grid the way the merge methods of the
    reference do (ndx.py:262-269, key.py:333-344, scores.py:441-448): the k-th own row goes to the k-th position of
    ``new_models`` that holds an own model.  That is the right row when the own sets are sorted (``new_*`` are sorted
    unions); with unsorted sets the reference permutes rows, and so does this."""
    out = numpy.zeros((new_models.shape[0], new_segs.shape[0]), dtype=dtype)
    ma = numpy.flatnonzero(numpy.isin(new_models, own_models))
    mb = numpy.flatnonzero(numpy.isin(own_models, new_models))
    sa = numpy.flatnonzero(numpy.isin(new_segs, own_segs))
    sb = numpy.flatnonzero(numpy.isin(own_segs, new_segs))
    out[ma[:, None], sa] = mat[mb[:, None], sb]
    return out


def _makedirs_for(path):
    d = os.path.dirname(path)
    if d != "" and not os.path.exists(d):
        os.makedirs(d)


class Key:
    """Trial key (key.py:49-110): ``tar`` / ``non`` (M, S) bool matrices over ``modelset`` x ``segset``."""

    def __init__(self, key_file_name=None, models=numpy.array([]), testsegs=numpy.array([]), trials=numpy.array([])):
        self.modelset = numpy.empty(0, dtype="|O")
        self.segset = numpy.empty(0, dtype="|O")
        self.tar = numpy.array([], dtype="bool")
        self.non = numpy.array([], dtype="bool")
        if key_file_name is not None:
            raise NotImplementedError("HDF5 Key files need h5py (not in this image); use Key.read_txt or pass models / testsegs / trials")
        models, testsegs, trials = numpy.asarray(models), numpy.asarray(testsegs), numpy.asarray(trials)
        if models.shape[0]:
            # key.py:79-97 vectorised: the LAST trial listed for a (model, segment) pair decides (dict(zip(...)))
            modelset, mi = numpy.unique(models, return_inverse=True)
            segset, si = numpy.unique(testsegs, return_inverse=True)
            tar = numpy.zeros((modelset.shape[0], segset.shape[0]), dtype="bool")
            non = numpy.zeros((modelset.shape[0], segset.shape[0]), dtype="bool")
            tar[mi, si] = trials == 'target'          # fancy assignment: the last write wins, like the dict
            non[mi, si] = trials == 'nontarget'
            self.modelset, self.segset, self.tar, self.non = modelset, segset, tar, non
            assert self.validate(), "Wrong Key format"

    @classmethod
    def create(cls, modelset, segset, tar, non):
        key = cls()
        key.modelset, key.segset, key.tar, key.non = modelset, segset, tar, non
        assert key.validate(), "Wrong Key format"
        return key

    @staticmethod
    def read_txt(input_file_name):
        """``model segment target|nontarget`` lines -> Key (key.py:262-304): sorted-unique model / segment sets, the LAST
        line of a (model, segment) pair decides, anything but the two labels leaves the trial unset."""
        rows = _read_columns(input_file_name, 3)
        col = lambda k: numpy.array([r[k] for r in rows], dtype="U")
        return Key(models=col(0), testsegs=col(1), trials=col(2)) if rows else Key()

    def write_txt(self, output_file_name):
        """key.py:151-164: per model, its target trials then its non-target trials, in ``segset`` order."""
        with open(output_file_name, "w") as fid:
            for m in range(self.modelset.shape[0]):
                for label, mask in (("target", self.tar), ("nontarget", self.non)):
                    fid.writelines("{} {} {}\n".format(self.modelset[m], seg, label) for seg in self.segset[mask[m, ]])

    def filter(self, modlist, seglist, keep):
        """key.py:166-205: keep (or drop) the listed models / segments; the order of the Key is kept."""
        mods, segs = set(numpy.asarray(modlist).tolist()), set(numpy.asarray(seglist).tolist())
        km = numpy.fromiter(((m in mods) == bool(keep) for m in self.modelset.tolist()), dtype=bool, count=self.modelset.shape[0])
        ks = numpy.fromiter(((x in segs) == bool(keep) for x in self.segset.tolist()), dtype=bool, count=self.segset.shape[0])
        out = Key()
        out.modelset, out.segset = self.modelset[km], self.segset[ks]
        out.tar, out.non = self.tar[km, :][:, ks], self.non[km, :][:, ks]
        assert out.validate()
        return out

    def merge(self, key_list):
        """key.py:305-367: union of the model / segment sets (sorted), target / non-target marks OR-ed; a trial that is a
        target in one key and a non-target in another is an error."""
        assert isinstance(key_list, list), "Input is not a list"
        for key2 in key_list:
            models = numpy.union1d(self.modelset, key2.modelset)
            segs = numpy.union1d(self.segset, key2.segset)
            tar = _expand(self.tar, self.modelset, self.segset, models, segs, bool) | _expand(key2.tar, key2.modelset, key2.segset, models, segs, bool)
            non = _expand(self.non, self.modelset, self.segset, models, segs, bool) | _expand(key2.non, key2.modelset, key2.segset, models, segs, bool)
            assert numpy.sum(tar & non) == 0, "Conflict in the new Key"
            self.modelset, self.segset, self.tar, self.non = models, segs, tar, non
            self.validate()

    def trial_indices(self):
        """Row-major flat indices of the target and of the non-target trials (``flatnonzero`` of ``tar`` / ``non``), cached:
        one Key usually selects the trials of several score matrices (cosine, PLDA, as-norm).  The cache is keyed on the
        identity and shape of the two matrices; rebinding ``tar`` / ``non`` invalidates it, writing into them in place
        does not."""
        tag = (id(self.tar), id(self.non), self.tar.shape)
        if getattr(self, "_idx_tag", None) != tag:
            self._idx = (numpy.flatnonzero(self.tar), numpy.flatnonzero(self.non))
            self._idx_tag = tag
        return self._idx

    def to_ndx(self):
        ndx = Ndx()
        ndx.modelset, ndx.segset, ndx.trialmask = self.modelset, self.segset, self.tar | self.non
        return ndx

    def validate(self):
        ok = isinstance(self.modelset, numpy.ndarray) and isinstance(self.segset, numpy.ndarray)
        ok &= isinstance(self.tar, numpy.ndarray) and isinstance(self.non, numpy.ndarray)
        ok &= self.modelset.ndim == 1 and self.segset.ndim == 1 and self.tar.ndim == 2 and self.non.ndim == 2
        ok &= self.tar.shape == self.non.shape == (self.modelset.shape[0], self.segset.shape[0])
        return bool(ok)


class Ndx:
    """Trial index: ``modelset`` (M,), ``segset`` (S,), ``trialmask`` (M, S) bool."""

    def __init__(self, ndx_file_name="", models=numpy.array([]), testsegs=numpy.array([])):
        self.modelset = numpy.empty(0, dtype="|O")
        self.segset = numpy.empty(0, dtype="|O")
        self.trialmask = numpy.array([], dtype="bool")
        if ndx_file_name != "":
            raise NotImplementedError("HDF5 Ndx files need h5py (not in this image); use Ndx.read_txt or set the fields directly")
        if len(models):
            # every (model, segment) pair listed is a trial (ndx.py:73-79), vectorised
            modelset, mi = numpy.unique(models, return_inverse=True)
            segset, si = numpy.unique(testsegs, return_inverse=True)
            mask = numpy.zeros((modelset.shape[0], segset.shape[0]), dtype="bool")
            mask[mi, si] = True
            self.modelset, self.segset, self.trialmask = modelset, segset, mask

    @classmethod
    def read_txt(cls, input_filename):
        """``model segment`` lines -> Ndx with sorted-unique sets (ndx.py:208-236).  Returns the object: the reference's
        ``check_path_existance`` decorator swallows the return value, so its own ``Ndx.read_txt`` yields None."""
        rows = _read_columns(input_filename, 2)
        ndx = cls(models=numpy.array([r[0] for r in rows], dtype="|O"), testsegs=numpy.array([r[1] for r in rows], dtype="|O"))
        assert ndx.validate(), "Wrong Ndx format"
        return ndx

    def merge(self, ndx_list):
        """ndx.py:239-283: union of the sets (sorted); a trial of any input is a trial of the result."""
        assert isinstance(ndx_list, list), "Input is not a list"
        self.validate()
        for ndx2 in ndx_list:
            models = numpy.union1d(self.modelset, ndx2.modelset)
            segs = numpy.union1d(self.segset, ndx2.segset)
            mask = _expand(self.trialmask, self.modelset, self.segset, models, segs, bool) | \
                _expand(ndx2.trialmask, ndx2.modelset, ndx2.segset, models, segs, bool)
            self.modelset, self.segset, self.trialmask = models, segs, mask

    def save_txt(self, output_file_name):
        """ndx.py:115-126: one ``model segment`` line per trial, row by row."""
        with open(output_file_name, "w") as fid:
            for m in range(self.modelset.shape[0]):
                fid.writelines("{} {}\n".format(self.modelset[m], s) for s in self.segset[self.trialmask[m, ]])

    def filter(self, modlist, seglist, keep):
        """Same semantics as ndx.py:128-165 (order of the Ndx kept, every occurrence kept), O(N) with hash sets."""
        mods, segs = set(numpy.asarray(modlist).tolist()), set(numpy.asarray(seglist).tolist())
        keepmod = numpy.fromiter(((m in mods) == bool(keep) for m in self.modelset.tolist()), dtype=bool,
                                 count=self.modelset.shape[0])
        keepseg = numpy.fromiter(((s in segs) == bool(keep) for s in self.segset.tolist()), dtype=bool,
                                 count=self.segset.shape[0])
        out = Ndx()
        out.modelset = self.modelset[keepmod]
        out.segset = self.segset[keepseg]
        all_m, all_s = bool(keepmod.all()), bool(keepseg.all())
        if all_m and all_s:
            # nothing is dropped (the usual case): the (M, S) mask is SHARED, not copied twice through boolean indexing
            # (2 x 400 MB at 20k x 20k); nothing in this package writes into a trialmask / scoremask in place
            out.trialmask = self.trialmask
        elif all_s:
            out.trialmask = self.trialmask[keepmod]
        elif all_m:
            out.trialmask = self.trialmask[:, keepseg]
        else:
            out.trialmask = self.trialmask[numpy.ix_(numpy.flatnonzero(keepmod), numpy.flatnonzero(keepseg))]
        assert out.validate(), "Wrong Ndx format"
        return out

    def validate(self):
        ok = isinstance(self.modelset, numpy.ndarray)
        ok &= isinstance(self.segset, numpy.ndarray)
        ok &= isinstance(self.trialmask, numpy.ndarray)
        ok &= self.modelset.ndim == 1
        ok &= self.segset.ndim == 1
        ok &= self.trialmask.ndim == 2
        ok &= self.trialmask.shape == (self.modelset.shape[0], self.segset.shape[0])
        return bool(ok)


class TrialList:
    """A trial list as three aligned 1-D arrays, one entry per trial in list order: ``enrolset`` / ``testset`` (ids) and
    ``labels`` (bool, True = target; None for an unlabelled list).  Unlike ``Key`` / ``Ndx`` it is never a (models x
    segments) matrix, so lists of VoxCeleb1-E / -H size (about 145 000 utterances, 580 000 trials) stay O(trials)."""

    def __init__(self, enrolset=(), testset=(), labels=None):
        self.enrolset = numpy.asarray(enrolset)
        self.testset = numpy.asarray(testset)
        self.labels = None if labels is None else numpy.asarray(labels, dtype=bool)
        if self.enrolset.ndim != 1 or self.testset.shape != self.enrolset.shape or \
                (self.labels is not None and self.labels.shape != self.enrolset.shape):
            raise ValueError("TrialList: enrolset, testset and labels must be aligned 1-D arrays")

    def __len__(self):
        return self.enrolset.shape[0]

    @classmethod
    def read_txt(cls, path):
        """The ``Key`` text format, ``model segment target|nontarget`` per line (what ``Key.write_txt`` writes), in file
        order.  A line with any other label is an error."""
        rows = _read_columns(path, 3)
        label = numpy.array([r[2] for r in rows], dtype="U")
        bad = (label != "target") & (label != "nontarget")
        if bad.any():
            raise ValueError("%s: label %r is neither 'target' nor 'nontarget'" % (path, label[bad][0]))
        return cls(numpy.array([r[0] for r in rows], dtype="U"), numpy.array([r[1] for r in rows], dtype="U"), label == "target")

    def write_txt(self, path):
        """One ``model segment target|nontarget`` line per trial, in list order (``Key.read_txt`` reads it)."""
        if self.labels is None:
            raise ValueError("TrialList.write_txt: the list has no labels")
        _makedirs_for(path)
        with open(path, "w") as fid:
            fid.writelines("{} {} {}\n".format(m, s, "target" if t else "nontarget")
                           for m, s, t in zip(self.enrolset.tolist(), self.testset.tolist(), self.labels.tolist()))

    @classmethod
    def read_voxceleb(cls, path):
        """The VoxCeleb list format, ``1|0 enrolment_path test_path`` per line (1 = target)."""
        rows = _read_columns(path, 3)
        label = numpy.array([r[0] for r in rows], dtype="U")
        bad = (label != "1") & (label != "0")
        if bad.any():
            raise ValueError("%s: label %r is neither 1 nor 0" % (path, label[bad][0]))
        return cls(numpy.array([r[1] for r in rows], dtype="U"), numpy.array([r[2] for r in rows], dtype="U"), label == "1")

    @classmethod
    def _from_mask(cls, modelset, segset, mask, tar=None):
        idx = numpy.flatnonzero(mask)            # row-major: the order of scoremat[trialmask] and score_trials
        n_seg = mask.shape[1]
        return cls(numpy.asarray(modelset)[idx // n_seg], numpy.asarray(segset)[idx % n_seg],
                   None if tar is None else tar.reshape(-1)[idx])

    @classmethod
    def from_key(cls, key):
        """The trials of a ``Key`` (targets and non-targets) in row-major ``tar | non`` order."""
        return cls._from_mask(key.modelset, key.segset, key.tar | key.non, key.tar)

    @classmethod
    def from_ndx(cls, ndx):
        """The trials of an ``Ndx`` in row-major ``trialmask`` order, unlabelled."""
        return cls._from_mask(ndx.modelset, ndx.segset, ndx.trialmask)

    def subset(self, keep):
        """The trials selected by a bool mask or an index array, in list order."""
        return TrialList(self.enrolset[keep], self.testset[keep], None if self.labels is None else self.labels[keep])

    def index(self, enrol_ids, test_ids):
        """``(rows, cols, keep)``: for the trials whose enrolment id is in ``enrol_ids`` and whose test id is in ``test_ids``
        (``keep``, a bool mask over the list), the int32 position of the FIRST occurrence of each id.  Other trials are
        dropped, as ``Ndx.filter`` drops unknown models / segments, and logged at INFO."""
        if max(len(enrol_ids), len(test_ids)) > numpy.iinfo(numpy.int32).max:
            raise ValueError("TrialList.index: more than 2^31 - 1 rows")
        etab = _first_index(enrol_ids)
        ttab = etab if test_ids is enrol_ids else _first_index(test_ids)
        n = len(self)
        rows = numpy.fromiter((etab.get(v, -1) for v in self.enrolset.tolist()), dtype=numpy.int64, count=n)
        cols = numpy.fromiter((ttab.get(v, -1) for v in self.testset.tolist()), dtype=numpy.int64, count=n)
        keep = (rows >= 0) & (cols >= 0)
        n_keep = int(keep.sum())
        if n_keep < n:
            logging.info('trials reduced from %d to %d (%d unknown enrolment ids, %d unknown test ids)', n, n_keep,
                         int((rows < 0).sum()), int((cols < 0).sum()))
            rows, cols = rows[keep], cols[keep]
        return rows.astype(numpy.int32), cols.astype(numpy.int32), keep


class TrialScores:
    """Scores of a ``TrialList``, one per trial in list order: ``trials`` (the trials scored), ``scores`` (host numpy,
    copied from ``scores_device`` when first read, like ``Scores.scoremat``)."""

    def __init__(self, trials, scores_device, np_dtype=None):
        self.trials = trials
        self.scores_device = scores_device
        self.scores_dtype = np_dtype         # numpy dtype of ``scores`` when it differs from the device tensor's
        self._scores = None

    @property
    def scores(self):
        if self._scores is None:
            self._scores = _device_to_numpy(self.scores_device, self.scores_dtype)
        return self._scores

    def get_tar_non(self):
        """Target and non-target score vectors, each in list order (``Scores.get_tar_non`` for a labelled list)."""
        if self.trials.labels is None:
            raise ValueError("TrialScores.get_tar_non: the trial list has no labels")
        s = self.scores
        return s[self.trials.labels], s[~self.trials.labels]


class Scores:
    """Score matrix container (scores.py:52-81).  ``scoremat`` is materialised lazily: the CUDA result stays on
    the device (``scoremat_device``, a torch tensor) until the numpy array is first read."""

    def __init__(self, scores_file_name=""):
        if scores_file_name != "":
            raise NotImplementedError("HDF5 Scores files need h5py (not in this image); use Scores.read_txt")
        self.modelset = numpy.empty(0, dtype="|O")
        self.segset = numpy.empty(0, dtype="|O")
        self.scoremask = numpy.array([], dtype="bool")
        self._scoremat = numpy.array([])
        self.scoremat_device = None
        self.scoremat_dtype = None          # numpy dtype of the materialised matrix when it differs from the device tensor's

    @property
    def scoremat(self):
        if self._scoremat is None:
            self._scoremat = _device_to_numpy(self.scoremat_device, self.scoremat_dtype)
        return self._scoremat

    @scoremat.setter
    def scoremat(self, value):
        self._scoremat = value

    def filter(self, modlist, seglist, keep):
        """scores.py:262-302: keep (or drop) the listed models / segments with their scores; order kept."""
        mods, segs = set(numpy.asarray(modlist).tolist()), set(numpy.asarray(seglist).tolist())
        km = numpy.fromiter(((m in mods) == bool(keep) for m in self.modelset.tolist()), dtype=bool, count=self.modelset.shape[0])
        ks = numpy.fromiter(((x in segs) == bool(keep) for x in self.segset.tolist()), dtype=bool, count=self.segset.shape[0])
        out = Scores()
        out.modelset, out.segset = self.modelset[km], self.segset[ks]
        out.scoremat, out.scoremask = self.scoremat[km, :][:, ks], self.scoremask[km, :][:, ks]
        return out

    def merge(self, score_list):
        """scores.py:414-467: both sides are sorted first (in place, like the reference), then laid out over the union of
        the sets; two scores for one trial are an error; the result is float64."""
        assert isinstance(score_list, list), "Input is not a list"
        self.validate()
        for scr2 in score_list:
            self.sort()
            scr2.sort()
            models = numpy.union1d(self.modelset, scr2.modelset)
            segs = numpy.union1d(self.segset, scr2.segset)
            mat1 = _expand(self.scoremat, self.modelset, self.segset, models, segs, numpy.float64)
            mask1 = _expand(self.scoremask, self.modelset, self.segset, models, segs, bool)
            mat2 = _expand(scr2.scoremat, scr2.modelset, scr2.segset, models, segs, numpy.float64)
            mask2 = _expand(scr2.scoremask, scr2.modelset, scr2.segset, models, segs, bool)
            assert numpy.sum(mask1 & mask2) == 0, "Conflict in the new scoremask"
            self.scoremat, self.scoremask, self.scoremat_device = mat1 + mat2, mask1 | mask2, None
            self.modelset, self.segset = models, segs
            assert self.validate(), 'Wrong Scores format'

    def get_score(self, modelID, segID):
        """scores.py:480-495: the (1, 1) block of the trial; raises when the model or the segment is unknown."""
        model_idx = numpy.argwhere(self.modelset == modelID)
        seg_idx = numpy.argwhere(self.segset == segID)
        if model_idx.shape[0] == 0:
            raise Exception('No such model as: %s', modelID)
        if seg_idx.shape[0] == 0:
            raise Exception('No such segment as: %s', segID)
        return self.scoremat[model_idx, seg_idx]

    def write_txt(self, output_file_name):
        """scores.py:118-131: one ``model segment score`` line per scored trial, scores printed as ``str`` of the
        matrix's own dtype (float32 for cosine / as-norm, float64 for PLDA).  The directory is created when missing (the
        reference also tries to create ``''`` for a bare file name and fails there; not reproduced)."""
        _makedirs_for(output_file_name)
        mat = self.scoremat
        with open(output_file_name, "w") as fid:
            for m in range(self.modelset.shape[0]):
                sel = self.scoremask[m, ]
                fid.writelines("{} {} {}\n".format(self.modelset[m], seg, sc) for seg, sc in zip(self.segset[sel], mat[m, sel]))

    @classmethod
    def read_txt(cls, input_file_name):
        """``model segment score`` lines -> Scores over the sorted-unique sets, float64, then ``sort()`` (scores.py:371-412).
        Returns the object (the reference's decorator swallows it, see ``Ndx.read_txt``)."""
        rows = _read_columns(input_file_name, 3)
        s = cls()
        models = numpy.array([r[0] for r in rows], dtype="|O")
        testsegs = numpy.array([r[1] for r in rows], dtype="|O")
        scores = numpy.array([float(r[2]) for r in rows], dtype=numpy.float64)
        modelset, mi = numpy.unique(models, return_inverse=True)
        segset, si = numpy.unique(testsegs, return_inverse=True)
        mask = numpy.zeros((modelset.shape[0], segset.shape[0]), dtype="bool")
        mat = numpy.zeros((modelset.shape[0], segset.shape[0]))
        mask[mi, si] = True
        mat[mi, si] = scores
        s.modelset, s.segset, s.scoremask, s.scoremat = modelset, segset, mask, mat
        assert s.validate(), "Wrong Scores format"
        s.sort()
        return s

    def validate(self):
        ok = self.scoremat.shape == self.scoremask.shape
        ok &= (self.scoremat.shape[0] == self.modelset.shape[0])
        ok &= (self.scoremat.shape[1] == self.segset.shape[0])
        return bool(ok)

    def get_tar_non(self, key):
        """scores.py:157-179: target and non-target score vectors selected by ``key``."""
        if (self.modelset.shape == key.modelset.shape and self.segset.shape == key.segset.shape
                and (key.modelset == self.modelset).all() and (key.segset == self.segset).all()
                and self.scoremask.shape == key.tar.shape):
            # the trials' flat indices (cached on the key), filtered by the score mask: a few 10^4 gathers instead of two
            # (M, S) boolean ANDs and two boolean-index passes; same row-major order as numpy's boolean indexing
            it, inn = key.trial_indices()
            mask = self.scoremask.reshape(-1)
            it, inn = it[mask[it]], inn[mask[inn]]
            if self._scoremat is None and self.scoremat_device is not None:
                # the matrix is still on the device: gather the trials there instead of copying the whole matrix
                # (3.2 GB of float64 at 20k x 20k) to the host first
                import torch
                dev = self.scoremat_device.device
                flat = self.scoremat_device.reshape(-1)
                both = flat[torch.from_numpy(numpy.concatenate([it, inn])).to(dev)].cpu().numpy()
                if self.scoremat_dtype is not None:
                    both = both.astype(self.scoremat_dtype)
                return both[:it.shape[0]], both[it.shape[0]:]
            flat = self.scoremat.reshape(-1)
            return flat[it], flat[inn]
        # The key lists other (or differently ordered) models / segments than the scores (scores.py:172-179 aligns a copy
        # of the whole matrix with the key first): map the key's rows / columns onto the score matrix with a hash join
        # and gather only the trials -- same vectors, in the key's row-major order, without an (M, S) intermediate.
        mtab, stab = _first_index(self.modelset), _first_index(self.segset)
        rows = numpy.array([mtab.get(m, -1) for m in numpy.asarray(key.modelset).tolist()], dtype=numpy.int64)
        cols = numpy.array([stab.get(x, -1) for x in numpy.asarray(key.segset).tolist()], dtype=numpy.int64)
        if (rows < 0).any():
            logging.info('models reduced from %d to %d', rows.shape[0], int((rows >= 0).sum()))
        if (cols < 0).any():
            logging.info('testsegs reduced from %d to %d', cols.shape[0], int((cols >= 0).sum()))
        n_seg = key.segset.shape[0]
        out = []
        for idx in key.trial_indices():
            r, c = rows[idx // n_seg], cols[idx % n_seg]
            ok = (r >= 0) & (c >= 0)
            r, c = r[ok], c[ok]
            keep = self.scoremask[r, c]
            out.append((r[keep], c[keep]))
        if self._scoremat is None and self.scoremat_device is not None:
            import torch
            dev = self.scoremat_device.device
            flat = self.scoremat_device.reshape(-1)
            n_col = self.scoremat_device.shape[1]
            lin = numpy.concatenate([o[0] * n_col + o[1] for o in out])
            both = flat[torch.from_numpy(lin).to(dev)].cpu().numpy()
            if self.scoremat_dtype is not None:
                both = both.astype(self.scoremat_dtype)
            tar, non = both[:out[0][0].shape[0]], both[out[0][0].shape[0]:]
        else:
            tar, non = self.scoremat[out[0]], self.scoremat[out[1]]
        assert numpy.all(numpy.isfinite(tar)) and numpy.all(numpy.isfinite(non)), 'Inifinite or Nan value in the scoremat'
        return tar, non

    def align_with_ndx(self, ndx):
        """scores.py:181-240: resized / reordered copy that follows ``ndx`` (a Key or an Ndx)."""
        aligned = Scores()
        aligned.modelset, aligned.segset = ndx.modelset, ndx.segset
        mtab, stab = _first_index(self.modelset), _first_index(self.segset)
        mlist, slist = numpy.asarray(ndx.modelset).tolist(), numpy.asarray(ndx.segset).tolist()
        hasmodel = numpy.fromiter((m in mtab for m in mlist), dtype=bool, count=len(mlist))
        hasseg = numpy.fromiter((s in stab for s in slist), dtype=bool, count=len(slist))
        rindx = numpy.array([mtab[m] for m in mlist if m in mtab], dtype=int)
        cindx = numpy.array([stab[s] for s in slist if s in stab], dtype=int)
        rows, cols = numpy.where(hasmodel)[0][:, None], numpy.where(hasseg)[0]
        aligned.scoremat = numpy.zeros((len(mlist), len(slist)))
        aligned.scoremask = numpy.zeros((len(mlist), len(slist)), dtype='bool')
        if rindx.size and cindx.size:
            aligned.scoremat[rows, cols] = self.scoremat[rindx[:, None], cindx]
            aligned.scoremask[rows, cols] = self.scoremask[rindx[:, None], cindx]
        if isinstance(ndx, Ndx):
            aligned.scoremask = aligned.scoremask & ndx.trialmask
        else:
            aligned.scoremask = aligned.scoremask & (ndx.tar | ndx.non)
        if hasmodel.sum() < len(mlist):
            logging.info('models reduced from %d to %d', len(mlist), hasmodel.sum())
        if hasseg.sum() < len(slist):
            logging.info('testsegs reduced from %d to %d', len(slist), hasseg.sum())
        assert numpy.all(numpy.isfinite(aligned.scoremat[aligned.scoremask])), 'Inifinite or Nan value in the scoremat'
        assert aligned.validate(), 'Wrong Score format'
        return aligned

    def sort(self):
        """scores.py:469-478: sort models and segments (in place)."""
        mi, si = numpy.argsort(self.modelset), numpy.argsort(self.segset)
        mask, mat = self.scoremask[mi[:, None], si], self.scoremat[mi[:, None], si]
        self.modelset.sort()
        self.segset.sort()
        self.scoremat, self.scoremask, self.scoremat_device = mat, mask, None
