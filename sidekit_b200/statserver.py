"""``StatServer`` as the container the scoring functions take (sidekit/statserver.py:202-304) plus the helpers on the
hot path (:656-684 align_*, :797-817 norm / rotate / center, :1357-1374 mean per model) and the embedding-conditioning
functions that feed PLDA (SURVEY.md 8f rank 3: :789-795 mean, :852-918 whitening, :920-1054 covariances / LDA / WCCN /
Mahalanobis, :1279-1333 spectral normalisation, :1335-1355 sums per model).  The per-speaker Python loops of the reference
are replaced by one pass over ``numpy.unique(..., return_inverse=True)`` (same float64 results up to summation order).
GMM / i-vector statistics, EM and HDF5 IO are out of scope.
"""
import copy

import numpy
import scipy.linalg

STAT_TYPE = numpy.float64


def _first_index(have, wanted):
    """Index of the FIRST occurrence of every wanted id (``numpy.argwhere(have == v)[0][0]``), O(N) hash join."""
    pos = {}
    for i, v in enumerate(have.tolist()):
        if v not in pos:
            pos[v] = i
    try:
        return numpy.fromiter((pos[v] for v in wanted.tolist()), dtype=numpy.int64, count=wanted.shape[0])
    except KeyError as e:       # the reference raises IndexError from argwhere(...)[0]
        raise IndexError("id %s not found" % (e,))


# D x D algebra of the conditioning functions, shared by the host methods below and by ``conditioning`` (the device path)
def _inverse_sqrt_factor(sigma):
    """``V diag(lambda^-1/2)`` of a symmetric matrix, eigenvalues in DESCENDING order (the column order fixes the
    coordinates of the whitened vectors, so it is part of the contract)."""
    lam, vec = scipy.linalg.eigh(sigma)
    order = numpy.argsort(lam.real)[::-1]
    return vec.real[:, order] / numpy.sqrt(lam.real[order])


def _cholesky_whitener(sigma):
    """Lower Cholesky factor of the precision ``sigma^-1`` (statserver.py:898-918)."""
    return scipy.linalg.cholesky(scipy.linalg.inv(sigma), lower=True)


def _lda_from_scatter(Sb, Sw, rank):
    """statserver.py:982-1018 from its two scatter matrices (including its ``eigh`` of the non-symmetric discrimination
    matrix)."""
    disc = numpy.dot(Sb, scipy.linalg.inv(Sw)).transpose()
    eigen_values, eigen_vectors = scipy.linalg.eigh(disc)
    idx = eigen_values.real.argsort()[-rank:][::-1]
    return eigen_vectors.real[:, idx]


def _wccn_from_scatter(class_normalised, n_models):
    """statserver.py:1030-1054 from the class-normalised within-class scatter."""
    return scipy.linalg.cholesky(scipy.linalg.inv(class_normalised / n_models)).T


class StatServer:
    def __init__(self, statserver_file_name=None):
        if statserver_file_name is not None and not isinstance(statserver_file_name, StatServer):
            raise NotImplementedError("StatServer file IO / IdMap construction is out of scope")
        self.modelset = numpy.empty(0, dtype="|O")
        self.segset = numpy.empty(0, dtype="|O")
        self.start = numpy.empty(0, dtype="|O")
        self.stop = numpy.empty(0, dtype="|O")
        self.stat0 = numpy.array([], dtype=STAT_TYPE)
        self.stat1 = numpy.array([], dtype=STAT_TYPE)

    @classmethod
    def from_embeddings(cls, ids, embeddings):
        """What ``extract_embeddings`` builds (xvector.py:1905-1914): stat1 = embeddings, stat0 = ones."""
        s = cls()
        s.modelset = numpy.asarray(ids)
        s.segset = numpy.asarray(ids)
        s.start = numpy.empty(len(ids), dtype="|O")
        s.stop = numpy.empty(len(ids), dtype="|O")
        s.stat0 = numpy.ones((len(ids), 1), dtype=STAT_TYPE)
        s.stat1 = numpy.asarray(embeddings, dtype=STAT_TYPE)
        return s

    def validate(self, warn=False):
        ok = self.modelset.ndim == 1 and self.modelset.shape == self.segset.shape == self.start.shape == self.stop.shape
        ok &= self.stat0.shape[0] == self.stat1.shape[0] == self.modelset.shape[0]
        return bool(ok)

    def _take(self, indx):
        self.segset = self.segset[indx]
        self.modelset = self.modelset[indx]
        self.start = self.start[indx]
        self.stop = self.stop[indx]
        self.stat0 = self.stat0[indx, :]
        self.stat1 = self.stat1[indx, :]

    def align_segments(self, segment_list):
        self._take(_first_index(self.segset, numpy.asarray(segment_list)))

    def align_models(self, model_list):
        self._take(_first_index(self.modelset, numpy.asarray(model_list)))

    def norm_stat1(self):
        """Length normalisation (statserver.py:797-802): rows scaled to unit Euclidean norm (norms floored at 1e-8)."""
        self.stat1 = self.stat1 / numpy.maximum(numpy.linalg.norm(self.stat1, axis=1, keepdims=True), 1e-08)

    def rotate_stat1(self, R):
        """statserver.py:804-810."""
        self.stat1 = self.stat1 @ R

    def center_stat1(self, mu):
        """statserver.py:812-817: ``stat1 -= stat0 (per distribution, broadcast over its block of stat1) * mu``."""
        block = self.stat1.shape[1] // self.stat0.shape[1]
        self.stat1 = self.stat1 - numpy.repeat(self.stat0, block, axis=1) * mu.astype(STAT_TYPE)

    def mean_stat_per_model(self):
        out = StatServer()
        out.modelset, inv = numpy.unique(self.modelset, return_inverse=True)
        out.segset = copy.deepcopy(out.modelset)
        n = out.modelset.shape[0]
        counts = numpy.bincount(inv, minlength=n).astype(STAT_TYPE)[:, None]
        out.stat0 = numpy.zeros((n, self.stat0.shape[1]), dtype=STAT_TYPE)
        out.stat1 = numpy.zeros((n, self.stat1.shape[1]), dtype=STAT_TYPE)
        numpy.add.at(out.stat0, inv, self.stat0)
        numpy.add.at(out.stat1, inv, self.stat1)
        out.stat0 /= counts
        out.stat1 /= counts
        out.start = numpy.empty(out.segset.shape, "|O")
        out.stop = numpy.empty(out.segset.shape, "|O")
        return out

    # ------------------------------------------------------------------ embedding conditioning (SURVEY.md 8f rank 3)
    def get_mean_stat1(self):
        """statserver.py:789-795."""
        return numpy.mean(self.stat1, axis=0)

    def get_model_stat0(self, mod_id):
        return self.stat0[self.modelset == mod_id, :]

    def get_model_stat1(self, mod_id):
        return self.stat1[self.modelset == mod_id, :]

    # accessors of statserver.py:574-654 (the k-th model is the k-th SORTED unique model id, a segment index is a row)
    def get_model_stat0_by_index(self, mod_idx):
        return self.stat0[self.modelset == numpy.unique(self.modelset)[mod_idx], :]

    def get_model_stat1_by_index(self, mod_idx):
        return self.stat1[self.modelset == numpy.unique(self.modelset)[mod_idx], :]

    def get_segment_stat0(self, seg_id):
        return self.stat0[self.segset == seg_id, :]

    def get_segment_stat1(self, seg_id):
        return self.stat1[self.segset == seg_id, :]

    def get_segment_stat0_by_index(self, seg_idx):
        return self.stat0[seg_idx, :]

    def get_segment_stat1_by_index(self, seg_idx):
        return self.stat1[seg_idx, :]

    def get_model_segments(self, mod_id):
        return self.segset[self.modelset == mod_id]

    def get_model_segments_by_index(self, mod_idx):
        # the reference indexes the 1-D segset with [mask, :] here (statserver.py:654) and raises IndexError; the intent is clear
        return self.segset[self.modelset == numpy.unique(self.modelset)[mod_idx]]

    def merge(*arg):
        """statserver.py:337-388: one StatServer with every distinct (model, segment, start, stop) session of the arguments
        (the later one wins when a session is repeated).  Rows come in first-occurrence order; the reference's row order is
        the iteration order of a Python ``set`` of strings, i.e. unspecified."""
        assert all(isinstance(ss, StatServer) and ss.validate() for ss in arg), "Arguments must be proper StatServers"
        d0, d1 = arg[0].stat0.shape[1], arg[0].stat1.shape[1]
        assert all(ss.stat0.shape[1] == d0 and ss.stat1.shape[1] == d1 for ss in arg), "Stat dimensions are not consistent"
        index, rows = {}, []
        for k, ss in enumerate(arg):
            for i, key in enumerate(zip(ss.modelset.tolist(), ss.segset.tolist(), map(str, ss.start), map(str, ss.stop))):
                if key not in index:
                    index[key] = len(rows)
                    rows.append((k, i))
                else:
                    rows[index[key]] = (k, i)
        if len(rows) != sum(ss.modelset.shape[0] for ss in arg):
            print("WARNING: duplicated segmentID in input StatServers")
        out = StatServer()
        n = len(rows)
        out.modelset, out.segset = numpy.empty(n, dtype="object"), numpy.empty(n, dtype="object")
        out.start, out.stop = numpy.empty(n, dtype="object"), numpy.empty(n, dtype="object")
        out.stat0, out.stat1 = numpy.zeros((n, d0), dtype=STAT_TYPE), numpy.zeros((n, d1), dtype=STAT_TYPE)
        for r, (k, i) in enumerate(rows):
            ss = arg[k]
            out.modelset[r], out.segset[r], out.start[r], out.stop[r] = ss.modelset[i], ss.segset[i], ss.start[i], ss.stop[i]
            out.stat0[r], out.stat1[r] = ss.stat0[i], ss.stat1[i]
        assert out.validate(), "Problem in StatServer Merging"
        return out

    def _classes(self):
        """(sorted unique models, class index of every session, sessions per class, class means)."""
        models, inv = numpy.unique(self.modelset, return_inverse=True)
        counts = numpy.bincount(inv, minlength=models.shape[0]).astype(STAT_TYPE)
        sums = numpy.zeros((models.shape[0], self.stat1.shape[1]), dtype=STAT_TYPE)
        numpy.add.at(sums, inv, self.stat1)
        return models, inv, counts, sums / counts[:, None]

    def sum_stat_per_model(self):
        """statserver.py:1335-1355: ``(StatServer of per-model sums, sessions per model)``."""
        out = StatServer()
        out.modelset, inv = numpy.unique(self.modelset, return_inverse=True)
        out.segset = copy.deepcopy(out.modelset)
        n = out.modelset.shape[0]
        out.stat0 = numpy.zeros((n, self.stat0.shape[1]), dtype=STAT_TYPE)
        out.stat1 = numpy.zeros((n, self.stat1.shape[1]), dtype=STAT_TYPE)
        numpy.add.at(out.stat0, inv, self.stat0)
        numpy.add.at(out.stat1, inv, self.stat1)
        out.start = numpy.empty(out.segset.shape, "|O")
        out.stop = numpy.empty(out.segset.shape, "|O")
        return out, numpy.bincount(inv, minlength=n).astype(STAT_TYPE)

    def whiten_stat1(self, mu, sigma, isSqrInvSigma=False):
        """statserver.py:852-896: centre, then whiten with a diagonal (1-D ``sigma``) or full (2-D) covariance; with
        ``isSqrInvSigma`` the 2-D argument already is the whitening matrix."""
        if sigma.ndim not in (1, 2):
            raise Exception('Wrong dimension of Sigma, must be 1 or 2')
        self.center_stat1(mu)
        if sigma.ndim == 1:
            self.stat1 = self.stat1 / numpy.sqrt(sigma.astype(STAT_TYPE))
        else:
            self.rotate_stat1(sigma if isSqrInvSigma else _inverse_sqrt_factor(sigma))

    def whiten_cholesky_stat1(self, mu, sigma):
        """statserver.py:898-918: as ``whiten_stat1`` with the lower Cholesky factor of the precision as whitening matrix."""
        if sigma.ndim not in (1, 2):
            raise Exception('Wrong dimension of Sigma, must be 1 or 2')
        self.center_stat1(mu)
        if sigma.ndim == 1:
            self.stat1 = self.stat1 / numpy.sqrt(sigma)
        else:
            self.stat1 = self.stat1 @ _cholesky_whitener(sigma)

    def get_total_covariance_stat1(self):
        """statserver.py:920-928."""
        C = self.stat1 - self.stat1.mean(axis=0)
        return numpy.dot(C.transpose(), C) / self.stat1.shape[0]

    def get_within_covariance_stat1(self):
        """statserver.py:940-956: sum_c sum_{x in c} (x - m_c)(x - m_c)' / N."""
        _, inv, _, means = self._classes()
        C = self.stat1 - means[inv]
        return numpy.dot(C.transpose(), C) / self.stat1.shape[0]

    def get_between_covariance_stat1(self):
        """statserver.py:958-980: sum_c n_c (m_c - mu)(m_c - mu)' / N."""
        _, _, counts, means = self._classes()
        D = means - self.get_mean_stat1()
        return numpy.dot(D.transpose() * counts, D) / self.stat1.shape[0]

    def _class_normalised_scatter(self):
        """sum_c (1 / n_c) sum_{x in c} (x - m_c)(x - m_c)' (the Sw of the LDA / the WCCN accumulator)."""
        models, inv, counts, means = self._classes()
        C = (self.stat1 - means[inv]) / numpy.sqrt(counts[inv])[:, None]
        return models, means, numpy.dot(C.transpose(), C)

    def get_lda_matrix_stat1(self, rank):
        """statserver.py:982-1018 (including its ``eigh`` of the non-symmetric discrimination matrix)."""
        _, means, Sw = self._class_normalised_scatter()
        class_means = means - self.get_mean_stat1()
        Sb = numpy.dot(class_means.transpose(), class_means)
        return _lda_from_scatter(Sb, Sw, rank)

    def get_mahalanobis_matrix_stat1(self):
        """statserver.py:1020-1028."""
        return scipy.linalg.inv(self.get_within_covariance_stat1())

    def get_wccn_choleski_stat1(self):
        """statserver.py:1030-1054."""
        models, _, scatter = self._class_normalised_scatter()
        return _wccn_from_scatter(scatter, models.shape[0])

    def estimate_spectral_norm_stat1(self, it=1, mode='efr'):
        """statserver.py:1279-1314: the (mean, covariance) pairs of ``it`` rounds of "whiten, then length-normalise", each
        estimated on the output of the round before.  ``mode``: 'efr' = total covariance, 'sphNorm' = within-class."""
        covariance_of = {'efr': StatServer.get_total_covariance_stat1, 'sphNorm': StatServer.get_within_covariance_stat1}
        work = copy.deepcopy(self)
        means, covs = [], []
        for _ in range(it):
            means.append(work.get_mean_stat1())
            if mode in covariance_of:                 # (any other mode: the reference appends no covariance and fails below)
                covs.append(covariance_of[mode](work))
            work.spectral_norm_stat1(means[-1:], covs[-1:])
        return means, covs

    def spectral_norm_stat1(self, spectral_norm_mean, spectral_norm_cov, is_sqr_inv_sigma=False):
        """statserver.py:1316-1333: apply the rounds estimated above."""
        assert len(spectral_norm_mean) == len(spectral_norm_cov), \
            'Number of mean vectors and covariance matrices is different'
        for mean, cov in zip(spectral_norm_mean, spectral_norm_cov):
            self.whiten_stat1(mean, cov, is_sqr_inv_sigma)
            self.norm_stat1()
