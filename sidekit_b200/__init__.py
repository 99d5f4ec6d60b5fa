"""sidekit_b200 -- B200-native drop-in for SIDEKIT's speaker-verification inference hot path.

Public surface mirrors the reference package for that path only (SURVEY.md 8b):
``Xtractor``, the front-end / pooling modules, ``StatServer`` / ``Ndx`` / ``Scores`` containers and
``cosine_scoring`` / ``PLDA_scoring`` / ``fast_PLDA_scoring`` / ``two_covariance_scoring`` / ``asnorm``.
All arithmetic runs in hand-written CUDA kernels for sm_100a behind ``libsidekit_b200.so``
(include/sidekit_b200.h); there is no CPU fallback.
"""
from . import _lib
from .nnet import Xtractor, MeanStdPooling, AttentivePooling, PreHalfResNet34, MfccFrontEnd, MelSpecFrontEnd
from .nnet.xsets import IdMap, IdMapSet

from .bosaris import Ndx, Scores, Key, TrialList, TrialScores
from .statserver import StatServer
from .iv_scoring import cosine_scoring, PLDA_scoring, fast_PLDA_scoring, full_PLDA_scoring, two_covariance_scoring, mahalanobis_scoring, score_matrix
from .iv_scoring import score_topk, cosine_topk, PLDA_topk, TopK
from .iv_scoring import score_pairs, cosine_scoring_trials, PLDA_scoring_trials
from .score_normalization import asnorm, znorm, tnorm, ztnorm, asnorm_trials
from . import detplot
from .detplot import pavx, rocch, rocch2eer, fast_minDCF, eer
from .factor_analyser import FactorAnalyser
from . import kaldi_io
from . import bulk
from . import conditioning
from .bulk import extract_embeddings

__version__ = "0.1.0"
