"""Outputs of the score-GEMM paths on seeded inputs, to compare two builds bit for bit.

    SKB_LIB_PATH=old/libsidekit_b200.so python tools/score_dump.py dump old.npz
    SKB_LIB_PATH=new/libsidekit_b200.so python tools/score_dump.py dump new.npz
    python tools/score_dump.py compare old.npz new.npz      # exit 1 unless every array is numpy.array_equal

Covers score_matrix (float32 / float64 / float16 output, D in {64, 200, 256, 320, 512}, passes 0 / 1 / 3, unit-norm and
N(0,1) rows, 1 x 33, 257 x 129 and 1000 x 777), score_trials (D <= 256, with and without a column term), score_topk
(k = 1, 10, 32, 100), the test side packed once, the symmetric as-norm matrix and its statistics, PLDA and Mahalanobis
scoring."""
import os
import sys

import numpy

SHAPES = ((1, 33), (257, 129), (1000, 777))
DIMS = (64, 200, 256, 320, 512)
PASSES = (0, 1, 3)


def dump(path):
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import sidekit_b200 as sk
    from sidekit_b200 import bulk, synth
    from sidekit_b200.iv_scoring import PackedEmbeddings, score_topk, score_trials

    dev = torch.device("cuda", 0)
    rng = numpy.random.default_rng(0)
    out = {}

    def put(name, t):
        out[name] = t.cpu().numpy() if torch.is_tensor(t) else numpy.asarray(t)

    def vec(n):
        return torch.from_numpy(rng.standard_normal(n).astype(numpy.float32)).to(dev)

    for D in DIMS:
        for unit in (True, False):
            for Ne, Nt in SHAPES:
                E = torch.from_numpy(synth.synth_embeddings(Ne, D, seed=Ne + D, unit_norm=unit)).float().to(dev)
                T = torch.from_numpy(synth.synth_embeddings(Nt, D, seed=Nt + D + 1, unit_norm=unit)).float().to(dev)
                r, q = vec(Ne), vec(Nt)
                mask = rng.random((Ne, Nt)) < 0.3
                for passes in PASSES:
                    key = "D%d_%s_%dx%d_p%d" % (D, "unit" if unit else "normal", Ne, Nt, passes)
                    for dt in (torch.float32, torch.float64, torch.float16):
                        put("matrix_%s_%s" % (key, str(dt)[6:]), sk.score_matrix(E, T, r, q, cst=0.25, alpha=1.5, passes=passes, out_dtype=dt))
                    if D <= 256:
                        put("trials_%s" % key, score_trials(E, T, mask, r, q, cst=0.25, alpha=1.5, passes=passes))
                        put("trials_noq_%s" % key, score_trials(E, T, mask, r, None, cst=0.25, alpha=1.5, passes=passes))
                    for k in (1, 10, 32, 100):
                        if k <= Nt:
                            v, i = score_topk(E, T, k, r, q, cst=0.25, alpha=1.5, passes=passes)
                            put("topk%d_val_%s" % (k, key), v)
                            put("topk%d_idx_%s" % (k, key), i)
                put("packed_D%d_%s_%dx%d" % (D, unit, Ne, Nt), sk.score_matrix(E, PackedEmbeddings(T), r, q, cst=0.25, alpha=1.5, passes=0))

    # symmetric as-norm: the column term ca takes the generic epilogue
    X = torch.nn.functional.normalize(torch.from_numpy(synth.synth_embeddings(700, 256, seed=21, unit_norm=False)).float(), dim=1).to(dev)
    coh = torch.nn.functional.normalize(torch.from_numpy(rng.standard_normal((1500, 256)).astype(numpy.float32)), dim=1).to(dev)
    mean, std = bulk._asnorm_stats_cuda(X, coh, 200)
    put("asnorm_mean", mean)
    put("asnorm_std", std)
    put("asnorm_matrix", bulk._asnorm_panel_cuda(X, 0, 700, mean, std))

    # PLDA and Mahalanobis scoring (the quadratic preparation's D x D GEMMs)
    for D in (64, 200, 256):
        E, T = synth.synth_embeddings(300, D, seed=31), synth.synth_embeddings(257, D, seed=32)
        ids_e = numpy.array(["m%03d" % i for i in range(300)])
        ids_t = numpy.array(["s%03d" % i for i in range(257)])
        ndx = sk.Ndx()
        ndx.modelset, ndx.segset, ndx.trialmask = ids_e, ids_t, rng.random((300, 257)) < 0.5
        ss = lambda ids, Y: sk.StatServer.from_embeddings(ids, Y)
        mu, F, Sigma = synth.synth_plda(D, D, seed=33)
        put("plda_D%d" % D, sk.PLDA_scoring(ss(ids_e, E), ss(ids_t, T), ndx, mu, F, numpy.zeros((D, 0)), Sigma).scoremat)
        M = numpy.linalg.inv(Sigma) + 0.05 * numpy.triu(F @ F.T)
        put("mahalanobis_D%d" % D, sk.mahalanobis_scoring(ss(ids_e, E), ss(ids_t, T), ndx, M).scoremat)
    numpy.savez(path, **out)
    print("%d arrays -> %s" % (len(out), path))


def compare(a_path, b_path):
    a, b = numpy.load(a_path), numpy.load(b_path)
    bad = sorted(set(a.files) ^ set(b.files))
    for name in sorted(set(a.files) & set(b.files)):
        if not numpy.array_equal(a[name], b[name]):
            bad.append(name)
    print("%d arrays compared, %d differ%s" % (len(set(a.files) | set(b.files)), len(bad), (": " + " ".join(bad)) if bad else ""))
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "dump":
        dump(sys.argv[2])
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
