"""Steady-state time of device embedding conditioning (sidekit_b200.conditioning), CUDA events, best of 3 windows after
warm-up, against the host StatServer path on the same data.

Data: 1 000 000 x 256 seeded float32 embeddings on the device in 5 994 classes of uneven size (VoxCeleb2-dev-sized; 1 GB,
larger than L2, so every timed pass reads X from HBM).  Reports scatter() split by Gram launch, whitening with a full sigma,
estimate_spectral_norm + spectral_norm (it = 2, both modes), LDA + WCCN end to end and the host path (including the
device-to-host copy).  Useful FLOPs: N D (D + 1) for a symmetric Gram, 2 N D D_out for an affine pass; rates are given as a
fraction of the float64 DMMA rate measured by tools/dmma_bench.cu (read from --dmma-file, its best all-SM line).
Prints the card's name and power limit first.  Usage: python tools/conditioning_probe.py [--dmma-file F] [--out FILE]"""
import argparse
import os
import re
import subprocess
import sys
import time

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import sidekit_b200 as sk  # noqa: E402
from sidekit_b200 import conditioning as cd  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--dmma-file", default=os.path.join(ROOT, "profiles", "r03_dmma_microbench.txt"))
ap.add_argument("--out", default=None, help="also write the printed lines to this file")
ap.add_argument("--n", type=int, default=1000000)
ap.add_argument("--skip-host", action="store_true")
args = ap.parse_args()
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


def best_ms(f, steps):
    for i in range(2):
        f(i)
    return min(bench.timed(f, steps, False) for _ in range(3)) / steps


emit("card: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True).stdout.strip())
rates = [float(m) for m in re.findall(r"([0-9.]+) TFLOP/s", open(args.dmma_file).read())]
dmma = max(rates)
emit("float64 DMMA rate used for the fractions: %.2f TFLOP/s (best all-SM line of %s)" % (dmma, os.path.basename(args.dmma_file)))

dev = torch.device("cuda", 0)
N, D, C = args.n, 256, 5994
rng = numpy.random.default_rng(2024)
sizes = rng.gamma(2.0, 1.0, C)
sizes = numpy.maximum(1, numpy.floor(sizes / sizes.sum() * N)).astype(numpy.int64)
sizes[numpy.argmax(sizes)] += N - sizes.sum()
lab_host = rng.permutation(numpy.repeat(numpy.arange(C), sizes))
lab = torch.from_numpy(lab_host).to(dev)
g = torch.Generator(device=dev).manual_seed(7)
centres = torch.randn((C, D), device=dev, generator=g, dtype=torch.float64) * 0.5
X = (centres[lab] + torch.randn((N, D), device=dev, generator=g, dtype=torch.float64) * 0.3 + 1.0).float()
del centres
emit("data: %d x %d float32 (%.2f GB), %d classes, sizes %d .. %d" % (N, D, N * D * 4 / 1e9, C, sizes.min(), sizes.max()))


def frac(flop, ms):
    return "%.2f TFLOP/s = %.2f of DMMA" % (flop / (ms * 1e-3) / 1e12, flop / (ms * 1e-3) / 1e12 / dmma)


gram_flop = N * D * (D + 1)
st = cd.scatter(X, lab)
classes = cd._Classes(lab, N, dev)
row_w = (1.0 / st.counts)[classes.idx.long()]
t_stats = best_ms(lambda i: cd._class_stats(X, classes), 5)
emit("scatter(X, labels), split:")
emit("  class statistics (mean + class sums, 2 passes)  %8.3f ms" % t_stats)
grams = [("total", lambda i: cd.gram(X, st.mean, scale=1.0 / N), gram_flop),
         ("within", lambda i: cd.gram(X, st.class_means, classes.idx, scale=1.0 / N), gram_flop),
         ("class_normalised", lambda i: cd.gram(X, st.class_means, classes.idx, row_w), gram_flop),
         ("between (C rows)", lambda i: cd.gram(st.class_means, st.mean, w=st.counts, scale=1.0 / N), C * D * (D + 1)),
         ("Sb (C rows)", lambda i: cd.gram(st.class_means, st.mean), C * D * (D + 1))]
t_three = 0.0
for name, f, fl in grams:
    t = best_ms(f, 5)
    if fl == gram_flop:
        t_three += t
    emit("  Gram %-42s %8.3f ms  %s" % (name, t, frac(fl, t)))
t_scatter = best_ms(lambda i: cd.scatter(X, lab), 3)
emit("  scatter() end to end (integer CUDA labels)      %8.3f ms = %.2f x its three N-row Grams (%.3f ms)"
     % (t_scatter, t_scatter / t_three, t_three))
t_total = best_ms(lambda i: cd.scatter(X), 5)
emit("  scatter() without labels (mean + total)         %8.3f ms" % t_total)

cov = st.total.cpu().numpy()
mu = st.mean.cpu().numpy()
aff_flop = 2.0 * N * D * D
for od in (torch.float32, torch.float64):
    t = best_ms(lambda i: cd.whiten(X, mu, cov, out_dtype=od), 5)
    emit("whiten, full sigma, float32 in, %s out          %8.3f ms  %s" % (str(od).split(".")[1], t, frac(aff_flop, t)))
t = best_ms(lambda i: cd.spectral_norm(X, [mu], [cov], out_dtype=torch.float32), 5)
emit("one spectral-norm round (whiten + unit norm, fused) %7.3f ms  %s" % (t, frac(aff_flop, t)))
for mode in ("efr", "sphNorm"):
    te = best_ms(lambda i: cd.estimate_spectral_norm(X, lab, 2, mode), 2)
    means, covs = cd.estimate_spectral_norm(X, lab, 2, mode)
    ta = best_ms(lambda i: cd.spectral_norm(X, means, covs), 3)
    emit("spectral norm %-7s it=2: estimate %8.3f ms, apply %8.3f ms" % (mode, te, ta))


def lda_wccn(i):
    s1 = cd.scatter(X, lab)
    L = cd.lda_matrix(s1, 200)
    Y = cd._affine(X, None, None, L, out_dtype=torch.float64)
    s2 = cd.scatter(Y, lab)
    return cd._affine(Y, None, None, cd.wccn_cholesky(s2), out_dtype=torch.float32)


t = best_ms(lda_wccn, 2)
emit("LDA (rank 200) + WCCN end to end (2 scatters, host algebra, 2 affine passes) %8.3f ms" % t)

if not args.skip_host:
    ids = lab_host
    t0 = time.perf_counter()
    Xh = X.cpu().numpy()
    ss = sk.StatServer.from_embeddings(ids, Xh)
    t1 = time.perf_counter()
    ss.get_total_covariance_stat1()
    t2 = time.perf_counter()
    ss.get_within_covariance_stat1()
    ss.get_between_covariance_stat1()
    t3 = time.perf_counter()
    L = ss.get_lda_matrix_stat1(200)
    ss.rotate_stat1(L)
    ss.rotate_stat1(ss.get_wccn_choleski_stat1())
    t4 = time.perf_counter()
    w = sk.StatServer.from_embeddings(ids, Xh)
    w.whiten_stat1(mu, cov)
    t5 = time.perf_counter()
    emit("host StatServer path (numpy / scipy, %d threads): D2H + widen %.0f ms, total cov %.0f ms, within + between %.0f ms, "
         "LDA + WCCN %.0f ms, whiten full sigma %.0f ms" % (torch.get_num_threads(), (t1 - t0) * 1e3, (t2 - t1) * 1e3,
                                                            (t3 - t2) * 1e3, (t4 - t3) * 1e3, (t5 - t4) * 1e3))
if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
