"""Pair-list scoring at VoxCeleb1-E shape: 145 160 unit-norm 256-d embeddings (one set serving as enrolment and test),
579 818 trials, a 5 994-row cohort, all generated from seeds on the device.

(a) skb_score_pairs kernel time (CUDA events over many launches, best of 3 windows after warm-up) for the trials in random
    order and grouped by enrolment row (as the real list is), and the gathered bytes per second against bench's HBM figure.
(b) asnorm_trials device time, split into the cohort statistics and the pair kernel with its as-norm epilogue.
(c) cosine_scoring_trials / asnorm_trials / PLDA_scoring_trials end to end through the API (TrialList + StatServer on the
    host -> host scores), wall clock around synchronised calls, with the host id join (TrialList.index) timed on its own.
(d) For context, VoxCeleb1-O shape (4 708 utterances, 37 720 trials, cohort 7 205): the dense path bench.py's
    vox1o_pipeline times (cosine_scoring + get_tar_non, asnorm + get_tar_non) and the pair-list path on the same trials.
Prints the card's name and power limit first.  Usage: python tools/trials_probe.py [--out FILE]."""
import argparse
import os
import subprocess
import sys
import time

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import sidekit_b200 as sk  # noqa: E402
from sidekit_b200 import bulk, synth  # noqa: E402
from sidekit_b200.iv_scoring import _score_pairs  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None, help="also write the printed lines to this file")
args = ap.parse_args()
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


def best_ms(f, steps):
    for i in range(3):
        f(i)
    return min(bench.timed(f, steps, False) for _ in range(3)) / steps


def wall(f, reps=3):
    """Median wall-clock seconds of f() ending in a device synchronise, after one warm-up call."""
    f()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        f()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return sorted(ts)[len(ts) // 2]


dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
emit("card: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True).stdout.strip())
peaks = bench.load_peaks()
emit("HBM bandwidth used for the fraction: %.0f GB/s (bench.load_peaks, source: %s)" % (peaks["hbm_gbs"], peaks["source"]))

N, D, n, C = 145160, 256, 579818, 5994
g = torch.Generator(device=dev).manual_seed(1234)
X = torch.nn.functional.normalize(torch.randn(N, D, device=dev, generator=g), dim=1)
coh = torch.randn(C, D, device=dev, generator=g)
rows = torch.randint(0, N, (n,), device=dev, generator=g, dtype=torch.int32)
cols = torch.randint(0, N, (n,), device=dev, generator=g, dtype=torch.int32)
order = torch.argsort(rows.long(), stable=True)
grouped = (rows[order].contiguous(), cols[order].contiguous())
emit("workload: %d x %d float32 embeddings (%.0f MB; L2 is 126 MB), %d trials, cohort %d x %d" % (N, D, N * D * 4 / 1e6, n, C, D))

# (a) the pair kernel
gathered = 2.0 * n * D * 4                       # the two rows of every trial
other = n * (4 + 4 + 4)                          # two indices and one score per trial
emit("(a) skb_score_pairs, %d trials: %.1f MB of rows gathered + %.1f MB of indices and scores per launch" % (n, gathered / 1e6, other / 1e6))
for name, (r, c) in (("random order", (rows, cols)), ("grouped by enrolment row", grouped)):
    ms = best_ms(lambda i: sk.score_pairs(X, X, r, c), 200)
    emit("  %-26s %.4f ms  %.3e trials/s  %.0f GB/s (rows + indices + scores) = %.2f of the HBM figure (L2 hits can exceed it)"
         % (name, ms, n / ms * 1e3, (gathered + other) / ms / 1e6, (gathered + other) / ms / 1e6 / peaks["hbm_gbs"]))
t_pairs = ms

# (b) asnorm_trials on the device: cohort statistics of all N rows, then the pairs with the as-norm epilogue
cohn = torch.nn.functional.normalize(coh, dim=1).contiguous()
t_stats = best_ms(lambda i: bulk._asnorm_stats_cuda(X, cohn, 200), 10)
mean, std = bulk._asnorm_stats_cuda(X, cohn, 200)
t_apair = best_ms(lambda i: _score_pairs(X, X, grouped[0], grouped[1], asnorm_stats=(mean, std, mean, std)), 200)
emit("(b) asnorm_trials device time: statistics %.3f ms (%d x %d cohort GEMM + top-200) + pairs with as-norm %.4f ms = %.3f ms"
     % (t_stats, N, C, t_apair, t_stats + t_apair))

# (c) through the API, host to host
ids = numpy.array(["id%05d/%011d/%05d.wav" % (10000 + i // 50, i // 7, i % 7) for i in range(N)])
host = X.double().cpu().numpy()
ss = sk.StatServer.from_embeddings(ids, host)
gr, gc = grouped[0].cpu().numpy(), grouped[1].cpu().numpy()
trials = sk.TrialList(ids[gr], ids[gc], numpy.arange(n) % 2 == 0)
cohort_host = coh.cpu()
mu, F, Sigma = synth.synth_plda(D, D, seed=3)
api = {}
emit("(c) API end to end (TrialList + one StatServer for both sides -> host scores), median of 3 after a warm-up:")
t_join = wall(lambda: trials.index(ss.modelset, ss.segset))
emit("  %-36s %.3f s" % ("host id join (TrialList.index)", t_join))
for name, f in (("cosine_scoring_trials", lambda: sk.cosine_scoring_trials(ss, ss, trials).scores),
                ("asnorm_trials", lambda: sk.asnorm_trials(ss, ss, trials, cohort_host).scores),
                ("PLDA_scoring_trials", lambda: sk.PLDA_scoring_trials(ss, ss, trials, mu, F, Sigma).scores)):
    api[name] = wall(f)
    emit("  %-36s %.3f s (join included)" % (name, api[name]))
tar, non = sk.asnorm_trials(ss, ss, trials, cohort_host).get_tar_non()
emit("  as-norm tar / non counts %d / %d; minDCF(0.01) of random embeddings %.4f" % (tar.shape[0], non.shape[0],
     sk.fast_minDCF(tar, non, numpy.log(0.01 / 0.99), normalize=True)[0]))

# (d) VoxCeleb1-O shape: dense path vs pair-list path on the same trials
No, no_ = 4708, 37720
rng = numpy.random.default_rng(55)
emb = synth.synth_embeddings(No, 256, seed=56).astype(numpy.float32)
oids = numpy.array(["utt%05d" % i for i in range(No)])
mi, si = rng.integers(0, No, no_), rng.integers(0, No, no_)
labels = numpy.where(numpy.arange(no_) % 2 == 0, "target", "nontarget")
key = sk.Key(models=oids[mi], testsegs=oids[si], trials=labels)
ndx = key.to_ndx()
oss = sk.StatServer.from_embeddings(oids, emb)
otr = sk.TrialList.from_key(key)
ocoh = torch.randn(7205, 256, generator=torch.Generator().manual_seed(57))


def dense_asnorm():
    Sm = sk.asnorm(torch.from_numpy(emb).to(dev), ocoh, None)
    sn = sk.Scores()
    sn.modelset, sn.segset, sn.scoremat, sn.scoremask = oids, oids, Sm, numpy.ones(Sm.shape, dtype=bool)
    return sn.get_tar_non(key)


emit("(d) VoxCeleb1-O shape (%d utterances, %d trials, cohort 7205), median wall clock of 3 after a warm-up:" % (No, len(otr)))
for name, f in (("dense cosine_scoring + get_tar_non", lambda: sk.cosine_scoring(oss, oss, ndx).get_tar_non(key)),
                ("cosine_scoring_trials + get_tar_non", lambda: sk.cosine_scoring_trials(oss, oss, otr).get_tar_non()),
                ("dense asnorm + get_tar_non", dense_asnorm),
                ("asnorm_trials + get_tar_non", lambda: sk.asnorm_trials(oss, oss, otr, ocoh).get_tar_non())):
    emit("  %-36s %.4f s" % (name, wall(f)))

emit("goals: pair kernel < 1 ms for 580 k trials: %s (%.3f ms grouped); asnorm_trials device time < 20 ms: %s (%.2f ms); "
     "API call < 1 s: %s (slowest %.3f s)" % ("met" if t_pairs < 1.0 else "missed", t_pairs, "met" if t_stats + t_apair < 20 else "missed",
                                              t_stats + t_apair, "met" if max(api.values()) < 1.0 else "missed", max(api.values())))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
