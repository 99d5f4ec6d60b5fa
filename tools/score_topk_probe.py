"""Steady-state time of top-k scoring (score_topk) against its baselines, CUDA events, best of 3 windows after warm-up.

(a) 20k x 20k x 256 unit-norm, gallery packed once: k = 1, 10, 32 (selection in the GEMM epilogue) and k = 100, 200 (row
    panels of the score matrix + per-row select); baselines: the trial-list mode at the vox1-O density and the float32
    score_matrix followed by torch.topk.
(b) 2 000 queries x 1 000 000-row gallery x 256, k = 10 (as a float32 matrix that would be 8 GB).
Prints the card's name and power limit first.  Usage: python tools/score_topk_probe.py [--out FILE] (--out also writes the
printed lines to FILE)."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import sidekit_b200 as sk  # noqa: E402
from sidekit_b200 import synth  # noqa: E402
from sidekit_b200.iv_scoring import PackedEmbeddings, TrialIndex, score_topk, score_trials  # noqa: E402

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


dev = torch.device("cuda", 0)
emit("card: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True).stdout.strip())
peaks = bench.load_peaks()
emit("bf16 sustained peak used for the fraction: %.1f TFLOP/s (%s)" % (peaks["tf_sustained"], peaks["source"]))

N, D = 20000, 256
E = torch.from_numpy(synth.synth_embeddings(N, D, seed=6)).float().to(dev)
T = torch.from_numpy(synth.synth_embeddings(N, D, seed=7)).float().to(dev)
Tp = PackedEmbeddings(T)
flop = 2.0 * N * N * D
g = torch.Generator(device=dev).manual_seed(99)
mask = torch.rand((N, N), device=dev, generator=g) < (37720.0 / 4708.0 ** 2)
idx = TrialIndex(mask, dev)
o32 = torch.empty((N, N), dtype=torch.float32, device=dev)
emit("(a) %d x %d x %d, unit-norm, gallery packed once, passes=0" % (N, N, D))
t_trial = best_ms(lambda i: score_trials(E, Tp, idx, passes=0), 20)
emit("  %-40s %.4f ms  %.3e trials/s  %.2f of the bf16 sustained peak" % ("trial list (vox1-O density)", t_trial, N * N / t_trial * 1e3,
                                                                         flop / (t_trial / 1e3) / 1e12 / peaks["tf_sustained"]))


def matrix_topk(k):
    sk.score_matrix(E, Tp, passes=0, out=o32)
    return torch.topk(o32, k, dim=1)


for k in (1, 10, 32, 100, 200):
    t = best_ms(lambda i: score_topk(E, Tp, k, passes=0), 10)
    tb = best_ms(lambda i: matrix_topk(k), 5)
    frac = " %.2f of the bf16 sustained peak" % (flop / (t / 1e3) / 1e12 / peaks["tf_sustained"]) if k <= 32 else ""
    emit("  k = %-4d %-6s score_topk %.4f ms  %.3e trials/s%s | matrix + torch.topk %.4f ms (%.2fx) | vs trial list %.2fx"
         % (k, "fused" if k <= 32 else "panel", t, N * N / t * 1e3, frac, tb, tb / t, t / t_trial))
# the selected values are the matrix entries
v, i = score_topk(E, Tp, 10, passes=0)
sk.score_matrix(E, Tp, passes=0, out=o32)
emit("  k = 10 values == score_matrix entries: %s" % bool(torch.equal(v, torch.gather(o32, 1, i))))
del o32, mask, idx, Tp, E, T
torch.cuda.empty_cache()

Nq, Ng = 2000, 1000000
Q = torch.nn.functional.normalize(torch.randn((Nq, D), device=dev, generator=g), dim=1)
G = torch.nn.functional.normalize(torch.randn((Ng, D), device=dev, generator=g), dim=1)
Gp = PackedEmbeddings(G)
del G
t = best_ms(lambda i: score_topk(Q, Gp, 10, passes=0), 5)
fl = 2.0 * Nq * Ng * D
emit("(b) %d queries x %d gallery x %d, k = 10: %.4f ms  %.3e trials/s  %.2f of the bf16 sustained peak"
     % (Nq, Ng, D, t, Nq * Ng / t * 1e3, fl / (t / 1e3) / 1e12 / peaks["tf_sustained"]))
if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
