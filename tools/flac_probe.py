"""FLAC decoding on the device at the size of one extraction batch: 1043 audio-seconds of 16 kHz, 16-bit mono, encoded the
way `flac -5` does (block size 4096, LPC order 8, partition order up to 5) by oracle/flac_ref.py; a few distinct
utterances repeated to fill the batch.

(a) device time of skb_flac_decode on the staged batch (CUDA events, after warm-up; min / median / max over windows),
    and the time of each of its three kernels (torch.profiler, a separate pass);
(b) audio-seconds decoded per second;
(c) bytes copied to the device: the compressed frames against the float32 samples the wav path copies;
(d) wall time of extract_embeddings over the same audio as .flac files and as .wav files (HalfResNet34, median of 3).
Prints the card's name and power limit first.  Usage: python tools/flac_probe.py [--out FILE]."""
import argparse
import os
import subprocess
import sys
import tempfile
import time
import wave

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sidekit_b200 as sk  # noqa: E402
from oracle import flac_ref as R  # noqa: E402
from sidekit_b200 import _lib, flac, synth  # noqa: E402
from tests.models import make_xtractor  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None, help="also write the printed lines to this file")
ap.add_argument("--seconds", type=float, default=1043.0)
args = ap.parse_args()
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


emit("card: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True).stdout.strip().splitlines()[0])
rate = 16000
lengths = [int(s * rate) for s in (4.2, 6.8, 8.1, 9.7, 5.5, 12.3, 7.4, 10.6)]
plan = lambda k: R.FramePlan(subs=[R.SubPlan(kind="lpc", order=8, precision=12, porder=5)])
utts = []
for i, L in enumerate(lengths):
    pcm = (synth.synth_wave(1, L, seed=3000 + i)[0].numpy() * 32768.0).clip(-32768, 32767).astype(numpy.int16)
    utts.append((pcm, R.encode(pcm, rate, 16, blocksize=4096, plan=plan)))
files, total = [], 0
while total < args.seconds * rate:
    files.append(utts[len(files) % len(utts)])
    total += files[-1][0].shape[0]
n_samples = sum(p.shape[0] for p, _ in files)
audio_s = n_samples / rate
emit("batch: %d files, %.1f audio-s, %d frames of 4096" % (len(files), audio_s, sum(-(-p.shape[0] // 4096) for p, _ in files)))

# correctness at this size first
out, n, _ = flac.decode([d for _, d in files])
ref = numpy.concatenate([p.astype(numpy.float32) / numpy.float32(32768) for p, _ in files])
assert numpy.array_equal(out.cpu().numpy(), ref), "decode mismatch"

# (a) the native call alone on a staged batch, as flac.decode makes it
infos = [flac.parse(d) for _, d in files]
blob = numpy.concatenate([numpy.frombuffer(d, numpy.uint8, offset=i.frames_begin) for (_, d), i in zip(files, infos)])
nb = numpy.array([i.frames_end - i.frames_begin for i in infos], numpy.int64)
tot = numpy.array([i.total_samples for i in infos], numpy.int64)
caps = numpy.minimum(-(-tot // numpy.array([i.min_blocksize for i in infos])) + 1, nb // 10 + 1)
table = numpy.stack([numpy.cumsum(nb) - nb, numpy.cumsum(nb), numpy.cumsum(tot) - tot, tot, numpy.cumsum(caps) - caps, caps,
                     numpy.full(len(files), rate), numpy.ones(len(files), numpy.int64), numpy.full(len(files), 16)], axis=1)
bytes_d = torch.from_numpy(blob).cuda()
table_d = torch.from_numpy(numpy.ascontiguousarray(table)).cuda()
out_d = torch.empty(int(tot.sum()), dtype=torch.float32, device="cuda")
status = torch.empty(len(files), dtype=torch.int32, device="cuda")
lib = _lib.lib()
work = torch.empty(int(lib.skb_flac_workspace_bytes(int(nb.sum()), len(files), int(caps.sum()))), dtype=torch.uint8, device="cuda")


def call():
    _lib.check(lib.skb_flac_decode(bytes_d.data_ptr(), int(nb.sum()), table_d.data_ptr(), len(files), int(caps.sum()),
                                   work.data_ptr(), work.numel(), out_d.data_ptr(), status.data_ptr(), _lib.stream_ptr()))


for _ in range(5):
    call()
torch.cuda.synchronize()
assert int(status.abs().sum()) == 0 and torch.equal(out_d, out)
reps, per = [], 20
for _ in range(7):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(per):
        call()
    e1.record()
    torch.cuda.synchronize()
    reps.append(e0.elapsed_time(e1) / per)
reps.sort()
emit("(a) skb_flac_decode device time per batch: min %.3f ms, median %.3f ms, max %.3f ms (7 windows x %d calls)"
     % (reps[0], reps[len(reps) // 2], reps[-1], per))
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(5):
        call()
    torch.cuda.synchronize()
for ev in prof.key_averages():
    if "flac_" in ev.key:
        emit("    %s: %.3f ms per call (torch.profiler, 5 calls)" % (ev.key.split("(")[0].replace("void skb::", ""),
                                                                   ev.device_time_total / 1e3 / 5))
emit("(b) %.2f M audio-s/s decoded (median)" % (audio_s / (reps[len(reps) // 2] * 1e-3) / 1e6))
emit("(c) host-to-device bytes: compressed frames %.2f MB, float32 samples %.2f MB (ratio %.3f); 16-bit PCM would be %.2f MB"
     % (blob.nbytes / 1e6, n_samples * 4 / 1e6, blob.nbytes / (n_samples * 4), n_samples * 2 / 1e6))

# (d) extract_embeddings, .flac against .wav files holding the same audio
m = make_xtractor("halfresnet34", 32, 256).cuda()
with tempfile.TemporaryDirectory() as d:
    for i, (pcm, data) in enumerate(files):
        with open(os.path.join(d, "u%d.flac" % i), "wb") as f:
            f.write(data)
        with wave.open(os.path.join(d, "u%d.wav" % i), "wb") as f:
            f.setnchannels(1); f.setsampwidth(2); f.setframerate(rate)
            f.writeframes(pcm.tobytes())
    im = sk.IdMap()
    im.leftids = numpy.array(["s%d" % i for i in range(len(files))], dtype="|O")
    im.rightids = numpy.array(["u%d" % i for i in range(len(files))], dtype="|O")
    im.start = numpy.empty(len(files), "|O")
    im.stop = numpy.empty(len(files), "|O")
    res = {}
    for ext in ("wav", "flac", "wav", "flac"):
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ss = sk.nnet.extract_embeddings(im, m, d, torch.device("cuda"), file_extension=ext)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        res.setdefault(ext, []).append(sorted(ts)[1])
        res[ext + "_emb"] = ss.stat1
    assert numpy.array_equal(res["wav_emb"], res["flac_emb"]), "flac and wav embeddings differ"
    emit("(d) extract_embeddings wall time over %.1f audio-s (median of 3, two alternating rounds): wav %s s, flac %s s; "
         "embeddings bit-identical" % (audio_s, " / ".join("%.3f" % t for t in res["wav"]), " / ".join("%.3f" % t for t in res["flac"])))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
