"""WAV / SPHERE decoding on the device at the size of one extraction batch: 1043 audio-seconds as 130 mono files, once as
16 kHz 16-bit WAV and once as 8 kHz mu-law NIST SPHERE; a few distinct utterances repeated to fill the batch.

(a) device time of skb_pcm_decode on the staged batch (CUDA events over repeated calls, after warm-up; min / median / max
    over windows), and the kernel's row in torch.profiler (a separate pass);
(b) bytes copied to the device per batch: the sample bytes against the float32 samples of a host decode;
(c) wall time of extract_embeddings over the 16-bit WAV files (HalfResNet34), median of several calls per round, with
    the embeddings compared bit for bit against read_wav + extract_varlen.  Then a breakdown of one call: reading the
    files, a batched decode call over them, and the rest (Python and extraction).
Prints the card's name and power limit first.  Usage: python tools/pcm_probe.py [--out FILE]."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sidekit_b200 as sk  # noqa: E402
from oracle import pcm_ref as R  # noqa: E402
from sidekit_b200 import audio, pcm, synth  # noqa: E402
from sidekit_b200.nnet import xsets  # noqa: E402
from tests.models import make_xtractor  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None, help="also write the printed lines to this file")
ap.add_argument("--seconds", type=float, default=1043.0)
ap.add_argument("--rounds", type=int, default=3)
args = ap.parse_args()
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


emit("card: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True).stdout.strip().splitlines()[0])
secs = (4.2, 6.8, 8.1, 9.7, 5.5, 12.3, 7.4, 10.6)
utts = [(synth.synth_wave(1, int(s * 16000), seed=3000 + i)[0].numpy() * 32768.0).clip(-32768, 32767).astype(numpy.int64)
        for i, s in enumerate(secs)]
files16, total = [], 0
while total < args.seconds * 16000:
    files16.append(utts[len(files16) % len(utts)])
    total += files16[-1].shape[0]
table_u = R.ulaw2lin(numpy.arange(256)).astype(numpy.int64)
order_u = numpy.argsort(table_u)
batches = {
    "16 kHz 16-bit WAV": [R.wav_bytes(x[:, None], 16000, "pcm", 2) for x in files16],
    "8 kHz mu-law SPHERE": [R.sph_bytes(order_u[numpy.clip(numpy.searchsorted(table_u[order_u], x[::2]), 0, 255)].astype(numpy.uint8)[:, None],
                                        8000, "ulaw", 1) for x in files16],
}
for label, datas in batches.items():
    infos = [pcm.parse(d) for d in datas]
    n = numpy.array([i.frames for i in infos], numpy.int64)
    rate = infos[0].sample_rate
    emit("batch %s: %d files, %.1f audio-s, %d samples" % (label, len(datas), n.sum() / rate, n.sum()))
    out, lengths, _ = audio.decode(datas)                             # correctness at this size first
    ref = numpy.concatenate([R.decode(d)[1] for d in datas])
    assert numpy.array_equal(out.cpu().numpy(), ref), "decode mismatch"
    # the native call alone on the batch staged as audio.decode stages it: each file's samples at a 16-byte boundary
    nbytes = [pcm.data_bytes(i) for i in infos]
    begin = numpy.cumsum([0] + [(b + 15) & ~15 for b in nbytes])[:-1]
    blob = numpy.zeros(int(begin[-1] + nbytes[-1]), numpy.uint8)
    for d, i, b0, nb in zip(datas, infos, begin, nbytes):
        blob[b0:b0 + nb] = numpy.frombuffer(d, numpy.uint8, count=nb, offset=i.data_begin)
    tab, n_tiles = pcm.table(infos, begin, numpy.cumsum(n) - n)
    bytes_d = torch.from_numpy(blob).cuda()
    tab_d = torch.from_numpy(tab).cuda()
    out_d = torch.empty(int(n.sum()), dtype=torch.float32, device="cuda")

    def call():
        pcm.launch(bytes_d.data_ptr(), tab_d.data_ptr(), len(datas), n_tiles, out_d.data_ptr())

    for _ in range(5):
        call()
    torch.cuda.synchronize()
    assert torch.equal(out_d, out)
    reps, per = [], 50
    for _ in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(per):
            call()
        e1.record()
        torch.cuda.synchronize()
        reps.append(e0.elapsed_time(e1) / per)
    reps.sort()
    med = reps[len(reps) // 2]
    emit("(a) skb_pcm_decode device time per batch: min %.4f ms, median %.4f ms, max %.4f ms (7 windows x %d calls); "
         "%.1f M audio-s/s, %.0f GB/s of bytes read + float32 written (working set in L2)"
         % (reps[0], med, reps[-1], per, n.sum() / rate / (med * 1e-3) / 1e6, (blob.nbytes + n.sum() * 4) / (med * 1e-3) / 1e9))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            call()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "pcm_" in ev.key:
            emit("    %s: %.4f ms per call (torch.profiler, 5 calls)" % (ev.key.split("(")[0].replace("void skb::", ""),
                                                                    ev.device_time_total / 1e3 / 5))
    emit("(b) host-to-device bytes per batch: samples %.2f MB (+ table %.1f kB) against %.2f MB as float32 (ratio %.3f)"
         % (blob.nbytes / 1e6, tab.nbytes / 1e3, n.sum() * 4 / 1e6, blob.nbytes / (n.sum() * 4)))

# (c) extract_embeddings from 16-bit WAV (the streamed window pipeline), checked against read_wav + extract_varlen
m = make_xtractor("halfresnet34", 32, 256).cuda()
with tempfile.TemporaryDirectory() as d:
    for i, data in enumerate(batches["16 kHz 16-bit WAV"]):
        with open(os.path.join(d, "u%d.wav" % i), "wb") as f:
            f.write(data)
    im = sk.IdMap()
    im.leftids = numpy.array(["s%d" % i for i in range(len(files16))], dtype="|O")
    im.rightids = numpy.array(["u%d" % i for i in range(len(files16))], dtype="|O")
    im.start = numpy.empty(len(files16), "|O")
    im.stop = numpy.empty(len(files16), "|O")

    def run():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ss = sk.nnet.extract_embeddings(im, m, d, torch.device("cuda"))
        torch.cuda.synchronize()
        return time.perf_counter() - t0, ss.stat1

    run()                                                            # warm-up: every batch geometry, the page cache
    res, emb = [], None
    for _ in range(args.rounds):
        ts = []
        for _ in range(3):
            t, emb = run()
            ts.append(t)
        res.append(sorted(ts)[1])
    ref = m.extract_varlen([xsets.read_wav(os.path.join(d, "u%d.wav" % i))[0].cuda() for i in range(len(files16))]).cpu().numpy()
    assert numpy.array_equal(emb, ref), "extract_embeddings differs from read_wav + extract_varlen"
    emit("(c) extract_embeddings wall time over %.1f audio-s of 16-bit WAV (median of 3 per round, %d rounds): %s s; "
         "embeddings bit-identical to read_wav + extract_varlen" % (total / 16000, args.rounds, " / ".join("%.3f" % t for t in res)))
    paths = [os.path.join(d, "u%d.wav" % i) for i in range(len(files16))]
    tr, td = [], []
    for _ in range(5):
        t0 = time.perf_counter()
        for p in paths:
            with open(p, "rb") as f:
                f.read()
        tr.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        audio.decode(paths, torch.device("cuda"))
        torch.cuda.synchronize()
        td.append(time.perf_counter() - t0)
    t_read, t_dec, t_all = sorted(tr)[2], sorted(td)[2], sorted(res)[len(res) // 2]
    emit("    device path breakdown (medians): reading the 130 files %.1f ms (%.0f %%), the whole decode call incl. that "
         "read, parse, staging and copy %.1f ms (%.0f %%), Python and extraction %.1f ms (%.0f %%) of %.1f ms"
         % (t_read * 1e3, 100 * t_read / t_all, t_dec * 1e3, 100 * t_dec / t_all, (t_all - t_dec) * 1e3,
            100 * (t_all - t_dec) / t_all, t_all * 1e3))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
