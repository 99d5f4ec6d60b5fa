"""Corpus extraction from disk: ``extract_xvectors.main`` over a synthetic corpus written from a seed, at world 1 and at
world = every visible GPU (spawned processes, NCCL).  Prints one JSON line per run.

The corpus: ``--files`` utterances of 2-20 s (the config-4 law, ``synth.synth_lengths``), 16-bit WAV, a tenth of them at
8 kHz and a tenth FLAC (``oracle.flac_ref.encode``; a few distinct encodes are reused, the pure-Python encoder being
slow).  It is written once and read once before the timed runs, so it is page-cached.

    python tools/corpus_probe.py --files 10000 --corpus /tmp/corpus --out <dir>   [--tree <other checkout>] [--worlds 1,8]

``--tree`` imports ``sidekit_b200`` from another checkout (an older commit: its ``main`` may lack the per-window
``stats``, then only wall-clock figures are printed; without ``sidekit_b200/corpus.py`` its ``main`` does not shard, so
only world 1 is run).  Per window the JSON gives the host seconds of reading, parsing and
staging (the reading thread) against the device seconds (CUDA events), and the share of wall time the device is idle.
"""
import argparse
import json
import os
import socket
import subprocess
import sys
import tempfile
import time

import numpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def write_corpus(d, n, seed):
    sys.path.insert(0, ROOT)
    from oracle import flac_ref, pcm_ref
    from sidekit_b200 import synth
    lengths = synth.synth_lengths(n, 2.0, 20.0, seed=seed)
    rng = numpy.random.default_rng(seed)
    kinds = rng.choice(3, size=n, p=[0.8, 0.1, 0.1])            # 0: WAV 16 kHz, 1: WAV 8 kHz, 2: FLAC 16 kHz
    flacs = []
    for k in range(4):
        x = (synth.synth_wave(1, 16000 * (3 + 2 * k), seed=seed + k)[0].numpy() * 32768).clip(-32768, 32767).astype(numpy.int64)[:, None]
        flacs.append(flac_ref.encode(x, 16000, 16, blocksize=4096))
    lines = []
    for i in range(n):
        if kinds[i] == 2:
            data, ext = flacs[i % len(flacs)], "flac"
        else:
            rate = 8000 if kinds[i] == 1 else 16000
            L = int(lengths[i]) * rate // 16000
            x = (numpy.random.default_rng(seed * 7919 + i).standard_normal(L) * 3000).astype(numpy.int64)[:, None]
            data, ext = pcm_ref.wav_bytes(x, rate, "pcm", 2), "wav"
        p = os.path.join(d, "u%06d.%s" % (i, ext))
        with open(p, "wb") as f:
            f.write(data)
        lines.append("utt%06d %s\n" % (i, p))
    with open(os.path.join(d, "wav.scp"), "w") as f:
        f.writelines(lines)
    return os.path.join(d, "wav.scp")


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return out.stdout.strip().splitlines()[0]
    except Exception:
        return "unknown"


def _worker(rank, world, port, tree, scp, out_dir, window_s, q):
    sys.path.insert(0, tree)
    import torch
    import torch.distributed as dist
    from sidekit_b200 import extract_xvectors as X
    from tests.models import make_xtractor
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    model = make_xtractor("halfresnet34", 32, 256).to(dev)
    # warm-up: the first windows of the corpus (engine buffers, resampler banks, NCCL)
    head = os.path.join(out_dir, "head_%d.scp" % rank)
    with open(scp) as f, open(head, "w") as g:
        g.writelines(f.readlines()[:200 * world])
    kw = {}
    import inspect
    if "stats" in inspect.signature(X.main).parameters:
        kw["stats"] = []
    X.main(model, head, os.path.join(out_dir, "warm_%d.scp" % rank), dev, window_audio_seconds=window_s)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    emb = X.main(model, scp, os.path.join(out_dir, "xv.scp"), dev, window_audio_seconds=window_s, **kw)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    q.put((rank, wall, kw.get("stats"), int(emb.shape[0]), float(emb.double().sum())))
    if world > 1:
        dist.destroy_process_group()


def run(tree, scp, world, out_dir, window_s):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = [ctx.Process(target=_worker, args=(r, world, port, tree, scp, out_dir, window_s, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=3600) for _ in range(world)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=300)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=4000)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--tree", default=ROOT)
    ap.add_argument("--label", default="")
    ap.add_argument("--worlds", default="")
    ap.add_argument("--window-audio-seconds", type=float, default=4800.0)
    ap.add_argument("--corpus", default="", help="directory holding wav.scp (written there when absent)")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    n_gpu = torch.cuda.device_count()
    if n_gpu == 0:
        raise SystemExit("corpus_probe measures on the GPU: no CUDA device is visible")
    corpus_dir = args.corpus or tempfile.mkdtemp(prefix="skb_corpus_")
    scp = os.path.join(corpus_dir, "wav.scp")
    if not os.path.exists(scp):
        write_corpus(corpus_dir, args.files, args.seed)
    with open(scp) as f:
        paths = [l.split(None, 1)[1].strip() for l in f]
    audio_s = 0.0
    sys.path.insert(0, ROOT)
    from sidekit_b200 import audio
    for p in paths:                                           # page-cache the corpus and total its audio
        with open(p, "rb") as f:
            frames, sr = audio.length(*audio.parse(f.read(), p))
        audio_s += frames / sr
    worlds = [int(w) for w in args.worlds.split(",")] if args.worlds else sorted({1, n_gpu})
    card = torch.cuda.get_device_name(0)
    shards = os.path.exists(os.path.join(args.tree, "sidekit_b200", "corpus.py"))
    for world in worlds:
        if world > 1 and not shards:
            # an older main embeds the whole corpus on every rank and every rank writes the same files: nothing to measure
            print(json.dumps({"probe": "corpus", "label": args.label, "world": world, "skipped": "this tree's main does not shard"}))
            continue
        out_dir = tempfile.mkdtemp(prefix="skb_probe_out_")
        res = run(os.path.abspath(args.tree), scp, world, out_dir, args.window_audio_seconds)
        wall = max(r[1] for r in res)
        line = {"probe": "corpus", "label": args.label, "world": world,
                "files": len(paths), "audio_s": round(audio_s, 1), "wall_s": round(wall, 3),
                "audio_s_per_s": round(audio_s / wall, 1), "files_per_s": round(len(paths) / wall, 1),
                "checksum": res[0][4], "card": card, "power_limit": _power_limit()}
        stats = res[0][2]
        if stats:
            w = len(stats)
            per = {k: round(sum(s[k] for s in stats) / w, 4) for k in ("read_s", "parse_s", "stage_s", "wait_s", "device_s")}
            line.update(windows_rank0=w, per_window_rank0=per,
                        device_idle_fraction_rank0=round(1.0 - sum(s["device_s"] for s in stats) / res[0][1], 3),
                        host_s_per_window_rank0=round(per["read_s"] + per["parse_s"] + per["stage_s"], 4))
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "corpus_probe.jsonl"), "a") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
