"""``sidekit/bin/extract_xvectors.py`` on the B200 path: Kaldi ``wav.scp`` in, x-vector ark / scp (and optional speaker
means) out, with the reference's function names and arguments (``read_wav_scp`` :18-35, ``prepare`` :37-72,
``load_model`` :74-91, ``main`` :93-173, the argparse block :175-203).

What changes against the reference: the utterances are not pushed through the model one by one (a few hundred small
launches and a device-to-host copy each) but streamed in windows of ~80 minutes of audio (host memory) through the
window pipeline of ``sidekit_b200.corpus``: a background thread reads and parses the next window while the current one
is on the device; a window's files go to the device in one copy, are decoded (one FLAC and one PCM call) straight into
their slots of the length-bucketed packed batches (``bulk.make_batches``), files at another rate through one resampling
call per rate (``preprocessor.Resample``), and are embedded by ``Xtractor.extract_packed`` without a synchronisation
until the window's rows come back; the ark is written window by window.  The packed engine is exact per utterance, so
the vectors are those of the one-by-one loop.  Under ``torchrun --nproc-per-node N`` the entries are sharded over the N
GPUs in contiguous blocks and rank 0 writes the same tables as one process.
Paths and pipe entries (``cat x.sph |``, ``sph2pipe -f wav x.sph |``) may hold FLAC, WAV or NIST SPHERE in every PCM
encoding (``sidekit_b200.audio``).
``--vad`` needs the silero model that the reference fetches with ``torch.hub`` at run time (no network here): it raises.
Tables are written with ``sidekit_b200.kaldi_io`` in the layout ``kaldiio.WriteHelper('ark,scp:...')`` produces.
"""
import contextlib
import os
import subprocess

import numpy
import torch

from . import audio, bulk, corpus, flac, kaldi_io
from .nnet.xsets import load_checkpoint


def read_wav_scp(wav_scp):
    """``utt -> [tokens of the second column onwards]`` in file order (extract_xvectors.py:18-35)."""
    utt2wav = {}
    with open(wav_scp) as ipf:
        for line in ipf:
            lns = line.strip().split()
            if lns:
                utt2wav[lns[0]] = lns[1:]
    return utt2wav


def _source(wav):
    return " ".join(wav) if not isinstance(wav, str) else wav


def _is_pipe(wav):
    return wav.strip().endswith("|")


def _read_source(wav):
    """A ``wav.scp`` entry -> ``(name, bytes)``: the file's bytes, or the standard output of a pipe command (``IOError``
    naming the entry when the command fails)."""
    wav = _source(wav)
    if _is_pipe(wav):
        try:
            with open(os.devnull, "w") as devnull:
                proc = subprocess.Popen(wav.strip()[:-1], stdout=subprocess.PIPE, shell=True, stderr=devnull)
                out = proc.communicate()[0]
            return wav, out
        except Exception as e:
            raise IOError("Error processing wav file: {}\n{}".format(wav, e))
    with open(wav, "rb") as f:
        return wav, f.read()


def _parse_source(name, data):
    """``(kind, info)`` of an entry's bytes; a pipe's output that is not a readable FLAC, WAV or NIST SPHERE stream raises
    ``IOError`` naming the command.  A FLAC stream without frames raises ``ValueError("<name>: no frames")``, as
    ``audio.decode`` does, whether it came from a path or a pipe."""
    if _is_pipe(name):
        try:
            kind, info = audio.parse(data, name)
        except Exception as e:
            raise IOError("Error processing wav file: {}\n{}".format(name, e))
    else:
        kind, info = audio.parse(data, name)
    if audio.no_frames(kind, info):
        raise ValueError("%s: no frames" % name)
    return kind, info


def _read_entry(wav):
    """A ``wav.scp`` entry -> ``(name, file bytes, sample_rate, frames)``, undecoded."""
    name, data = _read_source(wav)
    frames, sr = audio.length(*_parse_source(name, data))
    return name, data, sr, frames


def prepare(wav):
    """A ``wav.scp`` entry (a path, or a shell command ending in ``|`` whose standard output is an audio file) ->
    ``(float32 tensor (n,), sample_rate)`` scaled like ``soundfile.read`` / ``torchaudio.load`` (:37-72).  FLAC, WAV and
    NIST SPHERE in every PCM encoding (``sidekit_b200.audio.read``)."""
    name, data, _, _ = _read_entry(wav)
    return audio.read(data, name=name)


def load_model(model_path, device):
    """Checkpoint -> ``(xtractor in eval mode on device, checkpoint dict)`` (:74-91)."""
    model_config = torch.load(model_path, map_location="cpu", weights_only=False)
    return load_checkpoint(model_path, torch.device(device)), model_config


@torch.no_grad()
def main(xtractor, kaldi_wav_scp, out_file, device, vad=False, num_samples_per_window=2000, min_silence_samples=1500,
         model_sample_rate=16000, out_file_spk="", spk2utt_file="", max_audio_seconds=1200.0, window_audio_seconds=4800.0,
         stats=None):
    """Embed every utterance of ``kaldi_wav_scp`` and write ``<out_file stem>.ark`` + ``out_file`` (scp); with
    ``out_file_spk`` also the L2-normalised mean x-vector of every speaker of ``spk2utt_file`` (:93-173).  Returns the
    (n, E) float32 host tensor of the embeddings in ``wav.scp`` order.

    Under an initialised ``torch.distributed`` process group (one rank per GPU, ``device`` this rank's), the entries are
    cut into one contiguous block per rank, balanced by file size (``corpus.plan_blocks``); each rank embeds its block,
    one all-gather brings the rows together, rank 0 writes the tables -- the same bytes a one-process run writes -- and
    every rank returns the full tensor.  A bad entry on any rank makes every rank raise, naming it.
    ``stats`` (optional list) receives this rank's per-window timings (``corpus.run_windows``)."""
    if vad:
        raise NotImplementedError("--vad loads snakers4/silero-vad through torch.hub (network); run VAD upstream")
    device = flac.device_of(device)
    utt2wav = read_wav_scp(kaldi_wav_scp)
    keys, entries = list(utt2wav.keys()), [_source(w) for w in utt2wav.values()]
    xtractor.eval()
    xtractor.to(device)
    E = xtractor.embedding_size
    out_ark = os.path.realpath(os.path.join(os.path.dirname(out_file), os.path.splitext(os.path.basename(out_file))[0])) + ".ark"

    def prepare(win):
        """Reading thread: the window's length-sorted packing (largest batch first) and its decode straight into it."""
        lengths = corpus.model_lengths(win.frames, win.rates, model_sample_rate)
        order = numpy.argsort(lengths, kind="stable")
        batches = list(reversed(bulk.make_batches(order.tolist(), lengths, max_audio_seconds, sample_rate=model_sample_rate)))
        packed = numpy.array([i for b in batches for i in b], dtype=numpy.int64)
        slots = numpy.empty_like(lengths)
        slots[packed] = numpy.cumsum(lengths[packed]) - lengths[packed]
        with torch.cuda.device(device):
            win.prepared = (corpus.WindowDecode(win, model_sample_rate, slots, int(lengths.sum())), lengths, batches, packed)

    def embed(win):
        dec, lengths, batches, packed = win.prepared
        wave, _, status = dec.launch(device)
        emb = torch.empty((len(win), E), dtype=torch.float32, device=device)
        corpus.extract_batches(xtractor, wave, lengths, batches, emb)

        def finish():
            corpus.check_window(xtractor, dec, status, win.names)
            rows = torch.empty((len(win), E), dtype=torch.float32)
            rows[torch.from_numpy(packed)] = emb.cpu()
            return rows
        return finish

    _, rank, _ = bulk._dist()
    # The wav.scp is STREAMED in windows of `window_audio_seconds` of audio (host memory): a corpus of hundreds of hours
    # never sits in memory, and rank 0 writes the ark window by window in file order, like the reference's
    # one-file-at-a-time loop; the rows of the other ranks' blocks follow after the gather.
    with contextlib.ExitStack() as stack:
        writer = stack.enter_context(kaldi_io.ArkScpWriter(out_ark, os.path.realpath(out_file))) if rank == 0 else None

        def emit(index, rows):
            if writer is not None:
                for i, vec in zip(index, rows.numpy()):
                    writer(keys[i], vec[None, :])               # the reference writes the (1, E) output of the model
        with torch.cuda.device(device):
            emb, blocks = corpus.extract_sharded(entries, corpus.entry_weights([None if _is_pipe(e) else e for e in entries]),
                                                 _read_source, embed, E, window_audio_seconds, prepare, emit, _parse_source, device,
                                                 stats)
        if writer is not None:
            emit(range(blocks[0][1], len(keys)), emb[blocks[0][1]:])
    if out_file_spk and rank == 0:
        spk2utt = {}
        with open(spk2utt_file) as f:
            for line in f:
                lns = line.strip().split()
                if lns:
                    spk2utt[lns[0]] = lns[1:]
        kaldi_io.speaker_means(out_file, spk2utt, out_file_spk)
    return emb


if __name__ == "__main__":
    import argparse
    parser = argparse.ArgumentParser(description="Extract the x-vectors given a sidekit model")
    parser.add_argument("--model", type=str, required=True)
    parser.add_argument("--sample-rate", type=int, default=16000)
    parser.add_argument("--vad", action="store_true")
    parser.add_argument("--vad-num-samples-per-window", type=int, default=2000)
    parser.add_argument("--vad-min-silence-samples", type=int, default=1500)
    parser.add_argument("--wav-scp", type=str, required=True)
    parser.add_argument("--out-scp", type=str, required=True)
    parser.add_argument("--out-spk-scp", type=str, default="")
    parser.add_argument("--spk2utt-file", type=str, default="")
    parser.add_argument("--device", default="cuda", type=str)
    args = parser.parse_args()
    assert os.path.isfile(args.model), "NO SUCH FILE: %s" % args.model
    assert os.path.isfile(args.wav_scp), "NO SUCH FILE: %s" % args.wav_scp
    assert os.path.isdir(os.path.dirname(args.out_scp)), "NO SUCH DIRECTORY: %s" % args.out_scp
    if args.out_spk_scp:
        assert os.path.isdir(os.path.dirname(args.out_spk_scp)), "NO SUCH DIRECTORY: %s" % args.out_spk_scp
        assert os.path.isfile(args.spk2utt_file), "NO SUCH FILE: %s" % args.spk2utt_file
    device = args.device.strip().lower()
    if "LOCAL_RANK" in os.environ:           # under torchrun: one rank per GPU, NCCL from the environment
        import torch.distributed as dist
        device = "cuda:%d" % int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=torch.device(device))
    model, _ = load_model(args.model, device)
    main(model, args.wav_scp, args.out_scp, device, args.vad, args.vad_num_samples_per_window, args.vad_min_silence_samples,
         args.sample_rate, args.out_spk_scp, args.spk2utt_file)
    if "LOCAL_RANK" in os.environ:
        dist.destroy_process_group()
