"""``sidekit/bin/extract_xvectors.py`` on the B200 path: Kaldi ``wav.scp`` in, x-vector ark / scp (and optional speaker
means) out, with the reference's function names and arguments (``read_wav_scp`` :18-35, ``prepare`` :37-72,
``load_model`` :74-91, ``main`` :93-173, the argparse block :175-203).

What changes against the reference: the utterances are not pushed through the model one by one (a few hundred small
launches and a device-to-host copy each) but streamed in windows of ~80 minutes of audio (host memory), and each window
is embedded in length-bucketed packed batches (``bulk.make_batches`` + ``Xtractor.extract_varlen``), resampled on the
device where a file's rate differs from the model's (``preprocessor.Resample``); only the batch being embedded is on
the device, and the ark is written window by window.  The packed engine is exact per utterance, so the vectors are
those of the one-by-one loop.
Paths and pipe entries (``cat x.sph |``, ``sph2pipe -f wav x.sph |``) may hold FLAC, WAV or NIST SPHERE in every PCM
encoding; the entries of a window are read as bytes and decoded on the device in one batched call (``sidekit_b200.audio``).
``--vad`` needs the silero model that the reference fetches with ``torch.hub`` at run time (no network here): it raises.
Tables are written with ``sidekit_b200.kaldi_io`` in the layout ``kaldiio.WriteHelper('ark,scp:...')`` produces.
"""
import os
import subprocess

import numpy
import torch

from . import audio, bulk, kaldi_io
from .nnet.preprocessor import Resample
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


def _read_entry(wav):
    """A ``wav.scp`` entry -> ``(name, file bytes, sample_rate, frames)``, undecoded.  A pipe entry's output is checked to be
    a readable FLAC, WAV or NIST SPHERE stream here, so that a failing command raises ``IOError`` naming it."""
    wav = " ".join(wav) if not isinstance(wav, str) else wav
    if wav.strip().endswith("|"):
        try:
            with open(os.devnull, "w") as devnull:
                out = subprocess.Popen(wav.strip()[:-1], stdout=subprocess.PIPE, shell=True, stderr=devnull).communicate()[0]
            frames, sr = audio.length(*audio.parse(out, wav))
            return wav, out, sr, frames
        except Exception as e:
            raise IOError("Error processing wav file: {}\n{}".format(wav, e))
    with open(wav, "rb") as f:
        data = f.read()
    frames, sr = audio.length(*audio.parse(data, wav))
    return wav, data, sr, frames


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
         model_sample_rate=16000, out_file_spk="", spk2utt_file="", max_audio_seconds=1200.0, window_audio_seconds=4800.0):
    """Embed every utterance of ``kaldi_wav_scp`` and write ``<out_file stem>.ark`` + ``out_file`` (scp); with
    ``out_file_spk`` also the L2-normalised mean x-vector of every speaker of ``spk2utt_file`` (:93-173)."""
    if vad:
        raise NotImplementedError("--vad loads snakers4/silero-vad through torch.hub (network); run VAD upstream")
    device = torch.device(device)
    utt2wav = read_wav_scp(kaldi_wav_scp)
    xtractor.eval()
    xtractor.to(device)
    resamplers = {}
    out_ark = os.path.realpath(os.path.join(os.path.dirname(out_file), os.path.splitext(os.path.basename(out_file))[0])) + ".ark"
    all_emb = []

    def flush(window, writer):
        """Decode one window of entries (file bytes) in one call, embed it in length-bucketed packed batches and write its
        entries in file order.  Only the window's waveforms and the batch being embedded live on the device."""
        if not window:
            return
        out, n, _ = audio.decode([data for _, _, data, _ in window], device, names=[name for _, name, _, _ in window])
        window = [(key, x, sr) for (key, _, _, sr), x in zip(window, torch.split(out, n.tolist()))]
        lengths = numpy.array([-(-int(sig.shape[0]) * model_sample_rate // sr) for _, sig, sr in window], dtype=numpy.int64)
        order = numpy.argsort(lengths, kind="stable")
        emb = torch.empty((len(window), xtractor.embedding_size), dtype=torch.float32)
        for batch in reversed(bulk.make_batches(order.tolist(), lengths, max_audio_seconds, sample_rate=model_sample_rate)):
            waves = []
            for i in batch:
                _, sig, sr = window[i]
                sig = sig.to(device, non_blocking=True)
                if sr != model_sample_rate:
                    if sr not in resamplers:
                        resamplers[sr] = Resample(orig_freq=sr, new_freq=model_sample_rate)
                    sig = resamplers[sr](sig)
                waves.append(sig)
            emb[torch.as_tensor(batch)] = xtractor.extract_varlen(waves).cpu()
        for (key, _, _), vec in zip(window, emb.numpy()):
            writer(key, vec[None, :])                      # the reference writes the (1, E) output of the model
        all_emb.append(emb)

    # The wav.scp is STREAMED in windows of `window_audio_seconds` of audio (host memory; a pipe entry has no length until
    # it has been read): a corpus of hundreds of hours never sits in memory, and the ark grows window by window in file
    # order, like the reference's one-file-at-a-time loop.
    with kaldi_io.ArkScpWriter(out_ark, os.path.realpath(out_file)) as writer:
        window, window_s = [], 0.0
        for key, wav in utt2wav.items():
            name, data, sr, frames = _read_entry(wav)
            window.append((key, name, data, sr))           # decoded at flush time, with the window's other entries
            window_s += float(frames) / sr
            if window_s >= window_audio_seconds:
                flush(window, writer)
                window, window_s = [], 0.0
        flush(window, writer)
    emb = torch.cat(all_emb) if all_emb else torch.empty((0, xtractor.embedding_size), dtype=torch.float32)
    if out_file_spk:
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
    model, _ = load_model(args.model, args.device.strip().lower())
    main(model, args.wav_scp, args.out_scp, args.device, args.vad, args.vad_num_samples_per_window, args.vad_min_silence_samples,
         args.sample_rate, args.out_spk_scp, args.spk2utt_file)
