"""Front-end modules with the reference's names, constructor arguments and state_dict keys
(sidekit/nnet/preprocessor.py:61-124, :212-285; sidekit/nnet/augmentation.py:49-74).

The modules only hold the constant buffers (pre-emphasis filter, Hann window, Mel filterbank, DCT
matrix -- computed with the same float32 formulas as torchaudio so they are bit-identical to the
reference's buffers); the arithmetic runs in the fused CUDA front-end kernel (csrc/frontend.cu).
"""
import math

import torch


def melscale_fbanks(n_freqs, f_min, f_max, n_mels, sample_rate):
    """HTK triangular filterbank, norm=None (torchaudio.functional.melscale_fbanks) -> (n_freqs, n_mels)."""
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    m_min = 2595.0 * math.log10(1.0 + (f_min / 700.0))
    m_max = 2595.0 * math.log10(1.0 + (f_max / 700.0))
    m_pts = torch.linspace(m_min, m_max, n_mels + 2)
    f_pts = 700.0 * (10 ** (m_pts / 2595.0) - 1.0)
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    down_slopes = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up_slopes = slopes[:, 2:] / f_diff[1:]
    return torch.max(torch.zeros(1), torch.min(down_slopes, up_slopes))


def create_dct(n_mfcc, n_mels):
    """Orthonormal DCT-II matrix (torchaudio.functional.create_dct(norm='ortho')) -> (n_mels, n_mfcc)."""
    n = torch.arange(float(n_mels))
    k = torch.arange(float(n_mfcc)).unsqueeze(1)
    dct = torch.cos(math.pi / float(n_mels) * (n + 0.5) * k)
    dct[0] *= 1.0 / math.sqrt(2.0)
    dct *= math.sqrt(2.0 / float(n_mels))
    return dct.t().contiguous()


class PreEmphasis(torch.nn.Module):
    """y[t] = x[t] - coef * x[t-1] with reflect padding (augmentation.py:49-74); buffer only."""

    def __init__(self, coef: float = 0.97):
        super().__init__()
        self.coef = coef
        self.register_buffer("flipped_filter", torch.FloatTensor([-self.coef, 1.]).unsqueeze(0).unsqueeze(0))


class _Spectrogram(torch.nn.Module):
    def __init__(self, win_length):
        super().__init__()
        self.register_buffer("window", torch.hann_window(win_length))


class _MelScale(torch.nn.Module):
    def __init__(self, n_freqs, f_min, f_max, n_mels, sample_rate):
        super().__init__()
        self.register_buffer("fb", melscale_fbanks(n_freqs, f_min, f_max, n_mels, sample_rate))


class _MelSpectrogram(torch.nn.Module):
    """Container mirroring torchaudio.transforms.MelSpectrogram's buffers (.spectrogram.window, .mel_scale.fb)."""

    def __init__(self, sample_rate, n_fft, win_length, f_min, f_max, n_mels):
        super().__init__()
        self.spectrogram = _Spectrogram(win_length)
        self.mel_scale = _MelScale(n_fft // 2 + 1, f_min, f_max, n_mels, sample_rate)


class _MFCC(torch.nn.Module):
    def __init__(self, sample_rate, n_mfcc, melkwargs):
        super().__init__()
        self.register_buffer("dct_mat", create_dct(n_mfcc, melkwargs["n_mels"]))
        self.MelSpectrogram = _MelSpectrogram(sample_rate, melkwargs["n_fft"], melkwargs["win_length"],
                                              melkwargs["f_min"], melkwargs["f_max"], melkwargs["n_mels"])


class _FrontEndBase(torch.nn.Module):
    _owner = None     # set by Xtractor: the native front-end lives in the extractor's engine

    def _run(self, x):
        if x.dim() == 1:
            x = x.unsqueeze(0)
        owner = self.__dict__.get("_owner")
        if owner is None:
            raise RuntimeError("the front-end runs inside the fused CUDA engine: call it through Xtractor.preprocessor")
        return owner()._frontend(x)


class MelSpecFrontEnd(_FrontEndBase):
    """Log-Mel front-end of the ResNet archis (preprocessor.py:212-285); inference path only."""

    def __init__(self, pre_emphasis=0.97, sample_rate=16000, n_fft=1024, f_min=90, f_max=7600, win_length=400,
                 window_fn=torch.hann_window, hop_length=160, power=2.0, n_mels=80):
        super().__init__()
        if (n_fft, win_length, hop_length, power) != (1024, 400, 160, 2.0) or window_fn is not torch.hann_window:
            raise NotImplementedError("the CUDA front-end implements n_fft=1024, win=400, hop=160, power=2, Hann")
        self.pre_emphasis, self.sample_rate, self.n_fft, self.f_min, self.f_max = pre_emphasis, sample_rate, n_fft, f_min, f_max
        self.win_length, self.hop_length, self.power, self.n_mels = win_length, hop_length, power, n_mels
        self.PreEmphasis = PreEmphasis(self.pre_emphasis)
        self.MelSpec = _MelSpectrogram(sample_rate, n_fft, win_length, f_min, f_max, n_mels)

    def forward(self, x, is_eval=False):
        if not is_eval:
            raise NotImplementedError("training-time SpecAugment masking is out of scope (inference hot path only)")
        return self._run(x)


class MfccFrontEnd(_FrontEndBase):
    """MFCC front-end of the TDNN 'xvector' archi (preprocessor.py:61-124).

    ``forward`` accepts (and ignores) ``is_eval``: the reference's Xtractor passes it (xvector.py:885)
    although the reference's own MfccFrontEnd.forward lacks the parameter (SURVEY.md finding 4).
    """

    def __init__(self, pre_emphasis=0.97, sample_rate=16000, n_fft=2048, f_min=133.333, f_max=6855.4976,
                 win_length=1024, window_fn=torch.hann_window, hop_length=512, power=2.0, n_mels=100, n_mfcc=80):
        super().__init__()
        if (n_fft, win_length, hop_length, power) != (2048, 1024, 512, 2.0) or window_fn is not torch.hann_window:
            raise NotImplementedError("the CUDA front-end implements n_fft=2048, win=1024, hop=512, power=2, Hann")
        self.pre_emphasis, self.sample_rate, self.n_fft, self.f_min, self.f_max = pre_emphasis, sample_rate, n_fft, f_min, f_max
        self.win_length, self.hop_length, self.power, self.n_mels, self.n_mfcc = win_length, hop_length, power, n_mels, n_mfcc
        self.PreEmphasis = PreEmphasis(self.pre_emphasis)
        self.melkwargs = {"n_fft": n_fft, "f_min": f_min, "f_max": f_max, "win_length": win_length,
                          "hop_length": hop_length, "power": power, "n_mels": n_mels}
        self.MFCC = _MFCC(sample_rate, n_mfcc, self.melkwargs)

    def forward(self, x, is_eval=True):
        return self._run(x)


def sinc_resample_bank(orig_freq, new_freq, lowpass_filter_width=6, rolloff=0.99):
    """The polyphase filter bank of ``torchaudio.functional.resample`` (``sinc_interp_hann``), float64 -> float32 exactly
    as torchaudio builds it, in the compact form the kernel takes: ``(orig_r, new_r, width, bank[ntap][new_r], start[new_r])``.

    Taps whose argument is clamped to the edge of the window carry ``cos(pi / 2) ** 2 ~ 4e-33`` and are dropped; the
    remaining ones of phase ``ph`` are the ``ntap`` consecutive taps from ``start[ph]`` on (zero padded at the end)."""
    import numpy
    if int(orig_freq) != orig_freq or int(new_freq) != new_freq:
        raise Exception("Frequencies must be of integer type to ensure quality resampling computation.")
    if lowpass_filter_width <= 0:
        raise ValueError("Low pass filter width should be positive.")
    g = math.gcd(int(orig_freq), int(new_freq))
    orig_r, new_r = int(orig_freq) // g, int(new_freq) // g
    base = min(orig_r, new_r) * rolloff
    width = math.ceil(lowpass_filter_width * orig_r / base)
    idx = numpy.arange(-width, width + orig_r, dtype=numpy.float64)[None, :] / orig_r
    # torchaudio's phase offsets -ph / new are float32 (int64 arange / int under torch's true division), then float64
    phase = (numpy.arange(0, -new_r, -1).astype(numpy.float32) / numpy.float32(new_r)).astype(numpy.float64)
    t = (phase[:, None] + idx) * base
    inside = numpy.abs(t) < lowpass_filter_width
    t = numpy.clip(t, -lowpass_filter_width, lowpass_filter_width)
    window = numpy.cos(t * math.pi / lowpass_filter_width / 2) ** 2
    t = t * math.pi
    with numpy.errstate(invalid="ignore", divide="ignore"):
        kern = numpy.where(t == 0, 1.0, numpy.sin(t) / t)
    kern = (kern * window * (base / orig_r)).astype(numpy.float32)          # (new_r, 2 * width + orig_r)
    start = numpy.array([int(numpy.argmax(row)) if row.any() else 0 for row in inside], dtype=numpy.int32)
    count = inside.sum(axis=1)
    ntap = int(count.max())
    start = numpy.minimum(start, kern.shape[1] - ntap).astype(numpy.int32)
    bank = numpy.zeros((ntap, new_r), dtype=numpy.float32)
    for ph in range(new_r):
        seg = kern[ph, start[ph]:start[ph] + ntap].copy()
        seg[~inside[ph, start[ph]:start[ph] + ntap]] = 0.0
        bank[:, ph] = seg
    return orig_r, new_r, width, bank, start


class Resample(torch.nn.Module):
    """``torchaudio.transforms.Resample(orig_freq, new_freq)`` as the reference's feed path applies it to files whose rate
    differs from the model's (sidekit/nnet/xsets.py:435, :452; sidekit/bin/extract_xvectors.py:144), on the device
    (csrc/resample.cu).  ``forward`` takes a CUDA tensor ``(..., L)`` and returns ``(..., ceil(L * new / orig))``;
    ``resample_packed`` takes utterances of different lengths back to back."""

    def __init__(self, orig_freq=16000, new_freq=16000, resampling_method="sinc_interp_hann", lowpass_filter_width=6,
                 rolloff=0.99):
        super().__init__()
        if resampling_method not in ("sinc_interp_hann", "sinc_interpolation"):
            raise NotImplementedError("the CUDA resampler implements the Hann-windowed sinc (torchaudio's default)")
        self.orig_freq, self.new_freq = orig_freq, new_freq
        self.lowpass_filter_width, self.rolloff = lowpass_filter_width, rolloff
        self._bank = sinc_resample_bank(orig_freq, new_freq, lowpass_filter_width, rolloff) if orig_freq != new_freq else None
        self._dev = {}          # device -> (bank, start) tensors, uploaded once

    def out_length(self, n):
        if self._bank is None:
            return int(n)
        orig_r, new_r = self._bank[0], self._bank[1]
        return (int(n) * new_r + orig_r - 1) // orig_r

    def _device_bank(self, device):
        if device not in self._dev:
            bank, start = self._bank[3], self._bank[4]
            self._dev[device] = (torch.from_numpy(bank).to(device), torch.from_numpy(start).to(device))
        return self._dev[device]

    def resample_packed(self, wave, lengths):
        """``wave``: 1-D float32 CUDA tensor, the utterances back to back; ``lengths``: their sample counts."""
        import numpy
        from .. import _lib
        if self._bank is None:
            return wave
        if not wave.is_cuda:
            raise RuntimeError("sidekit_b200 has no CPU path: the waveform must be a CUDA tensor")
        orig_r, new_r, width = self._bank[:3]
        wave = wave.contiguous().float()
        n_in = numpy.asarray(lengths, dtype=numpy.int64).reshape(-1)
        assert wave.dim() == 1 and int(n_in.sum()) == wave.shape[0] and (n_in >= 0).all()
        n_out = (n_in * new_r + orig_r - 1) // orig_r
        out = torch.empty(int(n_out.sum()), dtype=torch.float32, device=wave.device)
        if out.numel() == 0:
            return out
        meta = numpy.stack([numpy.cumsum(n_in) - n_in, n_in, numpy.cumsum(n_out) - n_out, n_out], axis=1)
        with torch.cuda.device(wave.device):
            meta_dev = torch.from_numpy(meta).pin_memory().to(wave.device, non_blocking=True)
            self.launch(wave, meta_dev, out, int(n_out.max()))
        return out

    def launch(self, src, meta_dev, dst, max_out):
        """One ``skb_resample`` call on the current stream: row ``i`` of ``meta_dev`` (int64 CUDA tensor (n, 4), n <= 65535)
        resamples ``src[in_off : in_off + in_len]`` into ``dst[out_off : out_off + out_len]`` (``in_off, in_len, out_off,
        out_len``).  ``src`` and ``dst`` may be the same tensor when the rows' input and output ranges do not overlap."""
        from .. import _lib
        orig_r, new_r, width = self._bank[:3]
        bank, start = self._device_bank(dst.device)
        _lib.check(_lib.lib().skb_resample(src.data_ptr(), meta_dev.data_ptr(), int(meta_dev.shape[0]), int(max_out), orig_r, new_r,
                                           width, bank.data_ptr(), start.data_ptr(), bank.shape[0], dst.data_ptr(), _lib.stream_ptr()))

    def forward(self, waveform):
        if self._bank is None:
            return waveform
        shape = waveform.shape
        rows = waveform.reshape(-1, shape[-1])
        out = self.resample_packed(rows.reshape(-1), [shape[-1]] * rows.shape[0])
        return out.reshape(shape[:-1] + (self.out_length(shape[-1]),))
