"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

CPU restatement of the log-mel extraction TacotronSTFT.mel_spectrogram (SURVEY.md section 8(f) item 4):

    layers.py:63-80   mel_spectrogram: STFT magnitudes -> mel_basis @ magnitudes -> log(clamp(., 1e-5))
    stft.py:44-66     the windowed Fourier basis (real rows, then imaginary rows, of the first n/2 + 1 DFT bins,
                      multiplied by the zero-centre-padded periodic hann window)
    stft.py:69-94     transform: reflect-pad by n/2 on both sides, conv1d with stride = hop, magnitude
    audio_processing.py:78-84  dynamic_range_compression

Pinning: the STFT part is checked against the committed fixtures tests/golden/stft_mag.npz and stft_mag_settings.npz
produced by the reference's own ``stft.STFT`` (tools/make_golden.py, with functional stand-ins for the two librosa.util
helpers stft.py imports).  The mel filterbank is ``librosa.filters.mel`` of
librosa 0.6.0 (requirements.txt:5) -- a third-party dependency that is NOT in this image: ``mel_filterbank`` restates its
published algorithm (Slaney mel scale, htk=False; area normalisation norm=1) and is **parity unpinned** against librosa
itself; it is anchored only by its defining properties (tests/test_oracle_golden.py).
"""
import math

import numpy as np
import torch


def hann_periodic(n):
    """scipy.signal.get_window('hann', n, fftbins=True) (stft.py:58)."""
    return 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(n) / n)


def stft_forward_basis(filter_length, win_length):
    """(2 * (filter_length // 2 + 1), filter_length) float32: stft.py:44-63."""
    n, cutoff = filter_length, filter_length // 2 + 1
    k = np.arange(cutoff)[:, None] * np.arange(n)[None, :]
    ang = 2.0 * np.pi * k / n
    basis = np.concatenate([np.cos(ang), -np.sin(ang)], axis=0)          # rows of fft(eye): exp(-2 pi i k n / N)
    win = np.zeros(n)
    lpad = (n - win_length) // 2                                          # librosa.util.pad_center
    win[lpad:lpad + win_length] = hann_periodic(win_length)
    return (basis.astype(np.float32) * win.astype(np.float32)[None, :]).astype(np.float32)


def _hz_to_mel(f):
    f = np.asanyarray(f, dtype=np.float64)
    f_sp, min_log_hz = 200.0 / 3, 1000.0
    min_log_mel, logstep = min_log_hz / f_sp, math.log(6.4) / 27.0
    mels = f / f_sp
    return np.where(f >= min_log_hz, min_log_mel + np.log(np.maximum(f, 1e-30) / min_log_hz) / logstep, mels)


def _mel_to_hz(m):
    m = np.asanyarray(m, dtype=np.float64)
    f_sp, min_log_hz = 200.0 / 3, 1000.0
    min_log_mel, logstep = min_log_hz / f_sp, math.log(6.4) / 27.0
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), f_sp * m)


def mel_filterbank(sr, n_fft, n_mels, fmin, fmax):
    """librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax) of librosa 0.6.0 (htk=False, norm=1), float32 (n_mels, n_fft//2+1)."""
    fftfreqs = np.linspace(0.0, sr / 2.0, n_fft // 2 + 1)
    mel_f = _mel_to_hz(np.linspace(_hz_to_mel(fmin), _hz_to_mel(fmax if fmax is not None else sr / 2.0), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = mel_f[:, None] - fftfreqs[None, :]
    w = np.zeros((n_mels, n_fft // 2 + 1))
    for i in range(n_mels):
        w[i] = np.maximum(0.0, np.minimum(-ramps[i] / fdiff[i], ramps[i + 2] / fdiff[i + 1]))
    w *= (2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels]))[:, None]
    return w.astype(np.float32)


def stft_magnitude(y, filter_length=1024, hop_length=256, win_length=1024):
    """stft.py:69-91: y (B, n) -> magnitudes (B, filter_length // 2 + 1, 1 + n // hop)."""
    basis = torch.from_numpy(stft_forward_basis(filter_length, win_length))[:, None, :]
    x = torch.nn.functional.pad(y[:, None, None, :], (filter_length // 2, filter_length // 2, 0, 0), mode="reflect")[:, 0]
    ft = torch.nn.functional.conv1d(x, basis, stride=hop_length)
    cutoff = filter_length // 2 + 1
    return torch.sqrt(ft[:, :cutoff] ** 2 + ft[:, cutoff:] ** 2)


def mel_spectrogram(y, filter_length=1024, hop_length=256, win_length=1024, n_mel_channels=80, sampling_rate=22050,
                    mel_fmin=0.0, mel_fmax=8000.0, clip_val=1e-5):
    """layers.py:63-80 (the range asserts included)."""
    assert float(y.min()) >= -1 and float(y.max()) <= 1
    mag = stft_magnitude(y, filter_length, hop_length, win_length)
    mel_basis = torch.from_numpy(mel_filterbank(sampling_rate, filter_length, n_mel_channels, mel_fmin, mel_fmax))
    return torch.log(torch.clamp(torch.matmul(mel_basis, mag), min=clip_val))
