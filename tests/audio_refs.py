"""Host references for the audio-loss kernels (tests/test_audio_kernels_gpu.py), pinned on the CPU by
tests/test_audio_refs_cpu.py.  Plain torch, differentiable by autograd, in whatever dtype the inputs carry (float64 for
the references, float32 to measure the rounding floor of the same computation).

- `spec`: the power spectrogram of torchaudio.transforms.Spectrogram(n_fft, hop): periodic Hann window of length n_fft,
  center = True with reflect padding, one-sided, power 2.  Shape (..., n_fft/2 + 1, 1 + T // hop).
- `mss_loss`: one scale of the spectral loss (csrc/mss.cu, SSSLoss):
    l1    alpha * mean(w |log2(Sp + eps) - log2(St + eps)|) + mean(w |Sp - St|) over (batch, bins 1.., frames), with the
          time weight w[fr] = 2 fr / (F - 1) (1 - linspace(1, 0.9, F) normalised to mean 1; 1 when F = 1)
    rmse  sqrt(mean((log2(Sp + eps) - log2(St + eps))^2)) over (batch, all bins, frames)
- `filtered_noise`: DDSP filtered noise (csrc/noise.cu): x = 2 sigmoid(c)^2.3 + 1e-6, irfft(x, n = 2C - 1), rolled by
  C - 1 and windowed by a periodic Hann window of length 2C - 1, linearly convolved with each noise frame, overlap-added
  at stride L and cropped to T.
- `tone_signal`: seeded decaying tones over a white-noise floor, so every STFT bin sits far above eps.
None of it calls the package's kernels.
"""
import math

import torch
import torch.nn.functional as Fn


def spec(x, n, hop):
    """power spectrogram (..., n/2 + 1, 1 + T // hop) of x (..., T)"""
    shape = x.shape
    w = torch.hann_window(n, periodic=True, dtype=x.dtype)
    z = torch.stft(x.reshape(-1, shape[-1]), n, hop, win_length=n, window=w, center=True, pad_mode="reflect",
                   onesided=True, return_complex=True)
    S = torch.view_as_real(z).pow(2).sum(-1)          # |z|^2 without the kink of abs() at 0
    return S.reshape(*shape[:-1], S.shape[-2], S.shape[-1])


def time_weight(frames, dtype=torch.float64):
    if frames == 1:
        return torch.ones(1, dtype=dtype)
    return 2.0 * torch.arange(frames, dtype=dtype) / (frames - 1)


def mss_loss_from_spec(Sp, St, mode, alpha, eps):
    """the loss of one scale from the two power spectrograms (B, bins, frames); mode 'l1' or 'rmse'"""
    lp, lt = torch.log2(Sp + eps), torch.log2(St + eps)
    if mode == "rmse":
        return torch.sqrt(((lp - lt) ** 2).mean())
    w = time_weight(Sp.shape[-1], Sp.dtype)
    return (alpha * (w * (lp - lt).abs())[..., 1:, :].mean()) + (w * (Sp - St).abs())[..., 1:, :].mean()


def mss_loss(xp, xt, n, hop, mode, alpha=1.0, eps=1e-7):
    """one scale of the spectral loss between xp and xt (B, T)"""
    return mss_loss_from_spec(spec(xp, n, hop), spec(xt, n, hop), mode, alpha, eps)


def filter_ir(coeff):
    """windowed impulse responses (..., 2C - 1) of raw filter coefficients (..., C)"""
    C = coeff.shape[-1]
    N = 2 * C - 1
    x = 2.0 * torch.sigmoid(coeff) ** 2.3 + 1e-6
    h0 = torch.fft.irfft(x, n=N)
    return torch.roll(h0, C - 1, dims=-1) * torch.hann_window(N, periodic=True, dtype=coeff.dtype)


def filtered_noise(coeff, noise, T, gain=1.0):
    """filtered noise (B, T) from coefficients (B, F, C) and noise frames (B, F, L)"""
    B, F, C = coeff.shape
    L = noise.shape[-1]
    h = filter_ir(coeff)                                               # (B, F, N)
    N = h.shape[-1]
    # linear convolution of every frame with its own filter: a grouped conv1d with the flipped filter
    fr = Fn.conv1d(noise.reshape(1, B * F, L), torch.flip(h, [-1]).reshape(B * F, 1, N), padding=N - 1,
                   groups=B * F).reshape(B, F, L + N - 1) * gain
    pos = (torch.arange(F)[:, None] * L + torch.arange(L + N - 1)[None, :]).reshape(-1)
    y = torch.zeros(B, F * L + N - 1, dtype=coeff.dtype).index_add(1, pos, fr.reshape(B, -1))
    return y[:, :T]


def tone_signal(B, T, seed, sr=32000.0, tones=4, floor=0.3, dtype=torch.float64):
    """(B, T): `tones` decaying sinusoids of random frequency, phase and amplitude over white noise of rms `floor`"""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(T, dtype=torch.float64) / sr
    f = 100.0 + (0.45 * sr - 100.0) * torch.rand(B, tones, 1, generator=g, dtype=torch.float64)
    ph = 2 * math.pi * torch.rand(B, tones, 1, generator=g, dtype=torch.float64)
    a = 0.5 + torch.rand(B, tones, 1, generator=g, dtype=torch.float64)
    d = 5.0 + 60.0 * torch.rand(B, tones, 1, generator=g, dtype=torch.float64)
    y = (a * torch.exp(-d * t) * torch.sin(2 * math.pi * f * t + ph)).sum(1)
    return (y + floor * torch.randn(B, T, generator=g, dtype=torch.float64)).to(dtype)
