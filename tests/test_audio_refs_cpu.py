"""The host references of tests/test_audio_kernels_gpu.py (tests/audio_refs.py) checked against the goldens of the
original Python code and against explicit restatements of their definitions, without a GPU."""
import math

import numpy as np
import pytest
import torch

import audio_refs as refs
from conftest import golden


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.mark.parametrize("tag,mode", [("l1_a", "l1"), ("l1_b", "l1"), ("rmse", "rmse"), ("l1_2048", "l1")])
def test_mss_reference_matches_golden(tag, mode):
    """Per-scale losses <= 1e-5 relative (measured here: 2.5e-6), totals <= 2e-6 (5.6e-7); the gradient only to the
    golden's own fp32 error, <= 1.2e-2 rel-L2 (measured here: 1.0e-3 .. 8.9e-3)."""
    g = golden("mss_loss")
    pred = torch.tensor(g["pred"], dtype=torch.float64, requires_grad=True)
    true = torch.tensor(g["true"], dtype=torch.float64)
    per = [refs.mss_loss(pred, true, int(n), int(n) // 4, mode) for n in g[f"{tag}_nffts"]]
    got = np.array([float(x.detach()) for x in per])
    ref = g[f"{tag}_per_scale"]
    assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-5, (got, ref)
    total = sum(per)
    assert abs(float(total) - float(g[f"{tag}_loss"])) <= 2e-6 * abs(float(g[f"{tag}_loss"]))
    total.backward()
    assert _rel(pred.grad.numpy(), g[f"{tag}_grad"]) <= 1.2e-2


def test_spec_reference_matches_golden():
    """spec256 (B=3, T=8000, n=256, hop=64): <= 1e-6 of its maximum (measured here: 2.7e-7)."""
    g = golden("mss_loss")
    S = refs.spec(torch.tensor(g["pred"], dtype=torch.float64), 256, 64).numpy()
    assert S.shape == g["spec256"].shape
    assert np.abs(S - g["spec256"]).max() <= 1e-6 * np.abs(g["spec256"]).max()


@pytest.mark.parametrize("n,hop,T", [(8, 1, 5), (8, 3, 8), (16, 16, 9), (16, 5, 37), (32, 31, 17), (64, 64, 40),
                                     (64, 16, 97)])
def test_spec_reference_matches_explicit_dft(n, hop, T):
    """torch.stft as called by `spec` equals the definition written out: reflect-pad n/2 on each side, frame fr starts
    at padded position fr * hop, periodic Hann window, one-sided DFT, |.|^2; <= 1e-12 of the maximum.  Includes the
    smallest legal T = n/2 + 1, hop = 1, hop = n, hop not dividing n and a single frame."""
    x = refs.tone_signal(2, T, seed=n + hop + T)
    xn = x.numpy()
    frames = 1 + T // hop
    idx = np.arange(-(n // 2), T + n // 2)
    idx = np.where(idx < 0, -idx, idx)
    idx = np.where(idx >= T, 2 * (T - 1) - idx, idx)
    padded = xn[:, idx]
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(n) / n)
    k = np.arange(n // 2 + 1)
    D = np.exp(-2j * np.pi * np.outer(k, np.arange(n)) / n)
    ref = np.stack([np.abs((padded[:, fr * hop:fr * hop + n] * w) @ D.T) ** 2 for fr in range(frames)], -1)
    S = refs.spec(x, n, hop).numpy()
    assert S.shape == (2, n // 2 + 1, frames)
    assert np.abs(S - ref).max() <= 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize("mode", ["l1", "rmse"])
def test_mss_reference_identical_signals_give_zero(mode):
    x = refs.tone_signal(3, 1000, seed=4)
    for n, hop in ((64, 16), (256, 100), (8, 8)):
        assert float(refs.mss_loss(x, x.clone(), n, hop, mode)) == 0.0


def test_mss_reference_single_frame_has_weight_one():
    """T < hop: one frame, time weight 1 (the ramp's 0 / 0 is defined as 1), so the l1 loss is the plain mean."""
    assert refs.time_weight(1).tolist() == [1.0]
    w = refs.time_weight(5)
    assert torch.allclose(w, torch.tensor([0.0, 0.5, 1.0, 1.5, 2.0], dtype=torch.float64)) and float(w.mean()) == 1.0
    xp, xt = refs.tone_signal(2, 40, seed=1), refs.tone_signal(2, 40, seed=2)
    Sp, St = refs.spec(xp, 64, 64), refs.spec(xt, 64, 64)
    assert Sp.shape[-1] == 1
    lp, lt = torch.log2(Sp + 1e-7), torch.log2(St + 1e-7)
    plain = 0.5 * (lp - lt).abs()[:, 1:].mean() + (Sp - St).abs()[:, 1:].mean()
    assert abs(float(refs.mss_loss(xp, xt, 64, 64, "l1", 0.5)) - float(plain)) <= 1e-14 * float(plain)


def test_filtered_noise_reference_matches_golden():
    """FilteredNoise(2, 1000) with the golden's coefficient bank and seeded noise: audio <= 1e-6 rel-L2 (measured here:
    1.8e-7), gradient of sum(y * weight) to the bank <= 1e-6 (2.0e-7)."""
    g = golden("oscillator_r2")
    bank = torch.tensor(g["fn_bank"], dtype=torch.float64, requires_grad=True)
    B, F, C = bank.shape
    torch.manual_seed(int(g["fn_seed"]))
    noise = torch.rand(B, F, 64, dtype=torch.float32) * 2 - 1          # as FilteredNoise.forward draws it
    y = refs.filtered_noise(bank, noise.double(), 1000)
    assert _rel(y.detach().numpy(), g["fn_audio"]) <= 1e-6
    (y * torch.tensor(g["fn_weight"], dtype=torch.float64)).sum().backward()
    assert _rel(bank.grad.numpy(), g["fn_grad_bank"]) <= 1e-6


@pytest.mark.parametrize("C,L,F,T", [(2, 1, 4, 4), (3, 2, 6, 11), (5, 16, 3, 33), (9, 4, 7, 28), (4, 1, 9, 1)])
def test_filtered_noise_reference_matches_direct_sum(C, L, F, T):
    """The irfft / conv1d / index_add reference equals the closed form of the kernel's header evaluated term by term:
    h0[t] = (x_0 + 2 sum_k x_k cos(2 pi k t / N)) / N, h[t] = hann_N[t] h0[(t - C + 1) mod N],
    y[t] = gain sum_f sum_i noise_f[i] h_f[t - L f - i]; <= 1e-13 of the maximum.  Covers N < L, N > L and T < F L."""
    g = torch.Generator().manual_seed(C * 100 + L)
    coeff = torch.rand(2, F, C, generator=g, dtype=torch.float64) * 4 - 2
    noise = torch.rand(2, F, L, generator=g, dtype=torch.float64) * 2 - 1
    N = 2 * C - 1
    x = 2 * torch.sigmoid(coeff).numpy() ** 2.3 + 1e-6
    nz = noise.numpy()
    y = np.zeros((2, T))
    for b in range(2):
        for f in range(F):
            h = np.zeros(N)
            for t in range(N):
                t0 = (t - (C - 1)) % N
                h0 = (x[b, f, 0] + 2 * sum(x[b, f, k] * math.cos(2 * math.pi * k * t0 / N) for k in range(1, C))) / N
                h[t] = (0.5 - 0.5 * math.cos(2 * math.pi * t / N)) * h0
            for i in range(L):
                for tau in range(N):
                    t = L * f + i + tau
                    if t < T:
                        y[b, t] += 0.37 * nz[b, f, i] * h[tau]
    got = refs.filtered_noise(coeff, noise, T, 0.37).numpy()
    assert got.shape == (2, T)
    assert np.abs(got - y).max() <= 1e-13 * max(np.abs(y).max(), 1e-300)
