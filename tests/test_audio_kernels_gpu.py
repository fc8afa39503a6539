"""The audio-loss kernels one by one, through the native wrappers, against float64 references (tests/audio_refs.py).

The suite's other checks of these kernels compare with one golden of the original fp32 code at one shape, the gradient
at 1e-2 rel-L2: an error in the reflect-padding gather (n/2 samples at each end), in the DC bin (one bin of n/2 + 1) or
in the tail of a Hann-windowed noise filter shrinks below that over a whole signal.  Here:
  A  ds_stft_power                 float64 torch.stft; whole spectrogram, first / last frame, DC and Nyquist bins
  B  ds_mss_loss_fwd               the float64 loss of the same spectrograms, both modes, alpha, eps, frames == 1, B = 300
  C  ds_mss_loss_bwd               float64 autograd.  The linear l1 term (alpha = 0) is held tight over the whole signal
                                   and over its first and last n samples; the log terms divide by S + eps, so their bar
                                   scales with the float32 floor of the same reference, measured on the CPU per case
  D  ds_filtered_noise_fwd / _bwd  float64 irfft / conv1d / overlap-add and its autograd, per segment of L samples
  E  argument checks of the C ABI
Every bar states the value measured on an NVIDIA B200.  Helpers print what they measure (pytest -s shows it).
"""
import ctypes as C

import numpy as np
import pytest
import torch

import audio_refs as refs

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
PRIME_T = 7993                 # a prime near 8000: no hop divides it
MODES = {"l1": 0, "rmse": 1}
DS_ERR_ARG = -2

# bars: about 4x the worst error measured over every case of the test on an NVIDIA B200 (1000 W power limit)
STFT_BAR = 1.5e-6              # max |dS| / max S per signal; measured: 3.7e-7
STFT_FRAME_BAR = 1.5e-6        # first and last frame against their own maximum; measured: 3.7e-7
STFT_BIN_BAR = 8e-5            # DC and Nyquist bins against their own maximum (quieter than the peak); measured: 1.9e-5
FWD_BAR = 1e-5                 # |d loss| / loss; measured: 2.6e-6
LIN_BAR = 8e-6                 # l1, alpha = 0: gradient rel-L2 over the signal and over each edge window; measured: 1.9e-6
LOG_ABS_BAR = 1e-5             # log terms: rel-L2 <= max(LOG_ABS_BAR, LOG_K * float32 floor);
LOG_K = 15.0                   # measured: up to 3.9 x the floor (rmse, n = 4096, hop = 3), 0.52 of this bar
FN_BAR = 2e-6                  # filtered noise forward, rel-L2; measured: 4.5e-7
FN_SEG_BAR = 3e-5              # per segment: max |dy| / max(rms of the segment, 0.1 rms of the signal); measured: 7.3e-6
FN_GRAD_BAR = 3e-6             # filtered noise backward, rel-L2 and max |dg| / max |g|; measured: 6.7e-7


def _native():
    from diffsound_b200 import native
    return native


def _lib():
    from diffsound_b200 import _lib as L
    return L.load()


def _p(t):
    return C.c_void_p(t.data_ptr())


def _sweep():
    out = []
    for n in (8, 16, 64, 256, 1024, 4096):
        for hop in sorted({1, 3, n // 4, n - 1, n}):
            for T in (n // 2 + 1, n, PRIME_T):
                if hop == 1 and (n > 64 or T > 1000):      # keeps the float64 reference small
                    continue
                out.append((n, hop, T))
    return out


SWEEP = _sweep()


def _batch(n, hop, T):
    return 3 if (1 + T // hop) * n <= 1 << 22 else 1


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _pair(B, T, seed):
    """two independent fp32 test signals"""
    return (refs.tone_signal(B, T, seed, dtype=torch.float32),
            refs.tone_signal(B, T, seed + 1000, floor=0.2, dtype=torch.float32))


# ---------------------------------------------------------------------------------------------------------------------
# A. ds_stft_power
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,hop,T", SWEEP)
def test_stft_power_vs_fp64(n, hop, T):
    B = _batch(n, hop, T)
    x = refs.tone_signal(B, T, seed=n + 7 * hop + T, dtype=torch.float32)
    ref = refs.spec(x.double(), n, hop).numpy()
    got = _native().stft_power(x.to(DEV), n, hop).cpu().double().numpy()
    assert got.shape == ref.shape == (B, n // 2 + 1, 1 + T // hop)
    d = np.abs(got - ref)
    err = max(float(d[b].max() / ref[b].max()) for b in range(B))
    errs = {}
    for name, s in (("first frame", np.s_[:, 0]), ("last frame", np.s_[:, -1]), ("DC", np.s_[0, :]),
                    ("Nyquist", np.s_[-1, :])):
        errs[name] = max(float(d[b][s].max() / ref[b][s].max()) for b in range(B))
    print(f"stft n={n} hop={hop} T={T} B={B}: max|dS|/maxS {err:.2e}; " +
          ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert err <= STFT_BAR
    for k, v in errs.items():
        assert v <= (STFT_FRAME_BAR if k.endswith("frame") else STFT_BIN_BAR), k


# ---------------------------------------------------------------------------------------------------------------------
# B. ds_mss_loss_fwd
# ---------------------------------------------------------------------------------------------------------------------
def _fwd_cases():
    cases = [(_batch(n, hop, T), n, hop, T) for n, hop, T in SWEEP]
    # the one-warp reduction over B * frames partials: 300 single-frame signals, and 300 x 63 frames
    return cases + [(300, 8, 8, 5), (300, 64, 16, 1000)]


@pytest.mark.parametrize("B,n,hop,T", _fwd_cases())
def test_mss_loss_fwd_vs_fp64(B, n, hop, T):
    native = _native()
    xp, xt = _pair(B, T, seed=3 * n + hop + T)
    Sp, St = refs.spec(xp.double(), n, hop), refs.spec(xt.double(), n, hop)
    xpd, xtd = xp.to(DEV), xt.to(DEV)
    worst = 0.0
    for mode, alphas in (("l1", (0.0, 0.5, 1.0)), ("rmse", (1.0,))):
        for alpha in alphas:
            for eps in (1e-7, 1e-3):
                ref = float(refs.mss_loss_from_spec(Sp, St, mode, alpha, eps))
                loss, _ = native.mss_loss_fwd(xpd, xtd, n, hop, MODES[mode], alpha, eps)
                assert loss.dtype == torch.float64 and loss.dim() == 0
                e = abs(float(loss) - ref) / abs(ref)
                worst = max(worst, e)
                assert e <= FWD_BAR, (mode, alpha, eps, float(loss), ref)
    print(f"mss fwd B={B} n={n} hop={hop} T={T} frames={1 + T // hop}: max |dloss|/loss {worst:.2e}")


@pytest.mark.parametrize("n,hop,T", [(8, 3, 8), (8, 8, 5), (64, 1, 100), (256, 64, PRIME_T), (4096, 4096, 2049)])
def test_mss_identical_signals_give_exact_zero(n, hop, T):
    """pred == true: both losses are exactly 0 and both gradients exactly 0 (rmse takes its loss == 0 branch instead of
    dividing by the loss)."""
    native = _native()
    x = refs.tone_signal(3, T, seed=n + T, dtype=torch.float32).to(DEV)
    for mode in ("l1", "rmse"):
        loss, scratch = native.mss_loss_fwd(x, x.clone(), n, hop, MODES[mode], 1.0, 1e-7)
        gx = torch.full_like(x, float("nan"))
        native.mss_loss_bwd(x, x.clone(), n, hop, MODES[mode], 1.0, 1e-7, loss, 1.0, scratch, gx, False)
        print(f"identical n={n} hop={hop} T={T} {mode}: loss {float(loss):.3e}, max|g| {float(gx.abs().max()):.3e}")
        assert float(loss) == 0.0, mode
        assert bool(torch.isfinite(gx).all()) and float(gx.abs().max()) == 0.0, mode


# ---------------------------------------------------------------------------------------------------------------------
# C. ds_mss_loss_bwd
# ---------------------------------------------------------------------------------------------------------------------
BWD_SHAPES = [(8, 1, 5), (8, 3, 8), (8, 8, 5), (16, 5, 37), (64, 1, 1000), (64, 63, PRIME_T), (64, 64, 40),
              (128, 32, 700), (256, 64, PRIME_T), (256, 100, PRIME_T), (1024, 3, 1024), (1024, 1023, PRIME_T),
              (4096, 3, 2049), (4096, 1024, 2049), (4096, 4096, PRIME_T)]


def _ref_grad(xp, xt, n, hop, mode, alpha, eps, dtype):
    p = xp.to(dtype).clone().requires_grad_(True)
    refs.mss_loss(p, xt.to(dtype), n, hop, mode, alpha, eps).backward()
    return p.grad.double().numpy()


def _kernel_grad(xpd, xtd, n, hop, mode, alpha, eps, upstream, gx=None, accumulate=False):
    native = _native()
    loss, scratch = native.mss_loss_fwd(xpd, xtd, n, hop, MODES[mode], alpha, eps)
    gx = torch.empty_like(xpd) if gx is None else gx
    native.mss_loss_bwd(xpd, xtd, n, hop, MODES[mode], alpha, eps, loss, upstream, scratch, gx, accumulate)
    return gx


def _bwd_signals(n, hop, T):
    """pred, and a target that is half of it plus a little of another signal: the spectra differ by a factor near 4
    almost everywhere, so no bin sits where sign(Sp - St) could flip under fp32 rounding"""
    xp, other = _pair(2, T, seed=5 * n + hop + T)
    return xp, (0.5 * xp + 0.05 * other).float()


@pytest.mark.parametrize("n,hop,T", BWD_SHAPES)
def test_mss_loss_bwd_linear_term_vs_fp64(n, hop, T):
    """l1 with alpha = 0: the linear spectrum only, no 1 / (S + eps).  Whole signal and the edge windows [0, n) and
    [T - n, T) (where the reflect-padding images land) against their own norms; upstream 1 and -2.5; accumulate = 1
    onto a random pre-fill gives the pre-fill plus the gradient to fp32 rounding."""
    xp, xt = _bwd_signals(n, hop, T)
    ref = _ref_grad(xp, xt, n, hop, "l1", 0.0, 1e-7, torch.float64)
    xpd, xtd = xp.to(DEV), xt.to(DEV)
    worst = {}
    for up in (1.0, -2.5):
        got = _kernel_grad(xpd, xtd, n, hop, "l1", 0.0, 1e-7, up).cpu().double().numpy()
        r = up * ref
        m = min(n, T)
        for name, s in (("whole", np.s_[:, :]), ("left", np.s_[:, :m]), ("right", np.s_[:, T - m:])):
            worst[name] = max(worst.get(name, 0.0), _rel(got[s], r[s]))
    print(f"mss bwd l1 alpha=0 n={n} hop={hop} T={T}: rel-L2 " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    for k, v in worst.items():
        assert v <= LIN_BAR, k
    g = torch.Generator().manual_seed(T)
    pre = torch.randn(xp.shape, generator=g).to(DEV)
    plain = _kernel_grad(xpd, xtd, n, hop, "l1", 0.0, 1e-7, -2.5)
    acc = _kernel_grad(xpd, xtd, n, hop, "l1", 0.0, 1e-7, -2.5, gx=pre.clone(), accumulate=True)
    d = float(((acc - (pre + plain)).abs() / ((pre.abs() + plain.abs()) * 2.0 ** -23 + 1e-30)).max())
    print(f"  accumulate: max |acc - (pre + g)| = {d:.2f} fp32 ulp of |pre| + |g|")
    assert d <= 1.0


@pytest.mark.parametrize("n,hop,T", BWD_SHAPES)
def test_mss_loss_bwd_log_terms_vs_fp64(n, hop, T):
    """l1 with alpha = 0.5 (upstream 1) and rmse (upstream -2.5), eps = 1e-7: rel-L2 <= max(LOG_ABS_BAR,
    LOG_K * floor), the floor being the error of the same reference run in float32 on the CPU."""
    xp, xt = _bwd_signals(n, hop, T)
    xpd, xtd = xp.to(DEV), xt.to(DEV)
    for mode, alpha, up in (("l1", 0.5, 1.0), ("rmse", 1.0, -2.5)):
        ref = up * _ref_grad(xp, xt, n, hop, mode, alpha, 1e-7, torch.float64)
        floor = _rel(up * _ref_grad(xp, xt, n, hop, mode, alpha, 1e-7, torch.float32), ref)
        got = _kernel_grad(xpd, xtd, n, hop, mode, alpha, 1e-7, up).cpu().double().numpy()
        err = _rel(got, ref)
        m = min(n, T)
        edge = max(_rel(got[:, :m], ref[:, :m]), _rel(got[:, T - m:], ref[:, T - m:]))
        print(f"mss bwd {mode} alpha={alpha} n={n} hop={hop} T={T}: rel-L2 {err:.2e} (edges {edge:.2e}), "
              f"float32 floor {floor:.2e}")
        bar = max(LOG_ABS_BAR, LOG_K * floor)
        assert err <= bar, (mode, err, floor)
        assert edge <= 2 * bar, (mode, edge, floor)


def test_spectral_loss_modules_autograd_path():
    """SSSLoss / MSSLoss called the way training code calls them: float64 input, 3-D (batch, channel, T) input.  The
    gradient comes back in the input's dtype and shape and matches float64 autograd; the MSSLoss total is the sum of
    its scales."""
    from diffsound_b200.ddsp.mss_loss import MSSLoss, SSSLoss
    T = 1500
    xp32, other = _pair(6, T, seed=21)
    xt32 = (0.5 * xp32 + 0.05 * other).float()
    xp, xt = xp32.double().reshape(2, 3, T), xt32.double().reshape(2, 3, T)
    for typ, mode in (("l1_loss", "l1"), ("rmse_loss", "rmse")):
        m = MSSLoss([256, 128, 64], 32000, type=typ)
        p = xp.clone().to(DEV).requires_grad_(True)
        total = m(p, xt.to(DEV))
        per = [loss(p, xt.to(DEV)) for loss in m.losses]
        assert float(total.detach()) == float(sum(per).detach()), [float(x.detach()) for x in per]
        total.backward()
        assert p.grad.dtype == torch.float64 and p.grad.shape == (2, 3, T)
        ref = sum(_ref_grad(xp32, xt32, n, n // 4, mode, 1.0, 1e-7, torch.float64) for n in (256, 128, 64))
        floor = _rel(sum(_ref_grad(xp32, xt32, n, n // 4, mode, 1.0, 1e-7, torch.float32) for n in (256, 128, 64)), ref)
        err = _rel(p.grad.reshape(6, T).cpu().numpy(), ref)
        print(f"MSSLoss {typ} 3-D float64: rel-L2 {err:.2e}, float32 floor {floor:.2e}")
        assert err <= max(LOG_ABS_BAR, LOG_K * floor)
        s = SSSLoss(128, 32000, type=typ)
        q = xp.reshape(6, T).clone().to(DEV).requires_grad_(True)
        s(q, xt.reshape(6, T).to(DEV)).backward()
        assert q.grad.dtype == torch.float64 and q.grad.shape == (6, T)


# ---------------------------------------------------------------------------------------------------------------------
# D. ds_filtered_noise_fwd / _bwd
# ---------------------------------------------------------------------------------------------------------------------
def _fn_frames(C, L):
    """enough frames that later segments receive every frame that reaches them (L = 1, C = 129: 257 frames)"""
    return max(4, -(-(2 * C - 2) // L) + 3)


@pytest.mark.parametrize("C", [2, 3, 65, 128, 129])
@pytest.mark.parametrize("L", [1, 2, 63, 64, 256])
def test_filtered_noise_vs_fp64(C, L):
    native = _native()
    F = _fn_frames(C, L)
    worst = dict(whole=0.0, seg=0.0, grad=0.0, gmax=0.0)
    for i, T in enumerate((1, (F - 1) * L + 1, F * L - 1, F * L)):
        if T < 1:
            continue
        gain, B = ((1.0, 1), (0.37, 3), (1.0, 3), (0.37, 1))[i]
        g = torch.Generator().manual_seed(1000 * C + 10 * L + i)
        coeff = (torch.rand(B, F, C, generator=g) * 6 - 3).float()
        noise = (torch.rand(B, F, L, generator=g) * 2 - 1).float()
        gy = torch.randn(B, T, generator=g).float()
        c64 = coeff.double().requires_grad_(True)
        y64 = refs.filtered_noise(c64, noise.double(), T, gain)
        (y64 * gy.double()).sum().backward()
        ref, gref = y64.detach().numpy(), c64.grad.numpy()
        cd, nd = coeff.to(DEV), noise.to(DEV)
        y = native.filtered_noise_fwd(cd, nd, T, gain).cpu().double().numpy()
        gc = native.filtered_noise_bwd(cd, nd, gy.to(DEV), gain).cpu().double().numpy()
        assert y.shape == (B, T) and gc.shape == (B, F, C)
        d = np.abs(y - ref)
        if not ref.any():                              # T = 1: y[0] = noise h[0] and the window is 0 at 0
            assert not y.any() and not gc.any() and not gref.any()
            continue
        worst["whole"] = max(worst["whole"], _rel(y, ref))
        rms = np.sqrt((ref ** 2).mean())
        for s0 in range(0, T, L):
            seg = ref[:, s0:s0 + L]
            den = np.maximum(np.sqrt((seg ** 2).mean(1)), 0.1 * rms)
            worst["seg"] = max(worst["seg"], float((d[:, s0:s0 + L].max(1) / den).max()))
        worst["grad"] = max(worst["grad"], _rel(gc, gref))
        worst["gmax"] = max(worst["gmax"], float(np.abs(gc - gref).max() / np.abs(gref).max()))
    print(f"filtered noise C={C} L={L} F={F}: fwd rel-L2 {worst['whole']:.2e}, per segment {worst['seg']:.2e}; "
          f"bwd rel-L2 {worst['grad']:.2e}, max {worst['gmax']:.2e}")
    assert worst["whole"] <= FN_BAR
    assert worst["seg"] <= FN_SEG_BAR
    assert worst["grad"] <= FN_GRAD_BAR and worst["gmax"] <= FN_GRAD_BAR


# ---------------------------------------------------------------------------------------------------------------------
# E. argument checks
# ---------------------------------------------------------------------------------------------------------------------
SENT = -7.25


def test_mss_argument_checks():
    """Every rejected size returns DS_ERR_ARG from all three entry points and writes nothing.  The buffers are large
    enough for what a launch at these sizes would write."""
    lib = _lib()
    x = torch.zeros(1 << 20, device=DEV)
    S = torch.full((1 << 22,), SENT, device=DEV)
    scratch = torch.full((1 << 22,), SENT, device=DEV)
    gx = torch.full((1 << 20,), SENT, device=DEV)
    loss = torch.full((1,), SENT, dtype=torch.float64, device=DEV)
    cases = [(1, 100, 12, 3, "power of two"), (1, 100, 4, 1, "power of two"), (1, 9000, 8192, 2048, "power of two"),
             (1, 100, 64, 0, "hop"), (1, 100, 64, 65, "hop"), (2, 2048, 4096, 1024, "reflect padding"),
             (2, 4, 8, 2, "reflect padding"), (65536, 5, 8, 2, "bad sizes"), (0, 100, 64, 16, "bad sizes")]
    for B, T, n, hop, what in cases:
        rcs = [lib.ds_stft_power(_p(x), B, T, n, hop, _p(S), None),
               lib.ds_mss_loss_fwd(_p(x), _p(x), B, T, n, hop, 0, 1.0, 1e-7, _p(scratch), _p(loss), None),
               lib.ds_mss_loss_bwd(_p(x), _p(x), B, T, n, hop, 1, 1.0, 1e-7, _p(loss), 1.0, _p(scratch), _p(gx), 0, None)]
        msg = lib.ds_last_error().decode()
        print(f"B={B} T={T} n={n} hop={hop}: {rcs} '{msg}'")
        assert rcs == [DS_ERR_ARG] * 3 and what in msg, (B, T, n, hop, rcs, msg)
    torch.cuda.synchronize()
    for t in (S, scratch, gx, loss):
        assert bool((t == SENT).all())


def test_filtered_noise_argument_checks():
    lib = _lib()
    coeff = torch.zeros(1 << 20, device=DEV)
    noise = torch.zeros(1 << 20, device=DEV)
    gy = torch.zeros(1 << 20, device=DEV)
    y = torch.full((1 << 20,), SENT, device=DEV)
    g = torch.full((1 << 20,), SENT, device=DEV)
    cases = [(1, 4, 130, 64, 200, "filter_coeff_length"), (1, 4, 1, 64, 200, "filter_coeff_length"),
             (1, 4, 65, 257, 200, "frame_length"), (1, 4, 65, 0, 200, "frame_length"),
             (2, 2, 65, 64, 129, "do not cover"), (1, 300, 129, 1, 301, "do not cover"),
             (65536, 1, 2, 1, 1, "bad sizes"), (1, 4, 65, 64, 0, "bad sizes")]
    for B, F, Cn, L, T, what in cases:
        rcs = [lib.ds_filtered_noise_fwd(_p(coeff), _p(noise), B, F, Cn, L, T, 1.0, _p(y), None),
               lib.ds_filtered_noise_bwd(_p(coeff), _p(noise), _p(gy), B, F, Cn, L, T, 1.0, _p(g), None)]
        msg = lib.ds_last_error().decode()
        print(f"B={B} F={F} C={Cn} L={L} T={T}: {rcs} '{msg}'")
        assert rcs == [DS_ERR_ARG] * 2 and what in msg, (B, F, Cn, L, T, rcs, msg)
    torch.cuda.synchronize()
    assert bool((y == SENT).all()) and bool((g == SENT).all())
