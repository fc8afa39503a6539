// Multi-scale spectral loss: power spectrograms and the L1 / RMSE spectral losses, forward and backward, fused per
// STFT frame.
//
// Reference behaviour replaced: SSSLoss / MSSLoss (/root/reference/src/ddsp/mss_loss.py:70-147) on
// torchaudio.transforms.Spectrogram(n_fft, hop_length = n_fft / 4) -- win_length = n_fft, periodic Hann window,
// center = True with reflect padding, power = 2, one-sided -- as used by the material experiments
// (material_sync_train.py:123-125,159; material_real_train.py:109-110,119).  Loss types:
//   l1_loss   alpha * wl1(log2(S_p + eps), log2(S_t + eps)) + wl1(S_p, S_t),
//             wl1 = mean over (batch, bins 1.., frames) of w[frame] |a - b|, w = time ramp (mss_loss.py:55-66)
//   rmse_loss sqrt(mean((log2(S_p + eps) - log2(S_t + eps))^2))  (mss_loss.py:116-119; the -log2(eps) offsets cancel)
// ('geomloss' needs the third-party Sinkhorn solver, absent from this image and from the hot path.)
//
// The reference materialises four spectrograms per scale and differentiates through cuFFT.  Here one CTA owns one
// STFT frame of one signal pair: it windows the predicted and the target frame into the real and imaginary part of
// ONE complex radix-2 FFT in shared memory, separates the two spectra by symmetry, and reduces the frame's loss
// terms on the spot -- no spectrogram ever reaches HBM.  Backward: the same FFT again, dL/dS_p per bin, one inverse
// FFT of g_f X_f (the adjoint of the real DFT), the windowed frame gradient to a small scratch, and a gather kernel
// that sums every sample's contributions (overlapping frames + reflect-padding images) in a fixed order: no atomics.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"

namespace ds {

constexpr int MSS_MAXN = 4096;
constexpr int MSS_THREADS = 256;

struct Cplx { float re, im; };

// in-place radix-2 FFT of s[0..n) (bit-reversed input order expected), forward (sign -1) or inverse (+1, unnormalised)
__device__ void fft_smem(Cplx* s, const Cplx* tw, int n, int logn, bool inverse) {
    for (int st = 1; st <= logn; ++st) {
        const int half = 1 << (st - 1), tstep = n >> st;
        for (int j = threadIdx.x; j < n / 2; j += blockDim.x) {
            const int k = j & (half - 1);
            const int base = ((j - k) << 1) + k;
            Cplx w = tw[k * tstep];
            if (inverse) w.im = -w.im;
            const Cplx u = s[base], v0 = s[base + half];
            Cplx v;
            v.re = v0.re * w.re - v0.im * w.im;
            v.im = v0.re * w.im + v0.im * w.re;
            s[base].re = u.re + v.re;  s[base].im = u.im + v.im;
            s[base + half].re = u.re - v.re;  s[base + half].im = u.im - v.im;
        }
        __syncthreads();
    }
}

__device__ __forceinline__ int bitrev(int i, int logn) { return (int)(__brev((unsigned)i) >> (32 - logn)); }

__device__ __forceinline__ int64_t reflect_idx(int64_t p, int64_t T) {   // index into the signal of padded position p - n/2
    if (p < 0) p = -p;
    if (p >= T) p = 2 * (T - 1) - p;
    return p;
}

// shared memory: tw [n/2] | s [n]
__device__ void load_twiddles(Cplx* tw, int n) {
    for (int j = threadIdx.x; j < n / 2; j += blockDim.x) {
        float sn, cs;
        sincospif(-2.f * (float)j / (float)n, &sn, &cs);
        tw[j].re = cs; tw[j].im = sn;
    }
}

// s[bitrev(i)] = hann[i] * (a[i] + i b[i]) for the frame starting at padded position fr * hop.  Returns whether every
// sample this thread loaded has a[i] == b[i] (false without b).
__device__ bool load_frame(Cplx* s, const float* __restrict__ a, const float* __restrict__ b, int64_t T, int n, int logn,
                           int fr, int hop) {
    bool same = b != nullptr;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int64_t src = reflect_idx((int64_t)fr * hop + i - n / 2, T);
        const float w = 0.5f - 0.5f * cospif(2.f * (float)i / (float)n);
        Cplx v;
        v.re = w * a[src];
        v.im = b ? w * b[src] : 0.f;
        same = same && a[src] == b[src];
        s[bitrev(i, logn)] = v;
    }
    return same;
}

// spectra of the two real signals packed as re/im: A_f = (Z_f + conj(Z_{n-f})) / 2,  B_f = (Z_f - conj(Z_{n-f})) / (2i)
__device__ __forceinline__ void unpack2(const Cplx* s, int n, int f, Cplx& A, Cplx& B) {
    const Cplx z = s[f], zc = s[(n - f) & (n - 1)];
    A.re = 0.5f * (z.re + zc.re);  A.im = 0.5f * (z.im - zc.im);
    B.re = 0.5f * (z.im + zc.im);  B.im = -0.5f * (z.re - zc.re);
}

// ---- power spectrogram (materialised; SSSLoss.log_spec / .spec) ---------------------------------------
__global__ void __launch_bounds__(MSS_THREADS)
k_stft_power(const float* __restrict__ x, int64_t T, int n, int logn, int hop, int frames, float* __restrict__ S) {
    extern __shared__ __align__(8) unsigned char mss_smem[];
    Cplx* tw = reinterpret_cast<Cplx*>(mss_smem);
    Cplx* s = tw + n / 2;
    const int fr = blockIdx.x, b = blockIdx.y, bins = n / 2 + 1;
    load_twiddles(tw, n);
    load_frame(s, x + (size_t)b * T, nullptr, T, n, logn, fr, hop);
    __syncthreads();
    fft_smem(s, tw, n, logn, false);
    for (int f = threadIdx.x; f < bins; f += blockDim.x)
        S[((size_t)b * bins + f) * frames + fr] = s[f].re * s[f].re + s[f].im * s[f].im;
}

// time weight of weighted_l1_loss (mss_loss.py:59-61): w = 1 - linspace(1, 0.9, F), normalised to mean 1
__device__ __forceinline__ float time_weight(int fr, int frames) {
    if (frames == 1) return 1.f;       // linspace(1, .9, 1) = [1] -> w = 0 / 0 in the reference; keep it finite
    // w_i = 0.1 i / (F - 1); sum = 0.05 F; normalised: w_i * F / sum = 2 i / (F - 1)
    return 2.f * (float)fr / (float)(frames - 1);
}

// mode 0: l1_loss terms; mode 1: squared log difference.  partial[b * frames + fr] = the frame's sum (double)
__global__ void __launch_bounds__(MSS_THREADS)
k_mss_fwd(const float* __restrict__ xp, const float* __restrict__ xt, int64_t T, int n, int logn, int hop, int frames,
          int mode, float alpha, float eps, double* __restrict__ partial) {
    extern __shared__ __align__(8) unsigned char mss_smem[];
    Cplx* tw = reinterpret_cast<Cplx*>(mss_smem);
    Cplx* s = tw + n / 2;
    __shared__ double red[MSS_THREADS / 32];
    const int fr = blockIdx.x, b = blockIdx.y, bins = n / 2 + 1;
    load_twiddles(tw, n);
    // equal frames have equal spectra, but the packed FFT rounds A and B apart: take B = A, so that pred == true
    // gives a loss of exactly 0 (and rmse its zero gradient) instead of rounding noise
    const bool same = __syncthreads_and(load_frame(s, xp + (size_t)b * T, xt + (size_t)b * T, T, n, logn, fr, hop));
    fft_smem(s, tw, n, logn, false);
    const float wt = time_weight(fr, frames);
    double acc = 0.0;
    for (int f = threadIdx.x + (mode == 0 ? 1 : 0); f < bins; f += blockDim.x) {     // l1: the DC bin is dropped
        Cplx A, B;
        unpack2(s, n, f, A, B);
        if (same) B = A;
        const float Sp = A.re * A.re + A.im * A.im, St = B.re * B.re + B.im * B.im;
        const float lp = log2f(Sp + eps), lt = log2f(St + eps);
        // w |a - b|, not |w a - w b|: a contracted w a - w b is the rounding error of w b, not 0, when a == b
        if (mode == 0) acc += (double)(alpha * (wt * fabsf(lp - lt)) + wt * fabsf(Sp - St));
        else acc += (double)((lp - lt) * (lp - lt));
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < MSS_THREADS / 32; ++w) t += red[w];
        partial[(size_t)b * frames + fr] = t;
    }
}

__global__ void k_mss_reduce(const double* __restrict__ partial, int64_t count, double scale, int mode,
                             double* __restrict__ out) {
    // one warp, fixed order
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < count; i += 32) s += partial[i];
    s = warp_sum(s);
    if (threadIdx.x == 0) out[0] = mode == 0 ? s * scale : sqrt(s * scale);
}

// frame gradients: gframe[(b * frames + fr) * n + i] = hann[i] * d loss / d (windowed sample i of the frame)
__global__ void __launch_bounds__(MSS_THREADS)
k_mss_bwd_frames(const float* __restrict__ xp, const float* __restrict__ xt, int64_t T, int n, int logn, int hop,
                 int frames, int mode, float alpha, float eps, const double* __restrict__ loss, float upstream,
                 double scale, float* __restrict__ gframe) {
    extern __shared__ __align__(8) unsigned char mss_smem[];
    Cplx* tw = reinterpret_cast<Cplx*>(mss_smem);
    Cplx* s = tw + n / 2;
    Cplx* z = s + n;
    const int fr = blockIdx.x, b = blockIdx.y, bins = n / 2 + 1;
    load_twiddles(tw, n);
    // equal frames: B = A, as in k_mss_fwd
    const bool same = __syncthreads_and(load_frame(s, xp + (size_t)b * T, xt + (size_t)b * T, T, n, logn, fr, hop));
    fft_smem(s, tw, n, logn, false);
    const float wt = time_weight(fr, frames);
    // rmse: d sqrt(m) = d m / (2 sqrt(m)), m = scale * sum
    const float gscale = mode == 0 ? upstream * (float)scale
                                   : (loss[0] > 0.0 ? upstream * (float)(scale / (2.0 * loss[0])) : 0.f);
    const float inv_ln2 = 1.4426950408889634f;
    for (int f = threadIdx.x; f < n; f += blockDim.x) {
        Cplx o; o.re = 0.f; o.im = 0.f;
        if (f < bins && !(mode == 0 && f == 0)) {
            Cplx A, B;
            unpack2(s, n, f, A, B);
            if (same) B = A;
            const float Sp = A.re * A.re + A.im * A.im, St = B.re * B.re + B.im * B.im;
            const float lp = log2f(Sp + eps), lt = log2f(St + eps);
            float g;        // d loss / d S_p[f]
            if (mode == 0) {
                const float dl = lp - lt, ds_ = Sp - St;         // the signs of w (a - b): w >= 0
                const float sl = dl > 0.f ? 1.f : (dl < 0.f ? -1.f : 0.f), ss = ds_ > 0.f ? 1.f : (ds_ < 0.f ? -1.f : 0.f);
                g = gscale * wt * (alpha * sl * inv_ln2 / (Sp + eps) + ss);
            } else {
                g = gscale * 2.f * (lp - lt) * inv_ln2 / (Sp + eps);
            }
            o.re = g * A.re; o.im = g * A.im;
        }
        z[bitrev(f, logn)] = o;
    }
    __syncthreads();
    fft_smem(z, tw, n, logn, true);
    // d S / d y_i = 2 Re(X_f e^{+i theta}) summed over the one-sided bins
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float w = 0.5f - 0.5f * cospif(2.f * (float)i / (float)n);
        gframe[((size_t)b * frames + fr) * n + i] = 2.f * z[i].re * w;
    }
}

// gx[b, t] = sum over padded positions p that read sample t (itself + reflect images) and frames covering p
__global__ void k_mss_bwd_gather(const float* __restrict__ gframe, int64_t T, int n, int hop, int frames, int64_t B,
                                 float* __restrict__ gx, int accumulate) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= B * T) return;
    const int64_t b = idx / T, t = idx - b * T;
    const int64_t half = n / 2;
    int64_t pos[3];
    int np = 0;
    pos[np++] = t + half;
    if (t >= 1 && t <= half) pos[np++] = half - t;                                   // left reflection
    if (t <= T - 2 && 2 * (T - 1) - t < T + half) pos[np++] = half + 2 * (T - 1) - t;   // right reflection
    float s = 0.f;
    for (int q = 0; q < np; ++q) {
        const int64_t p = pos[q];
        int64_t f_hi = p / hop;
        if (f_hi > frames - 1) f_hi = frames - 1;
        int64_t f_lo = (p - n + hop) / hop;                                          // smallest f with f * hop + n > p
        if (p - n + 1 <= 0) f_lo = 0;
        for (int64_t f = f_lo; f <= f_hi; ++f) {
            const int64_t i = p - f * hop;
            if (i >= 0 && i < n) s += gframe[((size_t)b * frames + f) * n + i];
        }
    }
    if (accumulate) gx[idx] += s; else gx[idx] = s;
}

static int mss_check(const char* who, int64_t B, int64_t T, int n, int hop, int* logn) {
    DS_REQUIRE(B > 0 && B <= 65535 && T > 1, "%s: bad sizes (B=%lld T=%lld)", who, (long long)B, (long long)T);
    DS_REQUIRE(n >= 8 && n <= MSS_MAXN && (n & (n - 1)) == 0, "%s: n_fft=%d must be a power of two in [8, %d]", who, n, MSS_MAXN);
    DS_REQUIRE(hop >= 1 && hop <= n, "%s: hop=%d", who, hop);
    DS_REQUIRE(T > n / 2, "%s: reflect padding needs more than n_fft/2 = %d samples (T=%lld)", who, n / 2, (long long)T);
    int l = 0;
    while ((1 << l) < n) ++l;
    *logn = l;
    return DS_OK;
}

}  // namespace ds

using namespace ds;

extern "C" int ds_stft_frames(int64_t T, int hop) { return hop > 0 ? (int)(1 + T / hop) : -1; }

extern "C" int ds_stft_power(const float* x, int64_t B, int64_t T, int n_fft, int hop, float* S, void* stream) {
    DS_REQUIRE(x && S, "ds_stft_power: null argument");
    int logn;
    DS_TRY(mss_check("ds_stft_power", B, T, n_fft, hop, &logn));
    const int frames = (int)(1 + T / hop);
    const size_t smem = sizeof(Cplx) * (n_fft / 2 + n_fft);
    DS_CUDA(cudaFuncSetAttribute(k_stft_power, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ProfScope prof(PROF_OTHER, (cudaStream_t)stream);
    k_stft_power<<<dim3(frames, (unsigned)B), MSS_THREADS, smem, (cudaStream_t)stream>>>(x, T, n_fft, logn, hop, frames, S);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int64_t ds_mss_scratch_elems(int64_t B, int64_t T, int n_fft, int hop) {
    const int64_t frames = 1 + T / (hop > 0 ? hop : 1);
    return B * frames * (int64_t)n_fft + 2 * B * frames + 64;      // frame gradients (fp32) + partial sums (fp64 = 2 floats)
}

static double mss_scale(int mode, int64_t B, int n_fft, int frames) {
    const int bins = n_fft / 2 + 1;
    return 1.0 / ((double)B * (mode == 0 ? bins - 1 : bins) * frames);
}

extern "C" int ds_mss_loss_fwd(const float* x_pred, const float* x_true, int64_t B, int64_t T, int n_fft, int hop,
                               int mode, double alpha, double eps, float* scratch, double* loss, void* stream) {
    DS_REQUIRE(x_pred && x_true && scratch && loss, "ds_mss_loss_fwd: null argument");
    DS_REQUIRE(mode == 0 || mode == 1, "ds_mss_loss_fwd: mode must be 0 (l1_loss) or 1 (rmse_loss)");
    DS_REQUIRE((uintptr_t)scratch % 8 == 0, "ds_mss_loss_fwd: scratch must be 8-byte aligned");
    int logn;
    DS_TRY(mss_check("ds_mss_loss_fwd", B, T, n_fft, hop, &logn));
    const int frames = (int)(1 + T / hop);
    double* partial = reinterpret_cast<double*>(scratch);
    const size_t smem = sizeof(Cplx) * (n_fft / 2 + n_fft);
    DS_CUDA(cudaFuncSetAttribute(k_mss_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ProfScope prof(PROF_OTHER, (cudaStream_t)stream);
    k_mss_fwd<<<dim3(frames, (unsigned)B), MSS_THREADS, smem, (cudaStream_t)stream>>>(x_pred, x_true, T, n_fft, logn, hop,
                                                                                      frames, mode, (float)alpha, (float)eps, partial);
    DS_LAUNCH_CHECK();
    k_mss_reduce<<<1, 32, 0, (cudaStream_t)stream>>>(partial, B * frames, mss_scale(mode, B, n_fft, frames), mode, loss);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_mss_loss_bwd(const float* x_pred, const float* x_true, int64_t B, int64_t T, int n_fft, int hop,
                               int mode, double alpha, double eps, const double* loss, double upstream, float* scratch,
                               float* gx, int accumulate, void* stream) {
    DS_REQUIRE(x_pred && x_true && scratch && loss && gx, "ds_mss_loss_bwd: null argument");
    DS_REQUIRE(mode == 0 || mode == 1, "ds_mss_loss_bwd: mode must be 0 (l1_loss) or 1 (rmse_loss)");
    int logn;
    DS_TRY(mss_check("ds_mss_loss_bwd", B, T, n_fft, hop, &logn));
    const int frames = (int)(1 + T / hop);
    float* gframe = scratch + 2 * B * frames + 16;
    const size_t smem = sizeof(Cplx) * (n_fft / 2 + 2 * n_fft);
    DS_CUDA(cudaFuncSetAttribute(k_mss_bwd_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ProfScope prof(PROF_OTHER, (cudaStream_t)stream);
    k_mss_bwd_frames<<<dim3(frames, (unsigned)B), MSS_THREADS, smem, (cudaStream_t)stream>>>(
        x_pred, x_true, T, n_fft, logn, hop, frames, mode, (float)alpha, (float)eps, loss, (float)upstream,
        mss_scale(mode, B, n_fft, frames), gframe);
    DS_LAUNCH_CHECK();
    k_mss_bwd_gather<<<(unsigned)ceil_div(B * T, 256), 256, 0, (cudaStream_t)stream>>>(gframe, T, n_fft, hop, frames, B, gx,
                                                                                       accumulate);
    DS_LAUNCH_CHECK();
    return DS_OK;
}
