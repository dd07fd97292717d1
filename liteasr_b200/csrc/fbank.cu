// Kaldi-compatible log-mel filterbank features of a padded batch of waveforms (lasr_fbank, include/lasr_fbank.h): the
// torchaudio.compliance.kaldi.fbank definition with dither 0, the Povey window, snip_edges and a FLT_EPSILON log floor.
//
// One launch for the batch: grid (ceil(Fmax / 8), B), 8 warps per CTA, one warp per frame, no workspace.  Each warp reads its
// W samples straight from global memory into registers (lane l holds samples l + 32 i).  Neighbouring frames overlap by
// W / S ~ 2.5x; those re-reads hit L1 / L2, so HBM still reads every sample once, and every frame shift takes the same path.
//   1. mean: float64 warp sum (exact for int16 frames), rounded to fp32 and subtracted in fp32;
//   2. pre-emphasis with x[j - 1] from the neighbouring lane (lane 31 of the previous register for lane 0), the window from a
//      table, and a store into shared memory as z[n] = y[2n] + i y[2n + 1] at the bit-reversed position of n;
//   3. an NFFT/2-point radix-2 decimation-in-time FFT in shared memory, log2(NFFT/2) stages separated by __syncwarp;
//   4. the real-input split step X[k] = E[k] + w^k O[k] and P[k] = |X[k]|^2, written over the FFT buffer;
//   5. one lane per mel bin sums its contiguous range of P with fp32 weights, then logf(max(E, FLT_EPSILON)).
// Twiddles w^k = exp(-2 pi i k / NFFT), k < NFFT/2, are built per CTA with sincospif (the argument 2k / NFFT is exact).
// No tensor cores: a reduced-precision DFT-as-GEMM loses the weak bins, and a 10 ms frame is only ~25 kFLOP.
#include <cfloat>

#include "common.cuh"
#include "../../include/lasr_fbank.h"

namespace lasr {

constexpr int FB_WARPS = 8;  // frames per CTA

template <typename T> __device__ __forceinline__ float sample_f32(T v) { return (float)v; }

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int NFFT, typename T>
__global__ void __launch_bounds__(FB_WARPS * 32) fbank_kernel(const T* __restrict__ wave, long ld, const int64_t* __restrict__ nsamp,
                                                              long nmax, int W, int S, long Fmax, const float* __restrict__ window, int nb,
                                                              const int32_t* __restrict__ mel_lo, const int32_t* __restrict__ mel_off,
                                                              const float* __restrict__ mel_w, float* __restrict__ out) {
    constexpr int N2 = NFFT / 2;
    constexpr int LOG2N2 = NFFT == 256 ? 7 : (NFFT == 512 ? 8 : 9);
    constexpr int PER = NFFT / 32;  // samples per lane
    constexpr int BINS = N2 / 32;   // power-spectrum bins per lane
    static_assert(N2 == 1 << LOG2N2, "NFFT must be 256, 512 or 1024");
    __shared__ float2 tw[N2];
    __shared__ float2 zbuf[FB_WARPS][N2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.y;
    const long t = (long)blockIdx.x * FB_WARPS + warp;

    for (int k = threadIdx.x; k < N2; k += blockDim.x) {
        float s, c;
        sincospif(2.0f * k / NFFT, &s, &c);
        tw[k] = make_float2(c, -s);
    }
    __syncthreads();  // the only CTA-wide barrier: warps leave independently below
    if (t >= Fmax) return;

    long N = nsamp[b];
    N = N < 0 ? 0 : (N > nmax ? nmax : N);
    const long F = N < W ? 0 : 1 + (N - W) / S;
    float* orow = out + ((long)b * Fmax + t) * nb;
    if (t >= F) {
        for (int m = lane; m < nb; m += 32) orow[m] = 0.f;
        return;
    }

    // 1. frame mean
    const T* x = wave + (long)b * ld + t * S;
    float xr[PER];
    double sum = 0.0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int j = lane + 32 * i;
        xr[i] = j < W ? sample_f32(x[j]) : 0.f;
        sum += (double)xr[i];
    }
    const float mean = (float)(warp_sum_f64(sum) / W);

    // 2. pre-emphasis, window, bit-reversed store of the packed complex sequence (zero-padded to NFFT)
    float2* z = zbuf[warp];
    float* zf = reinterpret_cast<float*>(z);
    float cprev = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int j = lane + 32 * i;
        const float c = xr[i] - mean;
        float cm1 = __shfl_up_sync(0xffffffffu, c, 1);
        const float wrap = __shfl_sync(0xffffffffu, cprev, 31);
        if (lane == 0) cm1 = i ? wrap : c;  // x[max(j - 1, 0)]
        cprev = c;
        const float y = j < W ? (c - 0.97f * cm1) * __ldg(window + j) : 0.f;
        zf[2 * (__brev(j >> 1) >> (32 - LOG2N2)) + (j & 1)] = y;
    }
    __syncwarp();

    // 3. radix-2 DIT FFT of N2 points: stage s joins pairs h = 2^s apart with twiddle exp(-2 pi i p / 2h) = tw[p N2 / h]
#pragma unroll
    for (int s = 0; s < LOG2N2; ++s) {
        const int h = 1 << s;
#pragma unroll
        for (int q = 0; q < N2 / 64; ++q) {
            const int bf = lane + 32 * q;
            const int p = bf & (h - 1);
            const int i0 = ((bf >> s) << (s + 1)) + p, i1 = i0 + h;
            const float2 w = tw[p << (LOG2N2 - s)];
            const float2 u = z[i0], v0 = z[i1];
            const float2 v = make_float2(w.x * v0.x - w.y * v0.y, w.x * v0.y + w.y * v0.x);
            z[i0] = make_float2(u.x + v.x, u.y + v.y);
            z[i1] = make_float2(u.x - v.x, u.y - v.y);
        }
        __syncwarp();
    }

    // 4. split: E[k] = (Z[k] + conj Z[N2-k]) / 2, O[k] = (Z[k] - conj Z[N2-k]) / 2i, X[k] = E[k] + tw[k] O[k]
    float pw[BINS];
#pragma unroll
    for (int i = 0; i < BINS; ++i) {
        const int k = lane + 32 * i;
        const float2 zk = z[k], zn = z[(N2 - k) & (N2 - 1)];
        const float er = 0.5f * (zk.x + zn.x), ei = 0.5f * (zk.y - zn.y);
        const float orr = 0.5f * (zk.y + zn.y), oi = -0.5f * (zk.x - zn.x);
        const float2 w = tw[k];
        const float re = er + (w.x * orr - w.y * oi), im = ei + (w.x * oi + w.y * orr);
        pw[i] = re * re + im * im;
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < BINS; ++i) zf[lane + 32 * i] = pw[i];
    __syncwarp();

    // 5. sparse mel sum and log
    for (int m = lane; m < nb; m += 32) {
        const int lo = __ldg(mel_lo + m), o0 = __ldg(mel_off + m);
        int n = __ldg(mel_off + m + 1) - o0;
        if (lo < 0 || lo > N2) n = 0;
        n = n < N2 - lo ? n : N2 - lo;
        float e = 0.f;
        for (int k = 0; k < n; ++k) e = fmaf(__ldg(mel_w + o0 + k), zf[lo + k], e);
        orow[m] = logf(fmaxf(e, FLT_EPSILON));
    }
}

template <typename T>
static void launch_fbank(int nfft, dim3 grid, cudaStream_t st, const void* wave, long ld, const int64_t* nsamp, long nmax, int W, int S,
                         long Fmax, const float* window, int nb, const int32_t* mel_lo, const int32_t* mel_off, const float* mel_w,
                         float* out) {
    void (*k)(const T*, long, const int64_t*, long, int, int, long, const float*, int, const int32_t*, const int32_t*, const float*, float*);
    switch (nfft) {
        case 256: k = fbank_kernel<256, T>; break;
        case 512: k = fbank_kernel<512, T>; break;
        default: k = fbank_kernel<1024, T>; break;
    }
    k<<<grid, FB_WARPS * 32, 0, st>>>((const T*)wave, ld, nsamp, nmax, W, S, Fmax, window, nb, mel_lo, mel_off, mel_w, out);
}

}  // namespace lasr

extern "C" {
using namespace lasr;

int lasr_fbank(const void* wave, int dtype, int64_t ld, const int64_t* nsamp, int B, int64_t nmax, int frame_len, int frame_shift,
               const float* window, int nb, const int32_t* mel_lo, const int32_t* mel_off, const float* mel_w, float* out, void* stream) {
    LASR_REQUIRE(wave && nsamp && window && mel_lo && mel_off && mel_w && out && B > 0 && nmax >= 0 && ld >= nmax, "fbank: bad args");
    LASR_REQUIRE(B <= 65535, "fbank: B = %d exceeds the limit of 65535 utterances", B);
    LASR_REQUIRE(frame_shift >= 1, "fbank: frame_shift = %d samples, must be >= 1", frame_shift);
    LASR_REQUIRE(frame_len >= 2, "fbank: frame_len = %d samples, must be >= 2", frame_len);
    long nfft = 1;
    while (nfft < frame_len) nfft *= 2;
    LASR_REQUIRE(nfft >= 256 && nfft <= 1024,
                 "fbank: frame_len = %d samples needs a %ld-point FFT; supported are NFFT = 256, 512, 1024 (129 <= frame_len <= 1024)",
                 frame_len, nfft);
    LASR_REQUIRE(nb >= 4 && nb <= 128, "fbank: nb = %d mel bins outside the supported [4, 128]", nb);
    if (dtype != LASR_F32 && dtype != LASR_I16) { set_error("fbank: dtype %d is neither LASR_F32 nor LASR_I16", dtype); return LASR_ERR_BAD_ARG; }
    const long Fmax = nmax < frame_len ? 0 : 1 + (nmax - frame_len) / frame_shift;
    if (Fmax == 0) return LASR_OK;  // an empty (B, 0, nb) output
    const dim3 grid((unsigned)((Fmax + FB_WARPS - 1) / FB_WARPS), (unsigned)B);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == LASR_I16)
        launch_fbank<int16_t>((int)nfft, grid, st, wave, ld, nsamp, nmax, frame_len, frame_shift, Fmax, window, nb, mel_lo, mel_off, mel_w, out);
    else
        launch_fbank<float>((int)nfft, grid, st, wave, ld, nsamp, nmax, frame_len, frame_shift, Fmax, window, nb, mel_lo, mel_off, mel_w, out);
    return check_launch("fbank");
}

}  // extern "C"
