/* liblasr -- Kaldi-compatible log-mel filterbank features (the same library and conventions as lasr.h: device pointers, `stream`
 * as void*, no host synchronisation, CUDA-graph capturable, 0 or a negative LASR_ERR_* with lasr_last_error()).
 *
 * The output equals torchaudio.compliance.kaldi.fbank(w, num_mel_bins=nb, sample_frequency=sr, frame_length=fl,
 * frame_shift=fs, low_freq=lo, high_freq=hi, dither=0.0) with every other argument at its default, except for the log floor:
 * FLT_EPSILON (Kaldi's BaseFloat floor) where torchaudio takes the epsilon of the input dtype.  For utterance b with
 * N = nsamp[b] samples, W = frame_len, S = frame_shift samples (the caller's int(sr * fl / 1000), int(sr * fs / 1000)):
 *   NFFT = the next power of two >= W;  F = 0 if N < W, else 1 + (N - W) / S  (snip_edges)
 *   frame t takes samples [tS, tS + W) as fp32, then
 *     1. subtracts the frame mean (accumulated in float64, rounded to fp32, one fp32 subtraction per sample, so an integer
 *        constant frame becomes exactly 0),
 *     2. pre-emphasis: y[j] = x[j] - 0.97 x[max(j - 1, 0)],
 *     3. multiplies by window[j] (the Povey window (0.5 - 0.5 cos(2 pi j / (W - 1)))^0.85),
 *     4. zero-pads to NFFT and takes P[k] = |X[k]|^2, k = 0 .. NFFT/2 - 1 (the Nyquist bin has zero mel weight),
 *     5. E[m] = sum_k M[m, k] P[k] over Kaldi's triangular mel bank M (torchaudio get_mel_banks),
 *     6. out[m] = logf(max(E[m], FLT_EPSILON)).
 *   All arithmetic is fp32 except the mean; the FFT is a radix-2 complex FFT of NFFT/2 points with twiddles from sincospif and
 *   the real-input split step, so results match a float64 evaluation to fp32 rounding, not bit for bit.
 * Inputs:
 *   wave   (B, >= ld) samples, int16 (LASR_I16) or fp32 (LASR_F32), row stride ld >= nmax elements.  Samples are in int16
 *          scale, Kaldi's convention: a float waveform normalised to [-1, 1] must be multiplied by 32768 first.
 *   nsamp  (B,) int64, clamped to [0, nmax]; samples past nsamp[b] are never read.
 *   window (frame_len,) fp32.
 *   mel bank, sparse: bin m weights FFT bins [mel_lo[m], mel_lo[m] + mel_off[m+1] - mel_off[m]) with mel_w[mel_off[m] ..
 *          mel_off[m+1]), in ascending bin order; mel_lo (nb,) int32, mel_off (nb + 1,) int32, mel_w (mel_off[nb],) fp32.
 *          The kernel clamps each range to [0, NFFT/2).
 * Output: out (B, Fmax, nb) fp32, Fmax = the frame count of nmax.  Every row is written; rows t >= F_b are 0.0 (the padding
 *   value of the training and decoding input (xs, xlens)).
 * Limits: NFFT in {256, 512, 1024} (129 <= frame_len <= 1024), 4 <= nb <= 128, frame_shift >= 1, B <= 65535; anything else
 *   returns LASR_ERR_BAD_ARG with a message naming the bound.  The frequency limits of the mel bank are the table builder's
 *   (liteasr_b200/features.py).
 * One launch for the whole batch: 8 frames per CTA, one warp per frame; no workspace.
 */
#ifndef LASR_FBANK_H
#define LASR_FBANK_H

#include "lasr.h"

#define LASR_I16 2 /* int16 samples; only lasr_fbank takes it */

#ifdef __cplusplus
extern "C" {
#endif

int lasr_fbank(const void* wave, int dtype, int64_t ld, const int64_t* nsamp, int B, int64_t nmax, int frame_len, int frame_shift,
               const float* window, int nb, const int32_t* mel_lo, const int32_t* mel_off, const float* mel_w, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LASR_FBANK_H */
